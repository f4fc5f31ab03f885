/*
 * gpx.h -- C ABI of the B200-native batched-Paxos engine (gigapaxos hot path).
 *
 * This is the drop-in boundary (SURVEY.md 8b). gigapaxos has no FFI seam on this
 * path today; the seam defined here is the narrow waist already present in the
 * Java code.  Every entry point cites the reference interface it replaces
 * (paths relative to /root/reference/src/edu/umass/cs/gigapaxos/):
 *
 *   gpx_engine_create / gpx_config_from_properties
 *        <- PaxosConfig.java:64,83-90 (gigapaxos.properties), PaxosManager ctor
 *           PaxosManager.java:392-462
 *   gpx_create_groups        <- PaxosManager.createPaxosInstance :632, batch form :664-691,
 *                               HotRestoreInfo.createHRI paxosutil/HotRestoreInfo.java:145-157,
 *                               PaxosInstanceStateMachine.initiateRecovery :591-675
 *   gpx_destroy_groups       <- PaxosManager.kill :2162
 *   gpx_dump_rows/load_rows  <- PaxosManager pause/unpause :2284,:2370 (HotRestoreInfo field set)
 *   gpx_patch                <- PaxosAcceptor.handlePrepare :245-251 (ballot bump),
 *                               jumpSlot :564-578, forceStop :154; coordinator install/resign
 *   gpx_propose              <- RequestBatcher.enqueueImpl/dequeueImpl RequestBatcher.java:112-234,
 *                               PISM.handleRequest :767 / handleProposal :818,
 *                               PaxosCoordinatorState.propose :233-263
 *   gpx_handle_accepts       <- PISM.handleAccept :1080-1166 (+ AbstractPaxosLogger.logAndMessage :157)
 *   gpx_handle_accept_replies<- PISM.handleBatchedAcceptReply :1370 / handleAcceptReply :1248
 *   gpx_handle_decisions     <- PISM.handleBatchedCommit :1480 / handleCommittedRequest :1432 /
 *                               extractExecuteAndCheckpoint :1619 (EXEC records replace app.execute :1802)
 *   gpx_round                <- one full pass of the above for co-located replicas
 *                               (PaxosManager.send :2098-2128 routing incl. loopback)
 *   gpx_log_read             <- SQLPaxosLogger.journal :965-1036 / Journaler.appendToLogFile :814-826
 *   gpx_handle_prepares      <- PISM.handlePrepare :900-955, PaxosAcceptor.handlePrepare :239-297
 *   gpx_handle_prepare_replies <- PISM.handlePrepareReply :1017-1068, PaxosCoordinatorState.java:264-587 (phase 1b)
 *   gpx_select_groups / gpx_missing_decisions / gpx_clear_group_flags / gpx_pause_groups
 *                            <- PaxosManager.syncAndDeactivate :2806-2900 (the sweep over pinstances),
 *                               PISM.requestMissingDecisions :2292-2320, tryPause :2004-2035, pause(Map, dequeue) :2327-2366
 *   gpx_log_find / gpx_log_gather <- AbstractPaxosLogger.getLoggedDecisions :582 / getLoggedAccepts :568
 *                               (SQLPaxosLogger.getLoggedFromMessageLog :3674-3756, paxosutil/LogIndex.java:213-248)
 *   gpx_wire_*               <- paxospackets byte codecs (RequestPacket.java:819-1024,
 *                               AcceptPacket.java:95-138, BatchedAcceptReply.java:103-173,
 *                               BatchedCommit.java:184-252, PaxosPacket.java:443-476)
 *
 * Conventions (mirror the reference, SURVEY.md 8b): int return codes are for API
 * misuse only; protocol-level rejects (stopped group, stale ballot, unknown
 * acceptor, window overflow) are counted and dropped, never fatal.  The engine is
 * single-submitter and batch-synchronous: one call = one batch, per-group order
 * inside a batch is the order of the records in the batch.  The caller owns all
 * input and output buffers; the engine owns device memory.
 *
 * All records are little-endian, fixed size, 16-byte multiples.
 * A `gid` is a dense handle for one (paxosID, version) instance -- the analogue
 * of a PaxosInstanceStateMachine object reference; the version drop rule
 * (PISM :441-447) is applied where (paxosID, version) is mapped to a gid
 * (gpx_wire_decode_*).
 */
#ifndef GPX_H
#define GPX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPX_ABI_VERSION 2

#define GPX_MAX_GROUP_SIZE 16 /* PC.MAX_GROUP_SIZE, PaxosConfig.java:532 */
#define GPX_MAX_LANES 8       /* co-located replicas (lanes) per engine */
#define GPX_MAX_WINDOW 8      /* per-group in-flight slot window W (power of two) */
#define GPX_MAX_MSETS 4096    /* distinct member sets per engine */

/* return codes (API misuse / environment only) */
enum {
  GPX_OK = 0,
  GPX_EINVAL = -1,
  GPX_ENOMEM = -2,
  GPX_ECUDA = -3,
  GPX_ENOGPU = -4,
  GPX_ERANGE = -5,
  GPX_EIO = -6,
  GPX_EAGAIN = -7 /* log ring full (log_backpressure): drain + release, then repeat the call; nothing was done */
};

/* PaxosAcceptor.STATES ordinals (PaxosAcceptor.java:87-92); FREE = no instance */
enum {
  GPX_ST_RECOVERY = 0,
  GPX_ST_ACTIVE_1 = 1,
  GPX_ST_ACTIVE_2 = 2,
  GPX_ST_STOPPED = 3,
  GPX_ST_FREE = 255
};

/* record flags (uint16 `flags` of gpx_pvalue_hdr, low half of request/exec flags) */
#define GPX_F_STOP 0x0001u       /* RequestPacket.stop */
#define GPX_F_VOID 0x0002u       /* hole: ignore this record / frame */
#define GPX_F_ACCEPT 0x0004u     /* log frame / record is an ACCEPT (48 B + blob) */
#define GPX_F_DECISION 0x0008u   /* log frame / record is a DECISION (32 B) */
#define GPX_F_META 0x0010u       /* decision log frame is PValuePacket.getMetaDecision() form */
#define GPX_F_CKPT 0x0020u       /* exec: PISM.shouldCheckpoint() is true for this slot */
#define GPX_F_LOGGED 0x0040u     /* accept reply was released by a log append (LogMessagingTask) */
#define GPX_F_NACK 0x0080u       /* accept reply carries a ballot higher than the accept's */
#define GPX_F_EXTRA 0x0100u      /* exec/decision came from the reconstructDecision path */
#define GPX_F_PREPARE 0x0200u    /* log frame / record is a PREPARE (32 B pvalue header, slot = firstUndecidedSlot) */
#define GPX_F_FROM_LOG 0x0400u   /* prepare reply: journaling serves accepted pvalues from the log (GET_ACCEPTED_
                                  * PVALUES_FROM_DISK) and the preparer is behind this acceptor -> the host adds the
                                  * logged accepts of [firstUndecidedSlot, acceptor's slot) from the journal */

/* request status written by gpx_propose (one int32 per request) */
#define GPX_RS_BATCHED (-1)      /* latched into the batch of an earlier request of the group */
#define GPX_RS_FORWARD (-2)      /* coordinator is a remote node: forward PROPOSAL (host) */
#define GPX_RS_REFUSED_STOP (-3) /* PCS.propose refused: previous proposal is a STOP */
#define GPX_RS_BACKPRESSURE (-4) /* proposal window full (W in flight); resubmit later */
#define GPX_RS_DROPPED (-5)      /* group stopped / free (PISM :456-460) */
#define GPX_RS_PREACTIVE (-6)    /* coordinator exists but is not active: host slow path */
#define GPX_RS_NOCOORD (-7)      /* no usable coordinator on any local lane: host slow path */

/* ---- records -------------------------------------------------------------- */

/* client request handed to the RequestBatcher (RequestPacket essentials), 32 B */
typedef struct gpx_request_rec {
  uint32_t gid;
  uint32_t flags;       /* bit0 GPX_F_STOP; bits 8..11 entry lane */
  int64_t req_id;       /* RequestPacket.requestID */
  uint32_t payload_off; /* byte offset of requestValue in the batch payload arena */
  uint32_t payload_len;
  int32_t entry_node;   /* RequestPacket.entryReplica (node id) */
  uint32_t client;      /* opaque client handle, carried through */
} gpx_request_rec;

/* common prefix of ACCEPT and DECISION (PValuePacket), 32 B */
typedef struct gpx_pvalue_hdr {
  uint32_t gid;
  int32_t slot;      /* ProposalPacket.slot */
  int32_t bnum;      /* Ballot.ballotNumber */
  int32_t bcoord;    /* Ballot.coordinatorID (node id) */
  int32_t median_cp; /* PValuePacket.medianCheckpointedSlot */
  uint16_t flags;    /* GPX_F_* */
  uint16_t dst_mask; /* local lanes this record is addressed to */
  int64_t req_id;    /* requestID of the first request of the slot */
} gpx_pvalue_hdr;

typedef gpx_pvalue_hdr gpx_decision_rec; /* DECISION / one slot of a BATCHED_COMMIT, 32 B */

/* ACCEPT (AcceptPacket), 48 B.  The request body ("blob") lives in a payload
 * arena: nreq==1 -> the raw requestValue bytes; nreq>1 -> nreq x gpx_batch_ent
 * followed by the concatenated requestValues (RequestPacket.batched). */
typedef struct gpx_accept_rec {
  gpx_pvalue_hdr h;
  uint32_t payload_off;
  uint32_t payload_len;
  uint32_t nreq;
  int32_t sender; /* AcceptPacket.sender (node id) == coordinator that issued it */
} gpx_accept_rec;

/* per-request entry of a batched blob, 16 B */
typedef struct gpx_batch_ent {
  int64_t req_id;
  uint32_t len;
  uint32_t flags; /* bit0 STOP; bits 8.. entry lane (as gpx_request_rec.flags) */
} gpx_batch_ent;

/* ACCEPT_REPLY / one slot of a BATCHED_ACCEPT_REPLY, 32 B */
typedef struct gpx_accept_reply_rec {
  uint32_t gid;
  int32_t slot;   /* AcceptReplyPacket.slotNumber */
  int32_t bnum;   /* acceptor's ballot after handling the accept */
  int32_t bcoord;
  int32_t max_cp; /* AcceptReplyPacket.maxCheckpointedSlot (= acceptor slot - 1) */
  uint32_t who;   /* bits 0..7 acceptor member index, 8..15 destination member index
                     (the accept's sender), 16..31 flags (GPX_F_VOID|LOGGED|NACK) */
  int64_t req_id;
} gpx_accept_reply_rec;

#define GPX_WHO(acc_idx, dst_idx, flags) \
  ((uint32_t)(acc_idx) | ((uint32_t)(dst_idx) << 8) | ((uint32_t)(flags) << 16))
#define GPX_WHO_ACC(w) ((w) & 0xffu)
#define GPX_WHO_DST(w) (((w) >> 8) & 0xffu)
#define GPX_WHO_FLAGS(w) ((w) >> 16)

/* in-order execution record handed to the Replicable app, 24 B */
typedef struct gpx_exec_rec {
  uint32_t gid;
  int32_t slot;
  int64_t req_id;
  uint32_t payload_off; /* (byte offset of the blob in the lane's log ring) / 16 */
  uint32_t flags;       /* bits 0..11 GPX_F_STOP|VOID|CKPT|EXTRA; bits 12..15 lane; bits 16..31 nreq */
} gpx_exec_rec;

/* ---- log ring ---------------------------------------------------------------
 * One ring per lane.  A ring is a sequence of segments, one per kernel launch
 * that logs: [gpx_log_seg_hdr 64 B][n_slots record images][payload area].
 * ACCEPT segment (rec_bytes 48): the images are stored as two planes, n_slots x 32 B pvalue
 * headers followed by n_slots x 16 B {payload_off,payload_len,nreq,sender}, so that every image
 * moves as one 256-bit plus one 128-bit aligned store; image.payload_off is relative to the
 * segment's payload area; unlogged records have GPX_F_VOID.  Segments are 32-byte multiples.
 * DECISION segment: images are gpx_decision_rec (32 B), no payload area.
 * (SQLPaxosLogger.journal frames {int32 len}{packet bytes}, :1000-1003; gpx_wire_*
 * re-frames segments into that byte format.) */
#define GPX_SEG_MAGIC 0x53585047u /* "GPXS" */
typedef struct gpx_log_seg_hdr {
  uint32_t magic;
  uint16_t type; /* GPX_F_ACCEPT or GPX_F_DECISION */
  uint16_t lane;
  uint32_t n_slots;       /* record images reserved */
  uint32_t n_valid;       /* leading image slots in use (<= n_slots); some of them may be VOID holes */
  uint64_t payload_bytes; /* payload area bytes (ACCEPT segments) */
  uint64_t seq;           /* segment sequence number of this lane */
  uint64_t ring_off;      /* absolute ring offset of this header */
  uint32_t rec_bytes;     /* 48 or 32 */
  uint32_t reserved[5];
} gpx_log_seg_hdr;

/* ---- group management ------------------------------------------------------- */

/* HotRestoreInfo field set for one (lane, gid) row, paxosutil/HotRestoreInfo.java:31-120 */
typedef struct gpx_row {
  uint32_t gid;
  uint32_t lane;
  int32_t version;
  int32_t acc_slot;       /* accSlot */
  int32_t acc_bnum;       /* accBallot */
  int32_t acc_bcoord;
  int32_t acc_gc_slot;    /* accGCSlot */
  int32_t state;          /* GPX_ST_* */
  int32_t coord_exists;   /* coordBallot != null */
  int32_t coord_active;
  int32_t coord_bnum;
  int32_t coord_bcoord;
  int32_t next_proposal_slot;
  int32_t n_members;
  int32_t members[GPX_MAX_GROUP_SIZE];    /* sorted ascending node ids */
  int32_t node_slots[GPX_MAX_GROUP_SIZE]; /* PaxosCoordinatorState.nodeSlotNumbers */
  int32_t name_hash;      /* String.hashCode() of the paxosID (HotRestoreInfo.paxosID): getCPI :2694-2697 is a function of
                           * the paxosID, and a restored instance may get a different gid than it was created under */
} gpx_row;

#define GPX_INIT_BATCH 0   /* HotRestoreInfo.createHRI path (PaxosManager.java:664-691) */
#define GPX_INIT_DEFAULT 1 /* PISM.initiateRecovery + putInitialState path (:591-703) */

typedef struct gpx_group_desc {
  uint32_t gid;
  int32_t version;
  int32_t name_hash; /* Java String.hashCode() of the paxosID */
  int32_t n_members;
  int32_t members[GPX_MAX_GROUP_SIZE]; /* node ids, any order (sorted by the engine) */
  int32_t init_mode;                   /* GPX_INIT_* */
} gpx_group_desc;

/* host -> device state patch (slow path effects), applied between batches */
enum {
  GPX_PATCH_SET_BALLOT = 1,    /* acceptor ballot <- (a,b) if higher (handlePrepare) */
  GPX_PATCH_JUMP_SLOT = 2,     /* acceptor.jumpSlot(a) */
  GPX_PATCH_SET_STATE = 3,     /* acceptor state <- a (forceStop, setActive) */
  GPX_PATCH_INSTALL_COORD = 4, /* coordinator (bnum=a, bcoord=b, next=c, active=d) */
  GPX_PATCH_RESIGN_COORD = 5,  /* coordinator <- null */
  GPX_PATCH_SET_GC = 6,        /* acceptedGCSlot <- a */
  GPX_PATCH_SET_NODE_SLOT = 7  /* coordinator's nodeSlotNumbers[a] <- b if higher (recordSlotNumber :786-807 on a
                                * PREPARE_REPLY, host side of phase 1) */
};
typedef struct gpx_patch_rec {
  uint32_t gid;
  uint32_t lane;
  int32_t op;
  int32_t a, b, c, d;
  int32_t reserved;
} gpx_patch_rec;

/* ---- configuration ----------------------------------------------------------- */

typedef struct gpx_config {
  uint32_t abi_version;
  int32_t device;            /* CUDA device ordinal */
  uint32_t max_groups;       /* PINSTANCES_CAPACITY analogue: rows per lane */
  uint32_t n_lanes;          /* co-located replicas */
  int32_t lane_node[GPX_MAX_LANES]; /* node id served by each lane */
  uint32_t window;           /* W: 1,2,4,8 */
  uint32_t max_group_size;   /* <= GPX_MAX_GROUP_SIZE: node_slots columns allocated */
  uint64_t log_ring_bytes;   /* per lane, power of two; 0 => logging disabled (DISABLE_LOGGING) */
  uint32_t max_batch_recs;   /* largest record batch one call may carry */
  uint64_t max_batch_payload;/* largest payload arena one call may carry */
  /* gigapaxos.properties subset (PaxosConfig.java PC enum), same defaults */
  int32_t batching_enabled;        /* BATCHING_ENABLED :309 (true) */
  int32_t max_batch_size;          /* MAX_BATCH_SIZE :403 (2000) */
  int64_t max_batch_bytes;         /* min(NIO MAX_PAYLOAD_SIZE 4MB, MAX_LOG_MESSAGE_SIZE 5MB) */
  int32_t request_size_estimate;   /* RequestPacket.SIZE_ESTIMATE (:1351-1367) */
  int32_t checkpoint_interval;     /* CHECKPOINT_INTERVAL :410 (400) */
  double cpi_noise;                /* CPI_NOISE :746 (0) */
  int32_t gc_majority_executed;    /* GC_MAJORITY_EXECUTED :882 (true) */
  int32_t log_meta_decisions;      /* LOG_META_DECISIONS :588 (true) */
  int32_t journaling_enabled;      /* ENABLE_JOURNALING :240 (true): executed accepts leave memory */
  /* (BATCHED_ACCEPT_REPLIES :458, BATCHED_COMMITS :466, MIN_PP_BATCH_SIZE :860 shape how PaxosPacketBatcher packs
   * records into wire packets -- the engine exchanges fixed-size records, packing happens where packets are formed
   * (gpx_wire_*); SHORT_CIRCUIT_LOCAL :834 and DIGEST_REQUESTS :788 are host-side choices (DESIGN.md 2.3,
   * gpx_digest_requests): none of them is engine configuration, so none is carried here) */
  int32_t log_backpressure;        /* 1: a call that could overwrite log bytes not yet released by gpx_log_release is
                                    * refused with GPX_EAGAIN (log-then-message, AbstractPaxosLogger.java:691-716: the
                                    * journal must be drained before a ring position is reused); 0 (default): the ring
                                    * overwrites the oldest bytes */
  int32_t reserved[7];
} gpx_config;

typedef struct gpx_counters {
  uint64_t accepts_handled, accepts_acked, accepts_nacked, accepts_logged, accepts_dropped;
  uint64_t replies_handled, replies_ignored, preempted, coordinators_resigned;
  uint64_t decisions_made, decisions_handled, decisions_dropped, placeholders;
  uint64_t executed, stops_executed, checkpoints_due;
  uint64_t proposals, requests_batched, requests_rejected;
  uint64_t window_overflow, kernel_launches;
  uint64_t reserved[7];
} gpx_counters;

typedef struct gpx_engine gpx_engine;

/* ---- lifecycle ---------------------------------------------------------------- */
void gpx_config_defaults(gpx_config* cfg);
/* parse the gigapaxos.properties keys the engine consumes; unknown keys ignored */
int gpx_config_from_properties(const char* path, gpx_config* cfg);
int gpx_engine_create(const gpx_config* cfg, gpx_engine** out);
void gpx_engine_destroy(gpx_engine* e);
const char* gpx_last_error(void);
const char* gpx_build_info(void); /* "cuda sm_100a ..." or "oracle" */

/* ---- groups -------------------------------------------------------------------- */
int gpx_create_groups(gpx_engine* e, uint32_t n, const gpx_group_desc* descs);
int gpx_destroy_groups(gpx_engine* e, uint32_t n, const uint32_t* gids);
int gpx_dump_rows(gpx_engine* e, uint32_t n, const uint32_t* gids, uint32_t lane, gpx_row* out);
int gpx_load_rows(gpx_engine* e, uint32_t n, const gpx_row* rows);
int gpx_patch(gpx_engine* e, uint32_t n, const gpx_patch_rec* patches);

/* ---- data path: host buffers in, host buffers out (H2D and D2H inside) ---------- */

/* RequestBatcher + PCS.propose.  reqs must be grouped by gid (per-group FIFO order
 * preserved).  out_accepts capacity n; out_blob capacity blob_cap bytes (>= payload_bytes
 * + 16*n); status[n] receives the slot (>0) or a GPX_RS_* code. */
int gpx_propose(gpx_engine* e, uint32_t n, const gpx_request_rec* reqs, const uint8_t* payload,
                uint64_t payload_bytes, gpx_accept_rec* out_accepts, uint32_t* n_accepts,
                uint8_t* out_blob, uint64_t blob_cap, uint64_t* blob_bytes, int32_t* status);

/* handleAccept at every local lane in rec.dst_mask.  accepts must be grouped by gid.
 * out_replies[n * n_lanes] (index i*n_lanes+lane, GPX_F_VOID where not addressed/dropped).
 * out_extra_exec (cap extra_cap) receives EXEC records released by reconstructDecision. */
int gpx_handle_accepts(gpx_engine* e, uint32_t n, const gpx_accept_rec* accepts,
                       const uint8_t* blob, uint64_t blob_bytes, gpx_accept_reply_rec* out_replies,
                       gpx_exec_rec* out_extra_exec, uint32_t extra_cap, uint32_t* n_extra);

/* handleAcceptReply at the destination lane of each reply; replies grouped by gid.
 * out_decisions capacity n. */
int gpx_handle_accept_replies(gpx_engine* e, uint32_t n, const gpx_accept_reply_rec* replies,
                              gpx_decision_rec* out_decisions, uint32_t* n_decisions);

/* handleBatchedCommit per slot at every local lane in rec.dst_mask; grouped by gid.
 * out_exec[n * n_lanes] primary EXEC record per (decision, lane) (VOID if none);
 * further in-order executions released by the same decision go to out_extra_exec. */
int gpx_handle_decisions(gpx_engine* e, uint32_t n, const gpx_decision_rec* decisions,
                         gpx_exec_rec* out_exec, gpx_exec_rec* out_extra_exec, uint32_t extra_cap,
                         uint32_t* n_extra);

/* Fused co-located path (PaxosManager.sendOrLoopback :2116-2128): per ACCEPT, in batch order,
 * handleAccept at every addressed lane; replies addressed to a usable LOCAL coordinator lane are
 * handled at once (the others are returned in out_replies, VOID where consumed); a resulting
 * DECISION (out_decisions[n], VOID where none) is handled at every local lane before the next
 * ACCEPT.  out_exec[n * n_lanes].  EXEC records of one call are applied per group in slot order
 * (primary and extra records interleave). */
int gpx_handle_accepts_fused(gpx_engine* e, uint32_t n, const gpx_accept_rec* accepts, const uint8_t* blob,
                             uint64_t blob_bytes, gpx_accept_reply_rec* out_replies,
                             gpx_decision_rec* out_decisions, gpx_exec_rec* out_exec,
                             gpx_exec_rec* out_extra_exec, uint32_t extra_cap, uint32_t* n_extra);

/* ---- phase 1a at the acceptors ------------------------------------------------------------------
 * PREPARE = a gpx_pvalue_hdr whose `slot` is PreparePacket.firstUndecidedSlot and whose ballot is the would-be
 * coordinator's.  gpx_handle_prepares runs PISM.handlePrepare :896-955 / PaxosAcceptor.handlePrepare :239-275
 * at every addressed local lane: a stopped instance drops it; a higher ballot is adopted; the reply carries the
 * acceptor's ballot after that (NACK if it is higher than the PREPARE's), firstSlot =
 * getMaxGCSlotFirstUndecidedSlot :277-282 and -- unless NACKing -- the accepted pvalues with slot >=
 * firstUndecidedSlot in slot order (pruneAcceptedProposals :285-297).  When the ballot was raised the PREPARE is
 * appended to the lane's log ring before the reply is visible (LogMessagingTask, :940-944; segment type
 * GPX_F_PREPARE) and the reply is flagged GPX_F_LOGGED.  The coordinator side (PCS.isPrepareAcceptedByMajority,
 * combinePValuesOntoProposals) stays on the host and installs its result with gpx_patch. */
typedef struct gpx_accepted_pvalue { /* one accepted pvalue of a PREPARE_REPLY, 32 B (the accepted-window entry) */
  int32_t slot;
  int32_t bnum;
  int32_t bcoord;
  uint32_t frame_ref;   /* offset / 16 of the request blob in this acceptor's log ring (which wraps) */
  int64_t req_id;
  uint32_t payload_len;
  uint32_t flags;       /* bit1 STOP, bits 16.. nreq */
} gpx_accepted_pvalue;
typedef struct gpx_prepare_reply_rec { /* PrepareReplyPacket, 32 + 32 * GPX_MAX_WINDOW bytes */
  uint32_t gid;
  int32_t first_slot;   /* PrepareReplyPacket.firstSlot */
  int32_t bnum;         /* acceptor's ballot after handling the PREPARE */
  int32_t bcoord;
  uint32_t who;         /* GPX_WHO(acceptor idx, preparer idx, GPX_F_VOID | GPX_F_NACK | GPX_F_LOGGED | GPX_F_FROM_LOG) */
  uint32_t n_accepted;
  int64_t reserved;
  gpx_accepted_pvalue accepted[GPX_MAX_WINDOW];
} gpx_prepare_reply_rec;
/* out_replies[n * n_lanes] */
int gpx_handle_prepares(gpx_engine* e, uint32_t n, const gpx_pvalue_hdr* prepares, gpx_prepare_reply_rec* out_replies);

/* ---- phase 1b at the would-be coordinator -------------------------------------------------------
 * gpx_handle_prepare_replies runs, for a batch of elections (one candidate coordinator of one group each: the mass
 * fail-over after a node is lost is many groups electing at once), what PISM.handlePrepareReply :1017-1068 does per
 * PREPARE_REPLY and what follows a majority:
 *   PaxosCoordinator.getPreActivesIfPreempted :313-318 / PCS.isPreemptable :271-278   a reply with a higher ballot
 *       ends the election (GPX_EL_PREEMPTED; nothing is installed);
 *   PCS.canIgnorePrepareReply :287-316   lower ballot, not a member, already heard: ignored;
 *   PCS.isPrepareAcceptedByMajority :326-391   recordSlotNumber(PrepareReplyPacket) :786-807 with
 *       PrepareReplyPacket.getMinSlot :151-164 (= min(firstSlot, the accepted slots), wrap-aware), the pvalue of the
 *       highest ballot per slot is carried over, WaitforUtility majority;
 *   PCS.combinePValuesOntoProposals :393-444   the slots getMaxMinCarryoverSlot :921 .. getMaxPValueSlot :903 become
 *       the new coordinator's first proposals, carried-over pvalue or no-op (makeNoopPValue :886-897);
 *   PCS.processStop :478-554   every proposal carries the new ballot there (ProposalStateAtCoordinator's constructor
 *       :153-157 re-stamps it), so its two conversion branches cannot be taken; a regular request behind a STOP is the
 *       reference's `assert(false)` and is reported as GPX_ELF_STOP_ORDER; when a STOP was carried over and the last
 *       proposal is not a STOP, a fresh STOP is proposed behind it (:538-542);
 *   PCS.setCoordinatorActive :577-587   the coordinator is installed ACTIVE at `lane` with the recorded
 *       nodeSlotNumbers and nextProposalSlotNumber = the first slot of the plan; coordinators of a lower ballot at the
 *       other local lanes resign (PISM.handlePrepare would have removed them when the PREPARE arrived).
 * The plan is returned, not proposed: spawnCommandersForProposals :556-575 is the caller re-proposing plan[0..n_plan)
 * in order through gpx_propose / gpx_round (the request bodies of a carried-over pvalue are in the log ring of the
 * acceptor that reported it: reply index src_reply, ring offset frame_ref * 16).  The engine keeps no pre-active
 * proposals (a request that finds a pre-active coordinator gets GPX_RS_PREACTIVE and waits at the host), so
 * combinePValuesOntoProposals' preActives and reproposePreemptedProposals :460-468 have nothing to do here.
 *
 * A PREPARE_REPLY longer than GPX_MAX_WINDOW pvalues (accepts added from the journal, GPX_F_FROM_LOG) is given as
 * consecutive records of the same acceptor, all but the last flagged GPX_F_MORE in `who`.
 * Device rules (as for the slot window): more than GPX_MAX_CARRY distinct carried-over slots, or a plan range of more
 * than GPX_MAX_PLAN slots, gives GPX_EL_OVERFLOW and installs nothing -- the candidate is too far behind and syncs
 * first (PISM.syncLongDecisionGaps).  At most one election per gid per call (GPX_EINVAL otherwise). */
#define GPX_F_MORE 0x0800u /* prepare reply record: the same PREPARE_REPLY continues in the next record */
#define GPX_MAX_CARRY 32
#define GPX_MAX_PLAN 16
enum {
  GPX_EL_WAITING = 0,   /* no majority among the replies given */
  GPX_EL_MAJORITY = 1,  /* elected and installed */
  GPX_EL_PREEMPTED = 2, /* a reply carried a higher ballot */
  GPX_EL_DROPPED = 3,   /* no live instance at that lane / stopped / lane not a member (PISM :456-460) */
  GPX_EL_OVERFLOW = 4
};
enum {
  GPX_CO_NOOP = 0,     /* RequestPacket(0, NO_OP, false), entry replica = the new coordinator */
  GPX_CO_PVALUE = 1,   /* the carried-over pvalue's request(s), re-proposed under the new ballot */
  GPX_CO_STOP_NEW = 2  /* RequestPacket(0, STOP, true) :541 */
};
#define GPX_ELF_STOP_ORDER 1u /* a regular request lies behind a STOP in the plan: PCS.processStop's assert(false) */
typedef struct gpx_election_rec { /* one pre-active coordinator (PISM.checkRunForCoordinator :2090-2150), 32 B */
  uint32_t gid;
  uint32_t lane;        /* local lane of the candidate */
  int32_t bnum;         /* the ballot it sent its PREPARE with */
  int32_t bcoord;
  int32_t slot;         /* PCS ctor's nextProposalSlotNumber = paxosState.getSlot() (the PREPARE's firstUndecidedSlot) */
  uint32_t first_reply; /* replies[first_reply .. first_reply + n_replies) are handled in this order */
  uint32_t n_replies;
  uint32_t reserved;
} gpx_election_rec;
typedef struct gpx_carryover { /* one proposal of the view change, 48 B */
  int32_t slot;
  uint32_t kind;        /* GPX_CO_* */
  uint32_t src_reply;   /* GPX_CO_PVALUE: index into replies[] of the record that carried it */
  uint32_t reserved;
  gpx_accepted_pvalue pv; /* GPX_CO_PVALUE: as reported (its own, lower, ballot) */
} gpx_carryover;
typedef struct gpx_election_out { /* 16 + 64 + 17 * 48 = 896 B */
  uint32_t gid;
  int32_t verdict;      /* GPX_EL_* */
  int32_t next_slot;    /* GPX_EL_MAJORITY: the installed nextProposalSlotNumber (plan[0].slot when n_plan > 0) */
  uint16_t n_plan;
  uint16_t flags;       /* GPX_ELF_* */
  int32_t node_slots[GPX_MAX_GROUP_SIZE]; /* nodeSlotNumbers as recorded (-1 = not heard) */
  gpx_carryover plan[GPX_MAX_PLAN + 1];
} gpx_election_out;
/* replies: host array of n_reply_recs records; out[n] */
int gpx_handle_prepare_replies(gpx_engine* e, uint32_t n, const gpx_election_rec* elections, uint32_t n_reply_recs,
                               const gpx_prepare_reply_rec* replies, gpx_election_out* out);

/* One full round for co-located replicas.  gpx_round: RequestBatcher + propose, then the fused
 * accept -> tally -> commit per ACCEPT with replies, decisions and rows kept in registers.
 * gpx_round_phases: the same round phase by phase (all ACCEPTs, then all replies, then all
 * DECISIONs), inter-replica records going through HBM.  Host request buffers in, EXEC records out
 * (out_exec[*n_exec_slots], extras appended to out_extra_exec). */
int gpx_round(gpx_engine* e, uint32_t n, const gpx_request_rec* reqs, const uint8_t* payload,
              uint64_t payload_bytes, int32_t* status, gpx_exec_rec* out_exec, uint32_t* n_exec_slots,
              gpx_exec_rec* out_extra_exec, uint32_t extra_cap, uint32_t* n_extra);
int gpx_round_phases(gpx_engine* e, uint32_t n, const gpx_request_rec* reqs, const uint8_t* payload,
                     uint64_t payload_bytes, int32_t* status, gpx_exec_rec* out_exec, uint32_t* n_exec_slots,
                     gpx_exec_rec* out_extra_exec, uint32_t extra_cap, uint32_t* n_extra);

/* Pipelined form of gpx_round.  The reference's hot path is a pipeline of threads (RequestBatcher ->
 * PISM -> PaxosPacketBatcher / AbstractPaxosLogger.BatchedLogger -> Messenger): a batch is being collected
 * while the previous one is logged and the one before is executed.  gpx_round_submit enqueues the
 * host->device copy of a batch, the round kernels and the device->host copy of its results on three
 * streams and returns at once; up to GPX_PIPE_DEPTH rounds may be in flight, rounds execute in submission
 * order.  All host buffers of the io block must stay valid (and should be page-locked for the copies to
 * overlap) until gpx_round_wait(ticket) returns.
 *
 * Output modes:
 *   full (flags = 0)       status[n], exec[n * n_lanes] as gpx_round.
 *   GPX_ROUND_COMPACT      sum[n]: one 8-byte summary per REQUEST index.  lane_mask != 0: every lane in the
 *                          mask executed exactly this request at `slot`, as its next in-order execution
 *                          (flags: GPX_F_CKPT if PISM.shouldCheckpoint :2037 holds) -- the host runs
 *                          Replicable.execute from its own copy of the request.  lane_mask == 0: `slot` is
 *                          the request's status (slot number or GPX_RS_* code) and every execution it caused
 *                          is a full record in the extra queue.  EXEC records of one call are applied per
 *                          (lane, group) in slot order.
 *   GPX_ROUND_PACKED_REQS  (input) `reqs` holds n gpx_request_packed (16 B) instead of gpx_request_rec (32 B):
 *                          the payloads lie back to back in request order (payload_off = running sum of
 *                          payload_len), entry_node = the node of the entry lane, client = the request
 *                          index.  Halves the host->device bytes of a batch; the engine expands the records
 *                          on the device (k_unpack: block sums, scan, expand). */
#define GPX_PIPE_DEPTH 4
#define GPX_ROUND_COMPACT 1u
#define GPX_ROUND_PACKED_REQS 2u
typedef struct gpx_request_packed {
  uint32_t gid;
  uint16_t payload_len;
  uint16_t flags;  /* as gpx_request_rec.flags: bit0 GPX_F_STOP, bits 8..11 entry lane */
  int64_t req_id;
} gpx_request_packed;
typedef struct gpx_exec_sum {
  int32_t slot;       /* decided slot (lane_mask != 0) or the request's status */
  uint8_t lane_mask;  /* lanes that executed the request in order */
  uint8_t flags;      /* GPX_F_CKPT */
  uint16_t nreq;      /* requests executed with it (1) */
} gpx_exec_sum;
typedef struct gpx_round_io {
  uint32_t n;
  uint32_t flags;              /* GPX_ROUND_COMPACT | GPX_ROUND_PACKED_REQS */
  const gpx_request_rec* reqs; /* [n] host (gpx_request_packed[n] with GPX_ROUND_PACKED_REQS) */
  const uint8_t* payload;      /* host */
  uint64_t payload_bytes;
  int32_t* status;             /* [n] out, full mode */
  gpx_exec_rec* exec;          /* [n * n_lanes] out, full mode */
  gpx_exec_sum* sum;           /* [n] out, compact mode */
  gpx_exec_rec* extra;         /* [extra_cap] out: further executions (filled by gpx_round_wait; *n_extra >
                                * extra_cap = truncated.  compact mode needs up to n * n_lanes + the full mode's) */
  uint32_t extra_cap;
} gpx_round_io;
int gpx_round_submit(gpx_engine* e, const gpx_round_io* io, uint64_t* ticket);
/* blocks until round `ticket` is complete; rounds must be waited for in submission order */
int gpx_round_wait(gpx_engine* e, uint64_t ticket, uint32_t* n_exec_slots, uint32_t* n_extra);

/* Digest path (DIGEST_REQUESTS, paxospackets/RequestPacket.java:1414-1430, AcceptPacket.digest :162-170):
 * MD5 of every request's requestValue, 16 bytes each -- the digest a coordinator puts into an ACCEPT in
 * place of the request body and an acceptor checks against the body it received by broadcast
 * (paxosutil/PendingDigests.java:82-145, host side). */
int gpx_digest_requests(gpx_engine* e, uint32_t n, const gpx_request_rec* reqs, const uint8_t* payload,
                        uint64_t payload_bytes, uint8_t* out_digests);

/* ---- log ring ------------------------------------------------------------------- */
/* copy ring bytes [from, min(head, from+cap)) of `lane` into dst; *head receives the ring head */
int gpx_log_read(gpx_engine* e, uint32_t lane, uint64_t from, void* dst, uint64_t cap,
                 uint64_t* n_copied, uint64_t* head);

/* Drain without stopping the rounds (AbstractPaxosLogger.BatchedLogger :691-716 is a thread beside the protocol
 * threads; SQLPaxosLogger.journal :965-1036 / Journaler.appendToLogFile :814-826 append to the journal file).
 * gpx_log_drain_async enqueues, on the engine's own drain stream and behind the work already enqueued on
 * `after_stream` (a cudaStream_t; NULL = the engine's stream), the copy of the next undrained ring bytes of `lane`
 * -- [*from, *from + *n_bytes), at most cap, in ring order -- into dst (host memory; page-locked to overlap) and
 * returns at once.  The host tracks the ring heads itself (every logging call has a host-known size), so no device
 * read is involved.  gpx_log_drain_wait blocks until the enqueued copies are done; gpx_log_release(lane, upto) tells
 * the engine that everything before `upto` is durable elsewhere: with gpx_config.log_backpressure set, a call
 * that would overwrite unreleased bytes is refused with GPX_EAGAIN before it does anything. */
int gpx_log_drain_async(gpx_engine* e, uint32_t lane, void* dst, uint64_t cap, uint64_t* from, uint64_t* n_bytes,
                        void* after_stream);
int gpx_log_drain_wait(gpx_engine* e);
int gpx_log_drain_skip(gpx_engine* e); /* drop the backlog: drain cursor and tail <- current heads */
int gpx_log_release(gpx_engine* e, uint32_t lane, uint64_t upto);

/* ---- finding logged pvalues: the journal's index as a scan ---------------------------------------------------------
 * A replica that answers a SYNC_DECISIONS_REQUEST (PISM.handleSyncDecisionsPacket :2426-2510) or a PREPARE from a
 * lagging node (PISM.handlePrepare :900-955 with GET_ACCEPTED_PVALUES_FROM_DISK) needs decisions / accepts that have
 * left its memory: AbstractPaxosLogger.getLoggedDecisions :582 / getLoggedAccepts :568, which with journaling are
 * SQLPaxosLogger.getLoggedFromMessageLog :3674-3756 -- look the (paxosID, slot range) up in the per-group
 * paxosutil/LogIndex (:213-248), read those frames back from the journal files, and keep per slot the entry logged
 * LAST (`accepts.put(packet.slot, packet)` :3746 in log order).  The engine keeps no index on the hot path; the log ring
 * is in HBM, so the lookup is a scan of it: one thread walks the segment headers from `from` (a segment boundary:
 * 0 while the ring has not wrapped, else a position handed out by gpx_log_drain_async / gpx_log_release) to the head,
 * one thread per logged image matches (gid, slot) against the batch of wants (sorted by gid, one want per gid, at
 * most GPX_LOG_SPAN slots each), the LAST logged DECISION and ACCEPT image per wanted slot win.
 * out[i * GPX_LOG_SPAN + k] answers slot wants[i].min_slot + k: the two images (flags GPX_F_VOID where there is none;
 * accept.payload_off is relative to its segment's payload area as in the ring) and the absolute ring position of the
 * accept's request blob (gpx_log_read(lane, blob_pos, dst, accept.payload_len, ...)).  getActualDecisions :2539-2583
 * (a meta decision gets its value from the logged accept of the slot) is the caller joining the two. */
#define GPX_LOG_SPAN 16
typedef struct gpx_log_want { /* 16 B */
  uint32_t gid;
  int32_t min_slot;
  uint32_t n_slots;  /* <= GPX_LOG_SPAN */
  uint32_t reserved;
} gpx_log_want;
typedef struct gpx_log_hit { /* 96 B */
  gpx_decision_rec decision;
  gpx_accept_rec accept;
  uint64_t blob_pos;
  uint64_t reserved;
} gpx_log_hit;
int gpx_log_find(gpx_engine* e, uint32_t lane, uint64_t from, uint32_t n, const gpx_log_want* wants, gpx_log_hit* out);

/* Request bodies for a batch of gpx_log_find hits (or of carried-over pvalues: ring offset frame_ref * 16, which is the
 * position until the ring wraps) in ONE device->host copy: ranges[i] = {ring position, length, offset in dst (a multiple
 * of 16)}; range i lands at dst + dst_off rounded up to whole 16-byte chunks (the ring's payload areas are padded to
 * 16).  The journal analogue is SQLPaxosLogger.getJournaledMessage(FileOffsetLength[]) :3712 (frames in one pass). */
typedef struct gpx_log_range { /* 16 B */
  uint64_t pos;
  uint32_t len;
  uint32_t dst_off;
} gpx_log_range;
int gpx_log_gather(gpx_engine* e, uint32_t lane, uint32_t n, const gpx_log_range* ranges, void* dst, uint64_t dst_bytes);

/* ---- introspection ---------------------------------------------------------------- */
int gpx_get_counters(gpx_engine* e, gpx_counters* out);
int gpx_reset_counters(gpx_engine* e);
/* slow-path list: per-group flag byte of one lane (bit0 window overflow: a record beyond the
 * in-flight window W was dropped; bit1 needs sync: a commit could not be resolved locally ->
 * host runs PISM.syncLongDecisionGaps :1550 / requestMissingDecisions) */
#define GPX_GF_OVERFLOW_BIT 1u
#define GPX_GF_NEEDS_SYNC_BIT 2u
/* computed on the fly: the lane is NOT caught up -- PaxosAcceptor.caughtUp :452-459 (committedRequests empty, and
 * acceptedProposals empty unless journaling serves accepted pvalues from disk) or PCS.caughtUp :758 (myProposals
 * empty) is false.  PISM.tryPause :2004-2035 pauses an instance only when this bit is clear on every lane. */
#define GPX_GF_NOT_CAUGHT_UP_BIT 4u
int gpx_get_group_flags(gpx_engine* e, uint32_t lane, uint32_t n, const uint32_t* gids, uint8_t* out);
/* ---- the slow-path list (SURVEY.md 8b) / the candidates of a sweep --------------------------------------------------
 * PaxosManager's sweeps walk ALL instances (syncAndDeactivate :2806-2900 iterates pinstances; the failure detector's
 * checkRunForCoordinator pass likewise) and test each one; with millions of groups resident the test belongs where the
 * state is.  gpx_select_groups returns the live groups of `lane` whose flag byte -- exactly what gpx_get_group_flags
 * reports: GPX_GF_OVERFLOW_BIT | GPX_GF_NEEDS_SYNC_BIT | GPX_GF_NOT_CAUGHT_UP_BIT -- satisfies
 * (flags & mask) == value and whose acceptor is ACTIVE: mask = value = GPX_GF_NEEDS_SYNC_BIT lists the groups to sync
 * (PISM.syncLongDecisionGaps :1550), mask = GPX_GF_NOT_CAUGHT_UP_BIT, value = 0 the pause candidates
 * (PISM.tryPause :2004).  out_gids[0 .. min(*n_found, cap)) in ascending order; *n_found is the number that matched
 * (when it exceeds cap, which `cap` of them were returned is unspecified: ask again with a larger buffer). */
int gpx_select_groups(gpx_engine* e, uint32_t lane, uint32_t mask, uint32_t value, uint32_t* out_gids, uint32_t cap,
                      uint32_t* n_found);

/* What a listed group is missing: PISM.requestMissingDecisions :2292-2320 at `lane` for a batch of groups --
 * PaxosAcceptor.getMaxCommittedSlot :425-438 (the highest committed slot held, slot - 1 when there is none or the acceptor
 * is stopped), getMissingCommittedSlots(sizeLimit) :405-423 (from the next slot to execute up to the highest committed one:
 * no commit there, or a value-less commit without its accept) -- [slot] itself when nothing else is missing (:2297-2298) --
 * and isMissingTooMuch :2367-2370 = shouldSync(maxCommittedSlot, too_much_gap) :2341-2361 in its default mode (the
 * reference passes getMaxSyncDecisionsGap()).  These are the fields of the SYNC_DECISIONS_REQUEST the host sends
 * (SyncDecisionsPacket); whom to ask (:2305-2312) stays with the host.  With the bounded window a commit further than W
 * slots ahead is not held (it was dropped and flagged NEEDS_SYNC), so at most W - 1 slots are listed.
 * n_missing == 0: stopped / no live instance -- no request (getMissingCommittedSlots returns null). */
typedef struct gpx_missing_rec { /* 48 B */
  uint32_t gid;
  int32_t slot;               /* paxosState.getSlot(): the next slot to execute */
  int32_t max_decision_slot;  /* getMaxCommittedSlot() */
  uint16_t n_missing;
  uint8_t missing_too_much;
  uint8_t flags;              /* the group's flag byte (GPX_GF_*) */
  int32_t missing[GPX_MAX_WINDOW];
} gpx_missing_rec;
int gpx_missing_decisions(gpx_engine* e, uint32_t lane, uint32_t n, const uint32_t* gids, int32_t size_limit,
                          int32_t too_much_gap, gpx_missing_rec* out);

/* The OVERFLOW / NEEDS_SYNC bits are sticky: they stay until the host has dealt with the group (caught it up by a sync or
 * a checkpoint transfer) and says so -- out of the slow-path list.  Clears `mask` (of those two bits) at `lane` for
 * every gid given. */
int gpx_clear_group_flags(gpx_engine* e, uint32_t lane, uint32_t n, const uint32_t* gids, uint32_t mask);

/* ---- batched pause: the deactivation sweep (PaxosManager.Deactivator :2951 -> syncAndDeactivate :2806-2900 ->
 * pause(Map, dequeue) :2327-2366, PAUSE_BATCH_SIZE PaxosConfig.java:715) as one launch.  For every gid of the batch,
 * PISM.tryPause :2004-2035 at every local lane that hosts a replica: the group is paused only if it is live, every such
 * acceptor is ACTIVE and every lane is caught up (GPX_GF_NOT_CAUGHT_UP_BIT clear).  Then out_rows[i * n_lanes + lane]
 * = the HotRestoreInfo field set of every lane (what gpx_dump_rows returns; the caller turns them into the pause
 * table's strings, SQLPaxosLogger.pause) and the gid is free as after gpx_destroy_groups (forceStop + softCrash
 * :2284-2300).  out_paused[i] = 1 / 0; a group that does not pause is not touched and its rows are not written.
 * No gid may appear twice (GPX_EINVAL).  Unpause (PaxosManager.unpause :2370, PISM.hotRestore :677-690) =
 * gpx_load_rows. */
int gpx_pause_groups(gpx_engine* e, uint32_t n, const uint32_t* gids, gpx_row* out_rows, uint8_t* out_paused);
/* `active.<name>=host:port` entries (PaxosConfig.getActives :156-170) of the last
 * gpx_config_from_properties call, as "name=host:port\n" lines */
int gpx_properties_actives(char* out, size_t cap);

/* ---- device-resident API (bench `value`, multi-GPU shards): all pointers are device
 * pointers owned by the caller, `stream` is a cudaStream_t ------------------------------ */
typedef struct gpx_dev_round_bufs {
  const gpx_request_rec* reqs; /* [n] device */
  const uint8_t* payload;      /* device */
  uint64_t payload_bytes;
  uint32_t n;
  int32_t* status;             /* [n] device */
  gpx_exec_rec* exec;          /* [n * n_lanes] device */
} gpx_dev_round_bufs;
int gpx_round_device(gpx_engine* e, const gpx_dev_round_bufs* b, void* stream);        /* fused */
/* Form of the fused round.  0 / 1 (default): k_round_slow -- the general code for runs that are not the plain in-order
 * case -- is launched from the device, as a tail launch, by the first team that leaves a run over: a round without
 * such runs is ONE kernel on the stream.  2: the host launches k_round_slow behind every k_round (tuning / fallback). */
int gpx_set_round_mode(gpx_engine* e, int mode);
int gpx_round_device_phases(gpx_engine* e, const gpx_dev_round_bufs* b, void* stream); /* phase by phase */
/* gpx_propose + gpx_handle_accepts_fused on device buffers: ACCEPTs compacted at the front (exec[k * n_lanes + lane]
 * belongs to the k-th ACCEPT of the batch; the count is gpx_counters.proposals' increment), no per-request holes in
 * the log segments -- the form for batches in which many requests share a slot (RequestBatcher.java:198-219) */
int gpx_round_device_compact(gpx_engine* e, const gpx_dev_round_bufs* b, void* stream);
/* ---- device-resident phase calls: replicas of a group in DIFFERENT engines (spread placement:
 * one engine per GPU hosts one node; ACCEPT / ACCEPT_REPLY / DECISION records travel between engines
 * over NVLink).  Everything is asynchronous on `stream`; all pointers are device pointers unless
 * noted.  `ctl` is a caller-owned device block the kernels count into (the caller zeroes it). ---- */
typedef struct gpx_dev_ctl {
  uint32_t n_accepts;   /* gpx_propose_device: ACCEPTs written */
  uint32_t n_decisions; /* gpx_replies_device: DECISIONs appended (accumulates over calls) */
  uint32_t n_extra;     /* EXEC records appended to the extra queue */
  uint32_t any_batched;
  uint64_t blob1_used;  /* bytes of constructed (batched) blobs behind the payload arena */
  uint32_t n_todo;
  uint32_t pad;
} gpx_dev_ctl;
/* RequestBatcher + PISM.handleProposal / PCS.propose: out_accepts[<= n] (grouped by gid, dst_mask = all
 * members), payload_off relative to [payload arena | engine-owned batched blobs] */
int gpx_propose_device(gpx_engine* e, const gpx_request_rec* reqs, const uint8_t* payload, uint64_t payload_bytes,
                       uint32_t n, int32_t* status, gpx_accept_rec* out_accepts, gpx_dev_ctl* ctl, void* stream);
/* PaxosPacketBatcher per-destination grouping + PaxosManager.send unicast split (:2098-2128): bucket the
 * records of one kind (GPX_F_ACCEPT, GPX_F_DECISION, 0 = ACCEPT_REPLY) by destination node.
 * dest_nodes[n_dest <= 8] (host) lists the nodes served, the local one included (loopback).
 * out_recs[n_dest][cap], out_counts[n_dest] (zeroed by the caller); ACCEPTs also re-pack their blobs:
 * out_blob[n_dest][blob_cap], out_blob_units[n_dest] = bytes / 16.  Records of a group stay adjacent
 * and ordered inside a bucket.  *dropped counts records without a served destination / over capacity. */
int gpx_route_device(gpx_engine* e, uint32_t kind, const void* recs, const uint32_t* n_ptr, uint32_t n_max,
                     const uint8_t* payload, uint64_t payload_bytes, uint32_t n_dest, const int32_t* dest_nodes,
                     void* out_recs, uint32_t cap, uint32_t* out_counts, uint8_t* out_blob, uint64_t blob_cap,
                     uint32_t* out_blob_units, uint32_t* dropped, void* stream);
/* PISM.handleAccept at the local lanes for n received ACCEPTs = n_chunks concatenated buckets (chunk c ends
 * at record chunk_rec_end[c], its blob starts at chunk_blob_base[c] of `blob`; host arrays); payload_off of
 * the records is rebased in place.  out_replies[n * n_lanes]; executions released by
 * reconstructDecision go to out_extra[ctl->n_extra++]. */
int gpx_accepts_device(gpx_engine* e, gpx_accept_rec* recs, uint32_t n, const uint8_t* blob, uint64_t blob_bytes,
                       uint32_t n_chunks, const uint32_t* chunk_rec_end, const uint64_t* chunk_blob_base,
                       gpx_accept_reply_rec* out_replies, gpx_exec_rec* out_extra, uint32_t extra_cap,
                       gpx_dev_ctl* ctl, void* stream);
/* PaxosCoordinator.handleAcceptReply for n replies grouped by gid (one bucket of one acceptor at a time keeps
 * the replies of a group in one run); DECISIONs are appended at out_decisions[ctl->n_decisions++] */
int gpx_replies_device(gpx_engine* e, const gpx_accept_reply_rec* replies, uint32_t n,
                       gpx_decision_rec* out_decisions, gpx_dev_ctl* ctl, void* stream);
/* PISM.handleBatchedCommit + extractExecuteAndCheckpoint: out_exec[n * n_lanes], further executions in
 * out_extra[ctl->n_extra++].  (Received ACCEPT / DECISION records get their dst_mask -- a LOCAL lane mask --
 * rewritten in place to this engine's member lanes.) */
int gpx_decisions_device(gpx_engine* e, gpx_decision_rec* decisions, uint32_t n, gpx_exec_rec* out_exec,
                         gpx_exec_rec* out_extra, uint32_t extra_cap, gpx_dev_ctl* ctl, void* stream);

/* ---- SPREAD placement behind the C ABI (SURVEY.md 8e): the replicas of a group live in DIFFERENT engines -- one
 * single-lane engine per node, one node per GPU, replica j of a group on node (home + j) mod N
 * (PISM.roundRobinCoordinator :2251-2256) -- and the three inter-replica packet types of a round (ACCEPT,
 * ACCEPT_REPLY, DECISION; unicast fan-out paxosutil/PaxosMessenger.java:175-182, PaxosManager.send :2098-2128,
 * per-destination batching PaxosPacketBatcher.java:270-303) cross GPUs as fixed-capacity buckets whose record
 * count travels in-band: no host ever reads a count, a whole round is one asynchronous enqueue (optionally one
 * CUDA-graph launch) of  k_propose -> k_sp_route -> [exchange] -> k_sp_accept -> [exchange] -> k_sp_tally ->
 * [exchange] -> k_sp_commit.  The exchange is one ncclGroupStart / ncclSend + ncclRecv per peer / ncclGroupEnd per
 * packet type over NVLink (one process per GPU; libnccl.so.2 is loaded at run time), or plain device copies
 * when all nodes are engines of one process ("local" mode: tests on a single GPU).
 *
 * A Java PaxosManager would create one engine + one spread handle per GPU process, hand every batch of client
 * requests for the groups it coordinates to gpx_spread_round and apply the EXEC records it gets back; every
 * process of the spread group calls gpx_spread_round once per round (an empty batch still takes part in the
 * exchanges). */
#define GPX_SPREAD_MAX_NODES 8
#define GPX_SPREAD_GRAPH 1u /* capture a round into a CUDA graph per distinct io block and replay it */
#define GPX_SPREAD_P2P 2u   /* peer-memory transport: a node's send buckets ARE its peers' receive buckets (CUDA IPC between
                             * the per-GPU processes): k_sp_route / k_sp_accept / k_sp_tally store over NVLink, the exchange
                             * is a flag (k_sp_signal / k_sp_wait).  NCCL is then used once, to hand the IPC handles around */
typedef struct gpx_spread gpx_spread;
typedef struct gpx_spread_config {
  uint32_t n_nodes;                                         /* engines (nodes) of the spread group */
  int32_t node_ids[GPX_SPREAD_MAX_NODES];                   /* node id served by engine i (its lane 0) */
  uint32_t cap[GPX_SPREAD_MAX_NODES][GPX_SPREAD_MAX_NODES]; /* cap[s][d]: ACCEPTs node s may send node d in one round
                                                             * (>= groups s coordinates that d is a member of, times the
                                                             * slots a round may open per group); cap[s][s] is the
                                                             * loop-back bucket; 0 = the pair never exchanges.  The same
                                                             * matrix on every node. */
  uint32_t blob_per_rec; /* blob bytes a bucket reserves per record slot (multiple of 16): request bodies travel
                          * with their ACCEPT (AcceptPacket carries the RequestPacket, AcceptPacket.java:95-138) */
  uint32_t max_reqs;     /* requests one node submits per round (<= the engine's max_batch_recs) */
  uint32_t flags;        /* GPX_SPREAD_GRAPH | GPX_SPREAD_P2P */
  uint32_t reserved[8];
} gpx_spread_config;
/* what one node's buffers look like: byte offsets into its bucket arena, transfer sizes (0 = no transfer with that
 * peer), and the virtual index space of its receive side.  kind 0 = ACCEPT, 1 = ACCEPT_REPLY, 2 = DECISION.
 * Pure host arithmetic: send_bytes[k][d] of node s equals recv_bytes[k][s] of node d. */
typedef struct gpx_spread_plan {
  uint32_t n_nodes, rank;
  uint64_t send_off[3][GPX_SPREAD_MAX_NODES], send_bytes[3][GPX_SPREAD_MAX_NODES];
  uint64_t recv_off[3][GPX_SPREAD_MAX_NODES], recv_bytes[3][GPX_SPREAD_MAX_NODES];
  uint32_t vbase[GPX_SPREAD_MAX_NODES]; /* first virtual record index of the bucket received from node s */
  uint32_t vtotal;                      /* EXEC slots / log image slots per round at this node */
  uint64_t blob_off[GPX_SPREAD_MAX_NODES];
  uint64_t blob_vtotal;
  uint64_t arena_bytes;
} gpx_spread_plan;
int gpx_spread_plan_node(const gpx_spread_config* cfg, uint32_t rank, gpx_spread_plan* out);
/* per node and round: device pointers owned by the caller */
typedef struct gpx_spread_io {
  const gpx_request_rec* reqs; /* [n] requests for groups this node coordinates, grouped by gid (entry lane 0) */
  const uint8_t* payload;
  uint64_t payload_bytes;
  uint32_t n;
  uint32_t reserved;
  int32_t* status;    /* [n] */
  gpx_exec_rec* exec; /* [plan.vtotal]: EXEC record of the DECISION at that virtual index, VOID holes elsewhere */
  gpx_exec_rec* extra;
  uint32_t extra_cap;
  uint32_t reserved2;
  gpx_dev_ctl* ctl;   /* zeroed by the round; n_accepts / n_extra when it is done */
} gpx_spread_io;
/* 128-byte NCCL unique id (ncclGetUniqueId): made by one process, handed to the others by the host's own channel */
int gpx_spread_unique_id(void* out_id128);
/* one process per node: `e` is node `rank` of cfg->n_nodes; collective over the spread group (ncclCommInitRank) */
int gpx_spread_create_nccl(gpx_engine* e, const gpx_spread_config* cfg, uint32_t rank, const void* id128,
                           gpx_spread** out);
/* all cfg->n_nodes nodes are engines of this process (same device): the exchange is a set of device copies */
int gpx_spread_create_local(gpx_engine* const* engines, const gpx_spread_config* cfg, gpx_spread** out);
void gpx_spread_destroy(gpx_spread* sp);
/* one round, asynchronous on `stream`.  io[k] belongs to the k-th local node (NCCL mode: one; local mode: n_nodes) */
int gpx_spread_round(gpx_spread* sp, const gpx_spread_io* io, void* stream);
/* records k_sp_route could not place since creation (bucket too small / member node not in the spread group);
 * synchronises the device */
int gpx_spread_dropped(gpx_spread* sp, uint32_t local_index, uint32_t* out);

/* per-kernel CUDA-event timing of the last gpx_round_device calls (ms, accumulated) */
typedef struct gpx_kernel_times {
  double propose_ms, accept_ms, tally_ms, commit_ms;
  uint64_t launches;
} gpx_kernel_times;
int gpx_enable_kernel_timing(gpx_engine* e, int on);
int gpx_get_kernel_times(gpx_engine* e, gpx_kernel_times* out, int reset);

/* ---- helpers shared with the reference semantics ---------------------------------- */
int32_t gpx_java_string_hash(const char* s, size_t len); /* String.hashCode() */
/* PISM.roundRobinCoordinator :2251-2256 on sorted members */
int32_t gpx_round_robin_coordinator(int32_t name_hash, const int32_t* sorted_members, int32_t n,
                                    int32_t ballotnum);
/* PISM.getCPI :2694-2697 */
int32_t gpx_get_cpi(int32_t cpi, double noise, int32_t name_hash);

#ifdef __cplusplus
}
#endif
#endif /* GPX_H */
