/*
 * gpx_dev.cuh -- HBM state layout and per-record protocol transitions (device side).
 *
 * State is structure-of-arrays over a dense group index `gid`, one copy per co-located
 * replica ("lane").  Window arrays are laid out [lane][w][gid] so that groups advancing
 * in lockstep touch consecutive 32-byte entries (coalesced), and a straggling group
 * still costs exactly one 32-byte sector.
 *
 *   acc_row   int4  [L][G]      {_slot, ballotNum, ballotCoord, acceptedGCSlot}   PaxosAcceptor.java:94-99
 *   acc_aux   u32   [L][G]      state | committed-present mask | committed-valued mask | flags
 *   acc_win   2xint4[L][W][G]   accepted pvalue {slot,bnum,bcoord,frame_ref | reqID,plen,fl}  (acceptedProposals :108)
 *   com_win   2xint4[L][W][G]   committed decision {bnum,bcoord,medianCP,frame_ref | reqID,plen,fl} (committedRequests :109)
 *   coord_row int4  [L][G]      {myBallotNum, myBallotCoord, nextProposalSlotNumber, flags|outstanding<<8}
 *   node_slots i32  [L][R][G]   PaxosCoordinatorState.nodeSlotNumbers
 *   prop_win  int4  [L][W][G]   proposal {slot, votes|present|stop, reqID}  (myProposals + WaitforUtility bitmask)
 *   grp_meta  u32   [G]         member-set id | R | live
 *
 * All slot / ballot comparisons use Java's wrapping int subtraction (Ballot.java:60-66,
 * PaxosAcceptor.java:288,315,341,484).
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "gpx.h"
#include "gpx_logseg.cuh"

#define GPX_AUX_STATE(a) ((a) & 0xffu)
#define GPX_AUX_PRESENT(a) (((a) >> 8) & 0xffu)
#define GPX_AUX_VALUED(a) (((a) >> 16) & 0xffu)
#define GPX_AUX_FLAGS(a) ((a) >> 24)
#define GPX_GF_OVERFLOW 1u
#define GPX_GF_NEEDS_SYNC 2u

#define GPX_ENT_VALID 1u
#define GPX_ENT_STOP 2u

#define GPX_CF_EXISTS 1u
#define GPX_CF_ACTIVE 2u

#define GPX_PV_PRESENT (1u << 16)
#define GPX_PV_STOP (1u << 17)

#define GPX_META_LIVE (1u << 24)
#define GPX_META_IDENT (1u << 25) /* all R members are local lanes and lane l serves member index l */

/* counter indices == field order of gpx_counters */
enum {
  C_ACCEPTS_HANDLED = 0,
  C_ACCEPTS_ACKED,
  C_ACCEPTS_NACKED,
  C_ACCEPTS_LOGGED,
  C_ACCEPTS_DROPPED,
  C_REPLIES_HANDLED,
  C_REPLIES_IGNORED,
  C_PREEMPTED,
  C_COORD_RESIGNED,
  C_DECISIONS_MADE,
  C_DECISIONS_HANDLED,
  C_DECISIONS_DROPPED,
  C_PLACEHOLDERS,
  C_EXECUTED,
  C_STOPS_EXECUTED,
  C_CKPTS_DUE,
  C_PROPOSALS,
  C_REQS_BATCHED,
  C_REQS_REJECTED,
  C_WINDOW_OVERFLOW,
  C_KERNEL_LAUNCHES,
  /* aggregates of k_round's in-order fast path (folded into the public counters by gpx_get_counters): every lane
   * of a fast team handled + acked + logged one ACCEPT, handled one reply and one DECISION and executed once; every
   * team made one proposal (one request batched) and one decision */
  C_FAST_LANES = 24,
  C_FAST_TEAMS = 25,
  C_FAST_CKPT = 26,
  C_NCTR = 32
};
/* the global counter block is striped: block b adds into stripe b mod GPX_CTR_STRIPES (256 B apart), so the
 * per-block counter flushes of a large grid do not serialise on one L2 line */
#define GPX_CTR_STRIPES 64

struct MsetInfo { /* one sorted member set (PISM.groupMembers :205), 96 B */
  int32_t nodes[GPX_MAX_GROUP_SIZE];
  uint8_t lane_of_idx[GPX_MAX_GROUP_SIZE]; /* local lane hosting member idx, 0xff if remote */
  uint8_t idx_of_lane[GPX_MAX_LANES];      /* member idx served by lane, 0xff if lane not a member */
  uint16_t lane_mask;
  uint8_t R;
  uint8_t ident; /* lane l <-> member idx l for all l < R, R == n_lanes */
  uint32_t pad2;
};

struct DevState {
  uint32_t G, L, W, Rcap;
  int4* acc_row;
  uint32_t* acc_aux;
  int4* acc_win;
  uint8_t* acc_dirty; /* [L][G] journaling mode: 1 once a VALID accepted entry was stored for (lane, gid); while 0 the
                       * in-order path knows the window holds no accept without reading it */
  int4* com_win;
  int4* coord_row;
  int32_t* node_slots;
  int4* prop_win;
  uint32_t* grp_meta;
  int32_t* grp_cpi;
  const MsetInfo* msets;
  uint8_t* ring[GPX_MAX_LANES];
  uint64_t ring_cap;
  /* log position of every lane, {ring head (absolute byte offset), next segment sequence number}, kept TWICE:
   * a launch that logs reads copy `lp` and its block 0 writes copy `lp ^ 1` (the host flips `lp` with every such
   * launch), so nobody needs to know when the other blocks have read -- no ticket, no fence, no trailing kernel */
  unsigned long long* log_pos;   /* [2][GPX_MAX_LANES][2] */
  uint32_t lp;                   /* which copy this launch reads */
  unsigned long long* cur_seg;   /* [L] segment bases of the round in flight (k_round -> k_round_slow) */
  unsigned long long* ctr;       /* [GPX_CTR_STRIPES][C_NCTR] */
  unsigned int* tickets;         /* [8] words 6..7: the grid barrier of k_round_slow (the rest is unused since log_pos) */
  int32_t lane_node[GPX_MAX_LANES];
  int32_t cpi_const;
  int32_t cpi_per_group; /* CPI_NOISE != 0 */
  int32_t gc_majority_executed;
  int32_t log_meta;
  int32_t journaling;
  int32_t batching;
  int32_t max_batch_size;
  int32_t size_est;
  long long max_batch_bytes;
};

__device__ __forceinline__ int jsub(int a, int b) { return (int)((unsigned)a - (unsigned)b); }
/* Ballot.compareTo paxosutil/Ballot.java:60-66 */
__device__ __forceinline__ int bcmp(int an, int ac, int bn, int bc) { return an != bn ? jsub(an, bn) : jsub(ac, bc); }

__device__ __forceinline__ size_t row_idx(const DevState& S, uint32_t l, uint32_t gid) { return (size_t)l * S.G + gid; }
__device__ __forceinline__ size_t win_idx(const DevState& S, uint32_t l, uint32_t w, uint32_t gid) {
  return ((size_t)l * S.W + w) * S.G + gid;
}
__device__ __forceinline__ size_t ns_idx(const DevState& S, uint32_t l, uint32_t r, uint32_t gid) {
  return ((size_t)l * S.Rcap + r) * S.G + gid;
}

/* PISM :456-460: only an ACTIVE acceptor handles packets */
__device__ __forceinline__ bool st_usable(uint32_t aux) {
  uint32_t st = GPX_AUX_STATE(aux);
  return st == GPX_ST_ACTIVE_1 || st == GPX_ST_ACTIVE_2;
}

/* member set, replica count and liveness of one group */
struct GroupCtx {
  uint32_t R;
  const MsetInfo* ms;
  bool live;
};
__device__ __forceinline__ GroupCtx group_ctx(const DevState& S, uint32_t gid) {
  GroupCtx g;
  g.R = 0;
  g.ms = nullptr;
  g.live = false;
  if (gid < S.G) {
    const uint32_t meta = S.grp_meta[gid];
    g.ms = &S.msets[meta & 0xffffu];
    g.R = (meta >> 16) & 0xffu;
    g.live = (meta & GPX_META_LIVE) != 0;
  }
  return g;
}

/* ---- per-group helpers shared by the management kernels (gpx_kernels.cuh) and k_pause_groups (gpx_pause.cuh) ---- */
/* the HotRestoreInfo field set of (gid, lane) (paxosutil/HotRestoreInfo.java:40-58, PISM.tryPause :2004-2025) */
__device__ __forceinline__ void dump_row(const DevState& S, uint32_t lane, uint32_t gid, gpx_row& r) {
  memset(&r, 0, sizeof r);
  r.gid = gid;
  r.lane = lane;
  if (gid < S.G) {
    const uint32_t meta = S.grp_meta[gid];
    const size_t ri = row_idx(S, lane, gid);
    const int4 row = S.acc_row[ri];
    const int4 c = S.coord_row[ri];
    const bool live = (meta & GPX_META_LIVE) != 0;
    r.acc_slot = row.x;
    r.acc_bnum = row.y;
    r.acc_bcoord = row.z;
    r.acc_gc_slot = row.w;
    r.state = live ? (int)GPX_AUX_STATE(S.acc_aux[ri]) : GPX_ST_FREE;
    const bool ex = ((unsigned)c.w & GPX_CF_EXISTS) != 0;
    r.coord_exists = ex;
    r.coord_active = ex && (((unsigned)c.w & GPX_CF_ACTIVE) != 0);
    r.coord_bnum = ex ? c.x : 0;
    r.coord_bcoord = ex ? c.y : 0;
    r.next_proposal_slot = ex ? c.z : 0;
    if (live) {
      const MsetInfo* ms = &S.msets[meta & 0xffffu];
      const uint32_t R = (meta >> 16) & 0xffu;
      r.n_members = (int)R;
      for (uint32_t m = 0; m < R; m++) {
        r.members[m] = ms->nodes[m];
        r.node_slots[m] = ex ? S.node_slots[ns_idx(S, lane, m, gid)] : 0;
      }
    }
  }
}
/* gpx_get_group_flags' byte for (gid, lane), gid < S.G: the sticky group flags | NOT_CAUGHT_UP */
__device__ __forceinline__ uint32_t group_flags(const DevState& S, uint32_t lane, uint32_t gid) {
  const size_t ri = row_idx(S, lane, gid);
  const uint32_t aux = S.acc_aux[ri];
  /* PaxosAcceptor.caughtUp :452-459 / PCS.caughtUp :758 */
  bool busy = GPX_AUX_PRESENT(aux) != 0; /* committedRequests not empty */
  const int4 crow = S.coord_row[ri];
  if (((unsigned)crow.w & GPX_CF_EXISTS) && ((unsigned)crow.w >> 8)) busy = true; /* myProposals not empty */
  if (!S.journaling) { /* acceptedProposals not empty (journaling: accepted pvalues come from the log) */
    const int gc = S.acc_row[ri].w;
    for (uint32_t w = 0; w < S.W; w++) {
      const size_t ai = 2 * win_idx(S, lane, w, gid);
      const int4 a0 = S.acc_win[ai], a1 = S.acc_win[ai + 1];
      if (((unsigned)a1.w & GPX_ENT_VALID) && jsub(a0.x, gc) > 0) busy = true;
    }
  }
  return GPX_AUX_FLAGS(aux) | (busy ? GPX_GF_NOT_CAUGHT_UP_BIT : 0u);
}
/* PaxosManager.kill :2162 / softCrash :2284-2300: no instance behind this gid any more */
__device__ __forceinline__ void free_group(const DevState& S, uint32_t gid) {
  S.grp_meta[gid] = 0;
  for (uint32_t l = 0; l < S.L; l++) {
    const size_t ri = row_idx(S, l, gid);
    S.acc_row[ri] = make_int4(0, -1, -1, -1);
    S.acc_aux[ri] = GPX_ST_FREE;
    S.coord_row[ri] = make_int4(0, 0, 0, 0);
  }
}

__device__ __forceinline__ int4 ldg4(const void* p) { return *reinterpret_cast<const int4*>(p); }
__device__ __forceinline__ void stg4(void* p, int4 v) { *reinterpret_cast<int4*>(p) = v; }
/* streaming (read-once) 128-bit load: records and payloads are consumed exactly once */
__device__ __forceinline__ int4 ld_stream4(const void* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
/* streaming 128-bit store (outputs are read by a later kernel / the host, never by this one) */
__device__ __forceinline__ void st_stream4(void* p, int4 v) {
  asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
}

/* 256-bit (one full 32-byte sector) loads / stores: LDG.E.256 / STG.E.256 on sm_100a.  32-byte records
 * and window entries move in ONE instruction, so every store fills a sector instead of half of one. */
__device__ __forceinline__ void ld256(const void* p, int4& a, int4& b) {
  asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
               : "l"(p)
               : "memory");
}
/* every store of an accepted-window entry goes through here (keeps acc_dirty conservative) */
#define ST_ACC(S, lane, gid, idx, n0, n1)                                                    \
  do {                                                                                       \
    st256(&(S).acc_win[(idx)], (n0), (n1));                                                  \
    if ((S).journaling && ((unsigned)(n1).w & GPX_ENT_VALID)) (S).acc_dirty[(size_t)(lane) * (S).G + (gid)] = 1; \
  } while (0)

/* ---- TMA bulk copy (cp.async.bulk, SASS UBLKCP) of a contiguous record tile into shared memory, completion
 * signalled on an mbarrier: one elected thread arms the barrier with the byte count and issues the copy, every
 * thread waits on the phase.  Addresses and size are multiples of 16. ---- */
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, unsigned long long* bar) {
  const uint32_t b = (uint32_t)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(b)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  const uint32_t b = (uint32_t)__cvta_generic_to_shared(bar);
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(b), "r"(parity)
        : "memory");
  }
}

__device__ __forceinline__ void ld256_stream(const void* p, int4& a, int4& b) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
               : "l"(p));
}
__device__ __forceinline__ void st256(void* p, const int4 a, const int4 b) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w),
               "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}
__device__ __forceinline__ void st256_stream(void* p, const int4 a, const int4 b) {
  asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(a.x), "r"(a.y),
               "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}

/* up to 16 bytes from an arbitrarily aligned address, zero-padded to one 128-bit chunk */
__device__ __forceinline__ int4 load_chunk16(const uint8_t* src, uint32_t nbytes) {
  uint32_t w[4] = {0u, 0u, 0u, 0u};
  if (nbytes >= 16u && (((uintptr_t)src) & 3u) == 0) {
    const uint32_t* s4 = reinterpret_cast<const uint32_t*>(src);
    w[0] = s4[0];
    w[1] = s4[1];
    w[2] = s4[2];
    w[3] = s4[3];
  } else {
#pragma unroll
    for (int k = 0; k < 16; k++)
      if ((uint32_t)k < nbytes) w[k >> 2] |= (uint32_t)src[k] << (8 * (k & 3));
  }
  return make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]);
}

/* a pvalue in registers */
struct DPValue {
  int slot, bnum, bcoord, median_cp;
  long long req_id;
  unsigned frame_ref, plen, fl; /* fl: GPX_ENT_STOP | nreq<<16 */
  bool valued;
};

/* segment base of this launch for one lane: skip to the ring start if it would wrap */
__device__ __forceinline__ unsigned long long seg_base(const DevState& S, uint32_t l, unsigned long long reserved) {
  unsigned long long head = S.log_pos[((size_t)S.lp * GPX_MAX_LANES + l) * 2];
  unsigned long long pos = head & (S.ring_cap - 1);
  if (pos + reserved > S.ring_cap) head += S.ring_cap - pos;
  return head;
}
__device__ __forceinline__ unsigned long long seg_seq_of(const DevState& S, uint32_t l) {
  return S.log_pos[((size_t)S.lp * GPX_MAX_LANES + l) * 2 + 1];
}
/* block 0 of a logging launch: where the NEXT launch starts (written into the other copy) */
__device__ __forceinline__ void log_publish(const DevState& S, uint32_t l, unsigned long long new_head,
                                            unsigned long long new_seq) {
  unsigned long long* q = &S.log_pos[((size_t)(S.lp ^ 1u) * GPX_MAX_LANES + l) * 2];
  q[0] = new_head;
  q[1] = new_seq;
}
__device__ __forceinline__ uint8_t* ring_ptr(const DevState& S, uint32_t l, unsigned long long abs_off) {
  return S.ring[l] + (abs_off & (S.ring_cap - 1));
}

/* PaxosCoordinatorState.getMedianMinus :867-875 over node_slots[lane][0..R)[gid] */
__device__ __forceinline__ int median_minus(const DevState& S, uint32_t lane, uint32_t gid, uint32_t R) {
  if (R == 3) {
    int a = S.node_slots[ns_idx(S, lane, 0, gid)], b = S.node_slots[ns_idx(S, lane, 1, gid)],
        c = S.node_slots[ns_idx(S, lane, 2, gid)];
    return max(min(a, b), min(max(a, b), c));
  }
  int v[GPX_MAX_GROUP_SIZE];
  for (uint32_t k = 0; k < R; k++) v[k] = S.node_slots[ns_idx(S, lane, k, gid)];
  for (uint32_t k = 1; k < R; k++) { /* insertion sort, R <= 16 */
    int x = v[k];
    int m = (int)k - 1;
    while (m >= 0 && v[m] > x) {
      v[m + 1] = v[m];
      m--;
    }
    v[m + 1] = x;
  }
  return v[(R % 2 == 0) ? R / 2 - 1 : R / 2];
}

/* PCS.getMedianMinus :867-875 on a register array (R <= LP <= 8) */
template <int LP>
__device__ __forceinline__ int median_regs(const int (&ns)[LP], uint32_t R) {
  if (R == 1) return ns[0];
  if (LP >= 3 && R == 3) return max(min(ns[0], ns[1]), min(max(ns[0], ns[1]), ns[2]));
  int v[LP];
#pragma unroll
  for (int k = 0; k < LP; k++) v[k] = (uint32_t)k < R ? ns[k] : 2147483647;
#pragma unroll
  for (int a = 0; a < LP; a++) /* odd-even transposition sort, fully unrolled: no dynamic indexing */
#pragma unroll
    for (int b = (a & 1); b + 1 < LP; b += 2) {
      int lo = min(v[b], v[b + 1]), hi = max(v[b], v[b + 1]);
      v[b] = lo;
      v[b + 1] = hi;
    }
  const uint32_t idx = (R % 2 == 0) ? R / 2 - 1 : R / 2;
  int out = v[0];
#pragma unroll
  for (int k = 1; k < LP; k++)
    if ((uint32_t)k == idx) out = v[k];
  return out;
}

/* PaxosAcceptor.garbageCollectAccepted :476-494.  Entries <= gc die implicitly (an
 * accepted entry is alive iff valid && slot - gc > 0); garbageCollectDecisions :496-506
 * is a no-op here because committed entries only ever live in [_slot, _slot + W). */
__device__ __forceinline__ void gc_step(int4& row, int gcSlot) {
  if (jsub(row.x, gcSlot) <= 0) gcSlot = row.x - 1;
  if (jsub(gcSlot, row.w) > 0) row.w = gcSlot;
}

__device__ __forceinline__ gpx_exec_rec make_exec(const DevState& S, uint32_t gid, uint32_t lane, const DPValue& x,
                                                  bool extra) {
  int cpi = S.cpi_per_group ? S.grp_cpi[gid] : S.cpi_const;
  bool stop = (x.fl & GPX_ENT_STOP) != 0;
  bool ckpt = (x.slot % cpi == 0) || stop; /* PISM.shouldCheckpoint :2037-2041 */
  gpx_exec_rec r;
  r.gid = gid;
  r.slot = x.slot;
  r.req_id = x.req_id;
  r.payload_off = x.frame_ref;
  r.flags = (stop ? GPX_F_STOP : 0u) | (ckpt ? GPX_F_CKPT : 0u) | (extra ? GPX_F_EXTRA : 0u) | (lane << 12) |
            (x.fl & 0xffff0000u);
  return r;
}

__device__ __forceinline__ void store_exec(gpx_exec_rec* dst, const gpx_exec_rec& r) {
  /* 24 B = 3 x 8 B */
  const long long* s = reinterpret_cast<const long long*>(&r);
  long long* d = reinterpret_cast<long long*>(dst);
  d[0] = s[0];
  d[1] = s[1];
  d[2] = s[2];
}

/*
 * PISM.extractExecuteAndCheckpoint :1619-1701 around PaxosAcceptor.putAndRemoveNextExecutable
 * :325-366 / reconstructDecision :369-385 / executed :462-474, on register-resident row/aux.
 * The first execution goes to *primary (if non-null), further ones to the extra queue.
 * `acc_hint` may carry the already loaded accepted entry of d.slot (q0,q1) to skip a reload.
 */
__device__ __noinline__ void eec_impl(const DevState& S, uint32_t lane, uint32_t gid, int4& row, uint32_t& aux,
                                      const DPValue& d, gpx_exec_rec* primary, gpx_exec_rec* extra,
                                      uint32_t extra_cap, uint32_t* n_extra, unsigned int* s_ctr, bool all_extra) {
  const uint32_t Wm = S.W - 1;
  bool first = true;
  while (true) {
    if (GPX_AUX_STATE(aux) == GPX_ST_STOPPED) break;
    gc_step(row, d.median_cp); /* :340 */
    bool direct = false; /* d is next-in-line and valued: execute it without a com_win round trip */
    if (jsub(d.slot, row.x) >= 0) { /* :343 put decision unless a valued one is present */
      uint32_t w = (uint32_t)d.slot & Wm;
      bool present = (GPX_AUX_PRESENT(aux) >> w) & 1u, valued = (GPX_AUX_VALUED(aux) >> w) & 1u;
      if (!present || !valued) {
        if (d.slot == row.x && d.valued) {
          direct = true;
          aux |= (1u << (8 + w)) | (1u << (16 + w));
        } else {
          size_t ci = 2 * win_idx(S, lane, w, gid);
          S.com_win[ci] = make_int4(d.bnum, d.bcoord, d.median_cp, (int)d.frame_ref);
          S.com_win[ci + 1] = make_int4((int)(unsigned)(d.req_id & 0xffffffffll), (int)(d.req_id >> 32), (int)d.plen,
                                        (int)d.fl);
          aux |= (1u << (8 + w));
          if (d.valued)
            aux |= (1u << (16 + w));
          else
            aux &= ~(1u << (16 + w));
        }
      }
    }
    uint32_t w0 = (uint32_t)row.x & Wm;
    bool have = false;
    DPValue nx;
    if (direct) {
      nx = d;
      nx.fl = d.fl & ~GPX_ENT_VALID;
      have = true;
    } else if ((GPX_AUX_PRESENT(aux) >> w0) & 1u) { /* :352 */
      size_t ci = 2 * win_idx(S, lane, w0, gid);
      int4 c0 = S.com_win[ci], c1 = S.com_win[ci + 1];
      if ((GPX_AUX_VALUED(aux) >> w0) & 1u) {
        nx.slot = row.x;
        nx.bnum = c0.x;
        nx.bcoord = c0.y;
        nx.median_cp = c0.z;
        nx.frame_ref = (unsigned)c0.w;
        nx.req_id = ((long long)c1.y << 32) | (unsigned)c1.x;
        nx.plen = (unsigned)c1.z;
        nx.fl = (unsigned)c1.w;
        nx.valued = true;
        have = true;
      } else { /* reconstruct from the accept with an equal ballot :373-383 */
        size_t ai = 2 * win_idx(S, lane, w0, gid);
        int4 a0 = S.acc_win[ai], a1 = S.acc_win[ai + 1];
        bool alive = ((unsigned)a1.w & GPX_ENT_VALID) && jsub(a0.x, row.w) > 0 && a0.x == row.x;
        if (alive && a0.y == c0.x && a0.z == c0.y) {
          nx.slot = row.x;
          nx.bnum = a0.y;
          nx.bcoord = a0.z;
          nx.median_cp = c0.z;
          nx.frame_ref = (unsigned)a0.w;
          nx.req_id = ((long long)a1.y << 32) | (unsigned)a1.x;
          nx.plen = (unsigned)a1.z;
          nx.fl = (unsigned)a1.w & ~GPX_ENT_VALID;
          nx.valued = true;
          have = true;
        }
      }
    }
    {
      if (have) {
        aux &= ~((1u << (8 + w0)) | (1u << (16 + w0))); /* committedRequests.remove(slot) */
        row.x = (int)((unsigned)row.x + 1u);            /* executed(): _slot++ */
        if (nx.fl & GPX_ENT_STOP) {
          aux = (aux & ~0xffu) | GPX_ST_STOPPED; /* stop() */
          aux &= ~0x00ffff00u;                   /* committedRequests.clear() */
        }
        if (S.journaling) { /* acceptedProposals.remove(slot) :360-362 */
          size_t ai = 2 * win_idx(S, lane, w0, gid);
          int4 a0 = S.acc_win[ai];
          int4 a1 = S.acc_win[ai + 1];
          if (((unsigned)a1.w & GPX_ENT_VALID) && a0.x == nx.slot) {
            a1.w = (int)((unsigned)a1.w & ~GPX_ENT_VALID);
            S.acc_win[ai + 1] = a1;
          }
        }
      }
    }
    if (!have) break;
    atomicAdd(&s_ctr[C_EXECUTED], 1u);
    gpx_exec_rec er = make_exec(S, gid, lane, nx, all_extra || !first);
    if (er.flags & GPX_F_CKPT) atomicAdd(&s_ctr[C_CKPTS_DUE], 1u);
    if (first && !all_extra && primary) {
      store_exec(primary, er);
    } else if (n_extra) {
      uint32_t k = atomicAdd(n_extra, 1u);
      if (k < extra_cap) store_exec(extra + k, er);
    }
    first = false;
    if (nx.fl & GPX_ENT_STOP) {
      atomicAdd(&s_ctr[C_STOPS_EXECUTED], 1u);
      break;
    }
  }
}

/* call wrapper: only temporaries have their address taken, so the caller's row/aux stay in registers */
__device__ __forceinline__ void eec(const DevState& S, uint32_t lane, uint32_t gid, int4& row, uint32_t& aux,
                                    const DPValue& d, gpx_exec_rec* primary, gpx_exec_rec* extra, uint32_t extra_cap,
                                    uint32_t* n_extra, unsigned int* s_ctr, bool all_extra) {
  int4 r = row;
  uint32_t a = aux;
  DPValue dd = d;
  eec_impl(S, lane, gid, r, a, dd, primary, extra, extra_cap, n_extra, s_ctr, all_extra);
  row = r;
  aux = a;
}
