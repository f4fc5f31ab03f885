/*
 * gpx_kernels.cuh -- the four hot-path kernels (sm_100a) and the state-maintenance kernels.
 *
 *   k_propose  RequestBatcher.dequeueImpl (RequestBatcher.java:168-234) + PISM.handleProposal
 *              (:818-888) + PaxosCoordinatorState.propose (:233-263)
 *   k_accept   PISM.handleAccept (:1080-1166) incl. PaxosAcceptor.acceptAndUpdateBallot (:302-322),
 *              the toLog rule (:1146-1149) and the log append (AbstractPaxosLogger.logAndMessage :157)
 *   k_tally    PISM.handleBatchedAcceptReply (:1370) / PaxosCoordinator.handleAcceptReply (:210-250)
 *   k_commit   PISM.handleBatchedCommit (:1480-1528) / handleCommittedRequest (:1432-1478) /
 *              extractExecuteAndCheckpoint (:1619-1701)
 *
 *   k_act      accept -> tally -> commit fused per ACCEPT for co-located replicas: the reference's
 *              loopback path (PaxosManager.sendOrLoopback :2116-2128) with every inter-replica
 *              record kept in registers instead of HBM
 *
 * Work mapping: one thread per record; records of one group are adjacent in every stream
 * ("grouped by gid"), and the thread of the first record of a run processes the whole run
 * in order, which reproduces the per-instance `synchronized` of the reference
 * (PaxosAcceptor.java:302,325; PaxosCoordinator.java:210).  Different groups never share
 * state, so runs are independent.  Kernels are templated on the number of lanes so the
 * per-lane state of a record lives in registers and all of its independent loads
 * (L x {aux, row, window entry}) are issued before the first use.  32-byte records and window
 * entries move with ONE 256-bit LDG/STG (a full sector per thread per instruction), rows with
 * 128-bit ones.  Fixed-position outputs (reply i*L+lane, log image i, exec i*L+lane) need no
 * atomics; variable outputs (ACCEPTs, DECISIONs) are compacted with one atomic per block.
 */
#pragma once
#include "gpx_dev.cuh"

#define GPX_BLOCK 256
#ifndef GPX_ACT_MINB
#define GPX_ACT_MINB 2 /* resident CTAs per SM the fused kernel is compiled for (register cap = 64K/(256*MINB)) */
#endif
#ifndef GPX_PHASE_MINB
#define GPX_PHASE_MINB 3
#endif

struct RoundCtl { /* device-resident per-round counters */
  uint32_t n_accepts;
  uint32_t n_decisions;
  uint32_t n_extra;
  uint32_t any_batched;
  unsigned long long blob1_used;
  uint32_t n_todo;
  uint32_t pad[1];
};

/* every thread of the block calls; returns the first index reserved for this thread */
__device__ __forceinline__ uint32_t block_reserve(uint32_t cnt, uint32_t* counter, uint32_t* s_scan /*[GPX_BLOCK/32+1]*/) {
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= (uint32_t)d) incl += t;
  }
  if (lane == 31) s_scan[wid] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t tot = 0;
    for (uint32_t w = 0; w < GPX_BLOCK / 32; w++) {
      uint32_t v = s_scan[w];
      s_scan[w] = tot;
      tot += v;
    }
    uint32_t base = tot ? atomicAdd(counter, tot) : 0u;
    s_scan[GPX_BLOCK / 32] = base;
  }
  __syncthreads();
  uint32_t r = s_scan[GPX_BLOCK / 32] + s_scan[wid] + incl - cnt;
  __syncthreads();
  return r;
}

__device__ __forceinline__ void flush_counters(const DevState& S, unsigned int* s_ctr) {
  __syncthreads();
  if (threadIdx.x < C_NCTR) {
    unsigned int v = s_ctr[threadIdx.x];
    if (v) atomicAdd(&S.ctr[(blockIdx.x & (GPX_CTR_STRIPES - 1)) * C_NCTR + threadIdx.x], (unsigned long long)v);
  }
}

__device__ __forceinline__ bool usable(const DevState& S, uint32_t gid, uint32_t lane, uint32_t* aux_out) {
  uint32_t aux = S.acc_aux[row_idx(S, lane, gid)];
  *aux_out = aux;
  return st_usable(aux);
}

/* ============================== k_propose ===================================== */
struct ProposeArgs {
  const gpx_request_rec* reqs;
  uint32_t n;
  unsigned long long payload_bytes_al; /* request payload arena size, 16-B aligned */
  gpx_accept_rec* accepts;
  int32_t* status;
  uint32_t* copy_tab;
  uint32_t* copy_dst;
  RoundCtl* ctl;
};

__device__ __forceinline__ uint32_t batch_end(const DevState& S, const gpx_request_rec* reqs, uint32_t n, uint32_t k,
                                              uint32_t gid) {
  long long bytes = (long long)reqs[k].payload_len + S.size_est;
  int cnt = 1;
  uint32_t b = k + 1;
  if (S.batching)
    while (b < n && reqs[b].gid == gid) {
      bytes += (long long)reqs[b].payload_len + S.size_est;
      if (bytes > S.max_batch_bytes) break;
      cnt += 1;
      if (cnt > S.max_batch_size) break;
      b++;
    }
  return b;
}

/* `indexed`: the ACCEPT of the batch that starts at request k is written to A.accepts[k] (k_round) instead of
 * the compacted position base+emitted (k_propose) */
__device__ __noinline__ void propose_run(const DevState& S, const ProposeArgs& A, uint32_t i, uint32_t run_end,
                                         uint32_t nb, uint32_t base, unsigned int* s_ctr, bool indexed = false) {
  const gpx_request_rec* reqs = A.reqs;
  const uint32_t gid = reqs[i].gid;
  const uint32_t Wm = S.W - 1;
  uint32_t emitted = 0;
  int code = 0;
  uint32_t k = i;
  int clane = -1;
  const MsetInfo* ms = nullptr;
  uint32_t R = 0;
  do {
    uint32_t entry = (reqs[i].flags >> 8) & 0xfu;
    if (gid >= S.G || entry >= S.L) {
      code = GPX_RS_DROPPED;
      break;
    }
    uint32_t meta = S.grp_meta[gid];
    uint32_t aux;
    if (!(meta & GPX_META_LIVE) || !usable(S, gid, entry, &aux)) {
      code = GPX_RS_DROPPED;
      break;
    }
    ms = &S.msets[meta & 0xffffu];
    R = (meta >> 16) & 0xffu;
    int4 Ae = S.acc_row[row_idx(S, entry, gid)];
    int4 Ce = S.coord_row[row_idx(S, entry, gid)];
    if (((unsigned)Ce.w & GPX_CF_EXISTS) && bcmp(Ce.x, Ce.y, Ae.y, Ae.z) >= 0) { /* PaxosCoordinator.exists(c, ballot) */
      clane = (int)entry;
    } else {
      int fl = -1;
      for (uint32_t l = 0; l < S.L; l++)
        if (S.lane_node[l] == Ae.z) fl = (int)l;
      if (fl < 0) {
        code = GPX_RS_FORWARD;
        break;
      }
      if (fl == (int)entry) {
        code = GPX_RS_NOCOORD;
        break;
      }
      if (!usable(S, gid, (uint32_t)fl, &aux)) {
        code = GPX_RS_DROPPED;
        break;
      }
      int4 Af = S.acc_row[row_idx(S, fl, gid)];
      int4 Cf = S.coord_row[row_idx(S, fl, gid)];
      if (((unsigned)Cf.w & GPX_CF_EXISTS) && bcmp(Cf.x, Cf.y, Af.y, Af.z) >= 0)
        clane = fl;
      else {
        code = GPX_RS_NOCOORD;
        break;
      }
    }
  } while (false);

  if (code == 0) {
    int4 crow = S.coord_row[row_idx(S, clane, gid)];
    bool dirty = false;
    while (k < run_end) {
      uint32_t b = batch_end(S, reqs, A.n, k, gid);
      if (b > run_end) b = run_end;
      uint32_t nreq = b - k;
      const uint32_t w = (uint32_t)crow.z & Wm;
      if (((unsigned)crow.w >> 8) != 0) { /* proposals outstanding: only then can the window refuse */
        /* PCS.propose :235-239 refuse after a STOP that is still outstanding */
        int prev = (int)((unsigned)crow.z - 1u);
        int4 pe = S.prop_win[win_idx(S, clane, (uint32_t)prev & Wm, gid)];
        if (((unsigned)pe.y & GPX_PV_PRESENT) && pe.x == prev && ((unsigned)pe.y & GPX_PV_STOP)) {
          code = GPX_RS_REFUSED_STOP;
          break;
        }
        int4 pw = S.prop_win[win_idx(S, clane, w, gid)];
        if ((unsigned)pw.y & GPX_PV_PRESENT) { /* window full: W proposals in flight */
          code = GPX_RS_BACKPRESSURE;
          break;
        }
      }
      bool stop = false;
      for (uint32_t q = k; q < b; q++) stop = stop || (reqs[q].flags & GPX_F_STOP);
      int slot = crow.z;
      crow.z = (int)((unsigned)crow.z + 1u);
      crow.w = (int)((unsigned)crow.w + (1u << 8));
      dirty = true;
      long long rid = reqs[k].req_id;
      S.prop_win[win_idx(S, clane, w, gid)] =
          make_int4(slot, (int)(GPX_PV_PRESENT | (stop ? GPX_PV_STOP : 0u)), (int)(unsigned)(rid & 0xffffffffll),
                    (int)(rid >> 32));
      if (!((unsigned)crow.w & GPX_CF_ACTIVE)) { /* pre-active: queued, no ACCEPT yet :254-261 */
        for (uint32_t q = k; q < b; q++) A.status[q] = GPX_RS_PREACTIVE;
        k = b;
        continue;
      }
      int median = median_minus(S, (uint32_t)clane, gid, R);
      uint32_t off, plen;
      if (nreq == 1) {
        off = reqs[k].payload_off; /* zero copy: the blob is the request's own payload */
        plen = reqs[k].payload_len;
      } else {
        unsigned long long total = 16ull * nreq;
        for (uint32_t q = k; q < b; q++) total += reqs[q].payload_len;
        unsigned long long o1 = atomicAdd(&A.ctl->blob1_used, (total + 15ull) & ~15ull);
        off = (uint32_t)(A.payload_bytes_al + o1);
        plen = (uint32_t)total;
        unsigned long long run = 0;
        for (uint32_t q = k; q < b; q++) {
          A.copy_tab[q] = off + 16u * (q - k);
          A.copy_dst[q] = (uint32_t)(off + 16ull * nreq + run);
          run += reqs[q].payload_len;
        }
        A.ctl->any_batched = 1u;
      }
      gpx_accept_rec a;
      a.h.gid = gid;
      a.h.slot = slot;
      a.h.bnum = crow.x;
      a.h.bcoord = crow.y;
      a.h.median_cp = median;
      a.h.flags = (uint16_t)(GPX_F_ACCEPT | (stop ? GPX_F_STOP : 0u));
      a.h.dst_mask = ms->lane_mask;
      a.h.req_id = rid;
      a.payload_off = off;
      a.payload_len = plen;
      a.nreq = nreq;
      a.sender = crow.y;
      int4* dst = reinterpret_cast<int4*>(&A.accepts[indexed ? k : base + emitted]);
      const int4* src = reinterpret_cast<const int4*>(&a);
      dst[0] = src[0];
      dst[1] = src[1];
      dst[2] = src[2];
      emitted++;
      A.status[k] = slot;
      for (uint32_t q = k + 1; q < b; q++) A.status[q] = GPX_RS_BATCHED;
      atomicAdd(&s_ctr[C_PROPOSALS], 1u);
      atomicAdd(&s_ctr[C_REQS_BATCHED], nreq);
      k = b;
    }
    if (dirty) S.coord_row[row_idx(S, clane, gid)] = crow;
  }
  if (code != 0) {
    for (uint32_t q = k; q < run_end; q++) A.status[q] = code;
    atomicAdd(&s_ctr[C_REQS_REJECTED], run_end - k);
  }
  for (; !indexed && emitted < nb; emitted++) { /* reserved but unused: VOID keeps the run adjacent */
    gpx_accept_rec a;
    memset(&a, 0, sizeof a);
    a.h.gid = gid;
    a.h.flags = GPX_F_VOID;
    int4* dst = reinterpret_cast<int4*>(&A.accepts[base + emitted]);
    const int4* src = reinterpret_cast<const int4*>(&a);
    dst[0] = src[0];
    dst[1] = src[1];
    dst[2] = src[2];
  }
}

__global__ void __launch_bounds__(GPX_BLOCK) k_propose(const __grid_constant__ DevState S,
                                                       const __grid_constant__ ProposeArgs A) {
  __shared__ unsigned int s_ctr[C_NCTR];
  __shared__ uint32_t s_scan[GPX_BLOCK / 32 + 1];
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  bool head = false;
  uint32_t nb = 0, run_end = i + 1;
  if (i < A.n) {
    uint32_t gid = A.reqs[i].gid;
    head = (i == 0) || (A.reqs[i - 1].gid != gid);
    if (head) {
      if (i + 1 < A.n && A.reqs[i + 1].gid == gid) {
        uint32_t k = i;
        while (k < A.n && A.reqs[k].gid == gid) {
          k = batch_end(S, A.reqs, A.n, k, gid);
          nb++;
        }
        run_end = k;
      } else
        nb = 1;
    }
  }
  /* the plain case -- ONE request of the group in the batch, entering at the coordinator's own lane: everything the
   * proposal needs hangs off the request record, so it is fetched in one level, before (and overlapping) the block's
   * reservation of ACCEPT slots; validated afterwards, and anything else takes propose_run */
  gpx_request_rec rq;
  uint32_t meta = 0, aux = 0;
  int4 Ae = make_int4(0, 0, 0, 0), Ce = Ae;
  int ns[8];
  bool spec = false;
  size_t ri = 0;
  if (head && nb == 1 && run_end == i + 1) {
    rq = A.reqs[i];
    const uint32_t entry = (rq.flags >> 8) & 0xfu;
    /* (single-lane engines -- the nodes of a spread group -- only: with several lanes the coordinator is usually NOT the
     * entry lane, the guess would be wrong for most requests and the loads wasted: measured 127 -> 304 us at 1 M groups) */
    spec = S.L == 1u && rq.gid < S.G && entry < S.L;
    if (spec) {
      ri = row_idx(S, entry, rq.gid);
      meta = S.grp_meta[rq.gid];
      aux = S.acc_aux[ri];
      Ae = S.acc_row[ri];
      Ce = S.coord_row[ri];
#pragma unroll
      for (int m = 0; m < 8; m++) ns[m] = (uint32_t)m < S.Rcap ? S.node_slots[ns_idx(S, entry, (uint32_t)m, rq.gid)] : 0;
    }
  }
  uint32_t base = block_reserve(head ? nb : 0u, &A.ctl->n_accepts, s_scan);
  if (head) {
    const uint32_t R = (meta >> 16) & 0xffu;
    const bool fast = spec && (meta & GPX_META_LIVE) && st_usable(aux) && R <= 8u &&
                      ((unsigned)Ce.w & 0xffu) == (GPX_CF_EXISTS | GPX_CF_ACTIVE) && ((unsigned)Ce.w >> 8) == 0u &&
                      bcmp(Ce.x, Ce.y, Ae.y, Ae.z) >= 0; /* PaxosCoordinator.exists(c, ballot), active, nothing in flight */
    if (fast) { /* PCS.propose :233-263 + initCommander: exactly what propose_run does for this case */
      const uint32_t entry = (rq.flags >> 8) & 0xfu;
      const bool stop = (rq.flags & GPX_F_STOP) != 0;
      const int slot = Ce.z;
      Ce.z = (int)((unsigned)Ce.z + 1u);
      Ce.w = (int)((unsigned)Ce.w + (1u << 8));
      S.prop_win[win_idx(S, entry, (uint32_t)slot & (S.W - 1), rq.gid)] =
          make_int4(slot, (int)(GPX_PV_PRESENT | (stop ? GPX_PV_STOP : 0u)), (int)(unsigned)(rq.req_id & 0xffffffffll),
                    (int)(rq.req_id >> 32));
#pragma unroll
      for (int m = 0; m < 8; m++)
        if ((uint32_t)m >= R) ns[m] = 2147483647;
      gpx_accept_rec a;
      a.h.gid = rq.gid;
      a.h.slot = slot;
      a.h.bnum = Ce.x;
      a.h.bcoord = Ce.y;
      a.h.median_cp = median_regs<8>(ns, R);
      a.h.flags = (uint16_t)(GPX_F_ACCEPT | (stop ? GPX_F_STOP : 0u));
      a.h.dst_mask = S.msets[meta & 0xffffu].lane_mask;
      a.h.req_id = rq.req_id;
      a.payload_off = rq.payload_off;
      a.payload_len = rq.payload_len;
      a.nreq = 1;
      a.sender = Ce.y;
      int4* dst = reinterpret_cast<int4*>(&A.accepts[base]);
      const int4* src = reinterpret_cast<const int4*>(&a);
      dst[0] = src[0];
      dst[1] = src[1];
      dst[2] = src[2];
      A.status[i] = slot;
      S.coord_row[ri] = Ce;
      atomicAdd(&s_ctr[C_PROPOSALS], 1u);
      atomicAdd(&s_ctr[C_REQS_BATCHED], 1u);
    } else
      propose_run(S, A, i, run_end, nb, base, s_ctr);
  }
  if (i == 0) atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  flush_counters(S, s_ctr);
}

/* builds the blobs of batched slots: [nreq x gpx_batch_ent][payloads], one thread per request */
__global__ void __launch_bounds__(GPX_BLOCK) k_build_blobs(const __grid_constant__ ProposeArgs A,
                                                           const uint8_t* payload, uint8_t* blob1) {
  if (!A.ctl->any_batched) return;
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  if (i >= A.n) return;
  int st = A.status[i];
  bool batched = (st == GPX_RS_BATCHED) ||
                 (st > 0 && i + 1 < A.n && A.status[i + 1] == GPX_RS_BATCHED && A.reqs[i + 1].gid == A.reqs[i].gid);
  if (!batched) return;
  gpx_request_rec r = A.reqs[i];
  gpx_batch_ent be;
  be.req_id = r.req_id;
  be.len = r.payload_len;
  be.flags = r.flags;
  *reinterpret_cast<int4*>(blob1 + (A.copy_tab[i] - A.payload_bytes_al)) = *reinterpret_cast<const int4*>(&be);
  uint8_t* d = blob1 + (A.copy_dst[i] - A.payload_bytes_al);
  const uint8_t* s = payload + r.payload_off;
  for (uint32_t b = 0; b < r.payload_len; b++) d[b] = s[b];
}

/* ============================== shared per-lane steps ============================== */
struct AcceptArgs {
  const gpx_accept_rec* recs;
  const uint32_t* n_ptr; /* device count, or null */
  uint32_t n_max;        /* record slots reserved (grid covers these) */
  const uint8_t* blob0;  /* payload arena: offsets [0, blob0_bytes) */
  unsigned long long blob0_bytes;
  const uint8_t* blob1; /* constructed blobs: offsets [blob0_bytes, blob0_bytes+blob1_bytes) */
  unsigned long long blob1_bytes;
  const unsigned long long* blob1_used_ptr; /* device: bytes of blob1 actually used (overrides blob1_bytes) */
  gpx_accept_reply_rec* replies;            /* [n_max][L] */
  gpx_decision_rec* decisions;              /* k_act: [n_max], fixed position */
  uint8_t* out_mask;                        /* k_act: [n_max] lanes whose reply was NOT consumed locally (written) */
  gpx_exec_rec* exec;                       /* k_act: [n_max][L] */
  gpx_exec_rec* extra;
  uint32_t extra_cap;
  uint32_t* n_extra;
};

__device__ __forceinline__ const uint8_t* blob_ptr(const AcceptArgs& A, unsigned long long off) {
  return off < A.blob0_bytes ? A.blob0 + off : A.blob1 + (off - A.blob0_bytes);
}

/* per-lane state of one record, kept in registers across accept -> tally -> commit */
#define LS_HANDLED 1u   /* the acceptor processed the ACCEPT (row/aux may have changed) */
#define LS_STORE 2u     /* the accepted window entry still has to be written */
#define LS_LOGGED 4u    /* toLog: image + blob go to the log ring */
#define LS_RARE 8u      /* reconstructDecision path ran: window memory was touched */
#define LS_OCCVALID 16u /* the ring position held an entry with its valid bit set */
#define LS_ROWDIRTY 32u
#define LS_AUXDIRTY 64u
struct LaneSt {
  int4 row;
  uint32_t aux;
  int rbn, rbc, rmaxcp; /* ACCEPT_REPLY: acceptor ballot after the accept, maxCheckpointedSlot */
  uint32_t rwho;
  uint32_t frame_ref;
  uint32_t fl;
  uint32_t img_flags; /* flags | dst_mask<<16 of the ACCEPT log image */
};

__device__ __forceinline__ void make_entry(const int4 q0, const int4 q1, const int4 q2, uint32_t frame_ref, int4& n0,
                                           int4& n1) {
  const uint32_t rflags = (uint32_t)q1.y & 0xffffu;
  n0 = make_int4(q0.y, q0.z, q0.w, (int)frame_ref);
  n1 = make_int4(q1.z, q1.w, q2.y,
                 (int)(GPX_ENT_VALID | ((rflags & GPX_F_STOP) ? GPX_ENT_STOP : 0u) | ((uint32_t)q2.z << 16)));
}

/* PISM.handleAccept :1080-1166 for one ACCEPT at one lane, on register-resident state.  (e0,e1) is the
 * window entry at slot mod W as loaded.  The caller writes row/aux/entry back; if a commit had overtaken
 * this ACCEPT the reconstructDecision path runs here (rare) after the entry has been stored. */
__device__ __forceinline__ void accept_lane(const DevState& S, const AcceptArgs& A, uint32_t l, bool live,
                                            const MsetInfo* ms, uint32_t dstIdx, const int4 q0, const int4 q1,
                                            const int4 q2, const int4 e0, const int4 e1, unsigned frame_ref_new,
                                            LaneSt& st, unsigned int* s_ctr) {
  const uint32_t gid = (uint32_t)q0.x;
  const int slot = q0.y, bnum = q0.z, bcoord = q0.w, median_cp = q1.x;
  const uint32_t rflags = (uint32_t)q1.y & 0xffffu, dst_mask = (uint32_t)q1.y >> 16;
  const uint32_t Wm = S.W - 1;
  st.rbn = 0;
  st.rbc = 0;
  st.rmaxcp = 0;
  st.rwho = GPX_WHO(0xffu, 0xffu, GPX_F_VOID);
  st.img_flags = GPX_F_VOID | (dst_mask << 16);
  st.frame_ref = frame_ref_new;
  st.fl = ((unsigned)e1.w & GPX_ENT_VALID) ? LS_OCCVALID : 0u;
  if (!((dst_mask >> l) & 1u) || (rflags & GPX_F_VOID)) return;
  if (!live || !st_usable(st.aux)) { /* PISM :456-460 */
    atomicAdd(&s_ctr[C_ACCEPTS_DROPPED], 1u);
    return;
  }
  const uint32_t myIdx = ms->idx_of_lane[l];
  if (myIdx == 0xffu) {
    atomicAdd(&s_ctr[C_ACCEPTS_DROPPED], 1u);
    return;
  }
  int4& row = st.row;
  if (jsub(slot, row.x) >= (int)S.W) { /* beyond the in-flight window: drop + flag for the host */
    st.aux |= (GPX_GF_OVERFLOW << 24);
    st.fl |= LS_AUXDIRTY;
    atomicAdd(&s_ctr[C_WINDOW_OVERFLOW], 1u);
    atomicAdd(&s_ctr[C_ACCEPTS_DROPPED], 1u);
    return;
  }
  st.fl |= LS_HANDLED;
  atomicAdd(&s_ctr[C_ACCEPTS_HANDLED], 1u);
  const int4 row_in = row;
  /* prev = paxosState.getAccept(slot) :1123 */
  const bool ent_alive = ((unsigned)e1.w & GPX_ENT_VALID) && jsub(e0.x, row.w) > 0;
  const bool hasPrev = ent_alive && e0.x == slot;
  if (hasPrev && e0.y == bnum && e0.z == bcoord) st.frame_ref = (unsigned)e0.w; /* duplicate keeps its frame */
  /* acceptAndUpdateBallot :302-322 */
  bool store = false;
  if (bcmp(bnum, bcoord, row.y, row.z) >= 0) {
    row.y = bnum;
    row.z = bcoord;
    if (jsub(slot, row.w) > 0) {
      store = true;
      if (ent_alive && e0.x != slot) { /* ring conflict: never evict a live entry for a stale accept */
        bool staleNew = jsub(slot, row.x) < 0, occStale = jsub(e0.x, row.x) < 0;
        if (staleNew && !occStale) store = false;
      }
    }
  }
  gc_step(row, median_cp); /* :320 */
  /* AcceptReplyPacket :1139-1143 */
  int max_cp = row.x - 1;
  if (!S.gc_majority_executed) {
    int cpi = S.cpi_per_group ? S.grp_cpi[gid] : S.cpi_const;
    int s1 = row.x - 1;
    int lcp = s1 - s1 % cpi;
    if (lcp < 0) {
      lcp = jsub(lcp, cpi);
      if (lcp > 0) lcp = 2147483647 - 2147483647 % cpi;
    }
    max_cp = lcp;
  }
  /* toLog :1146-1149 */
  const bool toLog = bcmp(bnum, bcoord, row.y, row.z) >= 0 && jsub(slot, row.w) > 0 &&
                     (!hasPrev || bcmp(e0.y, e0.z, bnum, bcoord) < 0);
  const bool nack = bcmp(row.y, row.z, bnum, bcoord) > 0;
  st.rbn = row.y;
  st.rbc = row.z;
  st.rmaxcp = max_cp;
  st.rwho = GPX_WHO(myIdx, dstIdx, (toLog ? GPX_F_LOGGED : 0u) | (nack ? GPX_F_NACK : 0u));
  atomicAdd(&s_ctr[nack ? C_ACCEPTS_NACKED : C_ACCEPTS_ACKED], 1u);
  if (toLog) {
    atomicAdd(&s_ctr[C_ACCEPTS_LOGGED], 1u);
    st.fl |= LS_LOGGED;
    st.img_flags = rflags | ((1u << l) << 16);
  }
  if (store) st.fl |= LS_STORE;
  /* reconstructDecision(slot) -> handleCommittedRequest :1158-1161 (rare: a commit overtook its accept) */
  const int dslot = jsub(slot, row.x);
  if (dslot >= 0 && dslot < (int)S.W && ((GPX_AUX_PRESENT(st.aux) >> ((uint32_t)slot & Wm)) & 1u)) {
    const uint32_t w = (uint32_t)slot & Wm;
    const size_t ai = 2 * win_idx(S, l, w, gid);
    st.fl |= LS_RARE;
    if (store) { /* the entry must be visible to the commit path */
      int4 n0, n1;
      make_entry(q0, q1, q2, st.frame_ref, n0, n1);
      ST_ACC(S, l, gid, ai, n0, n1);
      st.fl &= ~LS_STORE;
    }
    int4 c0, c1;
    ld256(&S.com_win[ai], c0, c1);
    DPValue d;
    bool ok = false;
    if ((GPX_AUX_VALUED(st.aux) >> w) & 1u) {
      d.slot = slot;
      d.bnum = c0.x;
      d.bcoord = c0.y;
      d.median_cp = c0.z;
      d.frame_ref = (unsigned)c0.w;
      d.req_id = ((long long)c1.y << 32) | (unsigned)c1.x;
      d.plen = (unsigned)c1.z;
      d.fl = (unsigned)c1.w;
      d.valued = true;
      ok = true;
    } else {
      int4 n0, n1;
      ld256(&S.acc_win[ai], n0, n1);
      const bool alive = ((unsigned)n1.w & GPX_ENT_VALID) && jsub(n0.x, row.w) > 0 && n0.x == slot;
      if (alive && n0.y == c0.x && n0.z == c0.y) {
        d.slot = slot;
        d.bnum = n0.y;
        d.bcoord = n0.z;
        d.median_cp = c0.z;
        d.frame_ref = (unsigned)n0.w;
        d.req_id = ((long long)n1.y << 32) | (unsigned)n1.x;
        d.plen = (unsigned)n1.z;
        d.fl = (unsigned)n1.w;
        d.valued = true;
        ok = true;
      }
    }
    const uint32_t aux_b = st.aux;
    if (ok) eec(S, l, gid, row, st.aux, d, nullptr, A.extra, A.extra_cap, A.n_extra, s_ctr, true);
    if (st.aux != aux_b) st.fl |= LS_AUXDIRTY;
  }
  if (row.x != row_in.x || row.y != row_in.y || row.z != row_in.z || row.w != row_in.w) st.fl |= LS_ROWDIRTY;
}

/* PISM.handleAcceptReply :1248-1365 for one reply at the coordinator lane `cl` (row cached in `crow`) */
__device__ __forceinline__ bool tally_reply(const DevState& S, uint32_t cl, uint32_t gid, uint32_t R,
                                            const MsetInfo* ms, int4& crow, bool& dirty, int slot, int rb, int rc,
                                            int max_cp, uint32_t accIdx, gpx_decision_rec& d, unsigned int* s_ctr) {
  const uint32_t Wm = S.W - 1;
  bool decided = false;
  atomicAdd(&s_ctr[C_REPLIES_HANDLED], 1u);
  const uint32_t cf = (unsigned)crow.w & 0xffu;
  if ((cf & GPX_CF_EXISTS) && (cf & GPX_CF_ACTIVE)) { /* PaxosCoordinator.handleAcceptReply :212 */
    const int c = bcmp(rb, rc, crow.x, crow.y);
    const size_t pi = win_idx(S, cl, (uint32_t)slot & Wm, gid);
    if (c > 0) { /* handleAcceptReplyHigherBallot :661-675 */
      int4 pe = S.prop_win[pi];
      if (((unsigned)pe.y & GPX_PV_PRESENT) && pe.x == slot) {
        pe.y = (int)((unsigned)pe.y & ~GPX_PV_PRESENT);
        S.prop_win[pi] = pe;
        crow.w = (int)((unsigned)crow.w - (1u << 8));
        dirty = true;
        atomicAdd(&s_ctr[C_PREEMPTED], 1u);
      }
    } else if (c == 0) { /* handleAcceptReplyMyBallot :597-640 */
      if (accIdx < R) {  /* recordSlotNumber :809-825 (plain <) */
        const size_t ni = ns_idx(S, cl, accIdx, gid);
        if (S.node_slots[ni] < max_cp) S.node_slots[ni] = max_cp;
      }
      int4 pe = S.prop_win[pi];
      if (((unsigned)pe.y & GPX_PV_PRESENT) && pe.x == slot) {
        uint32_t vf = (unsigned)pe.y;
        if (accIdx < R) vf |= (1u << accIdx);      /* WaitforUtility.updateHeardFrom :51-62 */
        if (__popc(vf & 0xffffu) > (int)(R / 2)) { /* heardFromMajority :64-68 */
          d.gid = gid;
          d.slot = slot;
          d.bnum = crow.x;
          d.bcoord = crow.y;
          d.median_cp = median_minus(S, cl, gid, R); /* makeDecision(getMajorityCommittedSlot()) :630 */
          d.flags = (uint16_t)(GPX_F_DECISION | ((vf & GPX_PV_STOP) ? GPX_F_STOP : 0u));
          d.dst_mask = ms->lane_mask;
          d.req_id = ((long long)pe.w << 32) | (unsigned)pe.z;
          decided = true;
          pe.y = (int)(vf & ~GPX_PV_PRESENT);
          crow.w = (int)((unsigned)crow.w - (1u << 8));
          dirty = true;
          atomicAdd(&s_ctr[C_DECISIONS_MADE], 1u);
        } else
          pe.y = (int)vf;
        S.prop_win[pi] = pe;
      }
    }
  }
  /* nullifyCoordinatorIfPreemptedFully :1353-1356 */
  if ((((unsigned)crow.w) & GPX_CF_EXISTS) && bcmp(rb, rc, crow.x, crow.y) > 0 && (((unsigned)crow.w) >> 8) == 0) {
    crow = make_int4(0, 0, 0, 0);
    dirty = true;
    atomicAdd(&s_ctr[C_COORD_RESIGNED], 1u);
  }
  return decided;
}

template <int NR>
__device__ __forceinline__ bool tally_slot_core(const DevState& S, uint32_t cl, uint32_t gid, uint32_t R,
                                                const MsetInfo* ms, int4& crow, bool& dirty, int slot,
                                                const int4 (&r0)[NR], const int4 (&r1)[NR], uint32_t nrep, const int4 pe0,
                                                const int (&ns0)[8], gpx_decision_rec& d, unsigned int* s_ctr);

/* The replies to ONE ACCEPT (one slot) at the coordinator lane `cl`, with the coordinator row, the slot's proposal
 * entry and nodeSlotNumbers held in registers: what tally_reply does reply by reply against memory -- same order, same
 * effects -- with one load and at most one store per touched word (the R replies of a slot arrive together in the
 * batched exchange, PaxosPacketBatcher.java:270-303 / BatchedAcceptReply).  r0[k] = {gid, slot, bnum, bcoord},
 * r1[k] = {maxCheckpointedSlot, who, ...}; VOID replies are skipped.  R <= 8. */
template <int NR>
__device__ __forceinline__ bool tally_slot_regs(const DevState& S, uint32_t cl, uint32_t gid, uint32_t R,
                                                const MsetInfo* ms, int4& crow, bool& dirty, int slot,
                                                const int4 (&r0)[NR], const int4 (&r1)[NR], uint32_t nrep,
                                                gpx_decision_rec& d, unsigned int* s_ctr) {
  const uint32_t Wm = S.W - 1;
  const size_t pi = win_idx(S, cl, (uint32_t)slot & Wm, gid);
  const int4 pe0 = S.prop_win[pi];
  int ns0[8];
#pragma unroll
  for (int m = 0; m < 8; m++) ns0[m] = (uint32_t)m < R ? S.node_slots[ns_idx(S, cl, (uint32_t)m, gid)] : 2147483647;
  return tally_slot_core<NR>(S, cl, gid, R, ms, crow, dirty, slot, r0, r1, nrep, pe0, ns0, d, s_ctr);
}

/* the same with the proposal entry and nodeSlotNumbers already loaded (ns0[m] for m >= R is ignored) */
template <int NR>
__device__ __forceinline__ bool tally_slot_core(const DevState& S, uint32_t cl, uint32_t gid, uint32_t R,
                                                const MsetInfo* ms, int4& crow, bool& dirty, int slot,
                                                const int4 (&r0)[NR], const int4 (&r1)[NR], uint32_t nrep, const int4 pe0,
                                                const int (&ns0)[8], gpx_decision_rec& d, unsigned int* s_ctr) {
  const uint32_t Wm = S.W - 1;
  const size_t pi = win_idx(S, cl, (uint32_t)slot & Wm, gid);
  int4 pe = pe0;
  const int4 pe_in = pe;
  int ns[8], ns_in[8];
#pragma unroll
  for (int m = 0; m < 8; m++) {
    ns[m] = (uint32_t)m < R ? ns0[m] : 2147483647;
    ns_in[m] = ns[m];
  }
  bool decided = false;
  uint32_t handled = 0;
#pragma unroll
  for (int k = 0; k < NR; k++) {
    if ((uint32_t)k >= nrep) continue;
    const uint32_t who = (uint32_t)r1[k].y;
    if (GPX_WHO_FLAGS(who) & GPX_F_VOID) continue;
    handled++;
    const int rb = r0[k].z, rc = r0[k].w, max_cp = r1[k].x;
    const uint32_t accIdx = GPX_WHO_ACC(who);
    const uint32_t cf = (unsigned)crow.w & 0xffu;
    if ((cf & GPX_CF_EXISTS) && (cf & GPX_CF_ACTIVE)) { /* PaxosCoordinator.handleAcceptReply :212 */
      const int c = bcmp(rb, rc, crow.x, crow.y);
      if (c > 0) { /* handleAcceptReplyHigherBallot :661-675 */
        if (((unsigned)pe.y & GPX_PV_PRESENT) && pe.x == slot) {
          pe.y = (int)((unsigned)pe.y & ~GPX_PV_PRESENT);
          crow.w = (int)((unsigned)crow.w - (1u << 8));
          dirty = true;
          atomicAdd(&s_ctr[C_PREEMPTED], 1u);
        }
      } else if (c == 0) { /* handleAcceptReplyMyBallot :597-640 */
#pragma unroll
        for (int m = 0; m < 8; m++) /* recordSlotNumber :809-825 (plain <) */
          if ((uint32_t)m == accIdx && accIdx < R && ns[m] < max_cp) ns[m] = max_cp;
        if (((unsigned)pe.y & GPX_PV_PRESENT) && pe.x == slot) {
          uint32_t vf = (unsigned)pe.y;
          if (accIdx < R) vf |= (1u << accIdx);      /* WaitforUtility.updateHeardFrom :51-62 */
          if (__popc(vf & 0xffffu) > (int)(R / 2)) { /* heardFromMajority :64-68 */
            d.gid = gid;
            d.slot = slot;
            d.bnum = crow.x;
            d.bcoord = crow.y;
            d.median_cp = median_regs<8>(ns, R); /* makeDecision(getMajorityCommittedSlot()) :630 */
            d.flags = (uint16_t)(GPX_F_DECISION | ((vf & GPX_PV_STOP) ? GPX_F_STOP : 0u));
            d.dst_mask = ms->lane_mask;
            d.req_id = ((long long)pe.w << 32) | (unsigned)pe.z;
            decided = true;
            pe.y = (int)(vf & ~GPX_PV_PRESENT);
            crow.w = (int)((unsigned)crow.w - (1u << 8));
            dirty = true;
            atomicAdd(&s_ctr[C_DECISIONS_MADE], 1u);
          } else
            pe.y = (int)vf;
        }
      }
    }
    /* nullifyCoordinatorIfPreemptedFully :1353-1356 */
    if ((((unsigned)crow.w) & GPX_CF_EXISTS) && bcmp(rb, rc, crow.x, crow.y) > 0 && (((unsigned)crow.w) >> 8) == 0) {
      crow = make_int4(0, 0, 0, 0);
      dirty = true;
      atomicAdd(&s_ctr[C_COORD_RESIGNED], 1u);
    }
  }
  if (handled) atomicAdd(&s_ctr[C_REPLIES_HANDLED], handled);
  if (pe.y != pe_in.y) S.prop_win[pi] = pe;
#pragma unroll
  for (int m = 0; m < 8; m++)
    if ((uint32_t)m < R && ns[m] != ns_in[m]) S.node_slots[ns_idx(S, cl, (uint32_t)m, gid)] = ns[m];
  return decided;
}

/* PISM.handleBatchedCommit :1480-1528 (one slot) at one lane on register-resident row/aux; (a0,a1) is the
 * accepted window entry at slot mod W as currently in memory.  Produces the log image. */
__device__ __forceinline__ void commit_lane(const DevState& S, uint32_t l, uint32_t gid, int slot, int bnum,
                                            int bcoord, int median_cp, int4& row, uint32_t& aux, const int4 a0,
                                            const int4 a1, gpx_exec_rec* ex, gpx_exec_rec* extra, uint32_t extra_cap,
                                            uint32_t* n_extra, int4& img0, int4& img1, unsigned int* s_ctr) {
  if (jsub(slot, row.x) >= (int)S.W) {
    aux |= ((GPX_GF_OVERFLOW | GPX_GF_NEEDS_SYNC) << 24);
    atomicAdd(&s_ctr[C_WINDOW_OVERFLOW], 1u);
    atomicAdd(&s_ctr[C_DECISIONS_DROPPED], 1u);
    return;
  }
  atomicAdd(&s_ctr[C_DECISIONS_HANDLED], 1u);
  const bool a_alive = ((unsigned)a1.w & GPX_ENT_VALID) && jsub(a0.x, row.w) > 0 && a0.x == slot;
  DPValue d;
  d.slot = slot;
  d.bnum = bnum;
  d.bcoord = bcoord;
  d.median_cp = median_cp;
  if (a_alive && a0.y == bnum && a0.z == bcoord) { /* :1488 decision := the accept we hold */
    d.req_id = ((long long)a1.y << 32) | (unsigned)a1.x;
    d.frame_ref = (unsigned)a0.w;
    d.plen = (unsigned)a1.z;
    d.fl = (unsigned)a1.w & ~GPX_ENT_VALID;
    d.valued = true;
  } else { /* placeholder :1514-1522 */
    d.req_id = 0;
    d.frame_ref = 0;
    d.plen = 0;
    d.fl = 0;
    d.valued = false;
    atomicAdd(&s_ctr[C_PLACEHOLDERS], 1u);
  }
  /* logDecision :1446-1466 */
  if (d.valued || S.log_meta) {
    const bool meta = S.log_meta && a_alive && bcmp(a0.y, a0.z, d.bnum, d.bcoord) >= 0;
    const uint32_t lf = GPX_F_DECISION | (meta ? GPX_F_META : 0u) | ((d.fl & GPX_ENT_STOP) ? GPX_F_STOP : 0u);
    img0 = make_int4((int)gid, slot, d.bnum, d.bcoord);
    img1 = make_int4(meta ? -1 : d.median_cp, (int)(lf | ((1u << l) << 16)), (int)(unsigned)(d.req_id & 0xffffffffll),
                     (int)(d.req_id >> 32));
  }
  if (d.valued && slot == row.x && GPX_AUX_PRESENT(aux) == 0u) {
    /* the common case, in line: the decision is the accept we hold, it is next in line and nothing else is queued --
     * extractExecuteAndCheckpoint :1619-1701 runs exactly one execution (what eec_impl does in two loop iterations:
     * GC, execute, advance, drop the accept from memory when journaling, GC again) without the call and its frame */
    gc_step(row, d.median_cp);
    row.x = (int)((unsigned)row.x + 1u); /* executed(): _slot++ */
    const bool stop = (d.fl & GPX_ENT_STOP) != 0;
    if (stop) {
      aux = (aux & ~0xffu) | GPX_ST_STOPPED; /* stop() + committedRequests.clear() */
      aux &= ~0x00ffff00u;
    }
    if (S.journaling) { /* acceptedProposals.remove(slot) :360-362 */
      const size_t ai = 2 * win_idx(S, l, (uint32_t)slot & (S.W - 1), gid);
      S.acc_win[ai + 1] = make_int4(a1.x, a1.y, a1.z, (int)((unsigned)a1.w & ~GPX_ENT_VALID));
    }
    atomicAdd(&s_ctr[C_EXECUTED], 1u);
    const gpx_exec_rec er = make_exec(S, gid, l, d, false);
    if (er.flags & GPX_F_CKPT) atomicAdd(&s_ctr[C_CKPTS_DUE], 1u);
    if (ex) {
      store_exec(ex, er);
    } else if (n_extra) {
      const uint32_t k = atomicAdd(n_extra, 1u);
      if (k < extra_cap) store_exec(extra + k, er);
    }
    if (stop)
      atomicAdd(&s_ctr[C_STOPS_EXECUTED], 1u);
    else
      gc_step(row, d.median_cp);
    return;
  }
  const int slot_before = row.x;
  eec(S, l, gid, row, aux, d, ex, extra, extra_cap, n_extra, s_ctr, false);
  if (GPX_AUX_STATE(aux) != GPX_ST_STOPPED && !d.valued && jsub(slot, row.x) >= 0 && row.x == slot_before)
    aux |= (GPX_GF_NEEDS_SYNC << 24);
}

__device__ __forceinline__ void write_seg_hdr(const DevState& S, uint32_t l, unsigned long long base, uint16_t type,
                                              uint32_t n_slots, uint32_t n_valid, unsigned long long pay_bytes,
                                              uint32_t rec_bytes, unsigned long long seq) {
  gpx_log_seg_hdr h;
  memset(&h, 0, sizeof h);
  h.magic = GPX_SEG_MAGIC;
  h.type = type;
  h.lane = (uint16_t)l;
  h.n_slots = n_slots;
  h.n_valid = n_valid;
  h.payload_bytes = pay_bytes;
  h.seq = seq;
  h.ring_off = base;
  h.rec_bytes = rec_bytes;
  int4* hp = reinterpret_cast<int4*>(ring_ptr(S, l, base));
  const int4* sp = reinterpret_cast<const int4*>(&h);
  hp[0] = sp[0];
  hp[1] = sp[1];
  hp[2] = sp[2];
  hp[3] = sp[3];
}

/* copy one blob into the payload area of every logging lane (read once, written up to L times) */
template <int L>
__device__ __forceinline__ void copy_blob(const DevState& S, const AcceptArgs& A, uint32_t off, uint32_t plen,
                                          uint32_t logmask, const unsigned long long* payb) {
  const uint8_t* src = blob_ptr(A, off);
  if (((off | (uint32_t)(uintptr_t)src) & 15u) == 0) {
    for (uint32_t b = 0; b < plen; b += 16) {
      int4 v = ld_stream4(src + b);
#pragma unroll
      for (int l = 0; l < L; l++)
        if ((logmask >> l) & 1u) st_stream4(ring_ptr(S, l, payb[l] + off + b), v);
    }
  } else {
    for (uint32_t b = 0; b < plen; b++) {
      uint8_t v = src[b];
#pragma unroll
      for (int l = 0; l < L; l++)
        if ((logmask >> l) & 1u) *ring_ptr(S, l, payb[l] + off + b) = v;
    }
  }
}

/* ACCEPT segment: [64 B hdr][n x 32 B pvalue-header plane][n x 16 B extension plane][payload area];
 * the two planes let every image move as one 256-bit plus one 128-bit aligned store */
__device__ __forceinline__ void write_accept_image(const DevState& S, uint32_t l, unsigned long long segb,
                                                   uint32_t n_max, uint32_t j, const int4 q0, const int4 q1,
                                                   const int4 q2, uint32_t img_flags) {
  st256_stream(ring_ptr(S, l, segb + 64 + (unsigned long long)j * 32), q0, make_int4(q1.x, (int)img_flags, q1.z, q1.w));
  st_stream4(ring_ptr(S, l, segb + 64 + (unsigned long long)n_max * 32 + (unsigned long long)j * 16), q2);
}

__device__ __forceinline__ void store_void_exec(gpx_exec_rec* ex, uint32_t gid, int slot, uint32_t l) {
  gpx_exec_rec vx;
  vx.gid = gid;
  vx.slot = slot;
  vx.req_id = 0;
  vx.payload_off = 0;
  vx.flags = GPX_F_VOID | (l << 12);
  store_exec(ex, vx);
}

/* ============================== k_accept ====================================== */
template <int L>
__global__ void __launch_bounds__(GPX_BLOCK, GPX_PHASE_MINB) k_accept(const __grid_constant__ DevState S,
                                                      const __grid_constant__ AcceptArgs A) {
  __shared__ unsigned int s_ctr[C_NCTR];
  /* the block's tile of the incoming ACCEPT batch (its 256 records + the predecessor for the run-head test) is
   * staged in shared memory by ONE TMA bulk copy, overlapped with the segment bookkeeping below */
  __shared__ __align__(128) uint8_t s_tile[(GPX_BLOCK + 1) * sizeof(gpx_accept_rec)];
  __shared__ __align__(8) unsigned long long s_bar;
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  if (threadIdx.x == 0) mbar_init(&s_bar, 1);
  __syncthreads();
  uint32_t n = A.n_ptr ? *A.n_ptr : A.n_max;
  if (n > A.n_max) n = A.n_max;
  const uint32_t i0 = blockIdx.x * GPX_BLOCK, i = i0 + threadIdx.x;
  const uint32_t t0 = i0 ? i0 - 1u : 0u, t1 = min(n, i0 + GPX_BLOCK); /* records [t0, t1) are staged */
  const uint32_t tile_bytes = t1 > t0 ? (t1 - t0) * (uint32_t)sizeof(gpx_accept_rec) : 0u;
  if (threadIdx.x == 0 && tile_bytes) tma_load_1d(s_tile, &A.recs[t0], tile_bytes, &s_bar);
  const uint32_t Wm = S.W - 1;
  const unsigned long long pay_bytes = A.blob0_bytes + (A.blob1_used_ptr ? *A.blob1_used_ptr : A.blob1_bytes);
  const unsigned long long pay_rel = seg_pay_rel(A.n_max);
  const unsigned long long reserved = seg_align32(pay_rel + pay_bytes); /* = seg_accept_bytes(A.n_max, pay_bytes) */
  unsigned long long segb[L], payb[L];
#pragma unroll
  for (int l = 0; l < L; l++) {
    segb[l] = seg_base(S, l, reserved);
    payb[l] = segb[l] + pay_rel;
  }
  if (i == 0) {
#pragma unroll
    for (int l = 0; l < L; l++) {
      const unsigned long long sq = seg_seq_of(S, l);
      write_seg_hdr(S, l, segb[l], GPX_F_ACCEPT, A.n_max, n, pay_bytes, 48, sq);
      log_publish(S, l, segb[l] + reserved, sq + 1ull);
    }
    atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  }
  if (tile_bytes) mbar_wait(&s_bar, 0);
  if (i < n) {
    const int4* rp = reinterpret_cast<const int4*>(s_tile + (size_t)(i - t0) * sizeof(gpx_accept_rec));
    int4 q0 = rp[0], q1 = rp[1], q2 = rp[2];
    const uint32_t gid = (uint32_t)q0.x;
    const bool head = (i == 0) || ((uint32_t)rp[-3].x != gid);
    if (head) {
      const GroupCtx g = group_ctx(S, gid);
      uint32_t j = i;
      while (true) {
        const int slot = q0.y;
        const uint32_t payload_off = (uint32_t)q2.x;
        LaneSt st[L];
        int4 e0[L], e1[L];
#pragma unroll
        for (int l = 0; l < L; l++) { /* all independent loads first */
          st[l].aux = 0;
          st[l].row = make_int4(0, 0, 0, 0);
          e0[l] = e1[l] = make_int4(0, 0, 0, 0);
          if (g.live) {
            const size_t ri = row_idx(S, l, gid);
            st[l].aux = S.acc_aux[ri];
            st[l].row = S.acc_row[ri];
            ld256(&S.acc_win[2 * win_idx(S, l, (uint32_t)slot & Wm, gid)], e0[l], e1[l]);
          }
        }
        uint32_t dstIdx = 0xffu;
        if (g.live)
          for (uint32_t m = 0; m < g.R; m++)
            if (g.ms->nodes[m] == q2.w) dstIdx = m;
        uint32_t logmask = 0;
#pragma unroll
        for (int l = 0; l < L; l++) {
          const unsigned fr = (unsigned)(((payb[l] + payload_off) & (S.ring_cap - 1)) >> 4);
          accept_lane(S, A, l, g.live, g.ms, dstIdx, q0, q1, q2, e0[l], e1[l], fr, st[l], s_ctr);
          const size_t ri = row_idx(S, l, gid);
          if (st[l].fl & LS_STORE) {
            int4 n0, n1;
            make_entry(q0, q1, q2, st[l].frame_ref, n0, n1);
            ST_ACC(S, l, gid, 2 * win_idx(S, l, (uint32_t)slot & Wm, gid), n0, n1);
          }
          if (st[l].fl & LS_ROWDIRTY) S.acc_row[ri] = st[l].row;
          if (st[l].fl & LS_AUXDIRTY) S.acc_aux[ri] = st[l].aux;
          if (st[l].fl & LS_LOGGED) logmask |= 1u << l;
          st256_stream(&A.replies[(size_t)j * L + l], make_int4((int)gid, slot, st[l].rbn, st[l].rbc),
                       (GPX_WHO_FLAGS(st[l].rwho) & GPX_F_VOID) ? make_int4(0, (int)st[l].rwho, 0, 0)
                                                                : make_int4(st[l].rmaxcp, (int)st[l].rwho, q1.z, q1.w));
          write_accept_image(S, l, segb[l], A.n_max, j, q0, q1, q2, st[l].img_flags);
        }
        if (logmask) copy_blob<L>(S, A, payload_off, (uint32_t)q2.y, logmask, payb);
        j++;
        if (j >= n) break;
        /* the run continues in the staged tile, or -- across the block boundary -- in global memory */
        rp = j < t1 ? reinterpret_cast<const int4*>(s_tile + (size_t)(j - t0) * sizeof(gpx_accept_rec))
                    : reinterpret_cast<const int4*>(&A.recs[j]);
        const int4 nx = rp[0];
        if ((uint32_t)nx.x != gid) break;
        q0 = nx;
        q1 = rp[1];
        q2 = rp[2];
      }
    }
  }
  flush_counters(S, s_ctr);
}

/* ============================== k_tally ======================================= */
struct TallyArgs {
  const gpx_accept_reply_rec* replies;
  const uint32_t* n_ptr; /* device count of ACCEPTs (replies = n * mult), or null */
  uint32_t mult;
  uint32_t n_max; /* reply slots covered by the grid */
  gpx_decision_rec* decisions;
  uint32_t* n_decisions;
};

__global__ void __launch_bounds__(GPX_BLOCK) k_tally(const __grid_constant__ DevState S,
                                                     const __grid_constant__ TallyArgs A) {
  __shared__ unsigned int s_ctr[C_NCTR];
  __shared__ uint32_t s_scan[GPX_BLOCK / 32 + 1];
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  __syncthreads();
  uint32_t n = A.n_ptr ? (*A.n_ptr) * A.mult : A.n_max;
  if (n > A.n_max) n = A.n_max;
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  gpx_decision_rec dbuf[GPX_MAX_WINDOW];
  uint32_t nd = 0;
  if (i == 0) atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  if (i < n) {
    int4 q0, q1;
    ld256_stream(&A.replies[i], q0, q1);
    const uint32_t gid = (uint32_t)q0.x;
    const bool head = (i == 0) || (A.replies[i - 1].gid != gid);
    if (head) {
      int cl = -1;
      int4 crow = make_int4(0, 0, 0, 0);
      bool dirty = false;
      const GroupCtx g = group_ctx(S, gid);
      uint32_t j = i;
      while (true) {
        const uint32_t who = (uint32_t)q1.y;
        if (!(GPX_WHO_FLAGS(who) & GPX_F_VOID)) {
          const uint32_t dstIdx = GPX_WHO_DST(who);
          int lane = -1;
          uint32_t aux;
          if (g.live && dstIdx < g.R && g.ms->lane_of_idx[dstIdx] != 0xffu &&
              usable(S, gid, g.ms->lane_of_idx[dstIdx], &aux))
            lane = g.ms->lane_of_idx[dstIdx];
          if (lane < 0) {
            atomicAdd(&s_ctr[C_REPLIES_IGNORED], 1u);
          } else {
            if (lane != cl) {
              if (dirty) S.coord_row[row_idx(S, cl, gid)] = crow;
              cl = lane;
              crow = S.coord_row[row_idx(S, cl, gid)];
              dirty = false;
            }
            gpx_decision_rec d;
            if (tally_reply(S, (uint32_t)cl, gid, g.R, g.ms, crow, dirty, q0.y, q0.z, q0.w, q1.x, GPX_WHO_ACC(who), d,
                            s_ctr)) {
              if (nd < GPX_MAX_WINDOW) dbuf[nd] = d;
              nd++;
            }
          }
        }
        j++;
        if (j >= n) break;
        int4 t0, t1;
        ld256_stream(&A.replies[j], t0, t1);
        if ((uint32_t)t0.x != gid) break;
        q0 = t0;
        q1 = t1;
      }
      if (dirty) S.coord_row[row_idx(S, cl, gid)] = crow;
    }
  }
  if (nd > GPX_MAX_WINDOW) nd = GPX_MAX_WINDOW; /* cannot happen: <= W proposals outstanding */
  uint32_t base = block_reserve(nd, A.n_decisions, s_scan);
  for (uint32_t k = 0; k < nd; k++) {
    const int4* sp = reinterpret_cast<const int4*>(&dbuf[k]);
    st256_stream(&A.decisions[base + k], sp[0], sp[1]);
  }
  flush_counters(S, s_ctr);
}

/* k_tally_slots<L>: the replies of the phase pipeline lie as [ACCEPT j][lane l] (index j * L + l): one thread per
 * ACCEPT takes the L replies of its slot at once and tallies them in registers (tally_slot_regs); the thread of the
 * first ACCEPT of a group's run walks the run.  Replies addressed to different coordinator lanes inside one slot, or
 * groups of more than 8 members, take the reply-by-reply path. */
template <int L>
__global__ void __launch_bounds__(GPX_BLOCK) k_tally_slots(const __grid_constant__ DevState S,
                                                           const __grid_constant__ TallyArgs A) {
  __shared__ unsigned int s_ctr[C_NCTR];
  __shared__ uint32_t s_scan[GPX_BLOCK / 32 + 1];
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  __syncthreads();
  uint32_t n = A.n_ptr ? *A.n_ptr : A.n_max / (uint32_t)L; /* ACCEPTs */
  if (n > A.n_max / (uint32_t)L) n = A.n_max / (uint32_t)L;
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  gpx_decision_rec dbuf[GPX_MAX_WINDOW];
  uint32_t nd = 0;
  if (i == 0) atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  if (i < n) {
    const gpx_accept_reply_rec* rp = &A.replies[(size_t)i * L];
    int4 r0[L], r1[L];
#pragma unroll
    for (int l = 0; l < L; l++) ld256_stream(&rp[l], r0[l], r1[l]);
    const uint32_t gid = (uint32_t)r0[0].x;
    const uint32_t gprev = i ? A.replies[(size_t)(i - 1) * L].gid : 0xffffffffu;
    const uint32_t gnext = i + 1 < n ? A.replies[(size_t)(i + 1) * L].gid : 0xffffffffu;
    const bool head = (i == 0) || (gprev != gid);
    /* ---- the plain case in two load levels: ONE ACCEPT of the group in the batch, every reply addressed to the
     * same coordinator, and member index == lane (GPX_META_IDENT) so that the lane follows from the reply alone: the
     * group's meta word, the coordinator's aux / row, the slot's proposal entry and nodeSlotNumbers are all fetched
     * together, validated, and the slot is tallied in registers ---- */
    bool done = false;
    if (head && gnext != gid && gid < S.G) {
      uint32_t dst = 0xffu, nvalid = 0;
      bool same = true;
#pragma unroll
      for (int l = 0; l < L; l++) {
        const uint32_t who = (uint32_t)r1[l].y;
        if (GPX_WHO_FLAGS(who) & GPX_F_VOID) continue;
        if (nvalid++ == 0)
          dst = GPX_WHO_DST(who);
        else
          same = same && GPX_WHO_DST(who) == dst;
      }
      if (nvalid && same && dst < (uint32_t)L) {
        const int slot = r0[0].y;
        const uint32_t meta = S.grp_meta[gid];
        const size_t ri = row_idx(S, dst, gid);
        const uint32_t aux = S.acc_aux[ri];
        int4 crow = S.coord_row[ri];
        const int4 pe0 = S.prop_win[win_idx(S, dst, (uint32_t)slot & (S.W - 1), gid)];
        int ns0[8];
#pragma unroll
        for (int m = 0; m < 8; m++) ns0[m] = (uint32_t)m < S.Rcap ? S.node_slots[ns_idx(S, dst, (uint32_t)m, gid)] : 0;
        const uint32_t R = (meta >> 16) & 0xffu;
        if ((meta & (GPX_META_LIVE | GPX_META_IDENT)) == (GPX_META_LIVE | GPX_META_IDENT) && R <= 8u && st_usable(aux)) {
          bool dirty = false;
          gpx_decision_rec d;
          if (tally_slot_core<L>(S, dst, gid, R, &S.msets[meta & 0xffffu], crow, dirty, slot, r0, r1, (uint32_t)L, pe0, ns0,
                                 d, s_ctr)) {
            dbuf[0] = d;
            nd = 1;
          }
          if (dirty) S.coord_row[ri] = crow;
          done = true;
        }
      }
    }
    if (head && !done) {
      const GroupCtx g = group_ctx(S, gid);
      int cl = -1;
      int4 crow = make_int4(0, 0, 0, 0);
      bool dirty = false;
      uint32_t j = i;
      while (true) {
        /* the coordinator lane the slot's replies are addressed to (PISM drop rule :456-460: it must be usable) */
        int lane = -1;
        bool uniform = g.live && g.R <= 8u;
        uint32_t nvalid = 0;
#pragma unroll
        for (int l = 0; l < L; l++) {
          const uint32_t who = (uint32_t)r1[l].y;
          if (GPX_WHO_FLAGS(who) & GPX_F_VOID) continue;
          nvalid++;
          const uint32_t dstIdx = GPX_WHO_DST(who);
          const int ln = (g.live && dstIdx < g.R && g.ms->lane_of_idx[dstIdx] != 0xffu) ? (int)g.ms->lane_of_idx[dstIdx] : -1;
          if (lane == -1 && nvalid == 1)
            lane = ln;
          else if (ln != lane)
            uniform = false;
        }
        uint32_t aux;
        if (nvalid && uniform && lane >= 0 && usable(S, gid, (uint32_t)lane, &aux)) {
          if (lane != cl) {
            if (dirty) S.coord_row[row_idx(S, cl, gid)] = crow;
            cl = lane;
            crow = S.coord_row[row_idx(S, cl, gid)];
            dirty = false;
          }
          gpx_decision_rec d;
          if (tally_slot_regs<L>(S, (uint32_t)cl, gid, g.R, g.ms, crow, dirty, r0[0].y, r0, r1, (uint32_t)L, d, s_ctr)) {
            if (nd < GPX_MAX_WINDOW) dbuf[nd] = d;
            nd++;
          }
        } else if (nvalid) { /* reply by reply, against memory */
#pragma unroll
          for (int l = 0; l < L; l++) {
            const uint32_t who = (uint32_t)r1[l].y;
            if (GPX_WHO_FLAGS(who) & GPX_F_VOID) continue;
            const uint32_t dstIdx = GPX_WHO_DST(who);
            int ln = -1;
            if (g.live && dstIdx < g.R && g.ms->lane_of_idx[dstIdx] != 0xffu && usable(S, gid, g.ms->lane_of_idx[dstIdx], &aux))
              ln = g.ms->lane_of_idx[dstIdx];
            if (ln < 0) {
              atomicAdd(&s_ctr[C_REPLIES_IGNORED], 1u);
              continue;
            }
            if (ln != cl) {
              if (dirty) S.coord_row[row_idx(S, cl, gid)] = crow;
              cl = ln;
              crow = S.coord_row[row_idx(S, cl, gid)];
              dirty = false;
            }
            gpx_decision_rec d;
            if (tally_reply(S, (uint32_t)cl, gid, g.R, g.ms, crow, dirty, r0[l].y, r0[l].z, r0[l].w, r1[l].x,
                            GPX_WHO_ACC(who), d, s_ctr)) {
              if (nd < GPX_MAX_WINDOW) dbuf[nd] = d;
              nd++;
            }
          }
        }
        j++;
        if (j >= n) break;
        rp = &A.replies[(size_t)j * L];
        int4 t0, t1;
        ld256_stream(&rp[0], t0, t1);
        if ((uint32_t)t0.x != gid) break;
        r0[0] = t0;
        r1[0] = t1;
#pragma unroll
        for (int l = 1; l < L; l++) ld256_stream(&rp[l], r0[l], r1[l]);
      }
      if (dirty) S.coord_row[row_idx(S, cl, gid)] = crow;
    }
  }
  if (nd > GPX_MAX_WINDOW) nd = GPX_MAX_WINDOW; /* cannot happen: <= W proposals outstanding */
  uint32_t base = block_reserve(nd, A.n_decisions, s_scan);
  for (uint32_t k = 0; k < nd; k++) {
    const int4* sp = reinterpret_cast<const int4*>(&dbuf[k]);
    st256_stream(&A.decisions[base + k], sp[0], sp[1]);
  }
  flush_counters(S, s_ctr);
}

/* ============================== k_commit ====================================== */
struct CommitArgs {
  const gpx_decision_rec* decisions;
  const uint32_t* n_ptr;
  uint32_t n_max;
  gpx_exec_rec* exec; /* [n_max][L] */
  gpx_exec_rec* extra;
  uint32_t extra_cap;
  uint32_t* n_extra;
};

template <int L>
__global__ void __launch_bounds__(GPX_BLOCK, 2) k_commit(const __grid_constant__ DevState S,
                                                      const __grid_constant__ CommitArgs A) {
  __shared__ unsigned int s_ctr[C_NCTR];
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  __syncthreads();
  uint32_t n = A.n_ptr ? *A.n_ptr : A.n_max;
  if (n > A.n_max) n = A.n_max;
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  const uint32_t Wm = S.W - 1;
  const unsigned long long reserved = seg_decision_bytes(A.n_max);
  unsigned long long segb[L];
#pragma unroll
  for (int l = 0; l < L; l++) segb[l] = seg_base(S, l, reserved);
  if (i == 0) {
#pragma unroll
    for (int l = 0; l < L; l++) {
      const unsigned long long sq = seg_seq_of(S, l);
      write_seg_hdr(S, l, segb[l], GPX_F_DECISION, A.n_max, n, 0, 32, sq);
      log_publish(S, l, segb[l] + reserved, sq + 1ull);
    }
    atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  }
  if (i < n) {
    int4 q0, q1;
    ld256_stream(&A.decisions[i], q0, q1);
    const uint32_t gid = (uint32_t)q0.x;
    const bool head = (i == 0) || (A.decisions[i - 1].gid != gid);
    if (head) {
      const GroupCtx g = group_ctx(S, gid);
      uint32_t j = i;
      while (true) {
        const int slot = q0.y;
        const uint32_t rflags = (uint32_t)q1.y & 0xffffu, dst_mask = (uint32_t)q1.y >> 16;
        uint32_t aux[L];
        int4 row[L], e0[L], e1[L];
#pragma unroll
        for (int l = 0; l < L; l++) {
          aux[l] = 0;
          row[l] = e0[l] = e1[l] = make_int4(0, 0, 0, 0);
          if (g.live) {
            const size_t ri = row_idx(S, l, gid);
            aux[l] = S.acc_aux[ri];
            row[l] = S.acc_row[ri];
            ld256(&S.acc_win[2 * win_idx(S, l, (uint32_t)slot & Wm, gid)], e0[l], e1[l]);
          }
        }
#pragma unroll
        for (int l = 0; l < L; l++) {
          gpx_exec_rec* ex = &A.exec[(size_t)j * L + l];
          store_void_exec(ex, gid, slot, l);
          int4 img0 = q0, img1 = make_int4(q1.x, (int)(GPX_F_VOID | (dst_mask << 16)), q1.z, q1.w);
          if (((dst_mask >> l) & 1u) && !(rflags & GPX_F_VOID)) {
            if (!g.live || !st_usable(aux[l])) {
              atomicAdd(&s_ctr[C_DECISIONS_DROPPED], 1u);
            } else {
              const size_t ri = row_idx(S, l, gid);
              const int4 row_in = row[l];
              const uint32_t aux_in = aux[l];
              commit_lane(S, l, gid, slot, q0.z, q0.w, q1.x, row[l], aux[l], e0[l], e1[l], ex, A.extra, A.extra_cap,
                          A.n_extra, img0, img1, s_ctr);
              const int4 r2 = row[l];
              if (aux[l] != aux_in) S.acc_aux[ri] = aux[l];
              if (r2.x != row_in.x || r2.y != row_in.y || r2.z != row_in.z || r2.w != row_in.w) S.acc_row[ri] = r2;
            }
          }
          st256_stream(ring_ptr(S, l, segb[l] + 64 + (unsigned long long)j * 32), img0, img1);
        }
        j++;
        if (j >= n) break;
        int4 t0, t1;
        ld256_stream(&A.decisions[j], t0, t1);
        if ((uint32_t)t0.x != gid) break;
        q0 = t0;
        q1 = t1;
      }
    }
  }
  flush_counters(S, s_ctr);
}

/* ============================== k_act (fused) ================================== */
/* Per ACCEPT, in batch order: handleAccept at every addressed lane; replies addressed to a usable LOCAL
 * coordinator lane are tallied at once (the others are written to A.replies for the host); a resulting
 * DECISION is committed at every local lane before the next ACCEPT of the run.  Per lane it appends an
 * ACCEPT segment followed by a DECISION segment (image index = ACCEPT index).  On the fast path (the
 * in-order case) rows are read and written once, replies and the decision never touch HBM, and an entry
 * that is accepted and executed in the same pass is not written at all. */
template <int L>
__global__ void __launch_bounds__(GPX_BLOCK, GPX_ACT_MINB) k_act(const __grid_constant__ DevState S,
                                                   const __grid_constant__ AcceptArgs A) {
  __shared__ unsigned int s_ctr[C_NCTR];
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  __syncthreads();
  uint32_t n = A.n_ptr ? *A.n_ptr : A.n_max;
  if (n > A.n_max) n = A.n_max;
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  const uint32_t Wm = S.W - 1;
  const unsigned long long pay_bytes = A.blob0_bytes + (A.blob1_used_ptr ? *A.blob1_used_ptr : A.blob1_bytes);
  /* = seg_pay_rel(A.n_max), written out: calling the helper here reorders k_act's prologue */
  const unsigned long long pay_rel = 64ull + (unsigned long long)A.n_max * 48ull;
  const unsigned long long res_a = seg_align32(pay_rel + pay_bytes); /* = seg_accept_bytes(A.n_max, pay_bytes) */
  const unsigned long long res_d = seg_decision_bytes(A.n_max);
  unsigned long long segb[L], payb[L], dsegb[L];
#pragma unroll
  for (int l = 0; l < L; l++) {
    segb[l] = seg_base(S, l, res_a + res_d); /* both segments on one side of the ring wrap */
    payb[l] = segb[l] + pay_rel;
    dsegb[l] = segb[l] + res_a;
  }
  if (i == 0) {
#pragma unroll
    for (int l = 0; l < L; l++) {
      const unsigned long long sq = seg_seq_of(S, l);
      write_seg_hdr(S, l, segb[l], GPX_F_ACCEPT, A.n_max, n, pay_bytes, 48, sq);
      write_seg_hdr(S, l, dsegb[l], GPX_F_DECISION, A.n_max, n, 0, 32, sq + 1ull);
      log_publish(S, l, segb[l] + res_a + res_d, sq + 2ull);
    }
    atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  }
  if (i < n) {
    const int4* rp = reinterpret_cast<const int4*>(&A.recs[i]);
    int4 q0 = ld_stream4(rp), q1 = ld_stream4(rp + 1), q2 = ld_stream4(rp + 2);
    const uint32_t gid = (uint32_t)q0.x;
    const bool head = (i == 0) || (A.recs[i - 1].h.gid != gid);
    if (head) {
      const GroupCtx g = group_ctx(S, gid);
      uint32_t j = i;
      while (true) {
        const int slot = q0.y;
        const uint32_t payload_off = (uint32_t)q2.x;
        /* ---- all independent loads of this ACCEPT ---- */
        LaneSt st[L];
        int4 e0[L], e1[L];
#pragma unroll
        for (int l = 0; l < L; l++) {
          st[l].aux = 0;
          st[l].row = make_int4(0, 0, 0, 0);
          e0[l] = e1[l] = make_int4(0, 0, 0, 0);
          if (g.live) {
            const size_t ri = row_idx(S, l, gid);
            st[l].aux = S.acc_aux[ri];
            st[l].row = S.acc_row[ri];
            ld256(&S.acc_win[2 * win_idx(S, l, (uint32_t)slot & Wm, gid)], e0[l], e1[l]);
          }
        }
        uint32_t dstIdx = 0xffu;
        if (g.live)
          for (uint32_t m = 0; m < g.R; m++)
            if (g.ms->nodes[m] == q2.w) dstIdx = m;
        int cl = -1; /* the coordinator that issued this ACCEPT, if it is a local lane */
        if (g.live && dstIdx < g.R && g.ms->lane_of_idx[dstIdx] != 0xffu) cl = g.ms->lane_of_idx[dstIdx];
        int4 crow = make_int4(0, 0, 0, 0);
        if (cl >= 0) crow = S.coord_row[row_idx(S, cl, gid)];
        /* ---- accept at every lane ---- */
        uint32_t logmask = 0;
#pragma unroll
        for (int l = 0; l < L; l++) {
          const unsigned fr = (unsigned)(((payb[l] + payload_off) & (S.ring_cap - 1)) >> 4);
          accept_lane(S, A, l, g.live, g.ms, dstIdx, q0, q1, q2, e0[l], e1[l], fr, st[l], s_ctr);
          if (st[l].fl & LS_LOGGED) logmask |= 1u << l;
          write_accept_image(S, l, segb[l], A.n_max, j, q0, q1, q2, st[l].img_flags);
        }
        if (logmask) copy_blob<L>(S, A, payload_off, (uint32_t)q2.y, logmask, payb);
        /* ---- tally the replies addressed to a usable local coordinator (PISM drop rule :456-460) ---- */
        uint32_t caux = 0;
#pragma unroll
        for (int l = 0; l < L; l++)
          if (l == cl) caux = st[l].aux;
        const bool tally_here = cl >= 0 && st_usable(caux);
        gpx_decision_rec d;
        d.gid = gid;
        d.slot = slot;
        d.bnum = 0;
        d.bcoord = 0;
        d.median_cp = 0;
        d.flags = GPX_F_VOID;
        d.dst_mask = 0;
        d.req_id = 0;
        bool decided = false, cdirty = false;
        uint32_t omask = 0; /* replies that leave this engine (remote or unusable coordinator) */
#pragma unroll
        for (int l = 0; l < L; l++) {
          const bool is_void = (GPX_WHO_FLAGS(st[l].rwho) & GPX_F_VOID) != 0;
          if (is_void) continue;
          if (tally_here) { /* consumed locally: the reply never touches HBM */
            gpx_decision_rec dd;
            if (tally_reply(S, (uint32_t)cl, gid, g.R, g.ms, crow, cdirty, slot, st[l].rbn, st[l].rbc, st[l].rmaxcp,
                            GPX_WHO_ACC(st[l].rwho), dd, s_ctr) &&
                !decided) {
              d = dd;
              decided = true;
            }
          } else {
            omask |= 1u << l;
            st256_stream(&A.replies[(size_t)j * L + l], make_int4((int)gid, slot, st[l].rbn, st[l].rbc),
                         make_int4(st[l].rmaxcp, (int)st[l].rwho, q1.z, q1.w));
          }
        }
        A.out_mask[j] = (uint8_t)omask;
        if (cdirty) S.coord_row[row_idx(S, cl, gid)] = crow;
        {
          const int4* sp = reinterpret_cast<const int4*>(&d);
          st256_stream(&A.decisions[j], sp[0], sp[1]);
        }
        /* ---- commit the decision at every lane ---- */
#pragma unroll
        for (int l = 0; l < L; l++) {
          gpx_exec_rec* ex = &A.exec[(size_t)j * L + l];
          int4 img0 = make_int4((int)gid, slot, d.bnum, d.bcoord);
          int4 img1 = make_int4(d.median_cp, (int)(GPX_F_VOID | ((uint32_t)d.dst_mask << 16)),
                                (int)(unsigned)(d.req_id & 0xffffffffll), (int)(d.req_id >> 32));
          const size_t ai = 2 * win_idx(S, l, (uint32_t)slot & Wm, gid);
          const size_t ri = row_idx(S, l, gid);
          int4& row = st[l].row;
          uint32_t& aux = st[l].aux;
          if (!(decided && ((d.dst_mask >> l) & 1u))) {
            store_void_exec(ex, gid, slot, l);
          } else if (!g.live || !st_usable(aux)) {
            store_void_exec(ex, gid, slot, l);
            atomicAdd(&s_ctr[C_DECISIONS_DROPPED], 1u);
          } else {
            const int4 row_b = row;
            const uint32_t aux_b = aux;
            const bool fast = (st[l].fl & LS_STORE) && q0.z == d.bnum && q0.w == d.bcoord && slot == row.x &&
                              !((GPX_AUX_PRESENT(aux) >> ((uint32_t)slot & Wm)) & 1u);
            if (fast) {
              /* the accept stored a moment ago is the decided value and it is next in line:
               * handleBatchedCommit :1488-1501 + the first iteration of extractExecuteAndCheckpoint */
              atomicAdd(&s_ctr[C_DECISIONS_HANDLED], 1u);
              int4 n0, n1;
              make_entry(q0, q1, q2, st[l].frame_ref, n0, n1);
              const unsigned efl = (unsigned)n1.w;
              const bool metaf = S.log_meta != 0;
              const uint32_t lf = GPX_F_DECISION | (metaf ? GPX_F_META : 0u) | ((efl & GPX_ENT_STOP) ? GPX_F_STOP : 0u);
              img0 = make_int4((int)gid, slot, d.bnum, d.bcoord);
              img1 = make_int4(metaf ? -1 : d.median_cp, (int)(lf | ((1u << l) << 16)), n1.x, n1.y);
              gc_step(row, d.median_cp);
              DPValue x;
              x.slot = slot;
              x.bnum = d.bnum;
              x.bcoord = d.bcoord;
              x.median_cp = d.median_cp;
              x.req_id = ((long long)n1.y << 32) | (unsigned)n1.x;
              x.frame_ref = st[l].frame_ref;
              x.plen = (unsigned)n1.z;
              x.fl = efl & ~GPX_ENT_VALID;
              x.valued = true;
              row.x = (int)((unsigned)row.x + 1u); /* executed(): _slot++ */
              atomicAdd(&s_ctr[C_EXECUTED], 1u);
              gpx_exec_rec er = make_exec(S, gid, l, x, false);
              if (er.flags & GPX_F_CKPT) atomicAdd(&s_ctr[C_CKPTS_DUE], 1u);
              store_exec(ex, er);
              bool more = true;
              if (efl & GPX_ENT_STOP) {
                aux = (aux & ~0xffu) | GPX_ST_STOPPED; /* stop() + committedRequests.clear() */
                aux &= ~0x00ffff00u;
                atomicAdd(&s_ctr[C_STOPS_EXECUTED], 1u);
                more = false;
              }
              if (S.journaling) {
                /* acceptedProposals.remove(slot): the entry only has to reach HBM (invalidated) when it must
                 * hide an occupant of the ring position whose valid bit is set */
                if (st[l].fl & LS_OCCVALID) {
                  n1.w = (int)((unsigned)n1.w & ~GPX_ENT_VALID);
                  ST_ACC(S, l, gid, ai, n0, n1);
                }
              } else
                ST_ACC(S, l, gid, ai, n0, n1);
              st[l].fl &= ~LS_STORE;
              if (more) { /* second iteration: GC with the advanced slot, then any queued commits */
                gc_step(row, d.median_cp);
                if ((GPX_AUX_PRESENT(aux) >> ((uint32_t)row.x & Wm)) & 1u)
                  eec(S, l, gid, row, aux, x, nullptr, A.extra, A.extra_cap, A.n_extra, s_ctr, true);
              }
            } else {
              /* general path through memory: make the accepted entry visible, then commit */
              int4 a0, a1; /* rare path: re-read the entry instead of keeping L x 32 B of registers alive */
              if (st[l].fl & LS_STORE) {
                make_entry(q0, q1, q2, st[l].frame_ref, a0, a1);
                ST_ACC(S, l, gid, ai, a0, a1);
                st[l].fl &= ~LS_STORE;
              } else
                ld256(&S.acc_win[ai], a0, a1);
              store_void_exec(ex, gid, slot, l);
              commit_lane(S, l, gid, slot, d.bnum, d.bcoord, d.median_cp, row, aux, a0, a1, ex, A.extra, A.extra_cap,
                          A.n_extra, img0, img1, s_ctr);
            }
            if (aux != aux_b) st[l].fl |= LS_AUXDIRTY;
            if (row.x != row_b.x || row.y != row_b.y || row.z != row_b.z || row.w != row_b.w) st[l].fl |= LS_ROWDIRTY;
          }
          if (st[l].fl & LS_STORE) {
            int4 n0, n1;
            make_entry(q0, q1, q2, st[l].frame_ref, n0, n1);
            ST_ACC(S, l, gid, ai, n0, n1);
          }
          if (st[l].fl & LS_ROWDIRTY) S.acc_row[ri] = row;
          if (st[l].fl & LS_AUXDIRTY) S.acc_aux[ri] = aux;
          st256_stream(ring_ptr(S, l, dsegb[l] + 64 + (unsigned long long)j * 32), img0, img1);
        }
        j++;
        if (j >= n) break;
        rp = reinterpret_cast<const int4*>(&A.recs[j]);
        int4 t0 = ld_stream4(rp);
        if ((uint32_t)t0.x != gid) break;
        q0 = t0;
        q1 = ld_stream4(rp + 1);
        q2 = ld_stream4(rp + 2);
      }
    }
  }
  flush_counters(S, s_ctr);
}

/* ============================== state maintenance ============================== */
struct InitRec { /* host-preprocessed gpx_group_desc */
  uint32_t gid;
  uint32_t mset;
  int32_t coord0; /* roundRobinCoordinator(name, members, 0) */
  int32_t cpi;
  int32_t init_mode;
  uint32_t R;
};

/* PaxosManager.createPaxosInstance batch form :664-691 -> createHRI paxosutil/HotRestoreInfo.java:145-157,
 * or PISM.initiateRecovery :591-675 + putInitialState :692-699 */
__global__ void k_init_groups(const __grid_constant__ DevState S, const InitRec* recs, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const InitRec r = recs[i];
  const MsetInfo* ms = &S.msets[r.mset];
  S.grp_meta[r.gid] = r.mset | (r.R << 16) | GPX_META_LIVE | (ms->ident ? GPX_META_IDENT : 0u);
  S.grp_cpi[r.gid] = r.cpi;
  for (uint32_t l = 0; l < S.L; l++) {
    const size_t ri = row_idx(S, l, r.gid);
    S.acc_dirty[ri] = 0;
    for (uint32_t w = 0; w < S.W; w++) {
      const size_t wi = win_idx(S, l, w, r.gid);
      S.acc_win[2 * wi] = make_int4(0, 0, 0, 0);
      S.acc_win[2 * wi + 1] = make_int4(0, 0, 0, 0);
      S.com_win[2 * wi] = make_int4(0, 0, 0, 0);
      S.com_win[2 * wi + 1] = make_int4(0, 0, 0, 0);
      S.prop_win[wi] = make_int4(0, 0, 0, 0);
    }
    if (ms->idx_of_lane[l] == 0xffu) { /* lane is not a member: no instance here */
      S.acc_row[ri] = make_int4(0, -1, -1, -1);
      S.acc_aux[ri] = GPX_ST_FREE;
      S.coord_row[ri] = make_int4(0, 0, 0, 0);
      continue;
    }
    const bool batch = r.init_mode == GPX_INIT_BATCH;
    S.acc_row[ri] = make_int4(1, 0, r.coord0, batch ? -1 : 0);
    S.acc_aux[ri] = GPX_ST_ACTIVE_1;
    const bool am_coord = (r.coord0 == S.lane_node[l]);
    S.coord_row[ri] = am_coord ? make_int4(0, r.coord0, 1, (int)(GPX_CF_EXISTS | GPX_CF_ACTIVE)) : make_int4(0, 0, 0, 0);
    for (uint32_t m = 0; m < S.Rcap; m++) S.node_slots[ns_idx(S, l, m, r.gid)] = am_coord ? (batch ? 0 : -1) : 0;
  }
}

__global__ void k_destroy_groups(const __grid_constant__ DevState S, const uint32_t* gids, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t gid = gids[i];
  if (gid >= S.G) return;
  free_group(S, gid);
}

__global__ void k_dump_rows(const __grid_constant__ DevState S, const uint32_t* gids, uint32_t n, uint32_t lane,
                            gpx_row* out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  gpx_row r;
  dump_row(S, lane, gids[i], r);
  out[i] = r;
}

struct LoadRec {
  gpx_row row;
  uint32_t mset;
  int32_t cpi;
};
__global__ void k_load_rows(const __grid_constant__ DevState S, const LoadRec* recs, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const gpx_row& r = recs[i].row;
  const uint32_t gid = r.gid, l = r.lane;
  S.grp_meta[gid] = recs[i].mset | ((uint32_t)r.n_members << 16) | GPX_META_LIVE |
                    (S.msets[recs[i].mset].ident ? GPX_META_IDENT : 0u);
  S.grp_cpi[gid] = recs[i].cpi;
  const size_t ri = row_idx(S, l, gid);
  S.acc_row[ri] = make_int4(r.acc_slot, r.acc_bnum, r.acc_bcoord, r.acc_gc_slot);
  S.acc_aux[ri] = (uint32_t)r.state & 0xffu;
  S.acc_dirty[ri] = 0; /* every window entry is invalidated below */
  for (uint32_t w = 0; w < S.W; w++) {
    const size_t wi = win_idx(S, l, w, gid);
    S.acc_win[2 * wi + 1] = make_int4(0, 0, 0, 0);
    S.prop_win[wi] = make_int4(0, 0, 0, 0);
  }
  if (r.coord_exists) {
    S.coord_row[ri] =
        make_int4(r.coord_bnum, r.coord_bcoord, r.next_proposal_slot, (int)(GPX_CF_EXISTS | (r.coord_active ? GPX_CF_ACTIVE : 0u)));
    for (int m = 0; m < r.n_members && m < (int)S.Rcap; m++) S.node_slots[ns_idx(S, l, m, gid)] = r.node_slots[m];
  } else
    S.coord_row[ri] = make_int4(0, 0, 0, 0);
}

/* slow-path effects as state patches (SURVEY.md 8b): distinct (gid,lane) targets per call */
__global__ void k_patch(const __grid_constant__ DevState S, const gpx_patch_rec* p, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const gpx_patch_rec r = p[i];
  if (r.gid >= S.G || r.lane >= S.L) return;
  const size_t ri = row_idx(S, r.lane, r.gid);
  int4 row = S.acc_row[ri];
  uint32_t aux = S.acc_aux[ri];
  const uint32_t Wm = S.W - 1;
  switch (r.op) {
    case GPX_PATCH_SET_BALLOT: /* handlePrepare :245-251 */
      if (bcmp(r.a, r.b, row.y, row.z) > 0) {
        row.y = r.a;
        row.z = r.b;
      }
      break;
    case GPX_PATCH_JUMP_SLOT: /* jumpSlot :564-578 */
      while (jsub(row.x, r.a) < 0) {
        const uint32_t w = (uint32_t)row.x & Wm;
        aux &= ~((1u << (8 + w)) | (1u << (16 + w)));
        if (S.journaling) {
          const size_t ai = 2 * win_idx(S, r.lane, w, r.gid);
          int4 a0 = S.acc_win[ai], a1 = S.acc_win[ai + 1];
          if (((unsigned)a1.w & GPX_ENT_VALID) && a0.x == row.x) {
            a1.w = (int)((unsigned)a1.w & ~GPX_ENT_VALID);
            S.acc_win[ai + 1] = a1;
          }
        }
        row.x = (int)((unsigned)row.x + 1u);
      }
      break;
    case GPX_PATCH_SET_STATE:
      aux = (aux & ~0xffu) | ((uint32_t)r.a & 0xffu);
      if (((uint32_t)r.a & 0xffu) == GPX_ST_STOPPED) aux &= ~0x00ffff00u;
      break;
    case GPX_PATCH_INSTALL_COORD: {
      S.coord_row[ri] = make_int4(r.a, r.b, r.c, (int)(GPX_CF_EXISTS | (r.d ? GPX_CF_ACTIVE : 0u)));
      for (uint32_t m = 0; m < S.Rcap; m++) S.node_slots[ns_idx(S, r.lane, m, r.gid)] = -1;
      for (uint32_t w = 0; w < S.W; w++) S.prop_win[win_idx(S, r.lane, w, r.gid)] = make_int4(0, 0, 0, 0);
      break;
    }
    case GPX_PATCH_RESIGN_COORD:
      S.coord_row[ri] = make_int4(0, 0, 0, 0);
      for (uint32_t w = 0; w < S.W; w++) S.prop_win[win_idx(S, r.lane, w, r.gid)] = make_int4(0, 0, 0, 0);
      break;
    case GPX_PATCH_SET_GC: row.w = r.a; break;
    case GPX_PATCH_SET_NODE_SLOT: /* PCS.recordSlotNumber(PrepareReplyPacket) :786-807 */
      if ((((unsigned)S.coord_row[ri].w) & GPX_CF_EXISTS) && r.a >= 0 && (uint32_t)r.a < S.Rcap) {
        const size_t ni = ns_idx(S, r.lane, (uint32_t)r.a, r.gid);
        if (jsub(S.node_slots[ni], r.b) < 0) S.node_slots[ni] = r.b;
      }
      break;
    default: break;
  }
  S.acc_row[ri] = row;
  S.acc_aux[ri] = aux;
}

__global__ void k_get_flags(const __grid_constant__ DevState S, uint32_t lane, const uint32_t* gids, uint32_t n,
                            uint8_t* out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (gids[i] >= S.G) {
    out[i] = 0;
    return;
  }
  out[i] = (uint8_t)group_flags(S, lane, gids[i]);
}

/* ============================== digests (DIGEST_REQUESTS) ============================== */
/* RequestPacket.getDigest paxospackets/RequestPacket.java:1414-1430: MD5 of the requestValue bytes -- the
 * "accepted-pvalue digest" column.  One thread per request; RFC 1321. */
__device__ __forceinline__ uint32_t md5_rotl(uint32_t x, int c) { return (x << c) | (x >> (32 - c)); }
__constant__ uint32_t c_md5_k[64] = {
    0xd76aa478, 0xe8c7b756, 0x242070db, 0xc1bdceee, 0xf57c0faf, 0x4787c62a, 0xa8304613, 0xfd469501, 0x698098d8,
    0x8b44f7af, 0xffff5bb1, 0x895cd7be, 0x6b901122, 0xfd987193, 0xa679438e, 0x49b40821, 0xf61e2562, 0xc040b340,
    0x265e5a51, 0xe9b6c7aa, 0xd62f105d, 0x02441453, 0xd8a1e681, 0xe7d3fbc8, 0x21e1cde6, 0xc33707d6, 0xf4d50d87,
    0x455a14ed, 0xa9e3e905, 0xfcefa3f8, 0x676f02d9, 0x8d2a4c8a, 0xfffa3942, 0x8771f681, 0x6d9d6122, 0xfde5380c,
    0xa4beea44, 0x4bdecfa9, 0xf6bb4b60, 0xbebfbc70, 0x289b7ec6, 0xeaa127fa, 0xd4ef3085, 0x04881d05, 0xd9d4d039,
    0xe6db99e5, 0x1fa27cf8, 0xc4ac5665, 0xf4292244, 0x432aff97, 0xab9423a7, 0xfc93a039, 0x655b59c3, 0x8f0ccc92,
    0xffeff47d, 0x85845dd1, 0x6fa87e4f, 0xfe2ce6e0, 0xa3014314, 0x4e0811a1, 0xf7537e82, 0xbd3af235, 0x2ad7d2bb,
    0xeb86d391};
__constant__ uint8_t c_md5_s[64] = {7, 12, 17, 22, 7, 12, 17, 22, 7, 12, 17, 22, 7, 12, 17, 22, 5, 9,  14, 20, 5, 9,
                                    14, 20, 5, 9,  14, 20, 5, 9,  14, 20, 4, 11, 16, 23, 4, 11, 16, 23, 4, 11, 16, 23,
                                    4, 11, 16, 23, 6, 10, 15, 21, 6, 10, 15, 21, 6, 10, 15, 21, 6, 10, 15, 21};

__device__ __forceinline__ uint32_t md5_byte(const uint8_t* msg, uint64_t len, uint64_t padded, uint64_t idx) {
  if (idx < len) return msg[idx];
  if (idx == len) return 0x80u;
  if (idx >= padded - 8) return (uint32_t)(((len * 8ull) >> (8 * (idx - (padded - 8)))) & 0xffu);
  return 0u;
}

__global__ void __launch_bounds__(GPX_BLOCK) k_md5(const gpx_request_rec* reqs, uint32_t n, const uint8_t* payload,
                                                   uint8_t* out /* [n][16] */) {
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  if (i >= n) return;
  const uint8_t* msg = payload + reqs[i].payload_off;
  const uint64_t len = reqs[i].payload_len;
  const uint64_t padded = ((len + 8) / 64 + 1) * 64;
  uint32_t a0 = 0x67452301u, b0 = 0xefcdab89u, c0 = 0x98badcfeu, d0 = 0x10325476u;
  for (uint64_t off = 0; off < padded; off += 64) {
    uint32_t M[16];
#pragma unroll
    for (int w = 0; w < 16; w++) {
      const uint64_t p = off + 4ull * w;
      if (p + 4 <= len && ((uintptr_t)(msg + p) & 3u) == 0)
        M[w] = *reinterpret_cast<const uint32_t*>(msg + p);
      else
        M[w] = md5_byte(msg, len, padded, p) | (md5_byte(msg, len, padded, p + 1) << 8) |
               (md5_byte(msg, len, padded, p + 2) << 16) | (md5_byte(msg, len, padded, p + 3) << 24);
    }
    uint32_t A = a0, B = b0, Cc = c0, D = d0;
#pragma unroll
    for (int r = 0; r < 64; r++) {
      uint32_t F;
      int g;
      if (r < 16) {
        F = (B & Cc) | (~B & D);
        g = r;
      } else if (r < 32) {
        F = (D & B) | (~D & Cc);
        g = (5 * r + 1) & 15;
      } else if (r < 48) {
        F = B ^ Cc ^ D;
        g = (3 * r + 5) & 15;
      } else {
        F = Cc ^ (B | ~D);
        g = (7 * r) & 15;
      }
      F = F + A + c_md5_k[r] + M[g];
      A = D;
      D = Cc;
      Cc = B;
      B = B + md5_rotl(F, c_md5_s[r]);
    }
    a0 += A;
    b0 += B;
    c0 += Cc;
    d0 += D;
  }
  *reinterpret_cast<int4*>(out + 16ull * i) = make_int4((int)a0, (int)b0, (int)c0, (int)d0);
}
