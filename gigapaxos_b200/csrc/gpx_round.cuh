/*
 * gpx_round.cuh -- k_round: one launch advances every group of a request batch through a whole Paxos
 * round (RequestBatcher -> propose -> accept x R -> tally -> commit x R) for co-located replicas.
 *
 * Work mapping: a TEAM of L threads (adjacent lanes of one warp, 32/L teams per warp) owns one request index;
 * team thread `sub` is replica lane `sub` of the group.  Two kernels:
 *
 *   k_round       the in-order case, straight-line predicated code.  Every thread loads ITS lane's acceptor row,
 *                 aux word and coordinator row (+ the group's meta word and the first payload chunk); the entry
 *                 lane's and the coordinator lane's rows reach the team by full-warp __shfl_sync
 *                 (PISM.handleProposal :818-888, PCS.propose :233-263); a team vote (__ballot_sync) checks that every
 *                 lane is the plain case of PISM.handleAccept :1080-1166 (same ballot, next slot, nothing there);
 *                 the L ACCEPT_REPLYs (maxCheckpointedSlot :1139-1143) are exchanged by shuffles and tallied in
 *                 registers (recordSlotNumber :809-825, getMedianMinus :867-875, majority at reply L/2); each thread
 *                 then writes only the durable outputs of its lane (log image + blob, decision image, EXEC record or
 *                 summary, window entry, acceptor row) and thread 0 the status and the coordinator row.
 *                 The ACCEPT record, the replies, the DECISION and the proposal never exist in memory.  Block 0 writes
 *                 the segment headers and the NEXT launch's log positions (double-buffered by launch parity,
 *                 gpx_dev.cuh): no ticket, no fence, no publisher behind the kernel.
 *   k_round_slow  everything else (several requests of a group in the batch -> one batched slot, STOP, outstanding
 *                 proposals, a pre-active / missing / remote coordinator, an occupied window entry, a queued commit,
 *                 NACKs): teams that cannot take the in-order path append their request index to a todo list, and the
 *                 FIRST of them launches this kernel from the device as a tail launch (it starts when k_round has
 *                 completed and before anything else on the stream) -- a round without such runs is a single kernel;
 *                 gpx_set_round_mode(2) makes the host launch it behind every k_round instead.  Three grid-wide
 *                 phases separated by grid barriers: propose (one thread per run), blobs of batched slots + VOID
 *                 outputs (one thread per request of those runs), accept x L / tally / commit x L (one team per run:
 *                 propose_run / tally_reply against memory, decision broadcast to the lanes by shuffles).
 *
 * Semantics are those of gpx_propose followed by gpx_handle_accepts_fused (checked by the test-suite); record,
 * image and EXEC indices are REQUEST indices (holes are VOID).
 */
#pragma once
#include "gpx_kernels.cuh"

struct RoundArgs {
  ProposeArgs P;  /* reqs, n, payload_bytes_al, accepts (scratch, indexed by request), status, copy_*, ctl */
  AcceptArgs A;   /* blob0/blob1, replies, decisions, out_mask, exec, extra ... (recs/n_ptr unused) */
  uint8_t* blob1w; /* writable alias of A.blob1 (constructed blobs of batched slots) */
  unsigned long long blob1_res; /* payload-area bytes reserved for constructed blobs */
  uint32_t* todo;               /* request indices of the runs left to k_round_slow */
  uint32_t* todo_end;           /* [k] one past the last request of run todo[k] (written by k_round_slow's phase 1) */
  uint32_t* n_todo;
  uint8_t* mark;                /* [n] 1 = the request belongs to a run left to k_round_slow (written by k_round for every
                                 * request: phase 2 of the slow kernel is one thread per REQUEST) */
  RoundCtl* ctl_zero;           /* the control block the NEXT round will count into, zeroed by block 0 of k_round (null: the
                                 * host zeroes it) */
  uint32_t slow_grid;           /* grid of k_round_slow (all blocks resident: its phases are separated by grid barriers) */
  uint32_t tail_launch;         /* 1: the first team that leaves a run to k_round_slow launches it from the device as a
                                 * tail launch (runs when k_round has completed, before anything else on the stream);
                                 * 0: the host launches k_round_slow behind every k_round */
  /* launch constants of the two log segments of a lane (host-computed: no 64-bit arithmetic in the kernels) */
  unsigned long long pay_bytes; /* payload area of the ACCEPT segment = blob0_bytes + blob1_res */
  unsigned long long res_a;     /* ACCEPT segment bytes  = seg_accept_bytes(n, pay_bytes) (gpx_logseg.cuh) */
  unsigned long long res_d;     /* DECISION segment bytes = seg_decision_bytes(n) */
  uint32_t pay_rel;             /* payload area offset inside the ACCEPT segment = seg_pay_rel(n) */
  gpx_exec_sum* sum;            /* compact output mode (GPX_ROUND_COMPACT): one summary per request index instead of
                                 * n_lanes EXEC rows; everything that is not the plain in-order case goes to the
                                 * extra queue.  null = full EXEC rows */
};

__device__ __forceinline__ void store_sum(gpx_exec_sum* dst, int slot, uint32_t lane_mask, uint32_t flags, uint32_t nreq) {
  *reinterpret_cast<int2*>(dst) = make_int2(slot, (int)(lane_mask | (flags << 8) | (nreq << 16)));
}

#ifndef GPX_RBLOCK
#define GPX_RBLOCK 128 /* threads per block of the fast round kernel: finer-grained waves than 256 (measured +3%) */
#endif
#ifndef GPX_ROUND_MINB
#define GPX_ROUND_MINB 5 /* 48 registers per thread = 1,280 resident threads per SM; measured optimum (40 and 64 are slower) */
#endif

/* commit of decision d at one lane, state in registers (the per-lane part of k_act's commit phase) */
template <int L>
__device__ __forceinline__ void commit_team_lane(const DevState& S, const AcceptArgs& A, uint32_t l, uint32_t gid,
                                                 int slot, bool live, bool decided, const gpx_decision_rec& d,
                                                 const int4 q0, const int4 q1, const int4 q2, LaneSt& st, uint32_t j,
                                                 unsigned long long dseg, unsigned int* s_ctr) {
  const uint32_t Wm = S.W - 1;
  gpx_exec_rec* ex = &A.exec[(size_t)j * L + l];
  int4 img0 = make_int4((int)gid, slot, d.bnum, d.bcoord);
  int4 img1 = make_int4(d.median_cp, (int)(GPX_F_VOID | ((uint32_t)d.dst_mask << 16)),
                        (int)(unsigned)(d.req_id & 0xffffffffll), (int)(d.req_id >> 32));
  const size_t ai = 2 * win_idx(S, l, (uint32_t)slot & Wm, gid);
  const size_t ri = row_idx(S, l, gid);
  int4& row = st.row;
  uint32_t& aux = st.aux;
  if (!(decided && ((d.dst_mask >> l) & 1u))) {
    store_void_exec(ex, gid, slot, l);
  } else if (!live || !st_usable(aux)) {
    store_void_exec(ex, gid, slot, l);
    atomicAdd(&s_ctr[C_DECISIONS_DROPPED], 1u);
  } else {
    const int4 row_b = row;
    const uint32_t aux_b = aux;
    const bool fast = (st.fl & LS_STORE) && q0.z == d.bnum && q0.w == d.bcoord && slot == row.x &&
                      !((GPX_AUX_PRESENT(aux) >> ((uint32_t)slot & Wm)) & 1u);
    if (fast) {
      atomicAdd(&s_ctr[C_DECISIONS_HANDLED], 1u);
      int4 n0, n1;
      make_entry(q0, q1, q2, st.frame_ref, n0, n1);
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
      x.frame_ref = st.frame_ref;
      x.plen = (unsigned)n1.z;
      x.fl = efl & ~GPX_ENT_VALID;
      x.valued = true;
      row.x = (int)((unsigned)row.x + 1u);
      atomicAdd(&s_ctr[C_EXECUTED], 1u);
      gpx_exec_rec er = make_exec(S, gid, l, x, false);
      if (er.flags & GPX_F_CKPT) atomicAdd(&s_ctr[C_CKPTS_DUE], 1u);
      store_exec(ex, er);
      bool more = true;
      if (efl & GPX_ENT_STOP) {
        aux = (aux & ~0xffu) | GPX_ST_STOPPED;
        aux &= ~0x00ffff00u;
        atomicAdd(&s_ctr[C_STOPS_EXECUTED], 1u);
        more = false;
      }
      if (S.journaling) {
        if (st.fl & LS_OCCVALID) {
          n1.w = (int)((unsigned)n1.w & ~GPX_ENT_VALID);
          ST_ACC(S, l, gid, ai, n0, n1);
        }
      } else
        ST_ACC(S, l, gid, ai, n0, n1);
      st.fl &= ~LS_STORE;
      if (more) {
        gc_step(row, d.median_cp);
        if ((GPX_AUX_PRESENT(aux) >> ((uint32_t)row.x & Wm)) & 1u)
          eec(S, l, gid, row, aux, x, nullptr, A.extra, A.extra_cap, A.n_extra, s_ctr, true);
      }
    } else {
      int4 a0, a1;
      if (st.fl & LS_STORE) {
        make_entry(q0, q1, q2, st.frame_ref, a0, a1);
        ST_ACC(S, l, gid, ai, a0, a1);
        st.fl &= ~LS_STORE;
      } else
        ld256(&S.acc_win[ai], a0, a1);
      store_void_exec(ex, gid, slot, l);
      commit_lane(S, l, gid, slot, d.bnum, d.bcoord, d.median_cp, row, aux, a0, a1, ex, A.extra, A.extra_cap,
                  A.n_extra, img0, img1, s_ctr);
    }
    if (aux != aux_b) st.fl |= LS_AUXDIRTY;
    if (row.x != row_b.x || row.y != row_b.y || row.z != row_b.z || row.w != row_b.w) st.fl |= LS_ROWDIRTY;
  }
  if (st.fl & LS_STORE) {
    int4 n0, n1;
    make_entry(q0, q1, q2, st.frame_ref, n0, n1);
    ST_ACC(S, l, gid, ai, n0, n1);
  }
  if (st.fl & LS_ROWDIRTY) S.acc_row[ri] = row;
  if (st.fl & LS_AUXDIRTY) S.acc_aux[ri] = aux;
  st256_stream(ring_ptr(S, l, dseg + 64 + (unsigned long long)j * 32), img0, img1);
}

/* General path, phase 1, for the run that starts at request index i: RequestBatcher + PCS.propose by team thread 0
 * (propose_run writes the ACCEPTs at their request index, the status of every request of the run and, for batched
 * slots, where each request's table entry and body go).  Returns one past the last request of the run. */
__device__ __forceinline__ uint32_t round_propose(const DevState& S, const RoundArgs& RA, uint32_t i, uint32_t gid,
                                                  unsigned int* s_ctr) {
  const gpx_request_rec* reqs = RA.P.reqs;
  const uint32_t n = RA.P.n;
  uint32_t nb = 0, k = i;
  while (k < n && reqs[k].gid == gid) {
    k = batch_end(S, reqs, n, k, gid);
    nb++;
  }
  propose_run(S, RA.P, i, k, nb, i, s_ctr, true);
  return k;
}

/* General path, phase 2, for ONE request q of a left-over run: its entry and body in the blob of a batched slot,
 * [nreq x gpx_batch_ent][values] (RequestPacket.batched) */
__device__ __forceinline__ void round_build_blob(const RoundArgs& RA, uint32_t q, int st) {
  const gpx_request_rec* reqs = RA.P.reqs;
  const gpx_request_rec r = reqs[q];
  const bool batched = (st == GPX_RS_BATCHED) ||
                       (st > 0 && q + 1 < RA.P.n && RA.P.status[q + 1] == GPX_RS_BATCHED && reqs[q + 1].gid == r.gid);
  if (!batched) return;
  gpx_batch_ent be;
  be.req_id = r.req_id;
  be.len = r.payload_len;
  be.flags = r.flags;
  *reinterpret_cast<int4*>(RA.blob1w + (RA.P.copy_tab[q] - RA.A.blob0_bytes)) = *reinterpret_cast<const int4*>(&be);
  uint8_t* d = RA.blob1w + (RA.P.copy_dst[q] - RA.A.blob0_bytes);
  const uint8_t* sp = RA.A.blob0 + r.payload_off;
  uint32_t b = 0;
  if ((((uint32_t)(uintptr_t)d | (uint32_t)(uintptr_t)sp) & 15u) == 0)
    for (; b + 16 <= r.payload_len; b += 16) *reinterpret_cast<int4*>(d + b) = ld_stream4(sp + b);
  for (; b < r.payload_len; b++) d[b] = sp[b];
}

/* General path, phase 3, for the run [i, run_end): accept at every lane, coordinator work by team thread 0 against
 * memory (tally_reply), decision broadcast to the lanes by shuffles, commit at every lane. */
template <int L, int LP>
__device__ __forceinline__ void round_general(const DevState& S, const RoundArgs& RA, uint32_t i, uint32_t run_end,
                                              uint32_t sub, uint32_t tmask, uint32_t tbase, uint32_t gid,
                                              unsigned long long seg, unsigned long long dseg, unsigned long long payb,
                                              unsigned int* s_ctr) {
  const AcceptArgs& A = RA.A;
  const uint32_t n = RA.P.n;
  const uint32_t Wm = S.W - 1;
  const GroupCtx g = group_ctx(S, gid);
  for (uint32_t q = i; q < run_end;) {
    const int stq = RA.P.status[q];
    if (stq <= 0) break; /* refused / pre-active from here on (propose_run): no further ACCEPT in this run; the VOID
                          * outputs of request indices without an ACCEPT were written in phase 2 */
    const int4* rp = reinterpret_cast<const int4*>(&RA.P.accepts[q]);
    const int4 q0 = rp[0], q1 = rp[1], q2 = rp[2];
    const uint32_t q_next = q + max(1u, (uint32_t)q2.z); /* the next batch of the run starts behind this one's requests */
    const int slot = q0.y;
    uint32_t dstIdx = 0xffu;
    if (g.live)
      for (uint32_t m = 0; m < g.R; m++)
        if (g.ms->nodes[m] == q2.w) dstIdx = m;
    int cl2 = -1;
    if (g.live && dstIdx < g.R && g.ms->lane_of_idx[dstIdx] != 0xffu) cl2 = g.ms->lane_of_idx[dstIdx];
    LaneSt st;
    st.aux = 0;
    st.row = make_int4(0, 0, 0, 0);
    st.fl = 0;
    st.rwho = GPX_WHO(0xffu, 0xffu, GPX_F_VOID);
    st.rbn = st.rbc = st.rmaxcp = 0;
    if (sub < (uint32_t)L) {
      int4 e0 = make_int4(0, 0, 0, 0), e1 = e0;
      if (g.live) {
        const size_t ri = row_idx(S, sub, gid);
        st.aux = S.acc_aux[ri];
        st.row = S.acc_row[ri];
        ld256(&S.acc_win[2 * win_idx(S, sub, (uint32_t)slot & Wm, gid)], e0, e1);
      }
      const unsigned fr = (unsigned)(((payb + (uint32_t)q2.x) & (S.ring_cap - 1)) >> 4);
      accept_lane(S, A, sub, g.live, g.ms, dstIdx, q0, q1, q2, e0, e1, fr, st, s_ctr);
      write_accept_image(S, sub, seg, n, q, q0, q1, q2, st.img_flags);
      if (st.fl & LS_LOGGED) {
        const uint32_t off = (uint32_t)q2.x, plen = (uint32_t)q2.y;
        const uint8_t* src = blob_ptr(A, off);
        if (((off | (uint32_t)(uintptr_t)src) & 15u) == 0) {
          for (uint32_t b = 0; b < plen; b += 16) st_stream4(ring_ptr(S, sub, payb + off + b), ld_stream4(src + b));
        } else {
          for (uint32_t b = 0; b < plen; b++) *ring_ptr(S, sub, payb + off + b) = src[b];
        }
      }
    }
    uint32_t caux = 0;
    if (cl2 >= 0) caux = __shfl_sync(tmask, st.aux, tbase + (uint32_t)cl2);
    const bool tally_here = cl2 >= 0 && st_usable(caux);
    gpx_decision_rec d;
    d.gid = gid;
    d.slot = slot;
    d.bnum = 0;
    d.bcoord = 0;
    d.median_cp = 0;
    d.flags = GPX_F_VOID;
    d.dst_mask = 0;
    d.req_id = 0;
    int decided_i = 0;
    uint32_t omask = 0;
    int4 crow2 = make_int4(0, 0, 0, 0);
    bool cdirty = false;
    if (sub == 0 && tally_here) crow2 = S.coord_row[row_idx(S, (uint32_t)cl2, gid)];
#pragma unroll
    for (int l = 0; l < L; l++) {
      const uint32_t who = __shfl_sync(tmask, st.rwho, tbase + l);
      const int rb = __shfl_sync(tmask, st.rbn, tbase + l);
      const int rc = __shfl_sync(tmask, st.rbc, tbase + l);
      const int mcp = __shfl_sync(tmask, st.rmaxcp, tbase + l);
      if (GPX_WHO_FLAGS(who) & GPX_F_VOID) continue;
      if (!tally_here) {
        omask |= 1u << l;
        if (sub == (uint32_t)l)
          st256_stream(&A.replies[(size_t)q * L + l], make_int4((int)gid, slot, rb, rc),
                       make_int4(mcp, (int)who, q1.z, q1.w));
        continue;
      }
      if (sub == 0) {
        gpx_decision_rec dd;
        if (tally_reply(S, (uint32_t)cl2, gid, g.R, g.ms, crow2, cdirty, slot, rb, rc, mcp, GPX_WHO_ACC(who), dd,
                        s_ctr) &&
            !decided_i) {
          d = dd;
          decided_i = 1;
        }
      }
    }
    if (sub == 0) {
      if (cdirty) S.coord_row[row_idx(S, (uint32_t)cl2, gid)] = crow2;
      const int4* sp = reinterpret_cast<const int4*>(&d);
      st256_stream(&A.decisions[q], sp[0], sp[1]);
      A.out_mask[q] = (uint8_t)omask;
    }
    /* broadcast the decision of thread 0 to the lanes */
    decided_i = __shfl_sync(tmask, decided_i, tbase);
    {
      int4* dp = reinterpret_cast<int4*>(&d);
      dp[0].z = __shfl_sync(tmask, dp[0].z, tbase);
      dp[0].w = __shfl_sync(tmask, dp[0].w, tbase);
      dp[1].x = __shfl_sync(tmask, dp[1].x, tbase);
      dp[1].y = __shfl_sync(tmask, dp[1].y, tbase);
      dp[1].z = __shfl_sync(tmask, dp[1].z, tbase);
      dp[1].w = __shfl_sync(tmask, dp[1].w, tbase);
    }
    if (sub < (uint32_t)L)
      commit_team_lane<L>(S, A, sub, gid, slot, g.live, decided_i != 0, d, q0, q1, q2, st, q, dseg, s_ctr);
    if (RA.sum) { /* compact mode: the general path reports through the extra queue */
      if (sub < (uint32_t)L) {
        const gpx_exec_rec er = A.exec[(size_t)q * L + sub];
        if (!(er.flags & GPX_F_VOID) && A.n_extra) {
          const uint32_t k = atomicAdd(A.n_extra, 1u);
          if (k < A.extra_cap) store_exec(A.extra + k, er);
        }
      }
      if (sub == 0) store_sum(&RA.sum[q], stq, 0, 0, 0);
    }
    __syncwarp(tmask); /* the next ACCEPT of the run sees this one's coordinator/acceptor writes */
    q = q_next;
  }
}

template <int L, int LP>
__global__ void k_round_slow(const __grid_constant__ DevState S, const __grid_constant__ RoundArgs RA);

/*
 * The fast kernel.  The whole body is straight-line, predicated code: every shuffle and vote is a full-warp
 * operation outside divergent control flow (no per-team reconvergence bookkeeping), loads are issued in three
 * dependent levels (request -> rows of the group -> window entry / nodeSlotNumbers), and a team either takes
 * the in-order fast path or hands its request index to k_round_slow -- which the first such team launches from the
 * device as a tail launch, so that a round without left-over runs is ONE launch on the stream.  The ring heads are
 * published by block 0 into the other copy of log_pos (see DevState): warps retire right after their last store, no
 * fence, no arrival count.
 */
template <int L, int LP, bool DEF>
__global__ void __launch_bounds__(GPX_RBLOCK, GPX_ROUND_MINB * (256 / GPX_RBLOCK)) k_round(const __grid_constant__ DevState S,
                                                                     const __grid_constant__ RoundArgs RA) {
  static_assert(LP == L, "teams are exactly the L lanes of a group");
  /* DEF: the engine runs the reference's default configuration (ENABLE_JOURNALING, GC_MAJORITY_EXECUTED, LOG_META_DECISIONS
   * on, CPI_NOISE 0) -- the flags are compile-time constants and their branches fold away */
  const bool cf_journaling = DEF ? true : (S.journaling != 0);
  const bool cf_gcme = DEF ? true : (S.gc_majority_executed != 0);
  const bool cf_logmeta = DEF ? true : (S.log_meta != 0);
  const bool cf_cpi_pg = DEF ? false : (S.cpi_per_group != 0);
  constexpr uint32_t FULL = 0xffffffffu;
  constexpr uint32_t TPB = (GPX_RBLOCK / 32u) * (32u / LP); /* teams (= requests) per block */
  __shared__ unsigned int s_ctr[C_NCTR];
  /* the block's tile of the request batch (+ one neighbour on each side for the run tests) is staged in shared
   * memory by ONE TMA bulk copy */
  __shared__ __align__(128) gpx_request_rec s_req[TPB + 2];
  __shared__ __align__(8) unsigned long long s_bar;
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  if (threadIdx.x == 0) mbar_init(&s_bar, 1);
  __syncthreads();
  const AcceptArgs& A = RA.A;
  const gpx_request_rec* reqs = RA.P.reqs;
  const uint32_t n = RA.P.n;
  const uint32_t r0 = blockIdx.x * TPB; /* first request of the block; records [t0, t1) are staged */
  const uint32_t t0 = r0 ? r0 - 1u : 0u, t1 = min(n, r0 + TPB + 1u);
  const uint32_t tile_bytes = t1 > t0 ? (t1 - t0) * (uint32_t)sizeof(gpx_request_rec) : 0u;
  if (threadIdx.x == 0 && tile_bytes) tma_load_1d(s_req, &reqs[t0], tile_bytes, &s_bar);
  /* teams of L adjacent lanes; 32/L teams per warp (the 32 mod L last lanes of a warp idle) */
  const uint32_t lane_id = threadIdx.x & 31u;
  constexpr uint32_t TPW = 32u / LP;
  const uint32_t team_in_warp = lane_id / LP;
  const uint32_t sub = lane_id - team_in_warp * LP;
  const uint32_t tbase = team_in_warp * LP;
  constexpr uint32_t TEAM = (1u << LP) - 1u;
  const uint32_t i = team_in_warp < TPW ? (blockIdx.x * (GPX_RBLOCK / 32u) + (threadIdx.x >> 5)) * TPW + team_in_warp
                                        : 0xffffffffu;
  const uint32_t G = S.G, Wm = S.W - 1;
  /* per-lane log segments of this launch: [ACCEPT seg (n images + payload area)][DECISION seg] */
  const unsigned long long pay_bytes = RA.pay_bytes, res_a = RA.res_a, res_d = RA.res_d;
  const uint32_t pay_rel = RA.pay_rel;
  /* my lane's log position is read from the copy this launch owns (DevState.lp); block 0 writes the next launch's
   * position into the other copy and leaves the segment bases for k_round_slow -- the round needs neither a ticket
   * nor a fence nor a trailing kernel to finish */
  const unsigned long long seg = seg_base(S, sub, res_a + res_d);
  if (blockIdx.x == 0 && threadIdx.x < (uint32_t)L) { /* thread l writes lane l's two segment headers */
    const uint32_t t = threadIdx.x;
    const unsigned long long sq = seg_seq_of(S, t);
    write_seg_hdr(S, t, seg, GPX_F_ACCEPT, n, n, pay_bytes, 48, sq);
    write_seg_hdr(S, t, seg + res_a, GPX_F_DECISION, n, n, 0, 32, sq + 1ull);
    log_publish(S, t, seg + res_a + res_d, sq + 2ull);
    S.cur_seg[t] = seg;
    if (t == 0) {
      atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
      if (RA.ctl_zero) { /* the control block the next round counts into */
        int4* z = reinterpret_cast<int4*>(RA.ctl_zero);
        z[0] = make_int4(0, 0, 0, 0);
        z[1] = make_int4(0, 0, 0, 0);
      }
    }
  }

  /* ---- level A: the request record and the neighbours' gids (run-head / single-request tests) ---- */
  const bool valid = i < n;
  int4 rq0 = make_int4(0, 0, 0, 0), rq1 = rq0;
  uint32_t gprev = 0xffffffffu, gnext = 0xffffffffu;
  if (tile_bytes) mbar_wait(&s_bar, 0);
  if (valid) {
    const int4* rp = reinterpret_cast<const int4*>(&s_req[i - t0]);
    rq0 = rp[0];
    rq1 = rp[1];
    if (i > 0) gprev = s_req[i - t0 - 1].gid;
    if (i + 1 < n) gnext = s_req[i - t0 + 1].gid;
  }
  const uint32_t gid = (uint32_t)rq0.x, rflags = (uint32_t)rq0.y, entry = (rflags >> 8) & 0xfu;
  const uint32_t poff = (uint32_t)rq1.x, plen = (uint32_t)rq1.y;
  const bool head = valid && (i == 0 || gprev != gid);
  /* candidates for the in-order path: the only request of its group in this batch, no STOP */
  const bool cand = head && gnext != gid && gid < G && entry < (uint32_t)L && !(rflags & GPX_F_STOP);

  /* ---- level B (depends on gid only): group meta, my lane's acceptor + coordinator rows; the first chunk of
   * the payload rides along ---- */
  uint32_t meta = 0, my_aux = 0, my_dirty = 1;
  int ns_all[L];
#pragma unroll
  for (int c = 0; c < L; c++) ns_all[c] = 0;
  int4 my_row = make_int4(0, 0, 0, 0), my_crow = my_row, pv = my_row;
  const uint32_t ri = sub * G + gid; /* 32-bit plane indices: checked against 2^32 at engine creation */
  const uint8_t* const psrc = A.blob0 + poff;
  const bool pal = ((poff | (uint32_t)(uintptr_t)A.blob0) & 15u) == 0;
  if (cand) {
    meta = S.grp_meta[gid];
    my_aux = S.acc_aux[ri];
    my_row = S.acc_row[ri];
    my_crow = S.coord_row[ri];
    if (cf_journaling) my_dirty = S.acc_dirty[ri]; /* 0: no accept was ever stored here -> skip the window read */
#pragma unroll
    for (int c = 0; c < L; c++) /* nodeSlotNumbers[c][sub] of every lane that may turn out to coordinate: 4 B each, */
      ns_all[c] = S.node_slots[((uint32_t)c * S.Rcap + sub) * G + gid]; /* saves a whole dependent load level   */
    if (plen) {
      if (pal)
        pv = ld_stream4(psrc);
      else
        pv.x = psrc[0];
    }
  }
  /* a live group whose R members are exactly the L local lanes in member order */
  bool sf = cand && ((meta & (GPX_META_LIVE | GPX_META_IDENT)) == (GPX_META_LIVE | GPX_META_IDENT)) &&
            ((meta >> 16) & 0xffu) == (uint32_t)L;
  /* PISM.handleProposal :818-888: who coordinates?  the entry lane's rows come from its thread */
  const uint32_t esrc = tbase + entry;
  const int ae_y = __shfl_sync(FULL, my_row.y, esrc), ae_z = __shfl_sync(FULL, my_row.z, esrc);
  const int ce_x = __shfl_sync(FULL, my_crow.x, esrc), ce_y = __shfl_sync(FULL, my_crow.y, esrc);
  const int ce_w = __shfl_sync(FULL, my_crow.w, esrc);
  uint32_t cl = entry;
  if (!(((unsigned)ce_w & GPX_CF_EXISTS) && bcmp(ce_x, ce_y, ae_y, ae_z) >= 0)) {
    int fl = -1; /* forward to the coordinator of the entry lane's ballot, if it is a local lane */
#pragma unroll
    for (int l = 0; l < L; l++)
      if (S.lane_node[l] == ae_z) fl = l;
    sf = sf && fl >= 0 && fl != (int)entry;
    cl = fl >= 0 ? (uint32_t)fl : 0u;
  }
  const uint32_t csrc = tbase + cl;
  int4 crow;
  crow.x = __shfl_sync(FULL, my_crow.x, csrc);
  crow.y = __shfl_sync(FULL, my_crow.y, csrc);
  crow.z = __shfl_sync(FULL, my_crow.z, csrc);
  crow.w = __shfl_sync(FULL, my_crow.w, csrc);
  const int af_y = __shfl_sync(FULL, my_row.y, csrc), af_z = __shfl_sync(FULL, my_row.z, csrc);
  /* an ACTIVE coordinator whose ballot is not behind its acceptor, with no proposal outstanding; my lane must be
   * the plain in-order case: usable, same ballot, expecting exactly this slot, nothing committed there yet */
  const int slot = crow.z;
  sf = sf && ((unsigned)crow.w == (GPX_CF_EXISTS | GPX_CF_ACTIVE)) && bcmp(crow.x, crow.y, af_y, af_z) >= 0 &&
       st_usable(my_aux) && my_row.y == crow.x && my_row.z == crow.y && my_row.x == slot &&
       GPX_AUX_PRESENT(my_aux) == 0u && jsub(slot, my_row.w) > 0; /* no commit queued anywhere in the window: the
                                                                     * execution below is the only one (no EEC loop) */
  sf = ((__ballot_sync(FULL, sf) >> tbase) & TEAM) == TEAM;

  /* ---- level C (depends on the slot / the coordinator lane): window entry, nodeSlotNumbers ---- */
  int4 e0 = make_int4(0, 0, 0, 0), e1 = e0;
  int my_ns = 0;
  const uint32_t wi = 2u * ((sub * S.W + ((uint32_t)slot & Wm)) * G + gid);
  const uint32_t ni = (cl * S.Rcap + sub) * G + gid;
  if (sf) {
    if (my_dirty) ld256(&S.acc_win[wi], e0, e1);
#pragma unroll
    for (int c = 0; c < L; c++)
      if (cl == (uint32_t)c) my_ns = ns_all[c];
  }
  { /* an accept already sitting at this slot -> general path */
    const bool ent_live = ((unsigned)e1.w & GPX_ENT_VALID) && jsub(e0.x, my_row.w) > 0 && e0.x == slot;
    sf = ((__ballot_sync(FULL, sf && !ent_live) >> tbase) & TEAM) == TEAM;
  }
  int ns[LP];
#pragma unroll
  for (int k = 0; k < LP; k++) ns[k] = __shfl_sync(FULL, my_ns, tbase + k);
  const int median = median_regs<LP>(ns, (uint32_t)L); /* AcceptPacket.medianCheckpointedSlot (initCommander) */
  /* handleAccept at my lane: ballot equal, slot next-in-line, no previous accept -> ack + log */
  int4 row = my_row;
  gc_step(row, median);   /* acceptAndUpdateBallot -> garbageCollectAccepted :320 */
  const int cpi = cf_cpi_pg ? (sf ? S.grp_cpi[gid] : 1) : S.cpi_const;
  int max_cp = row.x - 1; /* AcceptReplyPacket.maxCheckpointedSlot :1139-1143 */
  if (!cf_gcme) {
    int lcp = max_cp - max_cp % cpi;
    if (lcp < 0) {
      lcp = jsub(lcp, cpi);
      if (lcp > 0) lcp = 2147483647 - 2147483647 % cpi;
    }
    max_cp = lcp;
  }
  /* tally (handleAcceptReplyMyBallot :597-640): replies arrive in lane order, all for my ballot; the decision is
   * made by reply number L/2 (0-based) with the nodeSlots recorded up to and including it */
  int nsd[LP], mine = my_ns;
#pragma unroll
  for (int k = 0; k < LP; k++) {
    const int mcp_k = __shfl_sync(FULL, max_cp, tbase + k);
    nsd[k] = ns[k];
    if (ns[k] < mcp_k) { /* recordSlotNumber :809-825 (plain <) */
      if (k <= L / 2) nsd[k] = mcp_k;
      if (sub == (uint32_t)k) mine = mcp_k;
    }
  }
  const int dmed = median_regs<LP>(nsd, (uint32_t)L); /* makeDecision(getMajorityCommittedSlot()) :630 */

  uint32_t c_lane = 0, c_team = 0, c_ckpt = 0; /* fast-path event counts, reduced once per warp at the end */
  if (sf) {
    /* ================= in-order fast path: nothing but the durable outputs touches HBM ================= */
    const int4 q0 = make_int4((int)gid, slot, crow.x, crow.y);
    /* my lane's two log segments are linear inside the ring (a launch never straddles the wrap) */
    uint8_t* const seg_p = ring_ptr(S, sub, seg);
    const unsigned frame_ref = (unsigned)(((seg + pay_rel + poff) & (S.ring_cap - 1)) >> 4);
    /* ACCEPT log image + my lane's copy of the blob (AbstractPaxosLogger.logAndMessage) */
    st256_stream(seg_p + 64 + (size_t)i * 32, q0,
                 make_int4(median, (int)(GPX_F_ACCEPT | ((1u << sub) << 16)), rq0.z, rq0.w));
    st_stream4(seg_p + 64 + (size_t)n * 32 + (size_t)i * 16, make_int4((int)poff, (int)plen, 1, crow.y));
    if (plen) {
      uint8_t* dst = seg_p + pay_rel + poff;
      if (pal) {
        st_stream4(dst, pv); /* the rest of a longer body is copied at the very end of the kernel (few live registers) */
      } else {
        dst[0] = (uint8_t)pv.x;
#pragma unroll 1
        for (uint32_t b = 1; b < plen; b++) dst[b] = psrc[b];
      }
    }
    /* commit (handleBatchedCommit :1488-1501 + extractExecuteAndCheckpoint): the accept is the decision */
    const bool metaf = cf_logmeta;
    st256_stream(seg_p + res_a + 64 + (size_t)i * 32, q0,
                 make_int4(metaf ? -1 : dmed, (int)((GPX_F_DECISION | (metaf ? GPX_F_META : 0u)) | ((1u << sub) << 16)),
                           rq0.z, rq0.w));
    gc_step(row, dmed);
    { /* EXEC record (PISM.execute hands the request to the app); shouldCheckpoint :2037-2041 */
      const bool ckpt = (slot % cpi) == 0;
      if (ckpt) c_ckpt++;
      gpx_exec_rec er;
      er.gid = gid;
      er.slot = slot;
      er.req_id = ((long long)rq0.w << 32) | (unsigned)rq0.z;
      er.payload_off = frame_ref;
      er.flags = (ckpt ? GPX_F_CKPT : 0u) | (sub << 12) | (1u << 16);
      if (!RA.sum) store_exec(&A.exec[(size_t)i * L + sub], er);
    }
    row.x = (int)((unsigned)row.x + 1u); /* executed(): _slot++ */
    if (cf_journaling) { /* acceptedProposals.remove(slot): only written to hide a valid occupant */
      if ((unsigned)e1.w & GPX_ENT_VALID)
        st256(&S.acc_win[wi], make_int4(slot, crow.x, crow.y, (int)frame_ref), /* VALID cleared: acc_dirty untouched */
              make_int4(rq0.z, rq0.w, (int)plen, (int)(1u << 16)));
    } else
      st256(&S.acc_win[wi], make_int4(slot, crow.x, crow.y, (int)frame_ref), /* not journaling: acc_dirty unused */
            make_int4(rq0.z, rq0.w, (int)plen, (int)(GPX_ENT_VALID | (1u << 16))));
    gc_step(row, dmed); /* second EEC iteration: GC with the advanced slot; nothing is queued (checked above) */
    S.acc_row[ri] = row;
    if (mine != my_ns) S.node_slots[ni] = mine; /* nodeSlotNumbers[cl][sub] */
    c_lane = 1;
    if (sub == 0) {
      constexpr uint32_t lane_mask = (1u << L) - 1u;
      if (RA.sum) /* every lane executed request i at `slot`, in order */
        store_sum(&RA.sum[i], slot, lane_mask, (slot % cpi) == 0 ? GPX_F_CKPT : 0u, 1u);
      else
        RA.P.status[i] = slot;
      crow.z = (int)((unsigned)crow.z + 1u); /* PCS.propose: nextProposalSlotNumber++ (proposal decided at once) */
      S.coord_row[cl * G + gid] = crow;
      /* the DECISION record and the reply out-mask are not written: every member is a local lane (IDENT), the
       * decision was committed above and gpx_round hands neither to the caller */
      c_team = 1;
    }
  } else if (head && sub == 0) {
    const uint32_t k = atomicAdd(RA.n_todo, 1u);
    RA.todo[k] = i; /* the run goes to k_round_slow */
    if (k == 0 && RA.tail_launch) /* the first left-over run of the round brings the second kernel in */
      k_round_slow<L, LP><<<RA.slow_grid, GPX_BLOCK, 0, cudaStreamTailLaunch>>>(S, RA);
  }
  if (valid && sub == 0) RA.mark[i] = sf ? 0 : 1;
  if (sf && pal && plen > 16u) { /* bodies longer than one chunk: four independent 128-bit loads in flight */
    uint8_t* const dst = ring_ptr(S, sub, seg) + pay_rel + poff;
    uint32_t b = 16;
#pragma unroll 1
    for (; b + 64 <= plen; b += 64) {
      const int4 a0 = ld_stream4(psrc + b), a1 = ld_stream4(psrc + b + 16), a2 = ld_stream4(psrc + b + 32),
                 a3 = ld_stream4(psrc + b + 48);
      st_stream4(dst + b, a0);
      st_stream4(dst + b + 16, a1);
      st_stream4(dst + b + 32, a2);
      st_stream4(dst + b + 48, a3);
    }
#pragma unroll 1
    for (; b < plen; b += 16) st_stream4(dst + b, ld_stream4(psrc + b));
  }
  /* fast-path events, counted in registers: one shared-memory update per warp */
  {
    const uint32_t nl = __reduce_add_sync(FULL, c_lane), nt = __reduce_add_sync(FULL, c_team);
    const uint32_t nc = __reduce_add_sync(FULL, c_ckpt);
    if (lane_id == 0 && (nl | nt)) { /* aggregates, expanded by gpx_get_counters */
      atomicAdd(&s_ctr[C_FAST_LANES], nl);
      atomicAdd(&s_ctr[C_FAST_TEAMS], nt);
      if (nc) atomicAdd(&s_ctr[C_FAST_CKPT], nc);
    }
  }
  flush_counters(S, s_ctr);
}

/* grid-wide barrier of a grid whose blocks are all resident (k_round_slow: at most 2 blocks per SM, launched behind
 * k_round): bar[0] counts arrivals, bar[1] is the generation */
__device__ __forceinline__ void grid_barrier(unsigned int* bar, unsigned int nblocks) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int gen = atomicAdd(&bar[1], 0u);
    if (atomicAdd(&bar[0], 1u) == nblocks - 1u) {
      bar[0] = 0u;
      __threadfence();
      atomicAdd(&bar[1], 1u);
    } else {
      while (atomicAdd(&bar[1], 0u) == gen) __nanosleep(100);
    }
    __threadfence();
  }
  __syncthreads();
}

/* The runs the fast kernel did not take (several requests of a group, STOPs, NACKs, coordinator changes, ...).
 * A fixed, small grid loops over the todo list in three phases separated by grid barriers:
 *   1  RequestBatcher + PCS.propose, one thread per run (propose_run)
 *   2  one thread per REQUEST of those runs (k_round marked them): its entry + body in the blob of a batched slot
 *      (RequestBatcher.java:198-219 packs up to MAX_BATCH_SIZE requests into one slot) and the VOID outputs of the
 *      request indices that carry no ACCEPT
 *   3  accept x L, tally, commit x L per ACCEPT of the run, one team of L threads per run
 * With an empty list the launch costs a few microseconds. */
template <int L, int LP>
__global__ void __launch_bounds__(GPX_BLOCK, 2) k_round_slow(const __grid_constant__ DevState S,
                                                             const __grid_constant__ RoundArgs RA) {
  __shared__ unsigned int s_ctr[C_NCTR];
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  __syncthreads();
  /* launched with programmatic stream serialization: the launch overlaps k_round's tail; wait for k_round's
   * completion (and memory flush) before looking at anything it wrote */
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const uint32_t ntodo = *RA.n_todo;
  if (ntodo == 0) return; /* host-launched form: nothing was left over */
  const AcceptArgs& A = RA.A;
  const uint32_t n = RA.P.n;
  const uint32_t lane_id = threadIdx.x & 31u;
  const unsigned long long pay_rel = RA.pay_rel, res_a = RA.res_a, res_d = RA.res_d;
  /* ---- phase 1: propose, one thread per run ---- */
  for (uint32_t k = blockIdx.x * GPX_BLOCK + threadIdx.x; k < ntodo; k += gridDim.x * GPX_BLOCK) {
    const uint32_t i = RA.todo[k];
    RA.todo_end[k] = round_propose(S, RA, i, RA.P.reqs[i].gid, s_ctr);
  }
  grid_barrier(&S.tickets[6], gridDim.x);
  /* ---- phase 2: one thread per REQUEST of the left-over runs ---- */
  {
    unsigned long long segl[L];
#pragma unroll
    for (int l = 0; l < L; l++) segl[l] = S.cur_seg[l]; /* k_round has moved the ring heads on already */
    for (uint32_t q = blockIdx.x * GPX_BLOCK + threadIdx.x; q < n; q += gridDim.x * GPX_BLOCK) {
      if (!RA.mark[q]) continue;
      const int st = RA.P.status[q];
      round_build_blob(RA, q, st);
      if (st > 0) continue;
      const uint32_t gid = RA.P.reqs[q].gid;
      const int4 z0 = make_int4((int)gid, 0, 0, 0), z1 = make_int4(0, (int)GPX_F_VOID, 0, 0);
#pragma unroll
      for (int l = 0; l < L; l++) {
        write_accept_image(S, l, segl[l], n, q, z0, z1, make_int4(0, 0, 0, 0), GPX_F_VOID);
        st256_stream(ring_ptr(S, l, segl[l] + res_a + 64 + (unsigned long long)q * 32), z0, z1);
        store_void_exec(&A.exec[(size_t)q * L + l], gid, 0, l);
      }
      st256_stream(&A.decisions[q], z0, z1);
      A.out_mask[q] = 0;
      if (RA.sum) store_sum(&RA.sum[q], st, 0, 0, 0);
    }
  }
  grid_barrier(&S.tickets[6], gridDim.x);
  /* ---- phase 3: one team per run ---- */
  {
    constexpr uint32_t TPW = 32u / LP;
    const uint32_t team_in_warp = lane_id / LP;
    const uint32_t sub = lane_id - team_in_warp * LP;
    const uint32_t tbase = team_in_warp * LP;
    const uint32_t tmask = ((1u << LP) - 1u) << tbase;
    const uint32_t nteams = gridDim.x * (GPX_BLOCK / 32u) * TPW;
    const uint32_t team = team_in_warp < TPW ? (blockIdx.x * (GPX_BLOCK / 32u) + (threadIdx.x >> 5)) * TPW + team_in_warp
                                             : 0xffffffffu;
    const uint32_t myl = sub < (uint32_t)L ? sub : 0u;
    const unsigned long long seg = S.cur_seg[myl]; /* same segments as the fast kernel */
    const unsigned long long payb = seg + pay_rel, dseg = seg + res_a;
    for (uint32_t k = team; k < ntodo; k += nteams) {
      const uint32_t i = RA.todo[k];
      round_general<L, LP>(S, RA, i, RA.todo_end[k], sub, tmask, tbase, RA.P.reqs[i].gid, seg, dseg, payb, s_ctr);
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  flush_counters(S, s_ctr);
}
