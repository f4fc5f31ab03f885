/*
 * gpx_spread.cuh -- the device side of SPREAD placement: the replicas of a group live in different engines
 * (one single-lane engine = one node = one GPU) and the three inter-replica packet types of a round travel
 * between them (SURVEY.md 8e; PISM.roundRobinCoordinator :2251-2256 places the coordinator,
 * paxosutil/PaxosMessenger.java:175-182 / PaxosManager.send :2098-2128 unicast the packets,
 * PaxosPacketBatcher.java:270-303 groups them per destination).
 *
 * Everything is sized and addressed so that NO count ever has to be read by a host:
 *
 *   bucket (s -> d, kind)  = [64-B header {count, blob_units}][cap(s,d) fixed-size records][blob area (ACCEPT only)]
 *
 * cap(s,d) is agreed when the spread group is created (gpx_spread_config.cap), so every transfer has a size both
 * ends know; the number of records actually in a bucket travels in-band in its header.  A round is
 *
 *   k_propose (+k_build_blobs)                      RequestBatcher + PCS.propose at the coordinator
 *   k_sp_route     ACCEPTs -> one bucket per member node (+ per-destination blob), remembers for every ACCEPT i and
 *                  member m the position pos[i][m] it took in that member's bucket
 *   == exchange ACCEPT buckets ==                   grouped ncclSend / ncclRecv (or device copies, local mode)
 *   k_sp_accept    PISM.handleAccept over the N received buckets in ONE launch (virtual index space: bucket s owns
 *                  [vbase[s], vbase[s] + cap)); the reply to the record at position j of the bucket from s is
 *                  written at position j of the reply bucket to s -- replies need no routing pass
 *   == exchange ACCEPT_REPLY buckets ==
 *   k_sp_tally     one thread per run of MY ACCEPTs gathers the R replies of every slot through pos[i][m]
 *                  (handleAcceptReply in member order, one read-modify-write of the coordinator row per run) and
 *                  writes the DECISION (or a VOID hole) at the SAME positions of the DECISION buckets
 *   == exchange DECISION buckets ==
 *   k_sp_commit    PISM.handleBatchedCommit + extractExecuteAndCheckpoint over the N received buckets; EXEC
 *                  records at the virtual index of the DECISION
 *
 * The loop-back bucket (s == d) is the same memory on both sides: nothing is copied for a node's own replica.
 */
#pragma once
#include "gpx_kernels.cuh"

#define GPX_SP_ND 8           /* nodes of a spread group (GPUs of one box) */
#define GPX_SP_NONE 0xffffffffu
#define GPX_SP_POS_BITS 28    /* pos[i][m] = dest << 28 | position */

struct SpHdr { /* 64 B, travels in front of every bucket */
  uint32_t count;      /* records in the bucket (ACCEPT: reserved by k_sp_route; REPLY / DECISION: mirrors it) */
  uint32_t blob_units; /* ACCEPT: blob bytes / 16 used */
  uint32_t pad[14];
};

struct SpBucket {
  uint8_t* base;               /* SpHdr, then the records, then (ACCEPT) the blob area */
  uint32_t cap;                /* record slots; 0 = this pair never exchanges */
  uint32_t vbase;              /* first virtual index of the bucket in the receiver's index space (256-aligned) */
  unsigned long long blob_off; /* ACCEPT: where this bucket's blob area starts in the receiver's log payload area */
};
__device__ __forceinline__ SpHdr* sp_hdr(const SpBucket& b) { return reinterpret_cast<SpHdr*>(b.base); }
__device__ __forceinline__ uint8_t* sp_recs(const SpBucket& b) { return b.base + 64; }
__device__ __forceinline__ uint8_t* sp_blob(const SpBucket& b) { return b.base + 64 + (size_t)b.cap * 48; }

struct SpArgs {
  uint32_t N, me;
  int32_t node_id[GPX_SP_ND];
  SpBucket sendA[GPX_SP_ND], recvA[GPX_SP_ND]; /* ACCEPT: me -> d, s -> me */
  SpBucket sendR[GPX_SP_ND], recvR[GPX_SP_ND]; /* ACCEPT_REPLY: me (acceptor) -> coordinator s; acceptor d -> me */
  SpBucket sendD[GPX_SP_ND], recvD[GPX_SP_ND]; /* DECISION: me -> d, s -> me */
  /* where k_sp_route counts the records of destination d: the header of the send bucket itself, or -- peer-memory
   * transport, where that header lives on another GPU -- a local scratch header that k_sp_signal copies over */
  SpHdr* cntA[GPX_SP_ND];
  uint32_t p2p;                     /* 1: send buckets ARE the peers' receive buckets (NVLink stores), see k_sp_signal */
  uint32_t* flags_local;            /* [3][GPX_SP_ND] round numbers signalled by the source nodes, per packet type */
  uint32_t* flags_peer[GPX_SP_ND];  /* node d's flags_local (mapped peer memory) */
  uint32_t* seq;                    /* [6] rounds signalled / awaited so far per packet type (device-resident: graph replay) */
  uint32_t vtotal;                  /* virtual record slots of the receive side (sum of 256-aligned caps) */
  unsigned long long blob_vtotal;   /* bytes of all received blob areas */
  uint32_t blob_per_rec;
  /* coordinator side */
  const gpx_accept_rec* accepts;    /* k_propose output, grouped by gid */
  const uint32_t* n_accepts;        /* device */
  uint32_t n_max;                   /* requests of the round (grid of the coordinator-side kernels) */
  const uint8_t* blob0;             /* request payload arena */
  unsigned long long blob0_bytes;
  const uint8_t* blob1;             /* constructed blobs of batched slots */
  uint32_t* pos;                    /* [n_max][Rcap] */
  uint32_t* dropped;                /* device counter: records that found no destination / no room */
  /* acceptor side */
  gpx_exec_rec* exec;               /* [vtotal] */
  gpx_exec_rec* extra;
  uint32_t extra_cap;
  uint32_t* n_extra;
};

__device__ __forceinline__ int sp_node_index(const SpArgs& A, int32_t node) {
  int d = -1;
#pragma unroll
  for (int k = 0; k < GPX_SP_ND; k++)
    if ((uint32_t)k < A.N && A.node_id[k] == node) d = k;
  return d;
}

/* ============================== k_sp_route (ACCEPTs out of the batcher) ============================== */
__global__ void __launch_bounds__(GPX_BLOCK) k_sp_route(const __grid_constant__ DevState S,
                                                        const __grid_constant__ SpArgs A) {
  __shared__ uint32_t s_cnt[GPX_SP_ND], s_units[GPX_SP_ND], s_base[GPX_SP_ND], s_ubase[GPX_SP_ND];
  if (threadIdx.x < GPX_SP_ND) s_cnt[threadIdx.x] = s_units[threadIdx.x] = 0;
  __syncthreads();
  uint32_t n = *A.n_accepts;
  if (n > A.n_max) n = A.n_max;
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  bool head = false;
  uint32_t gid = 0, run = 0, nrec = 0, nunits = 0, R = 0;
  const MsetInfo* ms = nullptr;
  uint32_t loc[GPX_SP_ND], uloc[GPX_SP_ND];
  int dest[GPX_SP_ND];
#pragma unroll
  for (int m = 0; m < GPX_SP_ND; m++) {
    loc[m] = uloc[m] = 0;
    dest[m] = -1;
  }
  if (i < n) {
    gid = A.accepts[i].h.gid;
    head = (i == 0) || (A.accepts[i - 1].h.gid != gid);
    if (head) {
      for (uint32_t j = i; j < n; j++) { /* pass 1: the run and what it carries */
        const int4* rp = reinterpret_cast<const int4*>(&A.accepts[j]);
        const int4 q0 = rp[0], q1 = rp[1];
        if ((uint32_t)q0.x != gid) break;
        run++;
        if ((uint32_t)q1.y & GPX_F_VOID) continue;
        nrec++;
        nunits += ((uint32_t)rp[2].y + 15u) >> 4;
      }
      bool ok = false;
      if (gid < S.G) {
        const uint32_t meta = S.grp_meta[gid];
        if (meta & GPX_META_LIVE) {
          ms = &S.msets[meta & 0xffffu];
          R = (meta >> 16) & 0xffu;
          ok = R <= GPX_SP_ND;
        }
      }
      if (!ok) {
        if (nrec && A.dropped) atomicAdd(A.dropped, nrec);
        nrec = 0;
        R = 0;
      }
      if (nrec)
#pragma unroll
        for (int m = 0; m < GPX_SP_ND; m++)
          if ((uint32_t)m < R) {
            const int d = sp_node_index(A, ms->nodes[m]);
            dest[m] = d;
            if (d < 0 || A.sendA[d].cap == 0) { /* member not served by this spread group */
              if (A.dropped) atomicAdd(A.dropped, nrec);
              dest[m] = -1;
            } else {
              loc[m] = atomicAdd(&s_cnt[d], nrec);
              uloc[m] = atomicAdd(&s_units[d], nunits);
            }
          }
    }
  }
  __syncthreads();
  if (threadIdx.x < GPX_SP_ND && threadIdx.x < A.N && s_cnt[threadIdx.x]) { /* one reservation per block + destination */
    SpHdr* h = A.cntA[threadIdx.x];
    s_base[threadIdx.x] = atomicAdd(&h->count, s_cnt[threadIdx.x]);
    s_ubase[threadIdx.x] = atomicAdd(&h->blob_units, s_units[threadIdx.x]);
  }
  __syncthreads();
  if (!head) return;
  const uint32_t Rcap = S.Rcap;
  uint32_t k = 0; /* non-VOID records of the run written so far */
  uint32_t ku = 0;
  for (uint32_t j = i; j < i + run; j++) {
    const int4* rp = reinterpret_cast<const int4*>(&A.accepts[j]);
    const int4 q0 = rp[0], q1 = rp[1], q2 = rp[2];
    const bool is_void = ((uint32_t)q1.y & GPX_F_VOID) != 0;
    const uint32_t plen = (uint32_t)q2.y, u = (plen + 15u) >> 4;
    const unsigned long long off = (uint32_t)q2.x;
    const uint8_t* src = off < A.blob0_bytes ? A.blob0 + off : A.blob1 + (off - A.blob0_bytes);
    const bool al = (((uint32_t)(uintptr_t)src) & 15u) == 0;
#pragma unroll
    for (int m = 0; m < GPX_SP_ND; m++) {
      if ((uint32_t)m >= Rcap) continue;
      uint32_t p = GPX_SP_NONE;
      const int d = dest[m];
      if (!is_void && d >= 0) {
        const SpBucket& b = A.sendA[d];
        const uint32_t pos = s_base[d] + loc[m] + k;
        const unsigned long long boff = ((unsigned long long)(s_ubase[d] + uloc[m] + ku)) << 4;
        if (pos >= b.cap || boff + ((unsigned long long)u << 4) > (unsigned long long)b.cap * A.blob_per_rec) {
          if (A.dropped) atomicAdd(A.dropped, 1u); /* the bucket is too small for this round */
        } else {
          int4* op = reinterpret_cast<int4*>(sp_recs(b) + (size_t)pos * 48);
          op[0] = q0;
          op[1] = q1;
          op[2] = make_int4((int)(uint32_t)boff, q2.y, q2.z, q2.w);
          uint8_t* dst = sp_blob(b) + boff; /* 16-byte aligned: whole chunks are stored, the tail zero-padded */
          uint32_t x = 0;
          if (al)
            for (; x + 16 <= plen; x += 16) st_stream4(dst + x, ld_stream4(src + x));
          for (; x < plen; x += 16) st_stream4(dst + x, load_chunk16(src + x, plen - x));
          p = ((uint32_t)d << GPX_SP_POS_BITS) | pos;
        }
      }
      A.pos[(size_t)j * Rcap + m] = p;
    }
    if (!is_void) {
      k++;
      ku += u;
    }
  }
}

/* which received bucket does the block that starts at virtual index v0 belong to (vbase is 256-aligned) */
__device__ __forceinline__ uint32_t sp_bucket_of(const SpBucket* rb, uint32_t N, uint32_t v0) {
  uint32_t s = 0;
#pragma unroll
  for (uint32_t k = 1; k < GPX_SP_ND; k++)
    if (k < N && rb[k].cap && rb[k].vbase <= v0) s = k;
  /* buckets with cap 0 share their successor's vbase: the loop keeps the last one with room, but bucket 0 may be
   * empty too */
  return s;
}

/* ============================== k_sp_accept ============================== */
/* PISM.handleAccept at this node's (single) lane for every record of the N received ACCEPT buckets. */
__global__ void __launch_bounds__(GPX_BLOCK, GPX_PHASE_MINB) k_sp_accept(const __grid_constant__ DevState S,
                                                                         const __grid_constant__ SpArgs A) {
  __shared__ unsigned int s_ctr[C_NCTR];
  __shared__ __align__(128) uint8_t s_tile[(GPX_BLOCK + 1) * sizeof(gpx_accept_rec)];
  __shared__ __align__(8) unsigned long long s_bar;
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  if (threadIdx.x == 0) mbar_init(&s_bar, 1);
  __syncthreads();
  const uint32_t v0 = blockIdx.x * GPX_BLOCK, v = v0 + threadIdx.x;
  const uint32_t s = sp_bucket_of(A.recvA, A.N, v0);
  const SpBucket& B = A.recvA[s];
  const uint32_t j0 = v0 - B.vbase;
  uint32_t cnt = B.cap ? sp_hdr(B)->count : 0u;
  if (cnt > B.cap) cnt = B.cap;
  const gpx_accept_rec* recs = reinterpret_cast<const gpx_accept_rec*>(sp_recs(B));
  /* stage the block's records (+ the predecessor for the run-head test) with one TMA bulk copy */
  const uint32_t t0 = j0 ? j0 - 1u : 0u, t1 = min(cnt, j0 + GPX_BLOCK);
  const uint32_t tile_bytes = (j0 < cnt && t1 > t0) ? (t1 - t0) * (uint32_t)sizeof(gpx_accept_rec) : 0u;
  if (threadIdx.x == 0 && tile_bytes) tma_load_1d(s_tile, &recs[t0], tile_bytes, &s_bar);
  const uint32_t Wm = S.W - 1;
  /* one ACCEPT segment per round: an image slot per virtual index, payload area = the received blob areas */
  const unsigned long long pay_rel = seg_pay_rel(A.vtotal);
  const unsigned long long reserved = seg_align32(pay_rel + A.blob_vtotal); /* = seg_accept_bytes(A.vtotal, blob_vtotal) */
  const unsigned long long segb = seg_base(S, 0, reserved);
  const unsigned long long payb = segb + pay_rel + B.blob_off;
  if (v == 0) {
    const unsigned long long sq = seg_seq_of(S, 0);
    write_seg_hdr(S, 0, segb, GPX_F_ACCEPT, A.vtotal, A.vtotal, A.blob_vtotal, 48, sq);
    log_publish(S, 0, segb + reserved, sq + 1ull);
    atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  }
  const uint32_t j = j0 + threadIdx.x;
  if (B.cap && j == 0) { /* the reply bucket back to s mirrors this one */
    SpHdr* h = sp_hdr(A.sendR[s]);
    h->count = cnt;
    h->blob_units = 0;
  }
  if (tile_bytes) mbar_wait(&s_bar, 0);
  AcceptArgs AA; /* what accept_lane needs */
  AA.extra = A.extra;
  AA.extra_cap = A.extra_cap;
  AA.n_extra = A.n_extra;
  if (v < A.vtotal && !(B.cap && j < cnt)) /* a hole of the virtual index space: VOID image */
    write_accept_image(S, 0, segb, A.vtotal, v, make_int4(0, 0, 0, 0), make_int4(0, 0, 0, 0), make_int4(0, 0, 0, 0),
                       GPX_F_VOID);
  if (B.cap && j < cnt) {
    const int4* rp = reinterpret_cast<const int4*>(s_tile + (size_t)(j - t0) * sizeof(gpx_accept_rec));
    int4 q0 = rp[0], q1 = rp[1], q2 = rp[2];
    const uint32_t gid = (uint32_t)q0.x;
    const bool head = (j == 0) || ((uint32_t)rp[-3].x != gid);
    if (head) {
      const GroupCtx g = group_ctx(S, gid);
      const uint32_t lanes = g.live ? g.ms->lane_mask : 0u; /* dst_mask is a per-engine notion: rewritten here */
      gpx_accept_reply_rec* replies = reinterpret_cast<gpx_accept_reply_rec*>(sp_recs(A.sendR[s]));
      uint32_t jj = j;
      while (true) {
        q1.y = (int)(((uint32_t)q1.y & 0xffffu) | (lanes << 16));
        const int slot = q0.y;
        const uint32_t payload_off = (uint32_t)q2.x;
        LaneSt st;
        int4 e0 = make_int4(0, 0, 0, 0), e1 = e0;
        st.aux = 0;
        st.row = make_int4(0, 0, 0, 0);
        if (g.live) {
          const size_t ri = row_idx(S, 0, gid);
          st.aux = S.acc_aux[ri];
          st.row = S.acc_row[ri];
          ld256(&S.acc_win[2 * win_idx(S, 0, (uint32_t)slot & Wm, gid)], e0, e1);
        }
        uint32_t dstIdx = 0xffu;
        if (g.live)
          for (uint32_t m = 0; m < g.R; m++)
            if (g.ms->nodes[m] == q2.w) dstIdx = m;
        const unsigned fr = (unsigned)(((payb + payload_off) & (S.ring_cap - 1)) >> 4);
        accept_lane(S, AA, 0, g.live, g.ms, dstIdx, q0, q1, q2, e0, e1, fr, st, s_ctr);
        if (g.live) {
          const size_t ri = row_idx(S, 0, gid);
          if (st.fl & LS_STORE) {
            int4 n0, n1;
            make_entry(q0, q1, q2, st.frame_ref, n0, n1);
            ST_ACC(S, 0, gid, 2 * win_idx(S, 0, (uint32_t)slot & Wm, gid), n0, n1);
          }
          if (st.fl & LS_ROWDIRTY) S.acc_row[ri] = st.row;
          if (st.fl & LS_AUXDIRTY) S.acc_aux[ri] = st.aux;
        }
        st256_stream(&replies[jj], make_int4((int)gid, slot, st.rbn, st.rbc),
                     (GPX_WHO_FLAGS(st.rwho) & GPX_F_VOID) ? make_int4(0, (int)st.rwho, 0, 0)
                                                           : make_int4(st.rmaxcp, (int)st.rwho, q1.z, q1.w));
        /* log image at the virtual index; payload_off of the image is relative to the segment's payload area */
        write_accept_image(S, 0, segb, A.vtotal, B.vbase + jj, q0, q1,
                           make_int4((int)(uint32_t)(B.blob_off + payload_off), q2.y, q2.z, q2.w), st.img_flags);
        if (st.fl & LS_LOGGED) {
          const uint32_t plen = (uint32_t)q2.y;
          const uint8_t* src = sp_blob(B) + payload_off;
          if (((payload_off | (uint32_t)(uintptr_t)src) & 15u) == 0) {
            for (uint32_t b = 0; b < plen; b += 16) st_stream4(ring_ptr(S, 0, payb + payload_off + b), ld_stream4(src + b));
          } else {
            for (uint32_t b = 0; b < plen; b++) *ring_ptr(S, 0, payb + payload_off + b) = src[b];
          }
        }
        jj++;
        if (jj >= cnt) break;
        rp = jj < t1 ? reinterpret_cast<const int4*>(s_tile + (size_t)(jj - t0) * sizeof(gpx_accept_rec))
                     : reinterpret_cast<const int4*>(&recs[jj]);
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

/* ============================== k_sp_tally ============================== */
/* PISM.handleBatchedAcceptReply / PaxosCoordinator.handleAcceptReply for every ACCEPT this node issued in the
 * round: the thread of the first ACCEPT of a group's run walks the run; per ACCEPT the replies of the members are
 * fetched from the reply buckets through pos[i][m] and handled in member order (the order in which a
 * coordinator that hosts all acceptors as lanes sees them).  The coordinator row is read and written once per
 * run.  The DECISION -- or a VOID hole when the slot is still undecided -- goes to the same position of every
 * member's DECISION bucket. */
__global__ void __launch_bounds__(GPX_BLOCK) k_sp_tally(const __grid_constant__ DevState S,
                                                        const __grid_constant__ SpArgs A) {
  __shared__ unsigned int s_ctr[C_NCTR];
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  __syncthreads();
  uint32_t n = *A.n_accepts;
  if (n > A.n_max) n = A.n_max;
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  if (i == 0) atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  if (blockIdx.x == 0 && threadIdx.x < A.N && A.sendD[threadIdx.x].cap) { /* DECISION buckets mirror the ACCEPT ones */
    SpHdr* h = sp_hdr(A.sendD[threadIdx.x]);
    uint32_t c = A.cntA[threadIdx.x]->count;
    if (c > A.sendA[threadIdx.x].cap) c = A.sendA[threadIdx.x].cap;
    h->count = c;
    h->blob_units = 0;
  }
  if (i < n) {
    const int4* rp = reinterpret_cast<const int4*>(&A.accepts[i]);
    int4 q0 = rp[0], q1 = rp[1];
    const uint32_t gid = (uint32_t)q0.x;
    const bool head = (i == 0) || (A.accepts[i - 1].h.gid != gid);
    if (head) {
      const GroupCtx g = group_ctx(S, gid);
      const uint32_t Rcap = S.Rcap;
      uint32_t aux = 0;
      const bool can = g.live && g.ms->idx_of_lane[0] != 0xffu && usable(S, gid, 0, &aux); /* PISM :456-460 */
      int4 crow = make_int4(0, 0, 0, 0);
      bool dirty = false;
      if (can) crow = S.coord_row[row_idx(S, 0, gid)];
      uint32_t j = i;
      while (true) {
        gpx_decision_rec d;
        d.gid = gid;
        d.slot = q0.y;
        d.bnum = d.bcoord = d.median_cp = 0;
        d.flags = GPX_F_VOID;
        d.dst_mask = 0;
        d.req_id = 0;
        bool decided = false;
        const bool is_void = ((uint32_t)q1.y & GPX_F_VOID) != 0;
        if (!is_void) { /* gather the R replies of the slot (member order), then tally them in registers */
          int4 r0[GPX_SP_ND], r1[GPX_SP_ND];
          uint32_t pp[GPX_SP_ND];
#pragma unroll
          for (int m = 0; m < GPX_SP_ND; m++) {
            pp[m] = (uint32_t)m < Rcap ? A.pos[(size_t)j * Rcap + m] : GPX_SP_NONE;
            r0[m] = make_int4(0, 0, 0, 0);
            r1[m] = make_int4(0, (int)GPX_WHO(0xffu, 0xffu, GPX_F_VOID), 0, 0);
            if (pp[m] != GPX_SP_NONE) {
              const SpBucket& rb = A.recvR[pp[m] >> GPX_SP_POS_BITS];
              ld256_stream(sp_recs(rb) + (size_t)(pp[m] & ((1u << GPX_SP_POS_BITS) - 1u)) * 32, r0[m], r1[m]);
              const uint32_t who = (uint32_t)r1[m].y;
              if (!(GPX_WHO_FLAGS(who) & GPX_F_VOID) &&
                  (!can || GPX_WHO_DST(who) >= g.R || g.ms->lane_of_idx[GPX_WHO_DST(who)] != 0)) {
                atomicAdd(&s_ctr[C_REPLIES_IGNORED], 1u); /* not addressed to a usable coordinator here */
                r1[m].y = (int)GPX_WHO(0xffu, 0xffu, GPX_F_VOID);
              }
            }
          }
          if (can && g.R <= 8u) {
            gpx_decision_rec dd;
            if (tally_slot_regs<GPX_SP_ND>(S, 0, gid, g.R, g.ms, crow, dirty, q0.y, r0, r1, (uint32_t)GPX_SP_ND, dd, s_ctr)) {
              d = dd;
              decided = true;
            }
          }
        }
        if (!is_void) {
          const int4* sp = reinterpret_cast<const int4*>(&d);
          for (uint32_t m = 0; m < Rcap && m < GPX_SP_ND; m++) {
            const uint32_t p = A.pos[(size_t)j * Rcap + m];
            if (p == GPX_SP_NONE) continue;
            const SpBucket& sb = A.sendD[p >> GPX_SP_POS_BITS];
            st256_stream(sp_recs(sb) + (size_t)(p & ((1u << GPX_SP_POS_BITS) - 1u)) * 32, sp[0], sp[1]);
          }
        }
        j++;
        if (j >= n) break;
        rp = reinterpret_cast<const int4*>(&A.accepts[j]);
        const int4 nx = rp[0];
        if ((uint32_t)nx.x != gid) break;
        q0 = nx;
        q1 = rp[1];
      }
      if (dirty) S.coord_row[row_idx(S, 0, gid)] = crow;
    }
  }
  flush_counters(S, s_ctr);
}

/* ============================== k_sp_commit ============================== */
/* PISM.handleBatchedCommit + extractExecuteAndCheckpoint at this node's lane for the N received DECISION buckets;
 * EXEC record and DECISION log image at the virtual index of the DECISION. */
__global__ void __launch_bounds__(GPX_BLOCK, GPX_PHASE_MINB) k_sp_commit(const __grid_constant__ DevState S,
                                                                         const __grid_constant__ SpArgs A) {
  __shared__ unsigned int s_ctr[C_NCTR];
  if (threadIdx.x < C_NCTR) s_ctr[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t v0 = blockIdx.x * GPX_BLOCK, v = v0 + threadIdx.x;
  const uint32_t s = sp_bucket_of(A.recvD, A.N, v0);
  const SpBucket& B = A.recvD[s];
  const uint32_t j = v - B.vbase;
  uint32_t cnt = B.cap ? sp_hdr(B)->count : 0u;
  if (cnt > B.cap) cnt = B.cap;
  const gpx_decision_rec* recs = reinterpret_cast<const gpx_decision_rec*>(sp_recs(B));
  const uint32_t Wm = S.W - 1;
  const unsigned long long reserved = seg_decision_bytes(A.vtotal);
  const unsigned long long segb = seg_base(S, 0, reserved);
  if (v == 0) {
    const unsigned long long sq = seg_seq_of(S, 0);
    write_seg_hdr(S, 0, segb, GPX_F_DECISION, A.vtotal, A.vtotal, 0, 32, sq);
    log_publish(S, 0, segb + reserved, sq + 1ull);
    atomicAdd(&s_ctr[C_KERNEL_LAUNCHES], 1u);
  }
  if (blockIdx.x == 0 && threadIdx.x < A.N && A.sendA[threadIdx.x].cap) { /* next round's k_sp_route counts from zero */
    SpHdr* h = A.cntA[threadIdx.x];
    h->count = 0;
    h->blob_units = 0;
  }
  const bool valid = B.cap && j < cnt;
  if (v < A.vtotal && !valid) { /* hole: VOID exec + VOID image */
    store_void_exec(&A.exec[v], 0, 0, 0);
    st256_stream(ring_ptr(S, 0, segb + 64 + (unsigned long long)v * 32), make_int4(0, 0, 0, 0),
                 make_int4(0, (int)GPX_F_VOID, 0, 0));
  }
  if (valid) {
    int4 q0, q1;
    ld256_stream(&recs[j], q0, q1);
    const uint32_t gid = (uint32_t)q0.x;
    const bool head = (j == 0) || (recs[j - 1].gid != gid);
    if (head) {
      const GroupCtx g = group_ctx(S, gid);
      const uint32_t lanes = g.live ? g.ms->lane_mask : 0u;
      uint32_t jj = j;
      while (true) {
        const int slot = q0.y;
        const uint32_t rflags = (uint32_t)q1.y & 0xffffu;
        const uint32_t vv = B.vbase + jj;
        gpx_exec_rec* ex = &A.exec[vv];
        store_void_exec(ex, gid, slot, 0);
        int4 img0 = q0, img1 = make_int4(q1.x, (int)(GPX_F_VOID | (lanes << 16)), q1.z, q1.w);
        if ((lanes & 1u) && !(rflags & GPX_F_VOID)) {
          const size_t ri = row_idx(S, 0, gid);
          uint32_t aux = S.acc_aux[ri];
          if (!st_usable(aux)) {
            atomicAdd(&s_ctr[C_DECISIONS_DROPPED], 1u);
          } else {
            int4 row = S.acc_row[ri], e0, e1;
            ld256(&S.acc_win[2 * win_idx(S, 0, (uint32_t)slot & Wm, gid)], e0, e1);
            const int4 row_in = row;
            const uint32_t aux_in = aux;
            commit_lane(S, 0, gid, slot, q0.z, q0.w, q1.x, row, aux, e0, e1, ex, A.extra, A.extra_cap, A.n_extra, img0,
                        img1, s_ctr);
            if (aux != aux_in) S.acc_aux[ri] = aux;
            if (row.x != row_in.x || row.y != row_in.y || row.z != row_in.z || row.w != row_in.w) S.acc_row[ri] = row;
          }
        }
        st256_stream(ring_ptr(S, 0, segb + 64 + (unsigned long long)vv * 32), img0, img1);
        jj++;
        if (jj >= cnt) break;
        int4 t0, t1;
        ld256_stream(&recs[jj], t0, t1);
        if ((uint32_t)t0.x != gid) break;
        q0 = t0;
        q1 = t1;
      }
    }
  }
  flush_counters(S, s_ctr);
}

/* ============================== peer-memory transport: k_sp_signal / k_sp_wait ============================== */
/* With GPX_SPREAD_P2P the send buckets of a node ARE the receive buckets of its peers (mapped peer memory: CUDA IPC
 * between the per-GPU processes, plain pointers between engines of one process): k_sp_route / k_sp_accept / k_sp_tally
 * store records, blobs, replies and decisions straight into the destination GPU over NVLink, and the "exchange" that
 * remains is a flag.  k_sp_signal runs behind the producing kernel (whose stores are complete and visible system-wide
 * when it has finished): it copies the ACCEPT counts into the peers' bucket headers, fences, and writes this round's
 * number into flag [kind][me] of every peer it sends to.  k_sp_wait runs in front of the consuming kernel and spins
 * until every source it receives from has signalled this round.  The round numbers live in device memory, so a
 * captured round replays unchanged.  Re-use of a bucket is safe without credits: a node writes the ACCEPT bucket of
 * round r+1 only after its tally of round r, i.e. after the peer's replies of round r, which the peer sent after it
 * had consumed the ACCEPT bucket of round r (and likewise for the other two kinds). */
__global__ void k_sp_signal(const __grid_constant__ SpArgs A, uint32_t kind) {
  const uint32_t t = threadIdx.x;
  const uint32_t round = A.seq[kind] + 1u;
  bool to = false;
  if (t < A.N) {
    const SpBucket& sb = kind == 0 ? A.sendA[t] : kind == 1 ? A.sendR[t] : A.sendD[t];
    to = sb.cap != 0;
    if (to && kind == 0) { /* the ACCEPT counts were taken in local scratch: into the (remote) bucket header */
      SpHdr* h = sp_hdr(sb);
      uint32_t c = A.cntA[t]->count;
      if (c > sb.cap) c = sb.cap;
      h->count = c;
      h->blob_units = A.cntA[t]->blob_units;
    }
  }
  __threadfence_system();
  __syncwarp();
  if (to) {
    volatile uint32_t* f = A.flags_peer[t] + kind * GPX_SP_ND + A.me;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"((uint32_t*)f), "r"(round) : "memory");
  }
  __syncwarp();
  if (t == 0) A.seq[kind] = round;
}

__global__ void k_sp_wait(const __grid_constant__ SpArgs A, uint32_t kind) {
  const uint32_t t = threadIdx.x;
  const uint32_t round = A.seq[3 + kind] + 1u;
  if (t < A.N) {
    const SpBucket& rb = kind == 0 ? A.recvA[t] : kind == 1 ? A.recvR[t] : A.recvD[t];
    if (rb.cap) {
      const uint32_t* f = A.flags_local + kind * GPX_SP_ND + t;
      uint32_t seen;
      do {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(f) : "memory");
        if ((int32_t)(seen - round) < 0) __nanosleep(100);
      } while ((int32_t)(seen - round) < 0);
    }
  }
  __syncwarp();
  if (t == 0) A.seq[3 + kind] = round;
}
