/*
 * gpx_prepare.cuh -- k_prepare: phase 1a at the acceptors (PISM.handlePrepare :896-955,
 * PaxosAcceptor.handlePrepare :239-275, pruneAcceptedProposals :285-297, getMaxGCSlotFirstUndecidedSlot :277-282).
 *
 * One thread per PREPARE record (a gpx_pvalue_hdr whose slot is firstUndecidedSlot); the thread of the first
 * record of a run of equal gids handles the run at every local lane.  Per lane: adopt a higher ballot, gather the
 * live accepted pvalues with slot >= firstUndecidedSlot from the W-entry window (slot order), write the reply
 * (32 B header + W x 32 B entries at the fixed position i * L + lane) and the PREPARE's log image (VOID unless the
 * ballot was raised: the promise must be durable before the reply is visible, LogMessagingTask :940-944).
 * View changes are rare: this kernel is written for clarity, not for the roofline.
 */
#pragma once
#include "gpx_kernels.cuh"

struct PrepareArgs {
  const gpx_pvalue_hdr* recs;
  uint32_t n;
  gpx_prepare_reply_rec* replies; /* [n * L] */
};

template <int L>
__global__ void __launch_bounds__(GPX_BLOCK) k_prepare(const __grid_constant__ DevState S,
                                                       const __grid_constant__ PrepareArgs A) {
  const uint32_t n = A.n;
  const uint32_t i = blockIdx.x * GPX_BLOCK + threadIdx.x;
  const unsigned long long reserved = seg_decision_bytes(n);
  unsigned long long segb[L];
#pragma unroll
  for (int l = 0; l < L; l++) segb[l] = seg_base(S, l, reserved);
  if (i == 0) {
#pragma unroll
    for (int l = 0; l < L; l++) {
      const unsigned long long sq = seg_seq_of(S, l);
      write_seg_hdr(S, l, segb[l], GPX_F_PREPARE, n, n, 0, 32, sq);
      log_publish(S, l, segb[l] + reserved, sq + 1ull);
    }
    atomicAdd(&S.ctr[C_KERNEL_LAUNCHES], 1ull);
  }
  if (i < n) {
    const uint32_t gid = A.recs[i].gid;
    const bool head = (i == 0) || (A.recs[i - 1].gid != gid);
    if (head) {
      const GroupCtx g = group_ctx(S, gid);
      for (uint32_t j = i; j < n && A.recs[j].gid == gid; j++) {
        const int4* rp = reinterpret_cast<const int4*>(&A.recs[j]);
        const int4 q0 = rp[0], q1 = rp[1];
        const int fus = q0.y, pbn = q0.z, pbc = q0.w; /* firstUndecidedSlot, the preparer's ballot */
        const uint32_t rflags = (uint32_t)q1.y & 0xffffu, dst_mask = (uint32_t)q1.y >> 16;
#pragma unroll
        for (int l = 0; l < L; l++) {
          gpx_prepare_reply_rec* rep = &A.replies[(size_t)j * L + l];
          int4* ro = reinterpret_cast<int4*>(rep);
          int4 img1 = make_int4(q1.x, (int)(GPX_F_VOID | (dst_mask << 16)), q1.z, q1.w);
          int4 h0 = make_int4((int)gid, 0, 0, 0), h1 = make_int4((int)GPX_WHO(0xffu, 0xffu, GPX_F_VOID), 0, 0, 0);
          gpx_accepted_pvalue acc[GPX_MAX_WINDOW];
          uint32_t na = 0;
          bool ok = ((dst_mask >> l) & 1u) && !(rflags & GPX_F_VOID) && g.live;
          uint32_t aux = 0;
          const size_t ri = row_idx(S, l, gid < S.G ? gid : 0);
          if (ok) {
            aux = S.acc_aux[ri];
            ok = st_usable(aux) && g.ms->idx_of_lane[l] != 0xffu; /* PISM :456-460: stopped / no instance -> dropped */
          }
          if (ok) {
            int4 row = S.acc_row[ri];
            const bool raised = bcmp(pbn, pbc, row.y, row.z) > 0; /* PaxosAcceptor.handlePrepare :245-251 */
            if (raised) {
              row.y = pbn;
              row.z = pbc;
              S.acc_row[ri] = row;
            }
            const bool nack = bcmp(row.y, row.z, pbn, pbc) > 0;
            if (!nack) { /* pruneAcceptedProposals :285-297, in slot order */
              for (uint32_t w = 0; w < S.W; w++) {
                int4 e0, e1;
                ld256(&S.acc_win[2 * win_idx(S, l, w, gid)], e0, e1);
                if (!((unsigned)e1.w & GPX_ENT_VALID) || jsub(e0.x, row.w) <= 0 || jsub(e0.x, fus) < 0) continue;
                gpx_accepted_pvalue pv;
                pv.slot = e0.x;
                pv.bnum = e0.y;
                pv.bcoord = e0.z;
                pv.frame_ref = (uint32_t)e0.w;
                pv.req_id = ((long long)e1.y << 32) | (unsigned)e1.x;
                pv.payload_len = (uint32_t)e1.z;
                pv.flags = (uint32_t)e1.w & ~GPX_ENT_VALID;
                uint32_t k = na++;
                while (k > 0 && jsub(acc[k - 1].slot, row.w) > jsub(pv.slot, row.w)) { /* insertion sort, <= W entries */
                  acc[k] = acc[k - 1];
                  k--;
                }
                acc[k] = pv;
              }
            }
            uint32_t dstIdx = 0xffu;
            for (uint32_t m = 0; m < g.R; m++)
              if (g.ms->nodes[m] == pbc) dstIdx = m;
            uint32_t fl = (nack ? GPX_F_NACK : 0u) | (raised ? GPX_F_LOGGED : 0u);
            if (!nack && S.journaling && jsub(fus, row.x) < 0) fl |= GPX_F_FROM_LOG; /* GET_ACCEPTED_PVALUES_FROM_DISK */
            const int first_slot = jsub(row.w, fus - 1) < 0 ? fus - 1 : row.w; /* getMaxGCSlotFirstUndecidedSlot */
            h0 = make_int4((int)gid, first_slot, row.y, row.z);
            h1 = make_int4((int)GPX_WHO(g.ms->idx_of_lane[l], dstIdx, fl), (int)na, 0, 0);
            if (raised) img1 = make_int4(q1.x, (int)(GPX_F_PREPARE | ((1u << l) << 16)), q1.z, q1.w);
          }
          ro[0] = h0;
          ro[1] = h1;
          for (uint32_t k = 0; k < GPX_MAX_WINDOW; k++) {
            int4 a0 = make_int4(0, 0, 0, 0), a1 = a0;
            if (k < na) {
              const int4* ap = reinterpret_cast<const int4*>(&acc[k]);
              a0 = ap[0];
              a1 = ap[1];
            }
            ro[2 + 2 * k] = a0;
            ro[3 + 2 * k] = a1;
          }
          st256_stream(ring_ptr(S, l, segb[l] + 64 + (unsigned long long)j * 32), q0, img1);
        }
      }
    }
  }
}
