/*
 * gpx_engine.cu -- host side of the engine and the C ABI of include/gpx.h.
 *
 * One engine == one GPU == one process (scale-out is one engine per rank, groups
 * sharded by paxosID hash; see gigapaxos_b200/shard.py).  The engine owns the SoA
 * state in HBM, the per-lane log rings and scratch streams; every entry point is a
 * thin marshalling layer around the kernels in gpx_kernels.cuh.  There is no CPU
 * fallback: without a CUDA device gpx_engine_create fails with GPX_ENOGPU.
 */
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h> /* types only: libnccl.so.2 is loaded at run time (gpx_spread_host.inc) */

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "gpx_round.cuh"
#include "gpx_route.cuh"
#include "gpx_spread.cuh"
#include "gpx_prepare.cuh"
#include "gpx_phase1b.cuh"
#include "gpx_pause.cuh"
#include "gpx_logfind.cuh"

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CK(call)                                                                        \
  do {                                                                                  \
    cudaError_t _e = (call);                                                            \
    if (_e != cudaSuccess)                                                              \
      return fail(GPX_ECUDA, std::string(#call) + ": " + cudaGetErrorString(_e));       \
  } while (0)

static inline uint32_t cdiv(uint64_t a, uint32_t b) { return (uint32_t)((a + b - 1) / b); }

/* where a launch helper counts and appends: the engine's scratch (gpx_engine::sink()) or a device-resident call's */
struct Sink {
  RoundCtl* ctl;
  gpx_accept_rec* accepts;
  gpx_exec_rec* extra;
  uint32_t extra_cap;
};

struct gpx_engine {
  gpx_config cfg;
  DevState S;
  std::vector<void*> allocs;
  cudaStream_t stream = nullptr;
  /* member sets */
  std::vector<MsetInfo> msets;
  std::map<std::vector<int32_t>, uint32_t> mset_ids;
  MsetInfo* d_msets = nullptr;
  /* host-side per-group info (name hash, version) for dump/load */
  std::vector<int32_t> h_version, h_name_hash;
  /* scratch streams */
  gpx_request_rec* d_reqs = nullptr;
  uint8_t* d_payload = nullptr;
  uint8_t* d_blob1 = nullptr;
  uint64_t blob1_cap = 0;
  gpx_accept_rec* d_accepts = nullptr;
  gpx_accept_reply_rec* d_replies = nullptr;
  gpx_decision_rec* d_decisions = nullptr;
  gpx_exec_rec* d_exec = nullptr;
  gpx_exec_rec* d_extra = nullptr;
  uint32_t extra_cap = 0;
  int32_t* d_status = nullptr;
  uint32_t* d_copy_tab = nullptr;
  uint32_t* d_copy_dst = nullptr;
  uint32_t* d_todo = nullptr; /* [2N] k_round's left-over runs: start index, end index */
  uint8_t* d_mark = nullptr;  /* [N] request belongs to a left-over run */
  uint8_t* d_out_mask = nullptr;
  std::vector<uint8_t> h_out_mask;
  RoundCtl* d_ctl = nullptr;
  RoundCtl* d_rctl = nullptr; /* [2] the round kernels' own control blocks: they alternate as the working block, each
                               * round zeroes the one the next round counts into */
  const RoundCtl* last_ctl = nullptr; /* where the last round left its counters */
  int round_mode = 0;         /* gpx_set_round_mode: 0 / 1 device tail launch of k_round_slow, 2 host-launched pair */
  uint32_t rparity = 0;
  RoundCtl* h_ctl = nullptr; /* pinned */
  void* d_misc = nullptr;    /* group-management staging */
  size_t misc_bytes = 0;
  /* pipelined rounds (gpx_round_submit / gpx_round_wait): per-slot staging, three streams */
  struct PipeSlot {
    gpx_request_rec* d_reqs = nullptr;
    uint8_t* d_payload = nullptr;
    int32_t* d_status = nullptr;
    gpx_exec_rec* d_exec = nullptr;
    gpx_exec_sum* d_sum = nullptr;
    gpx_request_packed* d_packed = nullptr;
    uint32_t* d_bsum = nullptr;
    gpx_exec_rec* d_extra = nullptr;
    RoundCtl* d_ctl = nullptr;
    RoundCtl* h_ctl = nullptr; /* pinned */
    cudaEvent_t ev_h2d = nullptr, ev_k = nullptr, ev_d2h = nullptr;
    bool busy = false;
    uint64_t ticket = 0;
    gpx_round_io io;
  };
  PipeSlot pipe[GPX_PIPE_DEPTH];
  bool pipe_ready = false;
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  uint64_t next_ticket = 0, next_wait = 0;
  /* host mirror of the per-lane log ring heads (every launch that logs has a size the host knows: the mirror is
   * exact and no device read is needed to drain; `head_exact` drops when a phase call sized its segment from a
   * device-resident count, the next drain / back-pressure check then re-reads the heads) */
  uint64_t h_head[GPX_MAX_LANES] = {0}, log_tail[GPX_MAX_LANES] = {0}, drain_pos[GPX_MAX_LANES] = {0};
  bool head_exact = true;
  cudaStream_t s_drain = nullptr;
  cudaEvent_t ev_drain = nullptr;
  /* timing */
  int n_sms = 148;
  bool timing = false;
  cudaEvent_t ev[5];
  gpx_kernel_times kt;

  template <typename T>
  int dalloc(T** p, size_t n) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T) + 16);
    if (e != cudaSuccess) return fail(GPX_ENOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    allocs.push_back(q);
    *p = (T*)q;
    return GPX_OK;
  }
  Sink sink() const { return {d_ctl, d_accepts, d_extra, extra_cap}; }
  /* a device-resident call: the caller's control block and, when given, the caller's extra EXEC queue */
  Sink sink(gpx_dev_ctl* ctl, gpx_exec_rec* extra = nullptr, uint32_t cap = 0) const {
    return {reinterpret_cast<RoundCtl*>(ctl), d_accepts, extra ? extra : d_extra, extra ? cap : extra_cap};
  }
  int ensure_misc(size_t bytes) {
    if (bytes <= misc_bytes) return GPX_OK;
    if (d_misc) cudaFree(d_misc);
    misc_bytes = bytes + (bytes >> 2) + 4096;
    cudaError_t e = cudaMalloc(&d_misc, misc_bytes);
    if (e != cudaSuccess) {
      d_misc = nullptr;
      misc_bytes = 0;
      return fail(GPX_ENOMEM, "cudaMalloc(misc)");
    }
    return GPX_OK;
  }
};

extern "C" {

const char* gpx_last_error(void) { return g_err.c_str(); }
const char* gpx_build_info(void) {
  return "gpx CUDA engine: hand-written kernels for sm_100a (compute_100a), nvcc " __DATE__;
}

void gpx_config_defaults(gpx_config* c) {
  memset(c, 0, sizeof *c);
  c->abi_version = GPX_ABI_VERSION;
  c->device = 0;
  c->max_groups = 1024;
  c->n_lanes = 3;
  c->lane_node[0] = 100; /* TC.TEST_START_NODE_ID testing/TESTPaxosConfig.java:100 */
  c->lane_node[1] = 101;
  c->lane_node[2] = 102;
  c->window = 8;
  c->max_group_size = 3;
  c->log_ring_bytes = 1ull << 26;
  c->max_batch_recs = 1u << 16;
  c->max_batch_payload = 1ull << 24;
  c->batching_enabled = 1;         /* PaxosConfig.java:309 */
  c->max_batch_size = 2000;        /* :403 */
  c->max_batch_bytes = 4 * 1024 * 1024; /* min(NIOTransport.MAX_PAYLOAD_SIZE, MAX_LOG_MESSAGE_SIZE) */
  c->request_size_estimate = 512;
  c->checkpoint_interval = 400;    /* :410 */
  c->cpi_noise = 0;                /* :746 */
  c->gc_majority_executed = 1;     /* :882 */
  c->log_meta_decisions = 1;       /* :588 */
  c->journaling_enabled = 1;       /* :240 */
}

/* ---- Java helpers (String.hashCode, Math.abs, PISM.roundRobinCoordinator, getCPI) ---- */
int32_t gpx_java_string_hash(const char* s, size_t len) {
  uint32_t h = 0;
  for (size_t i = 0; i < len; i++) h = 31u * h + (uint32_t)(unsigned char)s[i];
  return (int32_t)h;
}
static int32_t java_abs(int32_t v) { return v < 0 ? (int32_t)(0u - (uint32_t)v) : v; }
int32_t gpx_round_robin_coordinator(int32_t name_hash, const int32_t* m, int32_t n, int32_t ballotnum) {
  int32_t idx = java_abs((int32_t)((uint32_t)ballotnum + (uint32_t)name_hash)) % n;
  if (idx < 0) idx = -idx;
  return m[idx];
}
int32_t gpx_get_cpi(int32_t cpi, double noise, int32_t name_hash) {
  return (int32_t)(cpi * (1 - noise) + (java_abs(name_hash) % cpi) * 2 * noise);
}

/* ---- lifecycle -------------------------------------------------------------------- */
int gpx_engine_create(const gpx_config* cfg, gpx_engine** out) {
  if (!cfg || !out) return fail(GPX_EINVAL, "null argument");
  if (cfg->abi_version != GPX_ABI_VERSION) return fail(GPX_EINVAL, "abi_version mismatch");
  if (cfg->n_lanes == 0 || cfg->n_lanes > GPX_MAX_LANES) return fail(GPX_EINVAL, "n_lanes out of range");
  if (cfg->window == 0 || cfg->window > GPX_MAX_WINDOW || (cfg->window & (cfg->window - 1)))
    return fail(GPX_EINVAL, "window must be 1,2,4 or 8");
  if (cfg->max_group_size == 0 || cfg->max_group_size > GPX_MAX_GROUP_SIZE)
    return fail(GPX_EINVAL, "max_group_size out of range");
  if (cfg->log_ring_bytes < (1u << 16) || (cfg->log_ring_bytes & (cfg->log_ring_bytes - 1)))
    return fail(GPX_EINVAL, "log_ring_bytes must be a power of two >= 64 KiB");
  if (cfg->max_groups == 0 || cfg->max_batch_recs == 0) return fail(GPX_EINVAL, "zero capacity");
  { /* the kernels index the state planes with 32-bit element indices */
    const unsigned long long span = 2ull * cfg->n_lanes * cfg->max_groups *
                                    (cfg->window > cfg->max_group_size ? cfg->window : cfg->max_group_size);
    if (span >= (1ull << 32)) return fail(GPX_EINVAL, "max_groups * n_lanes * window too large for one engine");
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(GPX_ENOGPU, "no CUDA device: the gpx engine has no CPU fallback");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(GPX_EINVAL, "bad device ordinal");
  CK(cudaSetDevice(cfg->device));
  gpx_engine* e = new gpx_engine();
  e->cfg = *cfg;
  memset(&e->kt, 0, sizeof e->kt);
  DevState& S = e->S;
  memset(&S, 0, sizeof S);
  const size_t G = cfg->max_groups, L = cfg->n_lanes, W = cfg->window, R = cfg->max_group_size;
  S.G = (uint32_t)G;
  S.L = (uint32_t)L;
  S.W = (uint32_t)W;
  S.Rcap = (uint32_t)R;
  int rc;
#define TRY(x)            \
  if ((rc = (x)) != 0) {  \
    gpx_engine_destroy(e);\
    return rc;            \
  }
  TRY(e->dalloc(&S.acc_row, L * G));
  TRY(e->dalloc(&S.acc_aux, L * G));
  TRY(e->dalloc(&S.acc_win, 2 * L * W * G));
  TRY(e->dalloc(&S.acc_dirty, L * G));
  TRY(e->dalloc(&S.com_win, 2 * L * W * G));
  TRY(e->dalloc(&S.coord_row, L * G));
  TRY(e->dalloc(&S.node_slots, L * R * G));
  TRY(e->dalloc(&S.prop_win, L * W * G));
  TRY(e->dalloc(&S.grp_meta, G));
  TRY(e->dalloc(&S.grp_cpi, G));
  TRY(e->dalloc(&e->d_msets, (size_t)GPX_MAX_MSETS));
  S.msets = e->d_msets;
  S.ring_cap = cfg->log_ring_bytes;
  for (size_t l = 0; l < L; l++) {
    TRY(e->dalloc(&S.ring[l], (size_t)cfg->log_ring_bytes));
    cudaMemset(S.ring[l], 0, cfg->log_ring_bytes);
  }
  TRY(e->dalloc(&S.log_pos, (size_t)4 * GPX_MAX_LANES));
  TRY(e->dalloc(&S.cur_seg, (size_t)GPX_MAX_LANES));
  TRY(e->dalloc(&S.ctr, (size_t)C_NCTR * GPX_CTR_STRIPES));
  TRY(e->dalloc(&S.tickets, (size_t)8));
  cudaMemset(S.log_pos, 0, 4 * GPX_MAX_LANES * 8);
  S.lp = 0;
  cudaMemset(S.cur_seg, 0, GPX_MAX_LANES * 8);
  cudaMemset(S.ctr, 0, C_NCTR * GPX_CTR_STRIPES * 8);
  cudaMemset(S.tickets, 0, 8 * 4);
  cudaMemset(S.grp_meta, 0, G * 4);
  {
    /* every row starts FREE */
    std::vector<uint32_t> aux(L * G, (uint32_t)GPX_ST_FREE);
    cudaMemcpy(S.acc_aux, aux.data(), L * G * 4, cudaMemcpyHostToDevice);
    cudaMemset(S.coord_row, 0, L * G * sizeof(int4));
    cudaMemset(S.acc_win, 0, 2 * L * W * G * sizeof(int4));
    cudaMemset(S.acc_dirty, 0, L * G);
    cudaMemset(S.com_win, 0, 2 * L * W * G * sizeof(int4));
    cudaMemset(S.prop_win, 0, L * W * G * sizeof(int4));
  }
  for (size_t l = 0; l < GPX_MAX_LANES; l++) S.lane_node[l] = l < L ? cfg->lane_node[l] : INT32_MIN;
  S.cpi_const = cfg->checkpoint_interval;
  S.cpi_per_group = cfg->cpi_noise != 0.0;
  S.gc_majority_executed = cfg->gc_majority_executed;
  S.log_meta = cfg->log_meta_decisions;
  S.journaling = cfg->journaling_enabled;
  S.batching = cfg->batching_enabled;
  S.max_batch_size = cfg->max_batch_size;
  S.size_est = cfg->request_size_estimate;
  S.max_batch_bytes = cfg->max_batch_bytes;
  /* scratch */
  const size_t N = cfg->max_batch_recs;
  const uint64_t P = (cfg->max_batch_payload + 15) & ~15ull;
  TRY(e->dalloc(&e->d_reqs, N));
  TRY(e->dalloc(&e->d_payload, (size_t)P));
  e->blob1_cap = P + 16ull * N;
  TRY(e->dalloc(&e->d_blob1, (size_t)e->blob1_cap));
  TRY(e->dalloc(&e->d_accepts, N));
  TRY(e->dalloc(&e->d_replies, N * L));
  TRY(e->dalloc(&e->d_decisions, N * L));
  TRY(e->dalloc(&e->d_exec, N * L));
  e->extra_cap = (uint32_t)N;
  TRY(e->dalloc(&e->d_extra, N));
  TRY(e->dalloc(&e->d_status, N));
  TRY(e->dalloc(&e->d_copy_tab, N));
  TRY(e->dalloc(&e->d_copy_dst, N));
  TRY(e->dalloc(&e->d_todo, 2 * N));
  TRY(e->dalloc(&e->d_mark, N));
  TRY(e->dalloc(&e->d_out_mask, N));
  TRY(e->dalloc(&e->d_ctl, (size_t)1));
  TRY(e->dalloc(&e->d_rctl, (size_t)2));
  cudaMemset(e->d_rctl, 0, 2 * sizeof(RoundCtl));
#undef TRY
  if (cudaHostAlloc((void**)&e->h_ctl, sizeof(RoundCtl), cudaHostAllocDefault) != cudaSuccess) {
    gpx_engine_destroy(e);
    return fail(GPX_ENOMEM, "cudaHostAlloc");
  }
  {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) == cudaSuccess && prop.multiProcessorCount > 0)
      e->n_sms = prop.multiProcessorCount;
  }
  cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
  for (int i = 0; i < 5; i++) cudaEventCreate(&e->ev[i]);
  if (const char* rm = getenv("GPX_ROUND_MODE")) e->round_mode = atoi(rm) >= 0 && atoi(rm) <= 2 ? atoi(rm) : 0; /* tuning / tests */
  e->h_version.assign(G, 0);
  e->h_name_hash.assign(G, 0);
  cudaError_t err = cudaDeviceSynchronize();
  if (err != cudaSuccess) {
    gpx_engine_destroy(e);
    return fail(GPX_ECUDA, cudaGetErrorString(err));
  }
  *out = e;
  return GPX_OK;
}

void gpx_engine_destroy(gpx_engine* e) {
  if (!e) return;
  cudaDeviceSynchronize();
  for (void* p : e->allocs) cudaFree(p);
  if (e->d_misc) cudaFree(e->d_misc);
  if (e->h_ctl) cudaFreeHost(e->h_ctl);
  for (auto& ps : e->pipe) {
    if (ps.h_ctl) cudaFreeHost(ps.h_ctl);
    if (ps.ev_h2d) cudaEventDestroy(ps.ev_h2d);
    if (ps.ev_k) cudaEventDestroy(ps.ev_k);
    if (ps.ev_d2h) cudaEventDestroy(ps.ev_d2h);
  }
  if (e->s_drain) cudaStreamDestroy(e->s_drain);
  if (e->ev_drain) cudaEventDestroy(e->ev_drain);
  if (e->s_h2d) cudaStreamDestroy(e->s_h2d);
  if (e->s_d2h) cudaStreamDestroy(e->s_d2h);
  if (e->stream) {
    cudaStreamDestroy(e->stream);
    for (int i = 0; i < 5; i++) cudaEventDestroy(e->ev[i]);
  }
  delete e;
}

/* ---- groups ----------------------------------------------------------------------- */
static int intern_mset(gpx_engine* e, std::vector<int32_t> m, uint32_t* id, bool* added) {
  std::sort(m.begin(), m.end()); /* PISM ctor sorts groupMembers :205 */
  auto it = e->mset_ids.find(m);
  if (it != e->mset_ids.end()) {
    *id = it->second;
    return GPX_OK;
  }
  if (e->msets.size() >= GPX_MAX_MSETS) return fail(GPX_ERANGE, "too many distinct member sets");
  MsetInfo mi;
  memset(&mi, 0xff, sizeof mi);
  mi.R = (uint8_t)m.size();
  mi.lane_mask = 0;
  mi.ident = 0;
  mi.pad2 = 0;
  for (size_t i = 0; i < GPX_MAX_GROUP_SIZE; i++) mi.nodes[i] = i < m.size() ? m[i] : INT32_MIN;
  for (uint32_t l = 0; l < e->cfg.n_lanes; l++)
    for (size_t i = 0; i < m.size(); i++)
      if (m[i] == e->cfg.lane_node[l]) {
        mi.lane_of_idx[i] = (uint8_t)l;
        mi.idx_of_lane[l] = (uint8_t)i;
        mi.lane_mask |= (uint16_t)(1u << l);
      }
  bool ident = m.size() == e->cfg.n_lanes;
  for (uint32_t l = 0; ident && l < e->cfg.n_lanes; l++) ident = mi.idx_of_lane[l] == l && mi.lane_of_idx[l] == l;
  mi.ident = ident ? 1 : 0;
  *id = (uint32_t)e->msets.size();
  e->msets.push_back(mi);
  e->mset_ids[m] = *id;
  *added = true;
  return GPX_OK;
}
static int push_msets(gpx_engine* e) {
  CK(cudaMemcpyAsync(e->d_msets, e->msets.data(), e->msets.size() * sizeof(MsetInfo), cudaMemcpyHostToDevice,
                     e->stream));
  return GPX_OK;
}

int gpx_create_groups(gpx_engine* e, uint32_t n, const gpx_group_desc* d) {
  if (!e || (!d && n)) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  std::vector<InitRec> recs(n);
  bool added = false;
  for (uint32_t k = 0; k < n; k++) {
    if (d[k].gid >= e->cfg.max_groups) return fail(GPX_ERANGE, "gid >= max_groups");
    if (d[k].n_members <= 0 || d[k].n_members > (int)e->cfg.max_group_size)
      return fail(GPX_ERANGE, "group size exceeds max_group_size");
    std::vector<int32_t> m(d[k].members, d[k].members + d[k].n_members);
    std::sort(m.begin(), m.end());
    uint32_t id;
    int rc = intern_mset(e, m, &id, &added);
    if (rc) return rc;
    recs[k].gid = d[k].gid;
    recs[k].mset = id;
    recs[k].coord0 = gpx_round_robin_coordinator(d[k].name_hash, m.data(), (int32_t)m.size(), 0);
    recs[k].cpi = gpx_get_cpi(e->cfg.checkpoint_interval, e->cfg.cpi_noise, d[k].name_hash);
    recs[k].init_mode = d[k].init_mode;
    recs[k].R = (uint32_t)m.size();
    e->h_version[d[k].gid] = d[k].version;
    e->h_name_hash[d[k].gid] = d[k].name_hash;
  }
  if (added) {
    int rc = push_msets(e);
    if (rc) return rc;
  }
  int rc = e->ensure_misc(n * sizeof(InitRec));
  if (rc) return rc;
  CK(cudaMemcpyAsync(e->d_misc, recs.data(), n * sizeof(InitRec), cudaMemcpyHostToDevice, e->stream));
  k_init_groups<<<cdiv(n, 256), 256, 0, e->stream>>>(e->S, (const InitRec*)e->d_misc, n);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(e->stream));
  return GPX_OK;
}

int gpx_destroy_groups(gpx_engine* e, uint32_t n, const uint32_t* gids) {
  if (!e || (!gids && n)) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  int rc = e->ensure_misc(n * 4ull);
  if (rc) return rc;
  for (uint32_t k = 0; k < n; k++)
    if (gids[k] < e->cfg.max_groups) e->h_name_hash[gids[k]] = e->h_version[gids[k]] = 0;
  CK(cudaMemcpyAsync(e->d_misc, gids, n * 4ull, cudaMemcpyHostToDevice, e->stream));
  k_destroy_groups<<<cdiv(n, 256), 256, 0, e->stream>>>(e->S, (const uint32_t*)e->d_misc, n);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(e->stream));
  return GPX_OK;
}

int gpx_dump_rows(gpx_engine* e, uint32_t n, const uint32_t* gids, uint32_t lane, gpx_row* out) {
  if (!e || !gids || !out) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  if (n == 0) return GPX_OK;
  size_t goff = (n * sizeof(gpx_row) + 255) & ~(size_t)255;
  int rc = e->ensure_misc(goff + n * 4ull);
  if (rc) return rc;
  uint32_t* d_g = (uint32_t*)((uint8_t*)e->d_misc + goff);
  CK(cudaMemcpyAsync(d_g, gids, n * 4ull, cudaMemcpyHostToDevice, e->stream));
  k_dump_rows<<<cdiv(n, 128), 128, 0, e->stream>>>(e->S, d_g, n, lane, (gpx_row*)e->d_misc);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, e->d_misc, n * sizeof(gpx_row), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  for (uint32_t k = 0; k < n; k++)
    if (gids[k] < e->cfg.max_groups) {
      out[k].version = e->h_version[gids[k]];
      out[k].name_hash = e->h_name_hash[gids[k]];
    }
  return GPX_OK;
}

int gpx_load_rows(gpx_engine* e, uint32_t n, const gpx_row* rows) {
  if (!e || (!rows && n)) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  std::vector<LoadRec> recs(n);
  bool added = false;
  for (uint32_t k = 0; k < n; k++) {
    const gpx_row& r = rows[k];
    if (r.gid >= e->cfg.max_groups || r.lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "gid/lane");
    if (r.n_members <= 0 || r.n_members > (int)e->cfg.max_group_size) return fail(GPX_ERANGE, "n_members");
    std::vector<int32_t> m(r.members, r.members + r.n_members);
    uint32_t id;
    int rc = intern_mset(e, m, &id, &added);
    if (rc) return rc;
    recs[k].row = r;
    recs[k].mset = id;
    recs[k].cpi = gpx_get_cpi(e->cfg.checkpoint_interval, e->cfg.cpi_noise, r.name_hash); /* getCPI(paxosID) */
    e->h_version[r.gid] = r.version;
    e->h_name_hash[r.gid] = r.name_hash;
  }
  if (added) {
    int rc = push_msets(e);
    if (rc) return rc;
  }
  int rc = e->ensure_misc(n * sizeof(LoadRec));
  if (rc) return rc;
  CK(cudaMemcpyAsync(e->d_misc, recs.data(), n * sizeof(LoadRec), cudaMemcpyHostToDevice, e->stream));
  k_load_rows<<<cdiv(n, 128), 128, 0, e->stream>>>(e->S, (const LoadRec*)e->d_misc, n);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(e->stream));
  return GPX_OK;
}

int gpx_patch(gpx_engine* e, uint32_t n, const gpx_patch_rec* p) {
  if (!e || (!p && n)) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  for (uint32_t k = 0; k < n; k++) {
    if (p[k].gid >= e->cfg.max_groups || p[k].lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "gid/lane");
    if (p[k].op < GPX_PATCH_SET_BALLOT || p[k].op > GPX_PATCH_SET_NODE_SLOT) return fail(GPX_EINVAL, "bad patch op");
  }
  int rc = e->ensure_misc(n * sizeof(gpx_patch_rec));
  if (rc) return rc;
  /* patches to the same (gid,lane) must apply in order: launch them one wave at a time */
  std::vector<gpx_patch_rec> wave;
  std::vector<uint8_t> done(n, 0);
  uint32_t left = n;
  while (left) {
    wave.clear();
    std::map<std::pair<uint32_t, uint32_t>, int> seen;
    for (uint32_t k = 0; k < n; k++) {
      if (done[k]) continue;
      auto key = std::make_pair(p[k].gid, p[k].lane);
      if (seen.count(key)) continue;
      seen[key] = 1;
      wave.push_back(p[k]);
      done[k] = 1;
      left--;
    }
    CK(cudaMemcpyAsync(e->d_misc, wave.data(), wave.size() * sizeof(gpx_patch_rec), cudaMemcpyHostToDevice,
                       e->stream));
    k_patch<<<cdiv(wave.size(), 128), 128, 0, e->stream>>>(e->S, (const gpx_patch_rec*)e->d_misc,
                                                            (uint32_t)wave.size());
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
  }
  return GPX_OK;
}

/* every launch that appends to the log reads log_pos[lp] and writes log_pos[lp ^ 1]: flip after the launch */
static inline void log_flip(gpx_engine* e) { e->S.lp ^= 1u; }

/* ---- kernel launch helpers (device pointers) ------------------------------------- */
static int launch_propose(gpx_engine* e, const Sink& sk, const gpx_request_rec* d_reqs, const uint8_t* d_payload,
                          uint64_t payload_al, uint32_t n, int32_t* d_status, cudaStream_t st) {
  ProposeArgs A;
  A.reqs = d_reqs;
  A.n = n;
  A.payload_bytes_al = payload_al;
  A.accepts = sk.accepts;
  A.status = d_status;
  A.copy_tab = e->d_copy_tab;
  A.copy_dst = e->d_copy_dst;
  A.ctl = sk.ctl;
  k_propose<<<cdiv(n, GPX_BLOCK), GPX_BLOCK, 0, st>>>(e->S, A);
  k_build_blobs<<<cdiv(n, GPX_BLOCK), GPX_BLOCK, 0, st>>>(A, d_payload, e->d_blob1);
  CK(cudaGetLastError());
  return GPX_OK;
}

/* kernels are templated on the lane count so that per-lane state stays in registers */
#define GPX_DISPATCH_L(lanes, KERNEL, grid, st, ...)                                   \
  switch (lanes) {                                                                     \
    case 1: KERNEL<1><<<grid, GPX_BLOCK, 0, st>>>(__VA_ARGS__); break;                 \
    case 2: KERNEL<2><<<grid, GPX_BLOCK, 0, st>>>(__VA_ARGS__); break;                 \
    case 3: KERNEL<3><<<grid, GPX_BLOCK, 0, st>>>(__VA_ARGS__); break;                 \
    case 4: KERNEL<4><<<grid, GPX_BLOCK, 0, st>>>(__VA_ARGS__); break;                 \
    case 5: KERNEL<5><<<grid, GPX_BLOCK, 0, st>>>(__VA_ARGS__); break;                 \
    case 6: KERNEL<6><<<grid, GPX_BLOCK, 0, st>>>(__VA_ARGS__); break;                 \
    case 7: KERNEL<7><<<grid, GPX_BLOCK, 0, st>>>(__VA_ARGS__); break;                 \
    default: KERNEL<8><<<grid, GPX_BLOCK, 0, st>>>(__VA_ARGS__); break;                \
  }

static int launch_accept(gpx_engine* e, const Sink& sk, bool fused, const gpx_accept_rec* d_recs, const uint32_t* n_ptr,
                         uint32_t n_max, const uint8_t* blob0, uint64_t blob0_bytes, const uint8_t* blob1,
                         uint64_t blob1_bytes, const unsigned long long* blob1_used_ptr,
                         gpx_accept_reply_rec* d_replies, gpx_decision_rec* d_dec, gpx_exec_rec* d_exec,
                         cudaStream_t st) {
  AcceptArgs A;
  A.recs = d_recs;
  A.n_ptr = n_ptr;
  A.n_max = n_max;
  A.blob0 = blob0;
  A.blob0_bytes = blob0_bytes;
  A.blob1 = blob1;
  A.blob1_bytes = blob1_bytes;
  A.blob1_used_ptr = blob1_used_ptr;
  A.replies = d_replies;
  A.decisions = d_dec;
  A.out_mask = e->d_out_mask;
  A.exec = d_exec;
  A.extra = sk.extra;
  A.extra_cap = sk.extra_cap;
  A.n_extra = &sk.ctl->n_extra;
  const uint32_t grid = cdiv(n_max, GPX_BLOCK);
  if (fused) {
    GPX_DISPATCH_L(e->cfg.n_lanes, k_act, grid, st, e->S, A);
  } else {
    GPX_DISPATCH_L(e->cfg.n_lanes, k_accept, grid, st, e->S, A);
  }
  log_flip(e);
  CK(cudaGetLastError());
  return GPX_OK;
}

static int launch_tally(gpx_engine* e, const Sink& sk, const gpx_accept_reply_rec* d_replies, const uint32_t* n_ptr,
                        uint32_t mult, uint32_t n_max, gpx_decision_rec* d_dec, cudaStream_t st) {
  TallyArgs A;
  A.replies = d_replies;
  A.n_ptr = n_ptr;
  A.mult = mult;
  A.n_max = n_max;
  A.decisions = d_dec;
  A.n_decisions = &sk.ctl->n_decisions;
  if (mult > 1 && mult == e->cfg.n_lanes) { /* [ACCEPT][lane] layout of the phase pipeline: one thread per slot */
    GPX_DISPATCH_L(mult, k_tally_slots, cdiv(n_max / mult, GPX_BLOCK), st, e->S, A);
  } else
    k_tally<<<cdiv(n_max, GPX_BLOCK), GPX_BLOCK, 0, st>>>(e->S, A);
  CK(cudaGetLastError());
  return GPX_OK;
}

static int launch_commit(gpx_engine* e, const Sink& sk, const gpx_decision_rec* d_dec, const uint32_t* n_ptr,
                         uint32_t n_max, gpx_exec_rec* d_exec, cudaStream_t st) {
  CommitArgs A;
  A.decisions = d_dec;
  A.n_ptr = n_ptr;
  A.n_max = n_max;
  A.exec = d_exec;
  A.extra = sk.extra;
  A.extra_cap = sk.extra_cap;
  A.n_extra = &sk.ctl->n_extra;
  GPX_DISPATCH_L(e->cfg.n_lanes, k_commit, cdiv(n_max, GPX_BLOCK), st, e->S, A);
  log_flip(e);
  CK(cudaGetLastError());
  return GPX_OK;
}

/* k_round<L, LP, DEF>: LP = L (team width); DEF = the reference's default configuration folded at compile time */
extern "C++" {
template <int L, int LP>
static void launch_round_t(uint32_t grid, cudaStream_t st, const DevState& S, const RoundArgs& RA) {
  if (S.journaling && S.gc_majority_executed && S.log_meta && !S.cpi_per_group)
    k_round<L, LP, true><<<grid, GPX_RBLOCK, 0, st>>>(S, RA);
  else
    k_round<L, LP, false><<<grid, GPX_RBLOCK, 0, st>>>(S, RA);
  if (!RA.tail_launch) { /* host-launched pair; programmatic dependent launch hides k_round_slow's launch latency */
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(RA.slow_grid);
    cfg.blockDim = dim3(GPX_BLOCK);
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, k_round_slow<L, LP>, S, RA);
  }
}
}
/* payload-area bytes a round of n requests reserves for the blobs it constructs for batched slots */
static uint64_t blob1_res(const gpx_engine* e, uint32_t n, uint64_t pal) {
  return e->cfg.batching_enabled ? std::min<uint64_t>(e->blob1_cap, 16ull * n + pal) : 0;
}
static int launch_round(gpx_engine* e, const gpx_request_rec* d_reqs, const uint8_t* d_payload, uint64_t pal,
                        uint32_t n, int32_t* d_status, gpx_exec_rec* d_exec, cudaStream_t st,
                        RoundCtl* d_ctl = nullptr, gpx_exec_rec* d_extra = nullptr, uint32_t extra_cap = 0,
                        gpx_exec_sum* d_sum = nullptr) {
  /* the round counts into `working`: the engine's own blocks [0] / [1] alternate (each round zeroes the one the next
   * round uses); a caller-provided block is zeroed by the caller */
  RoundCtl* ctl_zero = nullptr;
  if (!d_ctl) {
    d_ctl = e->d_rctl + e->rparity;
    ctl_zero = e->d_rctl + (e->rparity ^ 1u);
    e->rparity ^= 1u;
  }
  e->last_ctl = d_ctl;
  if (!d_extra) {
    d_extra = e->d_extra;
    extra_cap = e->extra_cap;
  }
  RoundArgs RA;
  memset(&RA, 0, sizeof RA);
  RA.P.reqs = d_reqs;
  RA.P.n = n;
  RA.P.payload_bytes_al = pal;
  RA.P.accepts = e->d_accepts;
  RA.P.status = d_status;
  RA.P.copy_tab = e->d_copy_tab;
  RA.P.copy_dst = e->d_copy_dst;
  RA.P.ctl = d_ctl;
  RA.ctl_zero = ctl_zero;
  RA.sum = d_sum;
  RA.A.n_max = n;
  RA.A.blob0 = d_payload;
  RA.A.blob0_bytes = pal;
  RA.A.blob1 = e->d_blob1;
  RA.A.replies = e->d_replies;
  RA.A.decisions = e->d_decisions;
  RA.A.out_mask = e->d_out_mask;
  RA.A.exec = d_exec;
  RA.A.extra = d_extra;
  RA.A.extra_cap = extra_cap;
  RA.A.n_extra = &d_ctl->n_extra;
  RA.blob1w = e->d_blob1;
  RA.todo = e->d_todo;
  RA.todo_end = e->d_todo + e->cfg.max_batch_recs;
  RA.mark = e->d_mark;
  RA.n_todo = &d_ctl->n_todo;
  RA.blob1_res = blob1_res(e, n, pal);
  RA.A.blob1_bytes = RA.blob1_res;
  RA.pay_bytes = pal + RA.blob1_res;
  RA.pay_rel = (uint32_t)seg_pay_rel(n);
  RA.res_a = seg_accept_bytes(n, RA.pay_bytes);
  RA.res_d = seg_decision_bytes(n);
  const uint32_t L = e->cfg.n_lanes;
  const uint32_t teams_per_block = (GPX_RBLOCK / 32u) * (32u / L); /* teams of L adjacent lanes */
  const uint32_t grid = cdiv((uint64_t)n, teams_per_block);
  RA.slow_grid = std::min<uint32_t>(grid, 2u * (uint32_t)e->n_sms);
  RA.tail_launch = e->round_mode == 2 ? 0u : 1u; /* grid-stride over the todo list; all
                                                                            * blocks resident (grid barriers) */
  switch (L) {
    case 1: launch_round_t<1, 1>(grid, st, e->S, RA); break;
    case 2: launch_round_t<2, 2>(grid, st, e->S, RA); break;
    case 3: launch_round_t<3, 3>(grid, st, e->S, RA); break;
    case 4: launch_round_t<4, 4>(grid, st, e->S, RA); break;
    case 5: launch_round_t<5, 5>(grid, st, e->S, RA); break;
    case 6: launch_round_t<6, 6>(grid, st, e->S, RA); break;
    case 7: launch_round_t<7, 7>(grid, st, e->S, RA); break;
    default: launch_round_t<8, 8>(grid, st, e->S, RA); break;
  }
  log_flip(e);
  CK(cudaGetLastError());
  return GPX_OK;
}

/* ---- log ring bookkeeping on the host ------------------------------------------------------------------ */
/* What one API call appends to every lane: up to two reservations, in launch order (an unused one is 0 bytes).  A
 * reservation is what one seg_base takes on the device: a segment, or a pair of segments laid out back to back (k_act,
 * k_round).  exact = false: an ACCEPT segment's payload area is a count the kernels read on the device, and its size
 * here is an upper bound. */
struct LogSegs {
  uint64_t bytes[2];
  bool exact;
};
static LogSegs one_seg(uint64_t bytes) { return {{bytes, 0}, true}; }

enum class RoundForm {
  FUSED,   /* k_round (+ k_round_slow): outputs indexed by request */
  COMPACT, /* k_propose + k_act: one record, log image and EXEC row per ACCEPT */
  PHASES,  /* k_propose, k_accept, k_tally, k_commit */
};
static LogSegs round_segs(const gpx_engine* e, RoundForm form, uint32_t n, uint64_t payload_bytes) {
  const uint64_t pal = (payload_bytes + 15) & ~15ull;
  const uint64_t a = seg_accept_bytes(n, pal + blob1_res(e, n, pal)), d = seg_decision_bytes(n);
  if (form == RoundForm::PHASES) return {{a, d}, false};
  return {{a + d, 0}, form == RoundForm::FUSED};
}

/* the heads the next logging launch will start from, after everything enqueued so far on any stream */
static int read_device_heads(gpx_engine* e, uint64_t out[GPX_MAX_LANES]) {
  CK(cudaDeviceSynchronize());
  unsigned long long pos[2 * GPX_MAX_LANES]; /* {head, seq} per lane */
  CK(cudaMemcpy(pos, e->S.log_pos + (size_t)e->S.lp * 2 * GPX_MAX_LANES, sizeof pos, cudaMemcpyDeviceToHost));
  for (uint32_t l = 0; l < e->cfg.n_lanes; l++) out[l] = pos[2 * l];
  return GPX_OK;
}
static int log_resync(gpx_engine* e) {
  if (e->head_exact) return GPX_OK;
  int rc = read_device_heads(e, e->h_head);
  if (rc) return rc;
  e->head_exact = true;
  return GPX_OK;
}
/* what seg_base + the publishing block do on the device, on the mirror */
static void log_advance(gpx_engine* e, const LogSegs& s) {
  if (!s.exact) e->head_exact = false;
  if (!e->head_exact) return;
  const uint64_t cap = e->cfg.log_ring_bytes;
  for (const uint64_t reserved : s.bytes)
    for (uint32_t l = 0; l < e->cfg.n_lanes; l++) {
      uint64_t h = e->h_head[l];
      const uint64_t pos = h & (cap - 1);
      if (pos + reserved > cap) h += cap - pos;
      e->h_head[l] = h + reserved;
    }
}
/* With log_backpressure the call is refused (GPX_EAGAIN, nothing has happened yet) when it could overwrite bytes that
 * were not released (gpx_log_release): AbstractPaxosLogger.logAndMessage :157 logs THEN messages -- an ACCEPT_REPLY may
 * only leave once its ACCEPT is durable, so the journal must have been drained before the ring position is reused. */
static int ring_fits(gpx_engine* e, const LogSegs& s) {
  const uint64_t total = s.bytes[0] + s.bytes[1];
  if (total > e->cfg.log_ring_bytes) return fail(GPX_ERANGE, "batch does not fit the log ring; raise log_ring_bytes");
  if (e->cfg.log_backpressure) {
    int rc = log_resync(e);
    if (rc) return rc;
    for (uint32_t l = 0; l < e->cfg.n_lanes; l++) /* 2 x: a reservation may first skip to the ring start, and that skip
                                                    * is shorter than the reservation */
      if (e->h_head[l] - e->log_tail[l] + 2 * total > e->cfg.log_ring_bytes)
        return fail(GPX_EAGAIN, "log ring full: drain it (gpx_log_drain_async) and release the drained bytes (gpx_log_release)");
  }
  return GPX_OK;
}
static int check_batch(gpx_engine* e, uint32_t n, uint64_t payload_bytes) {
  if (n > e->cfg.max_batch_recs) return fail(GPX_ERANGE, "n > max_batch_recs");
  if (payload_bytes > e->cfg.max_batch_payload) return fail(GPX_ERANGE, "payload_bytes > max_batch_payload");
  return GPX_OK;
}
static int fetch_ctl(gpx_engine* e, const RoundCtl* src = nullptr) {
  CK(cudaMemcpyAsync(e->h_ctl, src ? src : e->d_ctl, sizeof(RoundCtl), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return GPX_OK;
}
/* the engine's extra EXEC queue, as counted in h_ctl, to the caller: at most cap records; *n_extra = the whole count */
static int copy_extra_out(gpx_engine* e, gpx_exec_rec* dst, uint32_t cap, uint32_t* n_extra) {
  const uint32_t nx = e->h_ctl->n_extra;
  if (n_extra) *n_extra = nx;
  const uint32_t cp = std::min(std::min(nx, cap), e->extra_cap);
  if (cp && dst) {
    CK(cudaMemcpyAsync(dst, e->d_extra, cp * sizeof(gpx_exec_rec), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
  }
  return GPX_OK;
}

/* ---- data path: host buffers -------------------------------------------------------- */
int gpx_propose(gpx_engine* e, uint32_t n, const gpx_request_rec* reqs, const uint8_t* payload,
                uint64_t payload_bytes, gpx_accept_rec* out_accepts, uint32_t* n_accepts, uint8_t* out_blob,
                uint64_t blob_cap, uint64_t* blob_bytes, int32_t* status) {
  if (!e || !n_accepts || !blob_bytes) return fail(GPX_EINVAL, "null argument");
  *n_accepts = 0;
  *blob_bytes = 0;
  if (n == 0) return GPX_OK;
  if (!reqs || !out_accepts || !status || (!payload && payload_bytes)) return fail(GPX_EINVAL, "null argument");
  int rc = check_batch(e, n, payload_bytes);
  if (rc) return rc;
  const uint64_t pal = (payload_bytes + 15) & ~15ull;
  cudaStream_t st = e->stream;
  CK(cudaMemsetAsync(e->d_ctl, 0, sizeof(RoundCtl), st));
  CK(cudaMemcpyAsync(e->d_reqs, reqs, n * sizeof(gpx_request_rec), cudaMemcpyHostToDevice, st));
  if (payload_bytes) CK(cudaMemcpyAsync(e->d_payload, payload, payload_bytes, cudaMemcpyHostToDevice, st));
  rc = launch_propose(e, e->sink(), e->d_reqs, e->d_payload, pal, n, e->d_status, st);
  if (rc) return rc;
  rc = fetch_ctl(e);
  if (rc) return rc;
  const uint32_t na = e->h_ctl->n_accepts;
  const uint64_t b1 = e->h_ctl->blob1_used;
  if (pal + b1 > blob_cap) return fail(GPX_ERANGE, "out_blob too small");
  CK(cudaMemcpyAsync(out_accepts, e->d_accepts, na * sizeof(gpx_accept_rec), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(status, e->d_status, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (out_blob) {
    if (payload_bytes) memcpy(out_blob, payload, payload_bytes);
    if (pal > payload_bytes) memset(out_blob + payload_bytes, 0, pal - payload_bytes);
    if (b1) CK(cudaMemcpyAsync(out_blob + pal, e->d_blob1, b1, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  *n_accepts = na;
  *blob_bytes = pal + b1;
  return GPX_OK;
}

int gpx_handle_accepts(gpx_engine* e, uint32_t n, const gpx_accept_rec* accepts, const uint8_t* blob,
                       uint64_t blob_bytes, gpx_accept_reply_rec* out_replies, gpx_exec_rec* out_extra_exec,
                       uint32_t extra_cap, uint32_t* n_extra) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (n_extra) *n_extra = 0;
  if (n == 0) return GPX_OK;
  if (!accepts || !out_replies || (!blob && blob_bytes)) return fail(GPX_EINVAL, "null argument");
  if (blob_bytes & 15) return fail(GPX_EINVAL, "blob_bytes must be a multiple of 16");
  if (n > e->cfg.max_batch_recs) return fail(GPX_ERANGE, "n > max_batch_recs");
  if (blob_bytes > e->blob1_cap) return fail(GPX_ERANGE, "blob too large");
  const LogSegs segs = one_seg(seg_accept_bytes(n, blob_bytes));
  int rc = ring_fits(e, segs);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  const uint32_t L = e->cfg.n_lanes;
  CK(cudaMemsetAsync(e->d_ctl, 0, sizeof(RoundCtl), st));
  CK(cudaMemcpyAsync(e->d_accepts, accepts, n * sizeof(gpx_accept_rec), cudaMemcpyHostToDevice, st));
  if (blob_bytes) CK(cudaMemcpyAsync(e->d_blob1, blob, blob_bytes, cudaMemcpyHostToDevice, st));
  log_advance(e, segs);
  rc = launch_accept(e, e->sink(), false, e->d_accepts, nullptr, n, e->d_blob1, blob_bytes, nullptr, 0, nullptr,
                     e->d_replies, nullptr, nullptr, st);
  if (rc) return rc;
  CK(cudaMemcpyAsync(out_replies, e->d_replies, (size_t)n * L * sizeof(gpx_accept_reply_rec), cudaMemcpyDeviceToHost,
                     st));
  rc = fetch_ctl(e);
  if (rc) return rc;
  return copy_extra_out(e, out_extra_exec, extra_cap, n_extra);
}

int gpx_handle_accept_replies(gpx_engine* e, uint32_t n, const gpx_accept_reply_rec* replies,
                              gpx_decision_rec* out_decisions, uint32_t* n_decisions) {
  if (!e || !n_decisions) return fail(GPX_EINVAL, "null argument");
  *n_decisions = 0;
  if (n == 0) return GPX_OK;
  if (!replies || !out_decisions) return fail(GPX_EINVAL, "null argument");
  if (n > (uint64_t)e->cfg.max_batch_recs * e->cfg.n_lanes) return fail(GPX_ERANGE, "n > max_batch_recs * n_lanes");
  cudaStream_t st = e->stream;
  CK(cudaMemsetAsync(e->d_ctl, 0, sizeof(RoundCtl), st));
  CK(cudaMemcpyAsync(e->d_replies, replies, n * sizeof(gpx_accept_reply_rec), cudaMemcpyHostToDevice, st));
  int rc = launch_tally(e, e->sink(), e->d_replies, nullptr, 1, n, e->d_decisions, st);
  if (rc) return rc;
  rc = fetch_ctl(e);
  if (rc) return rc;
  uint32_t nd = e->h_ctl->n_decisions;
  if (nd) {
    CK(cudaMemcpyAsync(out_decisions, e->d_decisions, nd * sizeof(gpx_decision_rec), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  *n_decisions = nd;
  return GPX_OK;
}

int gpx_handle_decisions(gpx_engine* e, uint32_t n, const gpx_decision_rec* decisions, gpx_exec_rec* out_exec,
                         gpx_exec_rec* out_extra_exec, uint32_t extra_cap, uint32_t* n_extra) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (n_extra) *n_extra = 0;
  if (n == 0) return GPX_OK;
  if (!decisions || !out_exec) return fail(GPX_EINVAL, "null argument");
  if (n > (uint64_t)e->cfg.max_batch_recs) return fail(GPX_ERANGE, "n > max_batch_recs");
  const LogSegs segs = one_seg(seg_decision_bytes(n));
  int rc = ring_fits(e, segs);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  const uint32_t L = e->cfg.n_lanes;
  CK(cudaMemsetAsync(e->d_ctl, 0, sizeof(RoundCtl), st));
  CK(cudaMemcpyAsync(e->d_decisions, decisions, n * sizeof(gpx_decision_rec), cudaMemcpyHostToDevice, st));
  log_advance(e, segs);
  rc = launch_commit(e, e->sink(), e->d_decisions, nullptr, n, e->d_exec, st);
  if (rc) return rc;
  CK(cudaMemcpyAsync(out_exec, e->d_exec, (size_t)n * L * sizeof(gpx_exec_rec), cudaMemcpyDeviceToHost, st));
  rc = fetch_ctl(e);
  if (rc) return rc;
  return copy_extra_out(e, out_extra_exec, extra_cap, n_extra);
}

/* phase 1a at the acceptors: PISM.handlePrepare for a batch of PREPAREs, host buffers */
int gpx_handle_prepares(gpx_engine* e, uint32_t n, const gpx_pvalue_hdr* prepares, gpx_prepare_reply_rec* out_replies) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  if (!prepares || !out_replies) return fail(GPX_EINVAL, "null argument");
  if (n > e->cfg.max_batch_recs) return fail(GPX_ERANGE, "n > max_batch_recs");
  const LogSegs segs = one_seg(seg_decision_bytes(n));
  int rc = ring_fits(e, segs);
  if (rc) return rc;
  const uint32_t L = e->cfg.n_lanes;
  const size_t out_bytes = (size_t)n * L * sizeof(gpx_prepare_reply_rec);
  rc = e->ensure_misc(out_bytes);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  CK(cudaMemcpyAsync(e->d_decisions, prepares, n * sizeof(gpx_pvalue_hdr), cudaMemcpyHostToDevice, st));
  PrepareArgs A;
  A.recs = e->d_decisions;
  A.n = n;
  A.replies = (gpx_prepare_reply_rec*)e->d_misc;
  log_advance(e, segs);
  GPX_DISPATCH_L(L, k_prepare, cdiv(n, GPX_BLOCK), st, e->S, A);
  log_flip(e);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out_replies, e->d_misc, out_bytes, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return GPX_OK;
}

/* phase 1b for a batch of elections: one launch of k_prepare_tally (gpx_phase1b.cuh) */
int gpx_handle_prepare_replies(gpx_engine* e, uint32_t n, const gpx_election_rec* elections, uint32_t n_reply_recs,
                               const gpx_prepare_reply_rec* replies, gpx_election_out* out) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  if (!elections || !out || (!replies && n_reply_recs)) return fail(GPX_EINVAL, "null argument");
  {
    std::vector<uint32_t> gids(n);
    for (uint32_t i = 0; i < n; i++) {
      if ((uint64_t)elections[i].first_reply + elections[i].n_replies > n_reply_recs)
        return fail(GPX_ERANGE, "election refers to replies beyond n_reply_recs");
      gids[i] = elections[i].gid;
    }
    std::sort(gids.begin(), gids.end());
    if (std::adjacent_find(gids.begin(), gids.end()) != gids.end())
      return fail(GPX_EINVAL, "more than one election for a group in one call");
  }
  const size_t el_bytes = (size_t)n * sizeof(gpx_election_rec);
  const size_t rep_bytes = (size_t)n_reply_recs * sizeof(gpx_prepare_reply_rec);
  const size_t out_bytes = (size_t)n * sizeof(gpx_election_out);
  int rc = e->ensure_misc(el_bytes + rep_bytes + out_bytes);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  uint8_t* base = (uint8_t*)e->d_misc;
  CK(cudaMemcpyAsync(base, elections, el_bytes, cudaMemcpyHostToDevice, st));
  if (rep_bytes) CK(cudaMemcpyAsync(base + el_bytes, replies, rep_bytes, cudaMemcpyHostToDevice, st));
  Phase1bArgs A;
  A.els = (const gpx_election_rec*)base;
  A.n = n;
  A.replies = (const gpx_prepare_reply_rec*)(base + el_bytes);
  A.out = (gpx_election_out*)(base + el_bytes + rep_bytes);
  k_prepare_tally<<<cdiv(n, GPX_P1B_BLOCK), GPX_P1B_BLOCK, 0, st>>>(e->S, A);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, A.out, out_bytes, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return GPX_OK;
}

/* handleAccept + loopback tally + commit per ACCEPT (k_act), host buffers */
int gpx_handle_accepts_fused(gpx_engine* e, uint32_t n, const gpx_accept_rec* accepts, const uint8_t* blob,
                             uint64_t blob_bytes, gpx_accept_reply_rec* out_replies, gpx_decision_rec* out_decisions,
                             gpx_exec_rec* out_exec, gpx_exec_rec* out_extra_exec, uint32_t extra_cap,
                             uint32_t* n_extra) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (n_extra) *n_extra = 0;
  if (n == 0) return GPX_OK;
  if (!accepts || !out_replies || !out_decisions || !out_exec || (!blob && blob_bytes))
    return fail(GPX_EINVAL, "null argument");
  if (blob_bytes & 15) return fail(GPX_EINVAL, "blob_bytes must be a multiple of 16");
  if (n > e->cfg.max_batch_recs) return fail(GPX_ERANGE, "n > max_batch_recs");
  if (blob_bytes > e->blob1_cap) return fail(GPX_ERANGE, "blob too large");
  const LogSegs segs = one_seg(seg_accept_bytes(n, blob_bytes) + seg_decision_bytes(n));
  int rc = ring_fits(e, segs);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  const uint32_t L = e->cfg.n_lanes;
  CK(cudaMemsetAsync(e->d_ctl, 0, sizeof(RoundCtl), st));
  CK(cudaMemcpyAsync(e->d_accepts, accepts, n * sizeof(gpx_accept_rec), cudaMemcpyHostToDevice, st));
  if (blob_bytes) CK(cudaMemcpyAsync(e->d_blob1, blob, blob_bytes, cudaMemcpyHostToDevice, st));
  log_advance(e, segs);
  rc = launch_accept(e, e->sink(), true, e->d_accepts, nullptr, n, e->d_blob1, blob_bytes, nullptr, 0, nullptr,
                     e->d_replies, e->d_decisions, e->d_exec, st);
  if (rc) return rc;
  /* replies consumed by a local coordinator never reach HBM: out_mask says which reply slots were written */
  e->h_out_mask.resize(n);
  CK(cudaMemcpyAsync(e->h_out_mask.data(), e->d_out_mask, n, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  bool any_out = false;
  for (uint32_t i = 0; i < n; i++) any_out = any_out || e->h_out_mask[i];
  if (any_out)
    CK(cudaMemcpyAsync(out_replies, e->d_replies, (size_t)n * L * sizeof(gpx_accept_reply_rec), cudaMemcpyDeviceToHost,
                       st));
  CK(cudaMemcpyAsync(out_decisions, e->d_decisions, (size_t)n * sizeof(gpx_decision_rec), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(out_exec, e->d_exec, (size_t)n * L * sizeof(gpx_exec_rec), cudaMemcpyDeviceToHost, st));
  rc = fetch_ctl(e);
  if (rc) return rc;
  for (uint32_t i = 0; i < n; i++) /* VOID where the reply was consumed locally or never produced */
    for (uint32_t l = 0; l < L; l++)
      if (!((e->h_out_mask[i] >> l) & 1u)) {
        gpx_accept_reply_rec& r = out_replies[(size_t)i * L + l];
        memset(&r, 0, sizeof r);
        r.gid = accepts[i].h.gid;
        r.slot = accepts[i].h.slot;
        r.who = GPX_WHO(0xffu, 0xffu, GPX_F_VOID);
      }
  return copy_extra_out(e, out_extra_exec, extra_cap, n_extra);
}

/* one round on device pointers; `segs` = round_segs(e, form, ...), already admitted by ring_fits */
static int round_on_stream(gpx_engine* e, RoundForm form, const LogSegs& segs, const gpx_request_rec* d_reqs,
                           const uint8_t* d_payload, uint64_t payload_bytes, uint32_t n, int32_t* d_status,
                           gpx_exec_rec* d_exec, cudaStream_t st) {
  const uint64_t pal = (payload_bytes + 15) & ~15ull;
  const uint32_t L = e->cfg.n_lanes;
  const bool tm = e->timing;
  const bool fused = form == RoundForm::FUSED, compact = form == RoundForm::COMPACT;
  if (!fused) CK(cudaMemsetAsync(e->d_ctl, 0, sizeof(RoundCtl), st)); /* the fused kernels keep their own block zero */
  log_advance(e, segs);
  if (tm) cudaEventRecord(e->ev[0], st);
  if (fused) { /* the whole round is ONE kernel */
    int rc1 = launch_round(e, d_reqs, d_payload, pal, n, d_status, d_exec, st);
    if (rc1) return rc1;
    if (tm) {
      cudaEventRecord(e->ev[1], st);
      cudaEventSynchronize(e->ev[1]);
      float ms;
      cudaEventElapsedTime(&ms, e->ev[0], e->ev[1]);
      e->kt.accept_ms += ms; /* reported as the dominant kernel of the fused path */
      e->kt.launches++;
    }
    return GPX_OK;
  }
  const Sink sk = e->sink();
  int rc = launch_propose(e, sk, d_reqs, d_payload, pal, n, d_status, st);
  if (rc) return rc;
  if (tm) cudaEventRecord(e->ev[1], st);
  /* the ACCEPT segment mirrors the payload arena plus the constructed blobs actually used */
  rc = launch_accept(e, sk, compact, sk.accepts, &sk.ctl->n_accepts, n, d_payload, pal, e->d_blob1, 0,
                     &sk.ctl->blob1_used, e->d_replies, e->d_decisions, d_exec, st);
  if (rc) return rc;
  if (tm) cudaEventRecord(e->ev[2], st);
  if (!compact) {
    rc = launch_tally(e, sk, e->d_replies, &sk.ctl->n_accepts, L, n * L, e->d_decisions, st);
    if (rc) return rc;
  }
  if (tm) cudaEventRecord(e->ev[3], st); /* compact: the tally and commit intervals are empty */
  if (!compact) {
    rc = launch_commit(e, sk, e->d_decisions, &sk.ctl->n_decisions, n, d_exec, st);
    if (rc) return rc;
  }
  if (tm) {
    cudaEventRecord(e->ev[4], st);
    cudaEventSynchronize(e->ev[4]);
    float ms;
    cudaEventElapsedTime(&ms, e->ev[0], e->ev[1]);
    e->kt.propose_ms += ms;
    cudaEventElapsedTime(&ms, e->ev[1], e->ev[2]);
    e->kt.accept_ms += ms;
    cudaEventElapsedTime(&ms, e->ev[2], e->ev[3]);
    e->kt.tally_ms += ms;
    cudaEventElapsedTime(&ms, e->ev[3], e->ev[4]);
    e->kt.commit_ms += ms;
    e->kt.launches++;
  }
  return GPX_OK;
}

int gpx_set_round_mode(gpx_engine* e, int mode) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (mode < 0 || mode > 2) return fail(GPX_EINVAL, "round mode: 0 / 1 device tail launch, 2 host-launched pair");
  e->round_mode = mode;
  return GPX_OK;
}

static int round_host(gpx_engine* e, RoundForm form, uint32_t n, const gpx_request_rec* reqs, const uint8_t* payload,
                      uint64_t payload_bytes, int32_t* status, gpx_exec_rec* out_exec, uint32_t* n_exec_slots,
                      gpx_exec_rec* out_extra_exec, uint32_t extra_cap, uint32_t* n_extra) {
  if (!e || !n_exec_slots) return fail(GPX_EINVAL, "null argument");
  *n_exec_slots = 0;
  if (n_extra) *n_extra = 0;
  if (n == 0) return GPX_OK;
  if (!reqs || !status || !out_exec || (!payload && payload_bytes)) return fail(GPX_EINVAL, "null argument");
  int rc = check_batch(e, n, payload_bytes);
  if (rc) return rc;
  const LogSegs segs = round_segs(e, form, n, payload_bytes);
  rc = ring_fits(e, segs);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  const uint32_t L = e->cfg.n_lanes;
  CK(cudaMemcpyAsync(e->d_reqs, reqs, n * sizeof(gpx_request_rec), cudaMemcpyHostToDevice, st));
  if (payload_bytes) CK(cudaMemcpyAsync(e->d_payload, payload, payload_bytes, cudaMemcpyHostToDevice, st));
  rc = round_on_stream(e, form, segs, e->d_reqs, e->d_payload, payload_bytes, n, e->d_status, e->d_exec, st);
  if (rc) return rc;
  CK(cudaMemcpyAsync(status, e->d_status, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  rc = fetch_ctl(e, form == RoundForm::FUSED ? e->last_ctl : nullptr);
  if (rc) return rc;
  /* fused: one EXEC row per REQUEST index (VOID where the request carries no ACCEPT); phases: one per DECISION */
  const uint32_t rows = form == RoundForm::FUSED ? n : e->h_ctl->n_decisions;
  if (rows) CK(cudaMemcpyAsync(out_exec, e->d_exec, (size_t)rows * L * sizeof(gpx_exec_rec), cudaMemcpyDeviceToHost, st));
  rc = copy_extra_out(e, out_extra_exec, extra_cap, n_extra);
  if (rc) return rc;
  CK(cudaStreamSynchronize(st));
  *n_exec_slots = rows * L;
  return GPX_OK;
}

int gpx_round(gpx_engine* e, uint32_t n, const gpx_request_rec* reqs, const uint8_t* payload, uint64_t payload_bytes,
              int32_t* status, gpx_exec_rec* out_exec, uint32_t* n_exec_slots, gpx_exec_rec* out_extra_exec,
              uint32_t extra_cap, uint32_t* n_extra) {
  return round_host(e, RoundForm::FUSED, n, reqs, payload, payload_bytes, status, out_exec, n_exec_slots,
                    out_extra_exec, extra_cap, n_extra);
}
int gpx_round_phases(gpx_engine* e, uint32_t n, const gpx_request_rec* reqs, const uint8_t* payload,
                     uint64_t payload_bytes, int32_t* status, gpx_exec_rec* out_exec, uint32_t* n_exec_slots,
                     gpx_exec_rec* out_extra_exec, uint32_t extra_cap, uint32_t* n_extra) {
  return round_host(e, RoundForm::PHASES, n, reqs, payload, payload_bytes, status, out_exec, n_exec_slots,
                    out_extra_exec, extra_cap, n_extra);
}

static int round_device(gpx_engine* e, RoundForm form, const gpx_dev_round_bufs* b, void* stream) {
  if (!e || !b) return fail(GPX_EINVAL, "null argument");
  if (b->n == 0) return GPX_OK;
  int rc = check_batch(e, b->n, b->payload_bytes);
  if (rc) return rc;
  const LogSegs segs = round_segs(e, form, b->n, b->payload_bytes);
  rc = ring_fits(e, segs);
  if (rc) return rc;
  return round_on_stream(e, form, segs, b->reqs, b->payload, b->payload_bytes, b->n, b->status, b->exec,
                         stream ? (cudaStream_t)stream : e->stream);
}
int gpx_round_device(gpx_engine* e, const gpx_dev_round_bufs* b, void* stream) {
  return round_device(e, RoundForm::FUSED, b, stream);
}
/* k_propose (ACCEPTs compacted at the front: one record, log image and EXEC row per ACCEPT, no per-request holes) +
 * k_act (accept -> tally -> commit per ACCEPT in registers): the form for batches in which most requests share a
 * slot with others (RequestBatcher.java:198-219) */
int gpx_round_device_compact(gpx_engine* e, const gpx_dev_round_bufs* b, void* stream) {
  return round_device(e, RoundForm::COMPACT, b, stream);
}
int gpx_round_device_phases(gpx_engine* e, const gpx_dev_round_bufs* b, void* stream) {
  return round_device(e, RoundForm::PHASES, b, stream);
}

/* ---- device-resident phase calls (spread placement) -------------------------------------- */
static_assert(sizeof(gpx_dev_ctl) == sizeof(RoundCtl), "gpx_dev_ctl mirrors RoundCtl");

int gpx_propose_device(gpx_engine* e, const gpx_request_rec* reqs, const uint8_t* payload, uint64_t payload_bytes,
                       uint32_t n, int32_t* status, gpx_accept_rec* out_accepts, gpx_dev_ctl* ctl, void* stream) {
  if (!e || !ctl) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  if (!reqs || !status || !out_accepts || (!payload && payload_bytes)) return fail(GPX_EINVAL, "null argument");
  int rc = check_batch(e, n, payload_bytes);
  if (rc) return rc;
  Sink sk = e->sink(ctl);
  sk.accepts = out_accepts;
  return launch_propose(e, sk, reqs, payload, (payload_bytes + 15) & ~15ull, n, status,
                        stream ? (cudaStream_t)stream : e->stream);
}

int gpx_route_device(gpx_engine* e, uint32_t kind, const void* recs, const uint32_t* n_ptr, uint32_t n_max,
                     const uint8_t* payload, uint64_t payload_bytes, uint32_t n_dest, const int32_t* dest_nodes,
                     void* out_recs, uint32_t cap, uint32_t* out_counts, uint8_t* out_blob, uint64_t blob_cap,
                     uint32_t* out_blob_units, uint32_t* dropped, void* stream) {
  if (!e || !recs || !dest_nodes || !out_recs || !out_counts) return fail(GPX_EINVAL, "null argument");
  if (kind != GPX_F_ACCEPT && kind != GPX_F_DECISION && kind != 0) return fail(GPX_EINVAL, "bad record kind");
  if (n_dest == 0 || n_dest > GPX_ROUTE_ND) return fail(GPX_EINVAL, "n_dest out of range");
  if (kind == GPX_F_ACCEPT && (!out_blob || !out_blob_units || (blob_cap & 15))) return fail(GPX_EINVAL, "blob buckets");
  if (n_max == 0) return GPX_OK;
  RouteArgs A;
  memset(&A, 0, sizeof A);
  A.recs = (const uint8_t*)recs;
  A.n_ptr = n_ptr;
  A.n_max = n_max;
  A.kind = kind;
  A.n_dest = n_dest;
  for (uint32_t d = 0; d < n_dest; d++) A.dest_node[d] = dest_nodes[d];
  A.out_recs = (uint8_t*)out_recs;
  A.cap = cap;
  A.out_counts = out_counts;
  A.blob0 = payload;
  A.blob0_bytes = (payload_bytes + 15) & ~15ull;
  A.blob1 = e->d_blob1;
  A.out_blob = out_blob;
  A.blob_cap = blob_cap;
  A.out_blob_units = out_blob_units;
  A.dropped = dropped;
  k_route<<<cdiv(n_max, GPX_BLOCK), GPX_BLOCK, 0, stream ? (cudaStream_t)stream : e->stream>>>(e->S, A);
  CK(cudaGetLastError());
  return GPX_OK;
}

int gpx_accepts_device(gpx_engine* e, gpx_accept_rec* recs, uint32_t n, const uint8_t* blob, uint64_t blob_bytes,
                       uint32_t n_chunks, const uint32_t* chunk_rec_end, const uint64_t* chunk_blob_base,
                       gpx_accept_reply_rec* out_replies, gpx_exec_rec* out_extra, uint32_t extra_cap,
                       gpx_dev_ctl* ctl, void* stream) {
  if (!e || !ctl) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  if (!recs || !out_replies || (!blob && blob_bytes)) return fail(GPX_EINVAL, "null argument");
  if (blob_bytes & 15) return fail(GPX_EINVAL, "blob_bytes must be a multiple of 16");
  if (n_chunks > GPX_ROUTE_ND || (n_chunks && (!chunk_rec_end || !chunk_blob_base))) return fail(GPX_EINVAL, "chunks");
  if (n > e->cfg.max_batch_recs) return fail(GPX_ERANGE, "n > max_batch_recs");
  const LogSegs segs = one_seg(seg_accept_bytes(n, blob_bytes));
  int rc = ring_fits(e, segs);
  if (rc) return rc;
  cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
  {
    IngestArgs R;
    memset(&R, 0, sizeof R);
    R.recs = (uint8_t*)recs;
    R.rec_bytes = 48;
    R.n = n;
    R.n_chunks = n_chunks;
    for (uint32_t c = 0; c < n_chunks; c++) {
      R.rec_end[c] = chunk_rec_end[c];
      R.blob_base[c] = chunk_blob_base[c];
    }
    k_ingest<<<cdiv(n, GPX_BLOCK), GPX_BLOCK, 0, st>>>(e->S, R);
  }
  log_advance(e, segs);
  return launch_accept(e, e->sink(ctl, out_extra, extra_cap), false, recs, nullptr, n, blob, blob_bytes, nullptr, 0,
                       nullptr, out_replies, nullptr, nullptr, st);
}

int gpx_replies_device(gpx_engine* e, const gpx_accept_reply_rec* replies, uint32_t n,
                       gpx_decision_rec* out_decisions, gpx_dev_ctl* ctl, void* stream) {
  if (!e || !ctl) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  if (!replies || !out_decisions) return fail(GPX_EINVAL, "null argument");
  return launch_tally(e, e->sink(ctl), replies, nullptr, 1, n, out_decisions, stream ? (cudaStream_t)stream : e->stream);
}

int gpx_decisions_device(gpx_engine* e, gpx_decision_rec* decisions, uint32_t n, gpx_exec_rec* out_exec,
                         gpx_exec_rec* out_extra, uint32_t extra_cap, gpx_dev_ctl* ctl, void* stream) {
  if (!e || !ctl) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  if (!decisions || !out_exec) return fail(GPX_EINVAL, "null argument");
  if (n > e->cfg.max_batch_recs) return fail(GPX_ERANGE, "n > max_batch_recs");
  const LogSegs segs = one_seg(seg_decision_bytes(n));
  int rc = ring_fits(e, segs);
  if (rc) return rc;
  cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
  {
    IngestArgs R;
    memset(&R, 0, sizeof R);
    R.recs = (uint8_t*)decisions;
    R.rec_bytes = 32;
    R.n = n;
    k_ingest<<<cdiv(n, GPX_BLOCK), GPX_BLOCK, 0, st>>>(e->S, R);
  }
  log_advance(e, segs);
  return launch_commit(e, e->sink(ctl, out_extra, extra_cap), decisions, nullptr, n, out_exec, st);
}

/* ---- pipelined rounds ---------------------------------------------------------------- */
static int pipe_init(gpx_engine* e) {
  if (e->pipe_ready) return GPX_OK;
  const size_t N = e->cfg.max_batch_recs, L = e->cfg.n_lanes;
  const uint64_t P = (e->cfg.max_batch_payload + 15) & ~15ull;
  int rc;
  for (auto& ps : e->pipe) {
    if ((rc = e->dalloc(&ps.d_reqs, N)) || (rc = e->dalloc(&ps.d_payload, (size_t)P)) ||
        (rc = e->dalloc(&ps.d_status, N)) || (rc = e->dalloc(&ps.d_exec, N * L)) || (rc = e->dalloc(&ps.d_sum, N)) ||
        (rc = e->dalloc(&ps.d_packed, N)) || (rc = e->dalloc(&ps.d_bsum, N / GPX_UNPACK_PER_BLOCK + 2)) ||
        (rc = e->dalloc(&ps.d_extra, N * (L + 1))) || /* compact mode: the general path reports here */ (rc = e->dalloc(&ps.d_ctl, (size_t)2)))
      return rc;
    if (cudaHostAlloc((void**)&ps.h_ctl, sizeof(RoundCtl), cudaHostAllocDefault) != cudaSuccess)
      return fail(GPX_ENOMEM, "cudaHostAlloc");
    CK(cudaMemset(ps.d_ctl, 0, 2 * sizeof(RoundCtl)));
    CK(cudaEventCreateWithFlags(&ps.ev_h2d, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ps.ev_k, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ps.ev_d2h, cudaEventDisableTiming));
  }
  CK(cudaStreamCreateWithFlags(&e->s_h2d, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&e->s_d2h, cudaStreamNonBlocking));
  e->pipe_ready = true;
  return GPX_OK;
}

int gpx_round_submit(gpx_engine* e, const gpx_round_io* io, uint64_t* ticket) {
  if (!e || !io || !ticket) return fail(GPX_EINVAL, "null argument");
  const uint32_t n = io->n;
  const bool compact = (io->flags & GPX_ROUND_COMPACT) != 0;
  const bool packed = (io->flags & GPX_ROUND_PACKED_REQS) != 0;
  if (io->flags & ~(GPX_ROUND_COMPACT | GPX_ROUND_PACKED_REQS)) return fail(GPX_EINVAL, "unknown round flags");
  if (n && (!io->reqs || (!io->payload && io->payload_bytes))) return fail(GPX_EINVAL, "null argument");
  if (n && (compact ? !io->sum : (!io->status || !io->exec))) return fail(GPX_EINVAL, "null output buffer");
  int rc = check_batch(e, n, io->payload_bytes);
  if (rc) return rc;
  const uint64_t pal = (io->payload_bytes + 15) & ~15ull;
  const LogSegs segs = round_segs(e, RoundForm::FUSED, n, io->payload_bytes);
  rc = ring_fits(e, segs);
  if (rc) return rc;
  rc = pipe_init(e);
  if (rc) return rc;
  gpx_engine::PipeSlot& ps = e->pipe[e->next_ticket % GPX_PIPE_DEPTH];
  if (ps.busy) return fail(GPX_ERANGE, "GPX_PIPE_DEPTH rounds in flight: call gpx_round_wait first");
  ps.busy = true;
  ps.ticket = e->next_ticket;
  ps.io = *io;
  *ticket = e->next_ticket++;
  if (n == 0) return GPX_OK;
  const uint32_t L = e->cfg.n_lanes;
  /* stream 1: inputs.  (the slot's previous round was waited for, so its buffers are free) */
  if (packed)
    CK(cudaMemcpyAsync(ps.d_packed, io->reqs, n * sizeof(gpx_request_packed), cudaMemcpyHostToDevice, e->s_h2d));
  else
    CK(cudaMemcpyAsync(ps.d_reqs, io->reqs, n * sizeof(gpx_request_rec), cudaMemcpyHostToDevice, e->s_h2d));
  if (io->payload_bytes)
    CK(cudaMemcpyAsync(ps.d_payload, io->payload, io->payload_bytes, cudaMemcpyHostToDevice, e->s_h2d));
  CK(cudaMemsetAsync(ps.d_ctl, 0, sizeof(RoundCtl), e->s_h2d)); /* the slot's control block: the round counts into it */
  CK(cudaEventRecord(ps.ev_h2d, e->s_h2d));
  /* stream 2: the round (serialised with every other engine call on the engine's stream) */
  CK(cudaStreamWaitEvent(e->stream, ps.ev_h2d, 0));
  if (packed) { /* expand the 16-byte requests: payload_off = running sum of payload_len */
    const uint32_t nb = cdiv(n, GPX_UNPACK_PER_BLOCK);
    k_unpack_sums<<<nb, GPX_BLOCK, 0, e->stream>>>(ps.d_packed, n, ps.d_bsum);
    k_unpack_scan<<<1, GPX_BLOCK, 0, e->stream>>>(ps.d_bsum, nb);
    k_unpack_expand<<<nb, GPX_BLOCK, 0, e->stream>>>(e->S, ps.d_packed, n, ps.d_bsum, ps.d_reqs);
    CK(cudaGetLastError());
  }
  log_advance(e, segs);
  rc = launch_round(e, ps.d_reqs, ps.d_payload, pal, n, ps.d_status, ps.d_exec, e->stream, ps.d_ctl, ps.d_extra,
                    (uint32_t)std::min<uint64_t>((uint64_t)e->cfg.max_batch_recs * (L + 1), 0xffffffffull),
                    compact ? ps.d_sum : nullptr);
  if (rc) return rc;
  CK(cudaEventRecord(ps.ev_k, e->stream));
  /* stream 3: results */
  CK(cudaStreamWaitEvent(e->s_d2h, ps.ev_k, 0));
  CK(cudaMemcpyAsync(ps.h_ctl, e->last_ctl, sizeof(RoundCtl), cudaMemcpyDeviceToHost, e->s_d2h));
  if (compact) {
    CK(cudaMemcpyAsync(io->sum, ps.d_sum, n * sizeof(gpx_exec_sum), cudaMemcpyDeviceToHost, e->s_d2h));
  } else {
    CK(cudaMemcpyAsync(io->status, ps.d_status, n * sizeof(int32_t), cudaMemcpyDeviceToHost, e->s_d2h));
    CK(cudaMemcpyAsync(io->exec, ps.d_exec, (size_t)n * L * sizeof(gpx_exec_rec), cudaMemcpyDeviceToHost, e->s_d2h));
  }
  CK(cudaEventRecord(ps.ev_d2h, e->s_d2h));
  return GPX_OK;
}

int gpx_round_wait(gpx_engine* e, uint64_t ticket, uint32_t* n_exec_slots, uint32_t* n_extra) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (n_exec_slots) *n_exec_slots = 0;
  if (n_extra) *n_extra = 0;
  if (ticket != e->next_wait || ticket >= e->next_ticket) return fail(GPX_EINVAL, "rounds are waited for in submission order");
  gpx_engine::PipeSlot& ps = e->pipe[ticket % GPX_PIPE_DEPTH];
  e->next_wait++;
  ps.busy = false;
  if (ps.io.n == 0) return GPX_OK;
  CK(cudaEventSynchronize(ps.ev_d2h));
  const uint32_t nx = ps.h_ctl->n_extra;
  const uint32_t cp = (uint32_t)std::min<uint64_t>(std::min(nx, ps.io.extra_cap),
                                                  (uint64_t)e->cfg.max_batch_recs * (e->cfg.n_lanes + 1));
  if (cp && ps.io.extra) { /* rare: executions beyond the one per (request, lane) */
    CK(cudaMemcpyAsync(ps.io.extra, ps.d_extra, cp * sizeof(gpx_exec_rec), cudaMemcpyDeviceToHost, e->s_d2h));
    CK(cudaStreamSynchronize(e->s_d2h));
  }
  if (n_exec_slots) *n_exec_slots = (ps.io.flags & GPX_ROUND_COMPACT) ? 0 : ps.io.n * e->cfg.n_lanes;
  if (n_extra) *n_extra = nx;
  return GPX_OK;
}

/* RequestPacket.getDigest :1414-1430 for a batch of requests (the digest column of DIGEST_REQUESTS mode) */
int gpx_digest_requests(gpx_engine* e, uint32_t n, const gpx_request_rec* reqs, const uint8_t* payload,
                        uint64_t payload_bytes, uint8_t* out_digests) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  if (!reqs || !out_digests || (!payload && payload_bytes)) return fail(GPX_EINVAL, "null argument");
  int rc = check_batch(e, n, payload_bytes);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  CK(cudaMemcpyAsync(e->d_reqs, reqs, n * sizeof(gpx_request_rec), cudaMemcpyHostToDevice, st));
  if (payload_bytes) CK(cudaMemcpyAsync(e->d_payload, payload, payload_bytes, cudaMemcpyHostToDevice, st));
  /* digests go to the blob scratch (16 B per request fits: blob1_cap >= 16 * max_batch_recs) */
  k_md5<<<cdiv(n, GPX_BLOCK), GPX_BLOCK, 0, st>>>(e->d_reqs, n, e->d_payload, e->d_blob1);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out_digests, e->d_blob1, 16ull * n, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return GPX_OK;
}

int gpx_enable_kernel_timing(gpx_engine* e, int on) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  e->timing = on != 0;
  return GPX_OK;
}
int gpx_get_kernel_times(gpx_engine* e, gpx_kernel_times* out, int reset) {
  if (!e || !out) return fail(GPX_EINVAL, "null argument");
  *out = e->kt;
  if (reset) memset(&e->kt, 0, sizeof e->kt);
  return GPX_OK;
}

/* ---- log ring ----------------------------------------------------------------------- */
int gpx_log_read(gpx_engine* e, uint32_t lane, uint64_t from, void* dst, uint64_t cap, uint64_t* n_copied,
                 uint64_t* head) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  uint64_t heads[GPX_MAX_LANES];
  int err = read_device_heads(e, heads);
  if (err) return err;
  const uint64_t h = heads[lane], rc = e->S.ring_cap;
  if (head) *head = h;
  uint64_t nb = 0;
  if (dst && from < h) {
    nb = std::min<uint64_t>(cap, h - from);
    if (h - from > rc) return fail(GPX_ERANGE, "requested bytes were already overwritten");
    uint64_t pos = from & (rc - 1);
    uint64_t first = std::min<uint64_t>(nb, rc - pos);
    CK(cudaMemcpy(dst, e->S.ring[lane] + pos, first, cudaMemcpyDeviceToHost));
    if (nb > first) CK(cudaMemcpy((uint8_t*)dst + first, e->S.ring[lane], nb - first, cudaMemcpyDeviceToHost));
  }
  if (n_copied) *n_copied = nb;
  return GPX_OK;
}

/* the journal's index as a scan: k_log_dir -> k_log_scan -> k_log_hits (gpx_logfind.cuh) */
int gpx_log_find(gpx_engine* e, uint32_t lane, uint64_t from, uint32_t n, const gpx_log_want* wants, gpx_log_hit* out) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  if (n == 0) return GPX_OK;
  if (!wants || !out) return fail(GPX_EINVAL, "null argument");
  if (from & 31) return fail(GPX_EINVAL, "from is not a segment boundary");
  for (uint32_t i = 0; i < n; i++) {
    if (wants[i].n_slots > GPX_LOG_SPAN) return fail(GPX_ERANGE, "n_slots > GPX_LOG_SPAN");
    if (i && wants[i - 1].gid >= wants[i].gid) return fail(GPX_EINVAL, "wants must be sorted by gid, one per group");
  }
  CK(cudaDeviceSynchronize()); /* rounds may have been issued on a caller's stream; the head is read on the device */
  const size_t cells = (size_t)n * GPX_LOG_SPAN;
  /* a segment is at least 96 bytes; a directory of 2^20 entries (32 MiB) covers every ring the launches of this engine
   * can fill with fewer segments than that, else LOGF_TOO_MANY */
  const uint64_t seg_cap64 = std::min<uint64_t>(e->cfg.log_ring_bytes / 96 + 2, 1ull << 20);
  const size_t want_bytes = ((size_t)n * sizeof(gpx_log_want) + 31) & ~(size_t)31;
  const size_t seg_bytes = (size_t)seg_cap64 * sizeof(LogSeg);
  const size_t best_bytes = 2 * cells * 8;
  const size_t hit_bytes = cells * sizeof(gpx_log_hit);
  int rc = e->ensure_misc(want_bytes + seg_bytes + 32 + best_bytes + hit_bytes);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  uint8_t* base = (uint8_t*)e->d_misc;
  LogFindArgs A;
  A.lane = lane;
  A.n = n;
  A.from = from;
  A.wants = (const gpx_log_want*)base;
  A.segs = (LogSeg*)(base + want_bytes);
  A.seg_cap = (uint32_t)seg_cap64;
  A.ctl = (unsigned long long*)(base + want_bytes + seg_bytes);
  A.best = A.ctl + 4;
  A.hits = (gpx_log_hit*)(base + want_bytes + seg_bytes + 32 + best_bytes);
  CK(cudaMemcpyAsync(base, wants, (size_t)n * sizeof(gpx_log_want), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(A.ctl, 0, 32 + best_bytes, st));
  k_log_dir<<<1, 32, 0, st>>>(e->S, A);
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device);
  k_log_scan<<<(unsigned)sms * 8u, GPX_LOGF_BLOCK, 0, st>>>(e->S, A);
  k_log_hits<<<cdiv(cells, GPX_LOGF_BLOCK), GPX_LOGF_BLOCK, 0, st>>>(e->S, A);
  CK(cudaGetLastError());
  unsigned long long ctl[4];
  CK(cudaMemcpyAsync(ctl, A.ctl, sizeof ctl, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(out, A.hits, hit_bytes, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (ctl[LOGF_ERR] == LOGF_OVERWRITTEN) return fail(GPX_ERANGE, "bytes from `from` on were already overwritten");
  if (ctl[LOGF_ERR] == LOGF_CORRUPT) return fail(GPX_EINVAL, "`from` is not a segment boundary");
  if (ctl[LOGF_ERR] == LOGF_TOO_MANY) return fail(GPX_ERANGE, "more log segments than the scan's directory holds");
  return GPX_OK;
}

/* the bodies of a batch of hits in one copy: k_log_gather (gpx_logfind.cuh) packs them into a staging buffer */
int gpx_log_gather(gpx_engine* e, uint32_t lane, uint32_t n, const gpx_log_range* ranges, void* dst, uint64_t dst_bytes) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  if (n == 0) return GPX_OK;
  if (!ranges || !dst) return fail(GPX_EINVAL, "null argument");
  uint64_t heads[GPX_MAX_LANES];
  int rc = read_device_heads(e, heads);
  if (rc) return rc;
  const uint64_t head = heads[lane], cap = e->S.ring_cap;
  std::vector<uint32_t> first(n + 1);
  uint64_t chunks = 0, top = 0;
  for (uint32_t i = 0; i < n; i++) {
    const uint64_t nc = ((uint64_t)ranges[i].len + 15) >> 4;
    if ((ranges[i].pos & 15) || (ranges[i].dst_off & 15)) return fail(GPX_EINVAL, "range not on a 16-byte boundary");
    if (ranges[i].pos + 16 * nc > head || head - ranges[i].pos > cap) return fail(GPX_ERANGE, "range outside the live ring bytes");
    if ((ranges[i].pos & (cap - 1)) + 16 * nc > cap) return fail(GPX_ERANGE, "range straddles the ring end");
    if ((uint64_t)ranges[i].dst_off + 16 * nc > dst_bytes) return fail(GPX_ERANGE, "range beyond dst");
    first[i] = (uint32_t)chunks;
    chunks += nc;
    top = std::max<uint64_t>(top, (uint64_t)ranges[i].dst_off + 16 * nc);
    if (chunks > 0xffffffffull) return fail(GPX_ERANGE, "too many bytes for one gather");
  }
  first[n] = (uint32_t)chunks;
  if (chunks == 0) return GPX_OK;
  const size_t r_bytes = ((size_t)n * sizeof(gpx_log_range) + 15) & ~(size_t)15;
  const size_t f_bytes = ((size_t)(n + 1) * 4 + 15) & ~(size_t)15;
  rc = e->ensure_misc(r_bytes + f_bytes + top);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  uint8_t* base = (uint8_t*)e->d_misc;
  CK(cudaMemcpyAsync(base, ranges, (size_t)n * sizeof(gpx_log_range), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(base + r_bytes, first.data(), (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, st));
  LogGatherArgs A;
  A.lane = lane;
  A.n = n;
  A.ranges = (const gpx_log_range*)base;
  A.first_chunk = (const uint32_t*)(base + r_bytes);
  A.out = (int4*)(base + r_bytes + f_bytes);
  CK(cudaMemsetAsync(A.out, 0, top, st)); /* gaps between ranges read as zero */
  k_log_gather<<<cdiv(chunks, GPX_LOGF_BLOCK), GPX_LOGF_BLOCK, 0, st>>>(e->S, A);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(dst, A.out, top, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return GPX_OK;
}

/* Asynchronous drain (SQLPaxosLogger.journal :965-1036 appends the batch to the journal file; here the caller's
 * page-locked buffer stands for the file's write buffer).  Everything is enqueued: the copy runs on the engine's
 * drain stream behind the work already enqueued on `after_stream` (NULL = the engine's stream) and overlaps later
 * rounds. */
int gpx_log_drain_async(gpx_engine* e, uint32_t lane, void* dst, uint64_t cap, uint64_t* from, uint64_t* n_bytes,
                        void* after_stream) {
  if (!e || !dst || !from || !n_bytes) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  int rc = log_resync(e);
  if (rc) return rc;
  if (!e->s_drain) {
    CK(cudaStreamCreateWithFlags(&e->s_drain, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&e->ev_drain, cudaEventDisableTiming));
  }
  const uint64_t rc_ = e->S.ring_cap, f = e->drain_pos[lane], h = e->h_head[lane];
  if (h - f > rc_) return fail(GPX_ERANGE, "undrained bytes were already overwritten (enable log_backpressure)");
  const uint64_t nb = std::min<uint64_t>(cap, h - f);
  *from = f;
  *n_bytes = nb;
  if (!nb) return GPX_OK;
  CK(cudaEventRecord(e->ev_drain, after_stream ? (cudaStream_t)after_stream : e->stream));
  CK(cudaStreamWaitEvent(e->s_drain, e->ev_drain, 0));
  const uint64_t pos = f & (rc_ - 1), first = std::min<uint64_t>(nb, rc_ - pos);
  CK(cudaMemcpyAsync(dst, e->S.ring[lane] + pos, first, cudaMemcpyDeviceToHost, e->s_drain));
  if (nb > first)
    CK(cudaMemcpyAsync((uint8_t*)dst + first, e->S.ring[lane], nb - first, cudaMemcpyDeviceToHost, e->s_drain));
  e->drain_pos[lane] = f + nb;
  return GPX_OK;
}
/* forget the undrained backlog: the drain cursor and the tail jump to the current heads (a caller that ran with the
 * journal disabled and now turns it on) */
int gpx_log_drain_skip(gpx_engine* e) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  int rc = log_resync(e);
  if (rc) return rc;
  for (uint32_t l = 0; l < e->cfg.n_lanes; l++) e->drain_pos[l] = e->log_tail[l] = e->h_head[l];
  return GPX_OK;
}
int gpx_log_drain_wait(gpx_engine* e) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (e->s_drain) CK(cudaStreamSynchronize(e->s_drain));
  return GPX_OK;
}
int gpx_log_release(gpx_engine* e, uint32_t lane, uint64_t upto) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  if (upto > e->drain_pos[lane]) return fail(GPX_EINVAL, "release beyond the drained position");
  if (upto > e->log_tail[lane]) e->log_tail[lane] = upto;
  return GPX_OK;
}

/* ---- introspection ------------------------------------------------------------------- */
int gpx_get_counters(gpx_engine* e, gpx_counters* out) {
  if (!e || !out) return fail(GPX_EINVAL, "null argument");
  CK(cudaDeviceSynchronize()); /* rounds may have been issued on a caller's stream (gpx_round_device) */
  std::vector<unsigned long long> rawv((size_t)C_NCTR * GPX_CTR_STRIPES);
  unsigned long long* raw = rawv.data();
  unsigned long long c[C_NCTR];
  CK(cudaMemcpy(raw, e->S.ctr, rawv.size() * 8, cudaMemcpyDeviceToHost));
  for (int i = 0; i < C_NCTR; i++) {
    c[i] = 0;
    for (int s = 0; s < GPX_CTR_STRIPES; s++) c[i] += raw[s * C_NCTR + i];
  }
  { /* fold the fast-path aggregates of k_round (gpx_dev.cuh) */
    const unsigned long long fl = c[C_FAST_LANES], ft = c[C_FAST_TEAMS], fc = c[C_FAST_CKPT];
    c[C_ACCEPTS_HANDLED] += fl;
    c[C_ACCEPTS_ACKED] += fl;
    c[C_ACCEPTS_LOGGED] += fl;
    c[C_REPLIES_HANDLED] += fl;
    c[C_DECISIONS_HANDLED] += fl;
    c[C_EXECUTED] += fl;
    c[C_CKPTS_DUE] += fc;
    c[C_PROPOSALS] += ft;
    c[C_REQS_BATCHED] += ft;
    c[C_DECISIONS_MADE] += ft;
  }
  memset(out, 0, sizeof *out);
  uint64_t* o = (uint64_t*)out;
  for (int i = 0; i < 24 && i < (int)(sizeof(gpx_counters) / 8); i++) o[i] = c[i];
  return GPX_OK;
}
int gpx_reset_counters(gpx_engine* e) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  CK(cudaMemset(e->S.ctr, 0, C_NCTR * GPX_CTR_STRIPES * 8));
  return GPX_OK;
}
int gpx_get_group_flags(gpx_engine* e, uint32_t lane, uint32_t n, const uint32_t* gids, uint8_t* out) {
  if (!e || !gids || !out) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  if (n == 0) return GPX_OK;
  size_t goff = ((size_t)n + 255) & ~(size_t)255;
  int rc = e->ensure_misc(goff + n * 4ull);
  if (rc) return rc;
  uint32_t* d_g = (uint32_t*)((uint8_t*)e->d_misc + goff);
  CK(cudaMemcpyAsync(d_g, gids, n * 4ull, cudaMemcpyHostToDevice, e->stream));
  k_get_flags<<<cdiv(n, 256), 256, 0, e->stream>>>(e->S, lane, d_g, n, (uint8_t*)e->d_misc);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, e->d_misc, n, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return GPX_OK;
}

/* the slow-path list / the candidates of a sweep: one launch of k_select_groups over all gids (gpx_pause.cuh) */
int gpx_select_groups(gpx_engine* e, uint32_t lane, uint32_t mask, uint32_t value, uint32_t* out_gids, uint32_t cap,
                      uint32_t* n_found) {
  if (!e || !n_found || (!out_gids && cap)) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  int rc = e->ensure_misc(16 + (size_t)cap * 4);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  uint8_t* base = (uint8_t*)e->d_misc;
  SelectArgs A;
  A.lane = lane;
  A.mask = mask;
  A.value = value;
  A.cap = cap;
  A.n_found = (unsigned long long*)base;
  A.gids = (uint32_t*)(base + 16);
  CK(cudaMemsetAsync(base, 0, 16, st));
  k_select_groups<<<cdiv(e->cfg.max_groups, GPX_PAUSE_BLOCK), GPX_PAUSE_BLOCK, 0, st>>>(e->S, A);
  CK(cudaGetLastError());
  unsigned long long found = 0;
  CK(cudaMemcpyAsync(&found, A.n_found, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const uint32_t got = (uint32_t)std::min<unsigned long long>(found, cap);
  if (got) {
    CK(cudaMemcpyAsync(out_gids, A.gids, (size_t)got * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    std::sort(out_gids, out_gids + got);
  }
  *n_found = (uint32_t)std::min<unsigned long long>(found, 0xffffffffull);
  return GPX_OK;
}

/* the fields of a SYNC_DECISIONS_REQUEST for a batch of groups: one launch of k_missing_decisions (gpx_pause.cuh) */
int gpx_missing_decisions(gpx_engine* e, uint32_t lane, uint32_t n, const uint32_t* gids, int32_t size_limit,
                          int32_t too_much_gap, gpx_missing_rec* out) {
  if (!e || ((!gids || !out) && n)) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  if (n == 0) return GPX_OK;
  const size_t gid_bytes = ((size_t)n * 4 + 15) & ~(size_t)15;
  int rc = e->ensure_misc(gid_bytes + (size_t)n * sizeof(gpx_missing_rec));
  if (rc) return rc;
  cudaStream_t st = e->stream;
  uint8_t* base = (uint8_t*)e->d_misc;
  CK(cudaMemcpyAsync(base, gids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  MissingArgs A;
  A.lane = lane;
  A.n = n;
  A.gids = (const uint32_t*)base;
  A.size_limit = size_limit;
  A.too_much_gap = too_much_gap;
  A.out = (gpx_missing_rec*)(base + gid_bytes);
  k_missing_decisions<<<cdiv(n, GPX_PAUSE_BLOCK), GPX_PAUSE_BLOCK, 0, st>>>(e->S, A);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, A.out, (size_t)n * sizeof(gpx_missing_rec), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return GPX_OK;
}

int gpx_clear_group_flags(gpx_engine* e, uint32_t lane, uint32_t n, const uint32_t* gids, uint32_t mask) {
  if (!e || (!gids && n)) return fail(GPX_EINVAL, "null argument");
  if (lane >= e->cfg.n_lanes) return fail(GPX_ERANGE, "lane");
  if (n == 0) return GPX_OK;
  { /* two threads must not read-modify-write the same word */
    std::vector<uint32_t> g(gids, gids + n);
    std::sort(g.begin(), g.end());
    if (std::adjacent_find(g.begin(), g.end()) != g.end()) return fail(GPX_EINVAL, "a gid appears twice in the batch");
  }
  int rc = e->ensure_misc((size_t)n * 4);
  if (rc) return rc;
  CK(cudaMemcpyAsync(e->d_misc, gids, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  k_clear_flags<<<cdiv(n, 128), 128, 0, e->stream>>>(e->S, lane, (const uint32_t*)e->d_misc, n, mask);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(e->stream));
  return GPX_OK;
}

/* the deactivation sweep: one launch of k_pause_groups (gpx_pause.cuh) */
int gpx_pause_groups(gpx_engine* e, uint32_t n, const uint32_t* gids, gpx_row* out_rows, uint8_t* out_paused) {
  if (!e) return fail(GPX_EINVAL, "null argument");
  if (n == 0) return GPX_OK;
  if (!gids || !out_rows || !out_paused) return fail(GPX_EINVAL, "null argument");
  {
    std::vector<uint32_t> g(gids, gids + n);
    std::sort(g.begin(), g.end());
    if (std::adjacent_find(g.begin(), g.end()) != g.end()) return fail(GPX_EINVAL, "a gid appears twice in the batch");
  }
  const uint32_t L = e->cfg.n_lanes;
  const size_t gid_bytes = ((size_t)n * 4 + 15) & ~(size_t)15;
  const size_t row_bytes = (size_t)n * L * sizeof(gpx_row);
  const size_t flag_off = gid_bytes + ((row_bytes + 15) & ~(size_t)15);
  int rc = e->ensure_misc(flag_off + n);
  if (rc) return rc;
  cudaStream_t st = e->stream;
  uint8_t* base = (uint8_t*)e->d_misc;
  CK(cudaMemcpyAsync(base, gids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  PauseArgs A;
  A.gids = (const uint32_t*)base;
  A.n = n;
  A.rows = (gpx_row*)(base + gid_bytes);
  A.paused = base + flag_off;
  k_pause_groups<<<cdiv(n, GPX_PAUSE_BLOCK), GPX_PAUSE_BLOCK, 0, st>>>(e->S, A);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out_paused, A.paused, n, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  /* only the rows of the paused groups were written: copy those (runs of consecutive paused entries) */
  for (uint32_t i = 0; i < n;) {
    if (!out_paused[i]) {
      i++;
      continue;
    }
    uint32_t j = i;
    while (j < n && out_paused[j]) j++;
    CK(cudaMemcpyAsync(out_rows + (size_t)i * L, A.rows + (size_t)i * L, (size_t)(j - i) * L * sizeof(gpx_row),
                       cudaMemcpyDeviceToHost, st));
    i = j;
  }
  CK(cudaStreamSynchronize(st));
  for (uint32_t i = 0; i < n; i++) { /* version and paxosID hash live on the host (as in gpx_dump_rows / _destroy_groups) */
    if (!out_paused[i] || gids[i] >= e->cfg.max_groups) continue;
    for (uint32_t l = 0; l < L; l++) {
      out_rows[(size_t)i * L + l].version = e->h_version[gids[i]];
      out_rows[(size_t)i * L + l].name_hash = e->h_name_hash[gids[i]];
    }
    e->h_name_hash[gids[i]] = e->h_version[gids[i]] = 0;
  }
  return GPX_OK;
}

#include "gpx_spread_host.inc"

} /* extern "C" */
