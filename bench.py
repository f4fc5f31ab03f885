#!/usr/bin/env python
"""bench.py -- Paxos decisions/sec of the B200 engine on BASELINE.json's metric.

A *step* is one full Paxos round over every group of the workload: one client request per
group enters the RequestBatcher, the coordinator proposes, all R co-located replicas accept +
log, the coordinator tallies the replies and all replicas commit + emit in-order EXEC records --
ONE kernel (k_round, the fused loopback path; the phase-by-phase kernels k_propose / k_accept /
k_tally / k_commit are timed beside it).  One step decides one slot per group.

  value  : decisions/s with the request batch already resident in HBM (gpx_round_device)
  e2e    : the same metric through the public C-ABI call gpx_round with HOST buffers
           (pinned), H2D of the requests and D2H of status + EXEC records inside the timing
  roofline: the kernel of the timed path (k_round), algorithmic bytes / CUDA-event duration
           vs the measured HBM copy peak; roofline_accept: the stand-alone accept-batch kernel
           (193+2P per ACCEPT at one acceptor, SURVEY.md 8d)
  cpu_baseline: the CPU oracle (a port of the Java path, reference JVM unavailable) on the
           host cores, groups sharded over threads

`--impl reference` times that CPU port alone with all host threads (the reference is
Java-only and no JVM exists in this image; see DESIGN.md).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg2": dict(name="3-replica, 100K groups, 1-byte NoopApp requests, single B200", G=100_000, R=3, P=1),
    "cfg3": dict(name="3-replica, 1M groups, 64-byte requests (per-GPU shard of BASELINE config 3)", G=1_000_000, R=3,
                 P=64),
    "1m1b": dict(name="3-replica, 1M groups, 1-byte requests, single B200 (north_star target size)", G=1_000_000,
                 R=3, P=1),
    "cfg4": dict(name="5-replica, 1M groups, mixed 1-1024 B requests with reconfiguration churn (0.1% of the groups "
                      "STOP and are re-created at the next epoch every round)", G=1_000_000, R=5, P=512),
    "cfg5": dict(name="3-replica, 10M groups resident, accept-batch sweep 1-1024 requests per batch on a 1% active "
                      "subset", G=10_000_000, R=3, P=1),
}
NODES = (100, 101, 102, 103, 104)


def b_acc(P: int) -> int:
    """Algorithmic bytes per ACCEPT at one acceptor (SURVEY.md 8d / BASELINE.md 3)."""
    return 193 + 2 * P


def b_slot(R: int, P: int) -> int:
    return R * (193 + 2 * P) + R * (64 + 8 * R) + 32 + R * 153


def b_act(R: int, P: int) -> int:
    """Algorithmic bytes per decided slot of the fused k_round kernel with all R replicas co-located
    (DESIGN.md 4): request 32 + blob P + status 4; per replica aux 4 + row 16 in + 16 out + window entry 32 in +
    ACCEPT log image 48 + blob P + DECISION log image 32 + EXEC 24; coordinator row 16 in + 16 out, nodeSlots
    4R in + 4R out.  (The DECISION record and the reply out-mask are no longer written by the fast path: every
    member is a local lane, nobody reads them.)"""
    return (32 + P + 4) + R * (4 + 16 + 16 + 32 + 48 + P + 32 + 24) + (32 + 8 * R)


def b_act_batched(R: int, P: int, b: int) -> int:
    """b_act for a slot that carries b requests of P bytes (SURVEY.md 8d: replace 2P by 2bP + 16b): b request records
    + bodies + statuses in, the constructed blob [b x 16 B entries][bodies] written once and logged by every replica."""
    blob = 16 * b + b * P
    return (32 * b + b * P + 4 * b) + blob + R * (4 + 16 + 16 + 32 + 48 + blob + 32 + 24) + (32 + 8 * R)


def java_hash_numbered(prefix: str, idx: np.ndarray) -> np.ndarray:
    """String.hashCode() of f"{prefix}{i}" for every i of idx, vectorised"""
    idx = np.asarray(idx, dtype=np.int64)
    h0 = np.uint32(java_hash(prefix) & 0xFFFFFFFF)
    out = np.zeros(len(idx), dtype=np.uint32)
    ndig = np.ones(len(idx), dtype=np.int64)
    t = idx // 10
    while np.any(t > 0):
        ndig += (t > 0)
        t //= 10
    for nd in np.unique(ndig):
        sel = np.nonzero(ndig == nd)[0]
        v = idx[sel]
        h = np.full(len(sel), h0, dtype=np.uint32)
        for k in range(int(nd) - 1, -1, -1):
            with np.errstate(over="ignore"):
                h = h * np.uint32(31) + ((v // (10 ** k)) % 10 + 48).astype(np.uint32)
        out[sel] = h
    return out.view(np.int32)


def make_descs_fast(abi, G, R, gid0=0, name0=0, prefix="NoopPaxosApp", version=0):
    d = np.zeros(G, dtype=abi.group_desc_dtype)
    d["gid"] = np.arange(gid0, gid0 + G, dtype=np.uint32)
    d["version"] = version
    d["name_hash"] = java_hash_numbered(prefix, np.arange(name0, name0 + G))
    d["n_members"] = R
    for i in range(R):
        d["members"][:, i] = NODES[i]
    d["init_mode"] = abi.INIT_BATCH
    return d


DUMP_LIMIT = 64_000_000  # bytes of all files together


def dump_round_outputs(out_dir, abi, status, exec_bytes, R):
    """What one gpx_round_device call returned, as float64 arrays under out_dir, one file per field: status [G] and the
    EXEC records [G, R] (req_id split into 32-bit halves, which float64 holds exactly).  When that exceeds DUMP_LIMIT,
    the same fields for a fixed sample of the groups (seed 0), whose indices go to group_index.npy."""
    ex = exec_bytes.view(abi.exec_dtype).reshape(-1, R)
    cols = {"status": status, "exec_gid": ex["gid"], "exec_slot": ex["slot"], "exec_req_id_hi": ex["req_id"] >> 32,
            "exec_req_id_lo": ex["req_id"] & 0xFFFFFFFF, "exec_payload_off": ex["payload_off"], "exec_flags": ex["flags"]}
    G, per_group = len(status), 8 * (1 + 6 * R)
    idx = np.arange(G)
    if G * per_group > DUMP_LIMIT:
        idx = np.sort(np.random.default_rng(0).choice(G, size=(DUMP_LIMIT - 4096) // (per_group + 8), replace=False))
        cols = {name: a[idx] for name, a in cols.items()}
        cols["group_index"] = idx
    os.makedirs(out_dir, exist_ok=True)
    for name, a in cols.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def java_hash(s: str) -> int:
    h = 0
    for ch in s:
        h = (31 * h + ord(ch)) & 0xFFFFFFFF
    return h - (1 << 32) if h >= (1 << 31) else h


def shard_names(G: int, rank: int, world: int, prefix="NoopPaxosApp"):
    """Groups of this rank: home_gpu(name) = |String.hashCode(name)| mod world (SURVEY.md 8e)."""
    names = []
    i = 0
    while len(names) < G:
        s = f"{prefix}{i}"
        if world == 1 or abs(java_hash(s)) % world == rank:
            names.append(s)
        i += 1
    return names


def make_descs(abi, names, R):
    d = np.zeros(len(names), dtype=abi.group_desc_dtype)
    d["gid"] = np.arange(len(names), dtype=np.uint32)
    d["name_hash"] = [java_hash(s) for s in names]
    d["n_members"] = R
    for i in range(R):
        d["members"][:, i] = NODES[i]
    d["init_mode"] = abi.INIT_BATCH  # TESTPaxosNode uses batch creation for NUM_GROUPS > 10000
    return d


def make_batch(abi, G, P, seed):
    rng = np.random.default_rng(seed)
    stride = P  # requests packed back to back, as the RequestBatcher concatenates them
    reqs = np.zeros(G, dtype=abi.request_dtype)
    reqs["gid"] = np.arange(G, dtype=np.uint32)
    reqs["flags"] = 0
    reqs["req_id"] = rng.integers(1, 1 << 62, size=G, dtype=np.int64)
    reqs["payload_off"] = np.arange(G, dtype=np.uint32) * stride
    reqs["payload_len"] = P
    reqs["entry_node"] = NODES[0]
    reqs["client"] = np.arange(G, dtype=np.uint32)
    alphabet = np.frombuffer(b"0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz", dtype=np.uint8)
    pay = np.zeros((G, stride), dtype=np.uint8)
    pay[:, :P] = alphabet[rng.integers(0, 62, size=(G, P))]
    return reqs, pay.reshape(-1)


def engine_config(lib, G, R, P, device):
    cfg = lib.config_defaults()
    cfg.device = device
    cfg.max_groups = G
    cfg.n_lanes = R
    for i in range(R):
        cfg.lane_node[i] = NODES[i]
    cfg.window = 8
    cfg.max_group_size = R
    cfg.max_batch_recs = G
    cfg.max_batch_payload = G * P + 16
    per_round = 64 + 48 * G + G * P + 64 + 32 * G + 64
    ring = 1 << 26
    while ring < 4 * per_round:
        ring <<= 1
    cfg.log_ring_bytes = ring
    return cfg


class L2Flush:
    """Flush the 126 MB L2 between timed steps, outside the timed events: a 256 MiB write (everything the previous step
    left is evicted) followed by a 256 MiB READ, so that the cache ends up full of CLEAN lines.  After a write-only
    flush the timed kernel would have to write back ~100 MB of the flush's own dirty lines before it can allocate
    anything -- a cost that belongs to the flush, not to the kernel (`--flush write` keeps that behaviour)."""

    def __init__(self, dev, mode="clean"):
        import torch
        self.torch, self.mode = torch, mode
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.rd = torch.zeros(64 << 20, dtype=torch.int32, device=dev)  # 256 MiB
        self.acc = torch.zeros(1, dtype=torch.int32, device=dev)

    def zero_(self):  # the call sites' name
        self.buf.zero_()
        if self.mode == "clean":
            self.torch.amax(self.rd, dim=0, keepdim=True, out=self.acc)  # a plain 256 MiB read

    def describe(self):
        return ("flushed between timed steps, outside the timed events: 256 MiB write then 256 MiB read (cold and clean)"
                if self.mode == "clean" else
                "flushed between timed steps (256 MiB write, outside the timed events; the flush's dirty lines are "
                "written back during the timed kernel)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile(prefix="gpx_clocks_", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "100"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                t = [x.strip() for x in line.split(",")]
                if len(t) < 9:
                    continue
                try:
                    sm.append(float(t[1]))
                    mx.append(float(t[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   t[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm))
        return out


# --------------------------------------------------------------------------------------------
# CPU arm: the oracle (port of the Java path) with groups sharded over host threads
# --------------------------------------------------------------------------------------------
def cpu_decisions_per_sec(G, R, P, budget_s, threads):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import oracle_library
    from gigapaxos_b200 import abi
    from gigapaxos_b200.abi import Engine

    lib = oracle_library()
    T = max(1, min(threads, G))
    per = [G // T + (1 if i < G % T else 0) for i in range(T)]
    engines, batches = [], []
    for t in range(T):
        cfg = engine_config(lib, per[t], R, P, 0)
        cfg.log_ring_bytes = 1 << 20
        e = Engine(lib, cfg)
        e.create_groups(make_descs(abi, [f"NoopPaxosApp{t}_{i}" for i in range(per[t])], R))
        engines.append(e)
        batches.append(make_batch(abi, per[t], P, 100 + t))

    fn = lib.fn("round")

    class Worker:
        def __init__(self, e, batch):
            self.e = e
            self.reqs, self.pay = batch
            n = len(self.reqs)
            self.status = np.zeros(n, np.int32)
            self.ex = np.zeros(n * R, abi.exec_dtype)
            self.extra = np.zeros(16, abi.exec_dtype)

        def round(self):
            n = len(self.reqs)
            ns, nx = C.c_uint32(0), C.c_uint32(0)
            rc = fn(self.e.handle, C.c_uint32(n), self.reqs.ctypes.data_as(C.c_void_p),
                    self.pay.ctypes.data_as(C.c_void_p), C.c_uint64(self.pay.size),
                    self.status.ctypes.data_as(C.c_void_p), self.ex.ctypes.data_as(C.c_void_p), C.byref(ns),
                    self.extra.ctypes.data_as(C.c_void_p), C.c_uint32(16), C.byref(nx))
            assert rc == 0 and ns.value == n * R

    workers = [Worker(e, b) for e, b in zip(engines, batches)]

    trunc = lib.fn("log_truncate")

    def run_rounds(k):
        def body(w):
            for it in range(k):
                w.round()
                if it % 8 == 7:  # the oracle's journal is an in-memory vector: drop it like a drained log
                    trunc(w.e.handle)
        ts = [threading.Thread(target=body, args=(w,)) for w in workers]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return time.perf_counter() - t0

    run_rounds(1)  # warm-up (page faults, allocator)
    t1 = run_rounds(1)
    k = int(max(1, min(20000, 0.25 * budget_s / max(t1, 1e-6))))
    dt = run_rounds(k)
    while dt < 0.8 * budget_s and k < 200000:  # the first estimate is cold: extend until the budget is used
        k2 = int(max(1, min(200000, (budget_s - dt) / max(dt / k, 1e-9))))
        dt += run_rounds(k2)
        k += k2
    for e in engines:
        e.close()
    return G * k / dt, k, dt, T


# --------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line: dict):
    """the ONE JSON line of the contract goes to the real stdout; everything else that libraries write to fd 1
    (e.g. NCCL's version banner) has been diverted to stderr"""
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--groups", type=int, default=0, help="override groups per GPU")
    ap.add_argument("--payload", type=int, default=0, help="override request payload bytes")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--flush", default="clean", choices=["clean", "write"],
                    help="clean (default): 256 MiB write + 256 MiB read between timed steps; write: the write only")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU work for cpu_baseline")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-large", action="store_true", help="skip the 1M-group roofline context measurement")
    ap.add_argument("--placement", default="auto", choices=["auto", "packed", "spread"],
                    help="auto (default): spread when the job has at least as many GPUs as replicas (SURVEY.md 8e), "
                         "else packed.  packed: all replicas of a group on its home GPU, no data-path collective; spread: "
                         "replica j on GPU (home+j) mod N, ACCEPT/REPLY/DECISION records exchanged over NCCL "
                         "(needs N >= replicas; with --gpus 1 the nodes are --spread-nodes engines on one GPU)")
    ap.add_argument("--spread-nodes", type=int, default=4)
    ap.add_argument("--spread-python", action="store_true",
                    help="spread placement through the host-orchestrated reference path (gigapaxos_b200/spread.py "
                         "SpreadCluster: torch.distributed exchanges, one host count read per exchange) instead of gpx_spread_*")
    ap.add_argument("--no-graph", action="store_true", help="spread: plain stream launches instead of one CUDA graph per round")
    ap.add_argument("--p2p", action="store_true",
                    help="spread: store the records straight into the peers' receive buckets over NVLink (GPX_SPREAD_P2P, CUDA "
                         "IPC between the ranks) instead of exchanging the buckets with grouped ncclSend/ncclRecv; falls back "
                         "to the NCCL exchange when the peer mapping cannot be set up")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last one returned (status and EXEC records of rank 0's "
                         "groups) as DIR/<name>.npy in float64, a fixed sample of the groups beyond 64 MB; "
                         "packed placement, workloads cfg2, cfg3 and 1m1b")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    wl = dict(WORKLOADS[args.workload])
    if args.groups:
        wl["G"] = args.groups
    if args.payload:
        wl["P"] = args.payload
    G, R, P = wl["G"], wl["R"], wl["P"]
    K, W = args.steps, max(args.warmup, 0)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.placement == "auto":
        args.placement = "spread" if (world >= R and world > 1) else "packed"
    if args.dump_outputs and (args.impl != "ours" or args.placement != "packed" or args.workload in ("cfg4", "cfg5")):
        ap.error("--dump-outputs covers the packed round path of workloads cfg2, cfg3 and 1m1b")
    metric = "paxos_decisions_per_sec"
    config = {
        "workload": wl["name"], "groups_per_gpu": G, "replicas": R, "payload_bytes": P, "window": 8,
        "requests_per_group_per_step": 1,
        "placement": "packed: all R replicas of a group on the GPU that owns the group; groups sharded by "
                     "|String.hashCode(paxosID)| mod n_gpus; no data-path collective"
                     + ("" if world >= R or world == 1 else f" (fewer GPUs than replicas: SURVEY.md 8e packs them)"),
        "l2": "none" if args.no_flush else L2Flush.describe(type("x", (), {"mode": args.flush})()),
        "init": "batch creation (HotRestoreInfo.createHRI)",
    }

    if args.impl == "reference":
        # The reference is Java-only and this image has no JVM: the CPU arm is the oracle port.
        if rank != 0:
            return
        threads = os.cpu_count() or 1
        v, k, dt, T = cpu_decisions_per_sec(G, R, P, max(5.0, min(60.0, 0.5 * (K + W))), threads)
        line = {
            "impl": "reference", "metric": metric, "value": v, "unit": "decisions/s", "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * dt / k, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": "decisions/s", "cores": T, "kind": "port",
                             "sample": f"{k} full rounds over {G} groups x {R} replicas (oracle = C++ port of the "
                                       f"Java path; reference JVM unavailable in this image), {dt:.1f} s"},
            "e2e": {"value": v, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        emit(line)
        return

    # (NCCL_DEBUG is left as the launcher set it: NCCL's log lines go to the diverted stdout = stderr)
    import torch
    import torch.distributed as dist

    import gigapaxos_b200
    from gigapaxos_b200 import abi
    from gigapaxos_b200.abi import DevRoundBufs, Engine, KernelTimes

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the gpx engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    lib = gigapaxos_b200.load_library()
    if args.placement == "spread":
        if args.workload == "cfg3" and world > 1 and not args.groups:
            G = wl["G"] // world  # BASELINE config 3 as written: 1 M groups sharded across the GPUs of the job
            config["groups_per_gpu"] = G
            config["workload"] = "3-replica, 1M groups, 64-byte requests, groups sharded across %d GPUs" % world
        (run_spread if args.spread_python else run_spread_c)(args, lib, dev, rank, world, G, R, P, K, max(W, 3), metric,
                                                              config)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.workload in ("cfg4", "cfg5"):
        (run_cfg4 if args.workload == "cfg4" else run_cfg5)(args, lib, dev, rank, world, wl, K, max(W, 3), metric, config)
        if world > 1:
            dist.destroy_process_group()
        return
    eng = Engine(lib, engine_config(lib, G, R, P, local_rank))
    names = shard_names(G, rank, world)
    eng.create_groups(make_descs(abi, names, R))

    NB = 4  # distinct synthetic request batches, cycled
    host_batches = [make_batch(abi, G, P, 1000 * rank + b) for b in range(NB)]
    d_reqs = [torch.from_numpy(b[0].view(np.uint8).copy()).to(dev) for b in host_batches]
    d_pay = [torch.from_numpy(b[1].copy()).to(dev) for b in host_batches]
    d_status = torch.zeros(G, dtype=torch.int32, device=dev)
    d_exec = torch.zeros(G * R * 24, dtype=torch.uint8, device=dev)
    flush_buf = L2Flush(dev, args.flush)
    round_dev = lib.fn("round_device")
    # everything below is issued on ONE explicit stream: the engine launches its kernels on the
    # stream handed to gpx_round_device and torch.cuda.Event only sees torch's current stream
    bench_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(bench_stream)

    def dev_round(b):
        bufs = DevRoundBufs(d_reqs[b].data_ptr(), d_pay[b].data_ptr(), d_pay[b].numel(), G, d_status.data_ptr(),
                            d_exec.data_ptr())
        st = torch.cuda.current_stream().cuda_stream
        assert st != 0, "bench must run on an explicit stream"
        rc = round_dev(eng.handle, C.byref(bufs), C.c_void_p(st))
        if rc != 0:
            raise RuntimeError(lib.last_error())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: device-resident rounds ------------------------------------------------
    for w in range(max(W, 3)):
        dev_round(w % NB)
    sampler = ClockSampler(local_rank)
    barrier()
    c0 = eng.counters()
    sampler.start()
    ev_s = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev_e = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    t_wall0 = time.perf_counter()
    for k in range(K):
        if not args.no_flush:
            flush_buf.zero_()
        ev_s[k].record()
        dev_round(k % NB)
        ev_e[k].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    step_ms = np.array([ev_s[k].elapsed_time(ev_e[k]) for k in range(K)])
    total_ms = float(step_ms.sum())
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    c1 = eng.counters()
    decided = c1["decisions_made"] - c0["decisions_made"]
    assert decided == G * K, f"expected {G * K} decisions in the timed region, engine made {decided}"
    assert c1["executed"] - c0["executed"] == G * K * R
    value = world * G * K / (total_ms / 1e3)
    if args.dump_outputs and rank == 0:  # before the legs below reuse d_status / d_exec
        dump_round_outputs(args.dump_outputs, abi, d_status.cpu().numpy(), d_exec.cpu().numpy(), R)

    # ---- roofline: per-kernel CUDA events inside the engine (same launches, same stream) ----
    def kernel_times(fn_name, K2):
        f = lib.fn(fn_name)
        lib.fn("enable_kernel_timing")(eng.handle, C.c_int(1))
        kt = KernelTimes()
        lib.fn("get_kernel_times")(eng.handle, C.byref(kt), C.c_int(1))
        for k in range(K2):
            if not args.no_flush:
                flush_buf.zero_()
            b = k % NB
            bufs = DevRoundBufs(d_reqs[b].data_ptr(), d_pay[b].data_ptr(), d_pay[b].numel(), G, d_status.data_ptr(),
                                d_exec.data_ptr())
            rc = f(eng.handle, C.byref(bufs), C.c_void_p(torch.cuda.current_stream().cuda_stream))
            if rc != 0:
                raise RuntimeError(lib.last_error())
        torch.cuda.synchronize()
        lib.fn("get_kernel_times")(eng.handle, C.byref(kt), C.c_int(1))
        lib.fn("enable_kernel_timing")(eng.handle, C.c_int(0))
        nl = max(kt.launches, 1)
        return {"propose": kt.propose_ms / nl, "accept": kt.accept_ms / nl, "tally": kt.tally_ms / nl,
                "commit": kt.commit_ms / nl}

    peak, peak_src = hbm_peak()
    kf = kernel_times("round_device", min(K, 20))          # fused: "accept" is k_act
    kp = kernel_times("round_device_phases", min(K, 20))   # phase by phase: the standalone kernels
    act_ms, acc_ms = kf["accept"], kp["accept"]
    act_bytes = G * b_act(R, P)
    acc_bytes = G * R * b_acc(P)
    roofline = {
        "kernel": "k_round (the whole round in one kernel: batch + propose, accept x R + log append, tally, commit x R)",
        "bound": "hbm", "achieved": act_bytes / (act_ms / 1e3) / 1e9 if act_ms > 0 else 0.0, "peak": peak,
        "unit": "GB/s", "peak_source": peak_src, "traffic": None,
        "algorithmic_bytes_per_launch": act_bytes, "bytes_per_decided_slot": b_act(R, P),
        "decided_slots_per_launch": G, "kernel_ms": act_ms,
        "kernel_ms_all": {"k_round": act_ms},
    }
    roofline["frac"] = roofline["achieved"] / peak
    # dram__bytes_read.sum + dram__bytes_write.sum per launch: measured with ncu on this very command by
    # tools/measure_traffic.py (profiles/traffic.json); null when no measurement of this workload is on file
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    wkey = args.workload if not (args.groups or args.payload) else None
    tr = traffic.get(f"{wkey}:k_round")
    roofline["traffic"] = tr["traffic"] if tr else None
    roofline["traffic_source"] = "profiles/traffic.json (tools/measure_traffic.py: ncu dram__bytes_read.sum + dram__bytes_write.sum)" if tr else None
    roofline_accept = {
        "kernel": "k_accept (stand-alone accept-batch kernel of the phase-by-phase pipeline, north_star kernel)",
        "bound": "hbm", "achieved": acc_bytes / (acc_ms / 1e3) / 1e9 if acc_ms > 0 else 0.0, "peak": peak,
        "unit": "GB/s", "peak_source": peak_src, "traffic": None, "algorithmic_bytes_per_launch": acc_bytes,
        "bytes_per_accept": b_acc(P), "accepts_per_launch": G * R, "kernel_ms": acc_ms,
        "kernel_ms_all": {"k_propose+k_build_blobs": kp["propose"], "k_accept": acc_ms, "k_tally_slots": kp["tally"],
                          "k_commit": kp["commit"]},
        "frac_all": {"k_accept": acc_bytes / (acc_ms / 1e3) / 1e9 / peak if acc_ms > 0 else 0.0,
                     "k_tally_slots (64 + 8R B per reply)": G * R * (64 + 8 * R) / (kp["tally"] / 1e3) / 1e9 / peak if kp["tally"] > 0 else 0.0,
                     "k_commit (153 B per decision per replica)": G * R * 153 / (kp["commit"] / 1e3) / 1e9 / peak if kp["commit"] > 0 else 0.0},
        "phase_pipeline_decisions_per_sec": G / ((kp["propose"] + acc_ms + kp["tally"] + kp["commit"]) / 1e3),
    }
    roofline_accept["frac"] = roofline_accept["achieved"] / peak
    tra = traffic.get(f"{wkey}:k_accept")
    roofline_accept["traffic"] = tra["traffic"] if tra else None
    roofline_accept["traffic_source"] = roofline["traffic_source"] if tra else None

    # ---- the same kernels on a batch that fills the GPU (context for the latency-bound 100K-group step) --------
    roofline_large = None
    if args.workload == "cfg2" and not args.groups and world == 1 and not args.skip_large:
        G2 = 1_000_000
        eng2 = Engine(lib, engine_config(lib, G2, R, P, local_rank))
        eng2.create_groups(make_descs(abi, shard_names(G2, rank, world), R))
        hb = [make_batch(abi, G2, P, 77 + b) for b in range(2)]
        r2 = [torch.from_numpy(b[0].view(np.uint8).copy()).to(dev) for b in hb]
        p2 = [torch.from_numpy(b[1].copy()).to(dev) for b in hb]
        st2 = torch.zeros(G2, dtype=torch.int32, device=dev)
        ex2 = torch.zeros(G2 * R * 24, dtype=torch.uint8, device=dev)
        res = {}
        for name in ("round_device", "round_device_phases"):
            f = lib.fn(name)
            lib.fn("enable_kernel_timing")(eng2.handle, C.c_int(0))
            kt = KernelTimes()
            for k in range(3 + 10):
                if k == 3:
                    torch.cuda.synchronize()
                    lib.fn("enable_kernel_timing")(eng2.handle, C.c_int(1))
                    lib.fn("get_kernel_times")(eng2.handle, C.byref(kt), C.c_int(1))
                if not args.no_flush:
                    flush_buf.zero_()
                bufs = DevRoundBufs(r2[k % 2].data_ptr(), p2[k % 2].data_ptr(), p2[k % 2].numel(), G2, st2.data_ptr(),
                                    ex2.data_ptr())
                if f(eng2.handle, C.byref(bufs), C.c_void_p(torch.cuda.current_stream().cuda_stream)) != 0:
                    raise RuntimeError(lib.last_error())
            torch.cuda.synchronize()
            lib.fn("get_kernel_times")(eng2.handle, C.byref(kt), C.c_int(1))
            lib.fn("enable_kernel_timing")(eng2.handle, C.c_int(0))
            res[name] = kt.accept_ms / max(kt.launches, 1)
        c2 = eng2.counters()
        assert c2["decisions_made"] == 2 * 13 * G2
        eng2.close()
        del r2, p2, st2, ex2
        km, ka = res["round_device"], res["round_device_phases"]
        roofline_large = {
            "workload": f"{G2} groups x {R} replicas, {P}-byte requests, one GPU (same kernels, batch fills the GPU)",
            "k_round": {"kernel_ms": km, "decisions_per_sec": G2 / (km / 1e3),
                        "achieved": G2 * b_act(R, P) / (km / 1e3) / 1e9, "frac": G2 * b_act(R, P) / (km / 1e3) / 1e9 / peak},
            "k_accept": {"kernel_ms": ka, "achieved": G2 * R * b_acc(P) / (ka / 1e3) / 1e9,
                         "frac": G2 * R * b_acc(P) / (ka / 1e3) / 1e9 / peak},
            "unit": "GB/s", "peak": peak,
        }

    # ---- e2e: public C-ABI calls with host (pinned) buffers -------------------------------
    # Headline: the pipelined form gpx_round_submit / gpx_round_wait with compact EXEC summaries -- every step
    # copies its request batch host->device and its result (one 8-byte summary per request + control block)
    # device->host inside the timed region; up to PIPE_DEPTH steps overlap.  The synchronous gpx_round with
    # full EXEC records (R x 24 B per decision) is reported beside it.
    e2e = None
    if not args.skip_e2e:
        from gigapaxos_b200.abi import (RoundIO, exec_sum_dtype, request_packed_dtype, PIPE_DEPTH, ROUND_COMPACT,
                                        ROUND_PACKED_REQS)
        fn = lib.fn("round")
        h_reqs = [torch.from_numpy(b[0].view(np.uint8).copy()).pin_memory() for b in host_batches]
        h_pay = [torch.from_numpy(b[1].copy()).pin_memory() for b in host_batches]
        h_status = torch.zeros(G, dtype=torch.int32).pin_memory()
        h_exec = torch.zeros(G * R * 24, dtype=torch.uint8).pin_memory()
        h_extra = torch.zeros(64 * 24, dtype=torch.uint8).pin_memory()
        ns, nx = C.c_uint32(0), C.c_uint32(0)

        def host_round(b):
            rc = fn(eng.handle, C.c_uint32(G), C.c_void_p(h_reqs[b].data_ptr()), C.c_void_p(h_pay[b].data_ptr()),
                    C.c_uint64(h_pay[b].numel()), C.c_void_p(h_status.data_ptr()), C.c_void_p(h_exec.data_ptr()),
                    C.byref(ns), C.c_void_p(h_extra.data_ptr()), C.c_uint32(64), C.byref(nx))
            if rc != 0:
                raise RuntimeError(lib.last_error())

        def allmax(dt):
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                return float(t.item())
            return dt

        for w in range(3):
            host_round(w % NB)
        K3 = min(K, 30)
        barrier()
        t0 = time.perf_counter()
        for k in range(K3):
            host_round(k % NB)
        torch.cuda.synchronize()
        dt_sync = allmax(time.perf_counter() - t0)
        assert ns.value == G * R
        ex = h_exec.numpy().view(abi.exec_dtype)
        assert int((ex["flags"] & abi.F_VOID).sum()) == 0, "e2e round left VOID exec records"

        # pipelined, compact summaries
        submit, wait = lib.fn("round_submit"), lib.fn("round_wait")
        h_sum = [torch.zeros(G * 8, dtype=torch.uint8).pin_memory() for _ in range(PIPE_DEPTH)]
        h_xtra = [torch.zeros(4096 * 24, dtype=torch.uint8).pin_memory() for _ in range(PIPE_DEPTH)]
        # 16-byte packed requests (GPX_ROUND_PACKED_REQS): gid, payload_len, flags, req_id; payloads back to back
        h_pk = []
        for b in range(NB):
            rq = host_batches[b][0]
            pk = np.zeros(G, dtype=request_packed_dtype)
            pk["gid"], pk["payload_len"], pk["flags"], pk["req_id"] = rq["gid"], rq["payload_len"], rq["flags"], rq["req_id"]
            assert np.array_equal(rq["payload_off"], np.arange(G, dtype=np.uint32) * P)
            h_pk.append(torch.from_numpy(pk.view(np.uint8).copy()).pin_memory())
        ios = []
        for d in range(PIPE_DEPTH * NB):
            b, q = d % NB, d % PIPE_DEPTH
            ios.append(RoundIO(G, ROUND_COMPACT | ROUND_PACKED_REQS, h_pk[b].data_ptr(), h_pay[b].data_ptr(),
                               h_pay[b].numel(), None, None, h_sum[q].data_ptr(), h_xtra[q].data_ptr(), 4096))
        tk = C.c_uint64(0)
        inflight = []

        def pipe_step(k):
            if len(inflight) == PIPE_DEPTH:
                pipe_wait()
            io = ios[k % (PIPE_DEPTH * NB)]
            rc = submit(eng.handle, C.byref(io), C.byref(tk))
            if rc != 0:
                raise RuntimeError(lib.last_error())
            inflight.append(tk.value)

        def pipe_wait():
            rc = wait(eng.handle, C.c_uint64(inflight.pop(0)), C.byref(ns), C.byref(nx))
            if rc != 0:
                raise RuntimeError(lib.last_error())
            assert nx.value == 0, "bench workload must stay on the in-order path"

        for w in range(2 * PIPE_DEPTH):
            pipe_step(w)
        while inflight:
            pipe_wait()
        K4 = max(K, 50)
        barrier()
        c0e = eng.counters()
        t0 = time.perf_counter()
        for k in range(K4):
            pipe_step(k)
        while inflight:
            pipe_wait()
        dt_pipe = allmax(time.perf_counter() - t0)
        c1e = eng.counters()
        assert c1e["decisions_made"] - c0e["decisions_made"] == G * K4
        assert c1e["executed"] - c0e["executed"] == G * K4 * R
        for q in range(PIPE_DEPTH):
            sm = h_sum[q].numpy().view(exec_sum_dtype)
            assert np.all(sm["lane_mask"] == (1 << R) - 1) and np.all(sm["slot"] > 0), "summaries incomplete"
        # decide latency of ONE batch end to end: submit -> wait with nothing else in flight
        lat = []
        for k in range(20):
            t1 = time.perf_counter()
            pipe_step(k)
            pipe_wait()
            lat.append(time.perf_counter() - t1)
        # ---- the same pipeline WITH the journal: every step's log segments (ACCEPT images + request bodies + DECISION
        # images of all R lanes) are drained to pinned host memory on the engine's drain stream and released
        # (AbstractPaxosLogger logs before it messages, SQLPaxosLogger.journal :965-1036 appends to a file; the pinned
        # buffer stands for the file's write buffer).  The first drain catches up with what the earlier legs left.
        per_round_log = 256 + 80 * G + 2 * (G * P + 16) + 16 * G
        dbuf = [[torch.zeros(2 * per_round_log, dtype=torch.uint8).pin_memory() for _ in range(R)]
                for _ in range(PIPE_DEPTH)]
        ring_b = int(eng.cfg.log_ring_bytes)
        drained_bytes = [0]

        def pipe_step_log(k):
            if len(inflight) == PIPE_DEPTH:
                pipe_wait_log()
            io = ios[k % (PIPE_DEPTH * NB)]
            if submit(eng.handle, C.byref(io), C.byref(tk)) != 0:
                raise RuntimeError(lib.last_error())
            q = k % PIPE_DEPTH
            ups = []
            for l in range(R):  # enqueue the drain of what this round appends (the copy waits for it on the device)
                f, nb = eng.log_drain_async(l, dbuf[q][l].data_ptr(), dbuf[q][l].numel())
                ups.append((l, f + nb))
                drained_bytes[0] += nb
            inflight.append((tk.value, ups))

        def pipe_wait_log():
            t, ups = inflight.pop(0)
            if wait(eng.handle, C.c_uint64(t), C.byref(ns), C.byref(nx)) != 0:
                raise RuntimeError(lib.last_error())
            eng.log_drain_wait()  # the journal bytes of this round are in host memory: release the ring
            for l, upto in ups:
                eng.log_release(l, upto)

        e2e_log = None
        try:
            # catch up: drop the backlog by re-creating the drain cursor at the current head
            lib.fn("log_drain_skip")(eng.handle)
            for w in range(2 * PIPE_DEPTH):
                pipe_step_log(w)
            while inflight:
                pipe_wait_log()
            barrier()
            drained_bytes[0] = 0
            c0l = eng.counters()
            t0 = time.perf_counter()
            for k in range(K4):
                pipe_step_log(k)
            while inflight:
                pipe_wait_log()
            dt_log = allmax(time.perf_counter() - t0)
            c1l = eng.counters()
            assert c1l["decisions_made"] - c0l["decisions_made"] == G * K4
            for l in range(R):
                f, nb = eng.log_drain_async(l, dbuf[0][l].data_ptr(), dbuf[0][l].numel())
                assert nb == 0, "every appended log byte was drained"
            e2e_log = {"value": world * G * K4 / dt_log, "ms_per_step": 1e3 * dt_log / K4,
                       "log_bytes_drained_per_step": drained_bytes[0] // K4}
        except Exception as ex:  # pragma: no cover
            e2e_log = {"error": repr(ex)}
            inflight.clear()

        e2e_nolog = {"value": world * G * K4 / dt_pipe, "unit": "decisions/s", "ms_per_step": 1e3 * dt_pipe / K4,
                     "d2h_bytes_per_step": int(G * 8 + 32),
                     "note": "the same pipeline without draining the log ring (DISABLE_LOGGING analogue on the host side: "
                             "the log images stay in HBM and are overwritten when the ring wraps)"}
        with_log = e2e_log is not None and "value" in e2e_log
        e2e = {"value": e2e_log["value"] if with_log else world * G * K4 / dt_pipe, "unit": "decisions/s",
               "h2d_bytes_per_step": int(G * 16 + h_pay[0].numel()),
               "d2h_bytes_per_step": int(G * 8 + 32 + (e2e_log["log_bytes_drained_per_step"] if with_log else 0)),
               "steps": K4, "ms_per_step": e2e_log["ms_per_step"] if with_log else 1e3 * dt_pipe / K4,
               "journal": ("drained: every step's log segments of all %d lanes copied to pinned host memory on the drain "
                           "stream (gpx_log_drain_async) and released (gpx_log_release) inside the timed region" % R)
               if with_log else "NOT drained (%r)" % (e2e_log,),
               "no_log": e2e_nolog,
               "p50_decide_latency_ms": 1e3 * float(np.median(lat)),
               "api": "gpx_round_submit / gpx_round_wait (include/gpx.h), GPX_ROUND_PACKED_REQS | GPX_ROUND_COMPACT: "
                      "pinned host buffers of 16-byte requests + payload in, one 8-byte EXEC summary per request out, "
                      "up to %d rounds in flight; "
                      "wall clock around submit..wait of all steps" % PIPE_DEPTH,
               "sync_full": {"value": world * G * K3 / dt_sync, "unit": "decisions/s", "steps": K3,
                             "ms_per_step": 1e3 * dt_sync / K3, "h2d_bytes_per_step": int(G * 32 + h_pay[0].numel()),
                             "d2h_bytes_per_step": int(G * 4 + 32 + G * R * 24),
                             "api": "gpx_round: synchronous call, status + R full EXEC records per decision out"}}

    # ---- cpu baseline (rank 0, N=1 only) --------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        threads = os.cpu_count() or 1
        v, k, dt, T = cpu_decisions_per_sec(G, R, P, args.cpu_budget, threads)
        cpu = {"value": v, "unit": "decisions/s", "cores": T, "kind": "port",
               "sample": f"{k} full rounds over the same {G} groups x {R} replicas, oracle (C++ port of the Java "
                         f"path; no JVM in this image) sharded over {T} threads, {dt:.1f} s"}

    if rank == 0:
        line = {
            "metric": metric, "value": value, "unit": "decisions/s", "n_gpus": world, "steps": K, "warmup": max(W, 3),
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic", "config": config, "roofline": roofline,
            "roofline_accept": roofline_accept, "roofline_1m_groups": roofline_large,
            "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks, "gpu_launches": K,  # one k_round per step (k_round_slow only when a run is left over)
            "p50_decide_latency_ms": float(np.median(step_ms)),
            "requests_per_sec": value, "wall_s_timed_region": t_wall,
        }
        emit(line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def _bench_common(dev, world):
    import torch
    import torch.distributed as dist

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x
    return barrier, allmax


def run_cfg4(args, lib, dev, rank, world, wl, K, W, metric, config):
    """BASELINE config 4: 5 replicas, request sizes uniform in 1..1024 B (seed 2), and reconfiguration churn INSIDE the
    timed region: every round 0.1 % of the groups receive a STOP (PISM.handleCommittedRequest stop path, executed in
    order on all 5 replicas), the stopped groups are killed and re-created at epoch + 1 with fresh state
    (PaxosManager.kill :2162 + createPaxosInstance :632 -> gpx_destroy_groups + gpx_create_groups; the version drop rule
    PISM :441-447 is where names map to gids).  Packed placement: groups sharded by paxosID hash, all 5 replicas of a
    group on its home GPU."""
    import torch
    from gigapaxos_b200 import abi
    from gigapaxos_b200.abi import DevRoundBufs, Engine
    G = args.groups or wl["G"] // max(world, 1)
    R = wl["R"]
    barrier, allmax = _bench_common(dev, world)
    churn = max(1, G // 1000)
    NB = 4
    rng = np.random.default_rng(2 + rank)
    host = []
    pay_max = 0
    for b in range(NB):
        lens = rng.integers(1, 1025, size=G).astype(np.uint32)
        stride = (lens + 15) // 16 * 16
        offs = np.concatenate([[0], np.cumsum(stride)[:-1]]).astype(np.uint32)
        reqs = np.zeros(G, dtype=abi.request_dtype)
        reqs["gid"] = np.arange(G, dtype=np.uint32)
        reqs["req_id"] = rng.integers(1, 1 << 62, size=G, dtype=np.int64)
        reqs["payload_off"], reqs["payload_len"] = offs, lens
        reqs["entry_node"] = NODES[0]
        reqs["client"] = np.arange(G, dtype=np.uint32)
        stop = rng.choice(G, size=churn, replace=False)
        reqs["flags"][stop] |= abi.F_STOP
        total = int(stride.sum())
        pay = rng.integers(48, 123, size=total, dtype=np.uint8)
        host.append((reqs, pay, np.sort(stop).astype(np.uint32), int(lens.sum())))
        pay_max = max(pay_max, total)
    cfg = lib.config_defaults()
    cfg.device = dev.index or 0
    cfg.max_groups, cfg.n_lanes, cfg.window, cfg.max_group_size = G, R, 8, R
    for i in range(R):
        cfg.lane_node[i] = NODES[i]
    cfg.max_batch_recs, cfg.max_batch_payload = G, pay_max + 16
    per_round = 256 + 80 * G + 2 * pay_max + 16 * G
    ring = 1 << 26
    while ring < 3 * per_round:
        ring <<= 1
    cfg.log_ring_bytes = ring
    eng = Engine(lib, cfg)
    eng.create_groups(make_descs_fast(abi, G, R, name0=rank * G))
    version = np.zeros(G, dtype=np.int32)
    name_hash = java_hash_numbered("NoopPaxosApp", np.arange(rank * G, rank * G + G))
    d_reqs = [torch.from_numpy(h[0].view(np.uint8).copy()).to(dev) for h in host]
    d_pay = [torch.from_numpy(h[1]).to(dev) for h in host]
    d_status = torch.zeros(G, dtype=torch.int32, device=dev)
    d_exec = torch.zeros(G * R * 24, dtype=torch.uint8, device=dev)
    flush_buf = L2Flush(dev, args.flush)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    round_dev = lib.fn("round_device")

    def step(k):
        b = k % NB
        bufs = DevRoundBufs(d_reqs[b].data_ptr(), d_pay[b].data_ptr(), d_pay[b].numel(), G, d_status.data_ptr(),
                            d_exec.data_ptr())
        if round_dev(eng.handle, C.byref(bufs), C.c_void_p(stream.cuda_stream)) != 0:
            raise RuntimeError(lib.last_error())
        # churn: the groups whose STOP was just decided and executed are killed and re-created at the next epoch
        dead = host[b][2]
        torch.cuda.current_stream().synchronize()  # the EXEC records of the STOPs are out (the host would apply them)
        version[dead] += 1
        nd = np.zeros(len(dead), dtype=abi.group_desc_dtype)
        nd["gid"], nd["version"], nd["name_hash"], nd["n_members"] = dead, version[dead], name_hash[dead], R
        for i in range(R):
            nd["members"][:, i] = NODES[i]
        nd["init_mode"] = abi.INIT_BATCH
        eng.destroy_groups(dead)
        eng.create_groups(nd)

    for w in range(W):
        step(w)
    sampler = ClockSampler(dev.index or 0)
    barrier()
    c0 = eng.counters()
    sampler.start()
    ev_s = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev_e = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev_r = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    for k in range(K):
        if not args.no_flush:
            flush_buf.zero_()
        ev_s[k].record()
        b = k % NB
        bufs = DevRoundBufs(d_reqs[b].data_ptr(), d_pay[b].data_ptr(), d_pay[b].numel(), G, d_status.data_ptr(),
                            d_exec.data_ptr())
        if round_dev(eng.handle, C.byref(bufs), C.c_void_p(stream.cuda_stream)) != 0:
            raise RuntimeError(lib.last_error())
        ev_r[k].record()
        dead = host[b][2]
        stream.synchronize()
        version[dead] += 1
        nd = np.zeros(len(dead), dtype=abi.group_desc_dtype)
        nd["gid"], nd["version"], nd["name_hash"], nd["n_members"] = dead, version[dead], name_hash[dead], R
        for i in range(R):
            nd["members"][:, i] = NODES[i]
        nd["init_mode"] = abi.INIT_BATCH
        eng.destroy_groups(dead)
        eng.create_groups(nd)
        ev_e[k].record()  # the stream is idle: this timestamp is taken when the synchronous churn calls have returned
    barrier()
    clocks = sampler.stop()
    step_ms = np.array([ev_s[k].elapsed_time(ev_e[k]) for k in range(K)])
    round_ms = np.array([ev_s[k].elapsed_time(ev_r[k]) for k in range(K)])
    total_ms = allmax(float(step_ms.sum()))
    c1 = eng.counters()
    assert c1["decisions_made"] - c0["decisions_made"] == G * K
    assert c1["executed"] - c0["executed"] == G * K * R
    assert c1["stops_executed"] - c0["stops_executed"] == churn * K * R
    value = world * G * K / (total_ms / 1e3)
    if rank == 0:
        peak, peak_src = hbm_peak()
        mean_len = float(np.mean([h[3] for h in host])) / G
        bytes_round = int(G * ((32 + 4) + R * (4 + 16 + 16 + 32 + 48 + 32 + 24) + (32 + 8 * R)) + (1 + R) * G * mean_len)
        rms = float(round_ms.mean())
        cfg_out = dict(config)
        cfg_out.update({"groups_per_gpu": G, "replicas": R, "payload_bytes": "uniform 1..1024 (seed 2)",
                        "churn": f"{churn} groups per round per GPU: STOP decided + executed on all {R} replicas, then "
                                 "gpx_destroy_groups + gpx_create_groups at version + 1, inside the timed region"})
        emit({"metric": metric, "value": value, "unit": "decisions/s", "n_gpus": world, "steps": K, "warmup": W,
              "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
              "dtype": "int32", "data": "synthetic", "config": cfg_out,
              "roofline": {"kernel": "k_round<5> + k_round_slow<5> (the round without the churn calls)", "bound": "hbm",
                           "achieved": bytes_round / (rms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                           "peak_source": peak_src, "traffic": None, "algorithmic_bytes_per_launch": bytes_round,
                           "kernel_ms": rms, "frac": bytes_round / (rms / 1e3) / 1e9 / peak},
              "churn_ms_per_step": float((step_ms - round_ms).mean()), "round_ms_per_step": rms,
              "cpu_baseline": None, "e2e": None, "clocks": clocks, "gpu_launches": 4 * K,
              "p50_decide_latency_ms": float(np.median(round_ms))})
    eng.close()


def run_cfg5(args, lib, dev, rank, world, wl, K, W, metric, config):
    """BASELINE config 5: 10 M groups resident (sharded over the GPUs), each round a 1 % subset is active and every active
    group receives b requests that the RequestBatcher packs into ONE slot (RequestBatcher.java:198-219); sweep
    b = 1, 2, 4, ..., 1024.  A round carries at most 4 M requests (active groups = min(1 % of the groups, 4 M / b)).
    Packed placement (all 3 replicas of a group on its home GPU)."""
    import torch
    from gigapaxos_b200 import abi
    from gigapaxos_b200.abi import DevRoundBufs, Engine
    GT = args.groups or wl["G"] // max(world, 1)
    R, P = wl["R"], wl["P"]
    barrier, allmax = _bench_common(dev, world)
    A1 = max(GT // 100, 1)
    MAXREQ = max(A1, min(4_000_000, A1 * 1024))
    cfg = lib.config_defaults()
    cfg.device = dev.index or 0
    cfg.max_groups, cfg.n_lanes, cfg.window, cfg.max_group_size = GT, R, 8, R
    for i in range(R):
        cfg.lane_node[i] = NODES[i]
    cfg.max_batch_recs, cfg.max_batch_payload = MAXREQ, MAXREQ * P + 16
    per_round = 256 + 80 * MAXREQ + 2 * MAXREQ * P + 16 * MAXREQ
    ring = 1 << 26
    while ring < 3 * per_round:
        ring <<= 1
    cfg.log_ring_bytes = ring
    eng = Engine(lib, cfg)
    t0 = time.perf_counter()
    for lo in range(0, GT, 2_000_000):
        n = min(2_000_000, GT - lo)
        eng.create_groups(make_descs_fast(abi, n, R, gid0=lo, name0=rank * GT + lo))
    create_s = time.perf_counter() - t0
    free_b, total_b = torch.cuda.mem_get_info(dev)
    flush_buf = L2Flush(dev, args.flush)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    round_dev = lib.fn("round_device")
    d_status = torch.zeros(MAXREQ, dtype=torch.int32, device=dev)
    d_exec = torch.zeros(MAXREQ * R * 24, dtype=torch.uint8, device=dev)
    peak, peak_src = hbm_peak()
    rng = np.random.default_rng(5 + rank)
    sweep, clocks_all = [], None
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    NB = 3
    for b in [1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024]:
        A = max(1, min(A1, MAXREQ // b))
        n = A * b
        d_reqs, d_pay = [], []
        for nb in range(NB):
            active = np.sort(rng.choice(GT, size=A, replace=False)).astype(np.uint32)
            reqs = np.zeros(n, dtype=abi.request_dtype)
            reqs["gid"] = np.repeat(active, b)
            reqs["req_id"] = rng.integers(1, 1 << 62, size=n, dtype=np.int64)
            reqs["payload_off"] = np.arange(n, dtype=np.uint32) * P
            reqs["payload_len"] = P
            reqs["entry_node"] = NODES[0]
            reqs["client"] = np.arange(n, dtype=np.uint32)
            d_reqs.append(torch.from_numpy(reqs.view(np.uint8)).to(dev))
            d_pay.append(torch.from_numpy(rng.integers(48, 123, size=n * P + 16, dtype=np.uint8)).to(dev))

        forms = {}
        for form, fname in (("fused_by_request", "round_device"), ("compact_fused", "round_device_compact"),
                            ("phases", "round_device_phases")):
            if form == "fused_by_request" and b > 64:
                pass  # still timed: it is the headline form's own curve
            fn = lib.fn(fname)

            def step(k):
                q = k % NB
                bufs = DevRoundBufs(d_reqs[q].data_ptr(), d_pay[q].data_ptr(), n * P, n, d_status.data_ptr(),
                                    d_exec.data_ptr())
                if fn(eng.handle, C.byref(bufs), C.c_void_p(stream.cuda_stream)) != 0:
                    raise RuntimeError(lib.last_error())
            for w in range(W):
                step(w)
            barrier()
            c0 = eng.counters()
            ev_s = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
            ev_e = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
            for k in range(K):
                if not args.no_flush:
                    flush_buf.zero_()
                ev_s[k].record()
                step(k)
                ev_e[k].record()
            barrier()
            ms = np.array([ev_s[k].elapsed_time(ev_e[k]) for k in range(K)])
            total_ms = allmax(float(ms.sum()))
            c1 = eng.counters()
            assert c1["decisions_made"] - c0["decisions_made"] == A * K, (b, form, c1["decisions_made"] - c0["decisions_made"])
            assert c1["executed"] - c0["executed"] == A * K * R
            assert c1["requests_batched"] - c0["requests_batched"] == n * K
            forms[form] = {"ms_per_step": total_ms / K, "p50_ms": float(np.median(ms))}
        bestf = min(forms, key=lambda f: forms[f]["ms_per_step"])
        per = forms[bestf]["ms_per_step"]
        bytes_round = A * b_act_batched(R, P, b)
        sweep.append({"requests_per_batch": b, "active_groups_per_gpu": A, "requests_per_step_per_gpu": n,
                      "form": bestf, "ms_per_step": per, "decisions_per_sec": world * A / (per / 1e3),
                      "requests_per_sec": world * n / (per / 1e3), "p50_ms": forms[bestf]["p50_ms"],
                      "roofline_frac": bytes_round / (per / 1e3) / 1e9 / peak, "algorithmic_bytes_per_step": bytes_round,
                      "ms_per_step_by_form": {f: v["ms_per_step"] for f, v in forms.items()}})
        del d_reqs, d_pay
    clocks = sampler.stop()
    if rank == 0:
        best = max(sweep, key=lambda x: x["requests_per_sec"])
        head = sweep[0]
        cfg_out = dict(config)
        cfg_out.update({"groups_per_gpu": GT, "groups_total": GT * world, "replicas": R, "payload_bytes": P,
                        "active_fraction": 0.01, "max_requests_per_step": MAXREQ,
                        "device_memory_used_gb": round((total_b - free_b) / 1e9, 2), "group_creation_s": round(create_s, 2)})
        emit({"metric": metric, "value": head["decisions_per_sec"], "unit": "decisions/s", "n_gpus": world, "steps": K,
              "warmup": W, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong",
              "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": cfg_out,
              "forms": {"fused_by_request": "gpx_round_device: k_round + k_round_slow, outputs indexed by request",
                        "compact_fused": "gpx_round_device_compact: k_propose + k_build_blobs + k_act, outputs per ACCEPT",
                        "phases": "gpx_round_device_phases: k_propose, k_accept, k_tally, k_commit"},
              "roofline": {"kernel": "k_round + k_round_slow at b = 1 (in-order fast path over the active 1 %)", "bound": "hbm",
                           "achieved": head["algorithmic_bytes_per_step"] / (head["ms_per_step"] / 1e3) / 1e9,
                           "peak": peak, "unit": "GB/s", "peak_source": peak_src, "traffic": None,
                           "algorithmic_bytes_per_launch": head["algorithmic_bytes_per_step"],
                           "kernel_ms": head["ms_per_step"], "frac": head["roofline_frac"]},
              "sweep": sweep, "best_requests_per_sec": best["requests_per_sec"],
              "best_requests_per_batch": best["requests_per_batch"], "cpu_baseline": None, "e2e": None,
              "clocks": clocks, "gpu_launches": 2 * K * len(sweep)})
    eng.close()


def spread_placement(N, G, R, node_ids):
    """G groups per coordinator node: names NoopPaxosApp<i>, i = 0, 1, ...; replica j of a group on node
    (home + j) mod N (SURVEY.md 8e), coordinator = PISM.roundRobinCoordinator(0).  Node c coordinates the global
    gids [c*G, (c+1)*G).  Returns (descs, member_of[N*G, N], coord[N*G])."""
    from gigapaxos_b200 import abi
    from gigapaxos_b200.spread import coordinator_of, members_of
    per, i, total = [[] for _ in range(N)], 0, 0
    while total < N * G:
        nm = f"NoopPaxosApp{i}"
        mem = [node_ids[m] for m in members_of(nm, N, R)]
        c = coordinator_of(nm, mem) - node_ids[0]
        if len(per[c]) < G:
            per[c].append((nm, mem))
            total += 1
        i += 1
    descs = np.zeros(N * G, dtype=abi.group_desc_dtype)
    member_of = np.zeros((N * G, N), dtype=bool)
    coord = np.repeat(np.arange(N), G)
    for c in range(N):
        for k, (nm, mem) in enumerate(per[c]):
            g = c * G + k
            descs[g]["gid"] = g
            descs[g]["name_hash"] = abi.java_string_hash(nm)
            descs[g]["n_members"] = R
            descs[g]["members"][:R] = mem
            descs[g]["init_mode"] = abi.INIT_BATCH
            member_of[g, [m - node_ids[0] for m in mem]] = True
    return descs, member_of, coord


def run_spread_c(args, lib, dev, rank, world, G, R, P, K, W, metric, config):
    """Spread placement behind the C ABI (gpx_spread_*, gigapaxos_b200/csrc/gpx_spread.cuh): one single-lane engine per
    GPU, every node coordinates G groups and is an acceptor of (R-1)*G more; a step = one request for every group; the
    ACCEPT / ACCEPT_REPLY / DECISION records cross GPUs as fixed-capacity buckets through grouped ncclSend/ncclRecv
    issued by libgpx itself (no Python and no host count read inside a round)."""
    import torch
    import torch.distributed as dist

    from gigapaxos_b200 import abi
    from gigapaxos_b200.abi import Engine
    from gigapaxos_b200.spread import Spread, spread_caps, spread_config
    N = world if world > 1 else args.spread_nodes
    if N < R:
        raise SystemExit(f"spread placement needs at least {R} nodes")
    node_ids = [NODES[0] + i for i in range(N)]
    descs, member_of, coord = spread_placement(N, G, R, node_ids)
    local = list(range(N)) if world == 1 else [rank]
    cap = spread_caps(coord, member_of)
    blob_per_rec = (P + 15) // 16 * 16
    scfg = spread_config(node_ids, cap, blob_per_rec=blob_per_rec, max_reqs=G, graph=not args.no_graph, p2p=args.p2p)
    engines = []
    for idx in local:
        n_in = int(member_of[:, idx].sum())
        vt = sum(((int(cap[s, idx]) + 255) // 256) * 256 for s in range(N))
        per_round = 256 + 80 * vt + n_in * blob_per_rec
        ring = 1 << 26
        while ring < 4 * per_round:
            ring <<= 1
        cfg = lib.config_defaults()
        cfg.device = dev.index or 0
        cfg.max_groups = N * G
        cfg.n_lanes = 1
        cfg.lane_node[0] = node_ids[idx]
        cfg.window = 8
        cfg.max_group_size = R
        cfg.max_batch_recs = G
        cfg.max_batch_payload = G * P + 16
        cfg.log_ring_bytes = ring
        e = Engine(lib, cfg)
        e.create_groups(descs[member_of[:, idx]])
        engines.append(e)
    transport = "p2p" if args.p2p else "nccl"
    if world > 1:
        def make(cfg_):
            ids = [Spread.unique_id(lib) if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0, device=dev)
            try:
                return Spread(lib, engines, cfg_, rank=rank, unique_id=ids[0]), 1
            except Exception as ex:  # e.g. CUDA IPC not permitted on this box
                print(f"[rank {rank}] spread group creation failed: {ex}", file=sys.stderr)
                return None, 0
        sp, ok = make(scfg)
        t = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        if int(t.item()) == 0 and args.p2p:  # every rank falls back to the NCCL bucket exchange together
            if sp is not None:
                sp.close()
            transport = "nccl (peer-memory transport unavailable: fell back)"
            scfg = spread_config(node_ids, cap, blob_per_rec=blob_per_rec, max_reqs=G, graph=not args.no_graph, p2p=False)
            sp, ok = make(scfg)
            t = torch.tensor([ok], dtype=torch.int32, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        if int(t.item()) == 0:
            raise SystemExit("could not create the spread group")
    else:
        sp = Spread(lib, engines, scfg)
    NB = 4
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    bufs = []  # per local node: device buffers
    for k, idx in enumerate(local):
        vt = sp.plans[k].vtotal
        b = {"status": torch.zeros(G, dtype=torch.int32, device=dev),
             "exec": torch.zeros(max(vt, 1) * 24, dtype=torch.uint8, device=dev),
             "extra": torch.zeros(4096 * 24, dtype=torch.uint8, device=dev),
             "ctl": torch.zeros(8, dtype=torch.int32, device=dev), "reqs": [], "pay": [], "h_reqs": [], "h_pay": []}
        for nb in range(NB):
            reqs, pay = make_batch(abi, G, P, 1000 * idx + nb)
            reqs["gid"] = np.arange(idx * G, (idx + 1) * G, dtype=np.uint32)
            reqs["entry_node"] = node_ids[idx]
            pay = np.concatenate([pay, np.zeros(16, np.uint8)])
            b["h_reqs"].append(torch.from_numpy(reqs.view(np.uint8).copy()).pin_memory())
            b["h_pay"].append(torch.from_numpy(pay).pin_memory())
            b["reqs"].append(b["h_reqs"][-1].to(dev))
            b["pay"].append(b["h_pay"][-1].to(dev))
        bufs.append(b)

    def make_ios(nb, reqs_key="reqs", pay_key="pay"):
        ios = []
        for b in bufs:
            io = abi.SpreadIO()
            io.reqs, io.payload, io.payload_bytes, io.n = b[reqs_key][nb].data_ptr(), b[pay_key][nb].data_ptr(), G * P, G
            io.status, io.exec = b["status"].data_ptr(), b["exec"].data_ptr()
            io.extra, io.extra_cap, io.ctl = b["extra"].data_ptr(), 4096, b["ctl"].data_ptr()
            ios.append(io)
        return ios

    ios = [make_ios(nb) for nb in range(NB)]
    flush_buf = L2Flush(dev, args.flush)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    st = stream.cuda_stream
    for w in range(max(W, 2 * NB)):
        sp.round(ios[w % NB], st)
    sampler = ClockSampler(dev.index or 0)
    barrier()
    c0 = [e.counters() for e in engines]
    sampler.start()
    # One round of a node touches every state row, window entry, bucket and log image of the (R x G) group replicas it
    # hosts: well over the 126 MB of L2 at the benchmark sizes (the line's config.working_set_mb says how much), so
    # consecutive rounds find nothing of their own in the cache ("inputs larger than L2"): the K steps are timed back to
    # back, one event per step boundary.  When the working set is smaller the L2 is flushed between steps instead.
    n_in0 = int(member_of[:, local[0]].sum())
    ws_mb = (n_in0 * (16 + 4 + 32 + 48 + 32 + 32 + 24 + 80 + 2 * blob_per_rec) + G * (32 + 48 + 16 + 16 + 12 + 32)) / 1e6
    use_flush = (not args.no_flush) and ws_mb < 160.0
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    ev_s = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    if not use_flush:
        ev[0].record()
    for k in range(K):
        if use_flush:
            flush_buf.zero_()
            if world > 1:  # the ranks are coupled by the exchanges: start the step together, or one rank's flush would be
                barrier()  # timed inside its peers' rounds
            ev_s[k].record()
        sp.round(ios[k % NB], st)
        ev[k + 1].record()
    barrier()
    clocks = sampler.stop()
    step_ms = np.array([(ev_s[k] if use_flush else ev[k]).elapsed_time(ev[k + 1]) for k in range(K)])
    total_ms = allmax(float(step_ms.sum()))
    c1 = [e.counters() for e in engines]
    for k, (a, b) in enumerate(zip(c0, c1)):
        n_in = int(member_of[:, local[k]].sum())
        assert b["decisions_made"] - a["decisions_made"] == G * K, "every coordinated group decides once per step"
        assert b["executed"] - a["executed"] == n_in * K, "every replica executes every decision"
        assert sp.dropped(k) == 0
    value = N * G * K / (total_ms / 1e3)
    b2b_ms = total_ms / K

    # per-kernel share of a round: CUDA events between the phases cannot be placed inside the C call (and inside a
    # graph), so a non-graph handle is timed phase by phase through the per-phase wall of the ncu launch list under
    # profiles/; here only the whole round is timed.

    # ---- e2e: host (pinned) request batches in, status + EXEC records out, copies inside the timed region ----------
    e2e = None
    if not args.skip_e2e:
        h_status = [torch.zeros(G, dtype=torch.int32).pin_memory() for _ in bufs]
        h_exec = [torch.zeros(b["exec"].numel(), dtype=torch.uint8).pin_memory() for b in bufs]
        for b in bufs:  # device staging the copies land in (fixed addresses: one graph)
            b["s_reqs"] = [torch.zeros_like(b["reqs"][0])]
            b["s_pay"] = [torch.zeros_like(b["pay"][0])]
        ios_e = make_ios(0, "s_reqs", "s_pay")

        def e2e_step(k):
            for b in bufs:
                b["s_reqs"][0].copy_(b["h_reqs"][k % NB], non_blocking=True)
                b["s_pay"][0].copy_(b["h_pay"][k % NB], non_blocking=True)
            sp.round(ios_e, st)
            for j, b in enumerate(bufs):
                h_status[j].copy_(b["status"], non_blocking=True)
                h_exec[j].copy_(b["exec"], non_blocking=True)

        for k in range(3):
            e2e_step(k)
        K3 = max(10, min(K, 30))
        barrier()
        t0 = time.perf_counter()
        for k in range(K3):
            e2e_step(k)
        torch.cuda.synchronize()
        dt = allmax(time.perf_counter() - t0)
        ex = h_exec[0].numpy().view(abi.exec_dtype)
        assert int(((ex["flags"] & abi.F_VOID) == 0).sum()) == int(member_of[:, local[0]].sum())
        assert np.all(h_status[0].numpy() > 0)
        e2e = {"value": N * G * K3 / dt, "unit": "decisions/s", "steps": K3, "ms_per_step": 1e3 * dt / K3,
               "h2d_bytes_per_step": int(G * 32 + G * P + 16), "d2h_bytes_per_step": int(G * 4 + h_exec[0].numel()),
               "api": "gpx_spread_round (include/gpx.h) per GPU process on request batches copied from pinned host "
                      "memory each step; status + one 24-byte EXEC record per executed (group, replica) copied back; "
                      "one stream, wall clock around all steps"}

    if rank == 0:
        n_in = int(member_of[:, local[0]].sum())
        peak, peak_src = hbm_peak()
        cfg = dict(config)
        link_bytes = int(sum(sp.plans[0].send_bytes[k][d] for k in range(3) for d in range(N) if d != local[0]))
        cfg.update({"groups_per_gpu": G, "accepts_in_per_node_per_step": n_in, "working_set_mb_per_gpu_per_step": round(ws_mb, 1),
                    "l2": (flush_buf.describe() if use_flush else
                           "not flushed: one step's working set (%.0f MB per GPU) exceeds the 126 MB L2, steps run back to back" % ws_mb),
                    "placement": f"spread: {N} nodes, one single-lane engine per "
                    + (("GPU; the kernels store records straight into the peers' fixed-capacity receive buckets over NVLink "
                        "(CUDA IPC; handles exchanged over NCCL), flag exchange per packet type" if transport == "p2p" else
                        "GPU; libgpx issues grouped ncclSend/ncclRecv of fixed-capacity buckets over NVLink")
                       if world > 1 else "node, all on ONE GPU")
                    + f"; replica j of a group on node (home+j) mod {N}; three record exchanges per round; "
                    + ("one CUDA graph launch per round" if not args.no_graph else "stream launches"),
                    "nvlink_bytes_sent_per_gpu_per_step": link_bytes, "transport": transport})
        ms = total_ms / K
        # algorithmic HBM bytes of one node's round: the phase pipeline's B_slot spread over the nodes (SURVEY.md 8d)
        bytes_round = G * b_slot(R, P)
        line = {
            "metric": metric, "value": value, "unit": "decisions/s", "n_gpus": world, "steps": K, "warmup": max(W, 2 * NB),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic", "config": cfg,
            "roofline": {"kernel": "one node's whole spread round (k_propose, k_build_blobs, k_sp_route, k_sp_accept, "
                                   "k_sp_tally, k_sp_commit + 3 bucket exchanges)", "bound": "hbm",
                         "achieved": bytes_round / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "peak_source": peak_src, "traffic": None, "algorithmic_bytes_per_launch": bytes_round,
                         "bytes_per_decided_slot": b_slot(R, P), "kernel_ms": ms,
                         "frac": bytes_round / (ms / 1e3) / 1e9 / peak,
                         "nvlink": {"bytes_sent_per_gpu": link_bytes, "min_ms_at_770GBs": link_bytes / 770e9 * 1e3}},
            "cpu_baseline": None, "e2e": e2e, "clocks": clocks,
            "gpu_launches": K * 6 * len(local), "p50_decide_latency_ms": float(np.median(step_ms)),
        }
        emit(line)
    sp.close()
    for e in engines:
        e.close()


def run_spread(args, lib, dev, rank, world, G, R, P, K, W, metric, config):
    """Spread placement: one node (single-lane engine) per GPU; every node coordinates G groups and is an acceptor of
    ~(R-1)*G more.  A step = one request for every group; the records cross GPUs three times (ACCEPT, ACCEPT_REPLY,
    DECISION) through gigapaxos_b200/spread.py."""
    import torch
    import torch.distributed as dist

    from gigapaxos_b200 import abi
    from gigapaxos_b200.spread import (DistExchange, LocalExchange, SpreadCluster, SpreadNode, coordinator_of,
                                       members_of)
    N = world if world > 1 else args.spread_nodes
    if N < R:
        raise SystemExit(f"spread placement needs at least {R} nodes")
    node_ids = [NODES[0] + i for i in range(N)]
    # group names NoopPaxosApp<i>, i = 0, 1, ...: keep the first G that every node coordinates
    per, i, total = [[] for _ in range(N)], 0, 0
    while total < N * G:
        nm = f"NoopPaxosApp{i}"
        mem = [node_ids[m] for m in members_of(nm, N, R)]
        c = coordinator_of(nm, mem) - node_ids[0]
        if len(per[c]) < G:
            per[c].append((nm, mem))
            total += 1
        i += 1
    descs = np.zeros(N * G, dtype=abi.group_desc_dtype)
    member_of = np.zeros((N * G, N), dtype=bool)
    for c in range(N):
        for k, (nm, mem) in enumerate(per[c]):
            g = c * G + k  # global gid: node c coordinates gids [c*G, (c+1)*G)
            descs[g]["gid"] = g
            descs[g]["name_hash"] = abi.java_string_hash(nm)
            descs[g]["n_members"] = R
            descs[g]["members"][:R] = mem
            descs[g]["init_mode"] = abi.INIT_BATCH
            member_of[g, [m - node_ids[0] for m in mem]] = True
    local = list(range(N)) if world == 1 else [rank]
    nodes = []
    for idx in local:
        n_in = int(member_of[:, idx].sum())
        ring = 1 << 26
        while ring < 4 * (128 + 80 * n_in + n_in * (P + 16)):
            ring <<= 1
        nd = SpreadNode(lib, idx, node_ids, dev, max_groups=N * G, max_batch=max(n_in, G), max_payload=G * P + 16,
                        max_group_size=R, window=8, log_ring_bytes=ring)
        nd.engine.create_groups(descs[member_of[:, idx]])
        nodes.append(nd)
    cluster = SpreadCluster(nodes, LocalExchange(N) if world == 1 else DistExchange(), N)
    NB = 4
    batches = []
    for b in range(NB):
        bb = {}
        for idx in local:
            reqs, pay = make_batch(abi, G, P, 1000 * idx + b)
            reqs["gid"] = np.arange(idx * G, (idx + 1) * G, dtype=np.uint32)
            reqs["entry_node"] = node_ids[idx]
            bb[idx] = (torch.from_numpy(reqs.view(np.uint8).copy()).to(dev),
                       torch.from_numpy(np.concatenate([pay, np.zeros(16, np.uint8)])).to(dev)[: pay.size], G)
        batches.append(bb)
    flush_buf = L2Flush(dev, args.flush)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for w in range(W):
        cluster.round(batches[w % NB])
    sampler = ClockSampler(dev.index or 0)
    barrier()
    c0 = [nd.engine.counters() for nd in nodes]
    sampler.start()
    cluster.timing = True
    step_ms, phase_ms = [], {}
    for k in range(K):
        if not args.no_flush:
            flush_buf.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = cluster.round(batches[k % NB])
        e1.record()
        torch.cuda.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        for name, ms in res[local[0]].get("ms", {}).items():
            phase_ms[name] = phase_ms.get(name, 0.0) + ms / K
    barrier()
    clocks = sampler.stop()
    total_ms = float(np.sum(step_ms))
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    c1 = [nd.engine.counters() for nd in nodes]
    for nd, a, b in zip(nodes, c0, c1):
        assert b["decisions_made"] - a["decisions_made"] == G * K, "every coordinated group decides once per step"
        assert b["executed"] - a["executed"] == int(member_of[:, nd.index].sum()) * K, "every replica executes"
    value = N * G * K / (total_ms / 1e3)
    if rank == 0:
        n_in = int(member_of[:, local[0]].sum())
        peak, peak_src = hbm_peak()
        acc_ms = phase_ms.get("accept+route", 0.0)
        cfg = dict(config)
        cfg.update({"groups_per_gpu": G, "placement": f"spread: {N} nodes, one single-lane engine per "
                    + ("GPU (NCCL point-to-point buckets over NVLink)" if world > 1 else "node, all on ONE GPU (device copies)")
                    + f"; replica j of a group on node (home+j) mod {N}; three record exchanges per round",
                    "accepts_in_per_node_per_step": n_in})
        line = {
            "metric": metric, "value": value, "unit": "decisions/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic", "config": cfg,
            "roofline": {"kernel": "accept phase of one node: k_ingest + k_accept<1> + k_route(replies)", "bound": "hbm",
                         "achieved": n_in * b_acc(P) / (acc_ms / 1e3) / 1e9 if acc_ms > 0 else 0.0, "peak": peak,
                         "unit": "GB/s", "peak_source": peak_src, "traffic": None,
                         "algorithmic_bytes_per_launch": n_in * b_acc(P), "kernel_ms": acc_ms,
                         "frac": (n_in * b_acc(P) / (acc_ms / 1e3) / 1e9 / peak) if acc_ms > 0 else 0.0},
            "phase_ms": phase_ms, "cpu_baseline": None, "e2e": None, "clocks": clocks,
            "gpu_launches": K * (2 + 3 + 2 + N + 1 + 2) * len(local),
            "p50_decide_latency_ms": float(np.median(step_ms)),
        }
        emit(line)
    for nd in nodes:
        nd.engine.close()


if __name__ == "__main__":
    main()
