"""The host's copy of the log ring heads against the device's, after every kind of call that logs.

gpx_log_drain_async hands out [from, from + n_bytes) from the host's copy of the heads (no device read while that copy
is exact); gpx_log_read reads the head from the device.  After each logging entry point, both ends must agree, before
and after the ring has wrapped.  The device-resident rounds are checked against the ring like every other logging
call: a batch whose segments exceed the ring is refused with GPX_ERANGE, and with log_backpressure a round that would
overwrite unreleased bytes is refused with GPX_EAGAIN until the ring is drained and released.
"""
import ctypes as C

import numpy as np
import pytest

from helpers import Engine, GpxErrorT, abi, group_descs, make_config, make_requests

pytestmark = pytest.mark.gpu

RING = 1 << 16  # the smallest ring an engine takes: a few passes over the entry points wrap it


class Heads:
    """drains every lane after each call (so no undrained byte is overwritten) and compares both ends of the ring"""

    def __init__(self, eng):
        import torch
        self.eng = eng
        self.buf = torch.zeros(int(eng.cfg.log_ring_bytes), dtype=torch.uint8).pin_memory()

    def check(self, what):
        eng = self.eng
        heads = []
        for l in range(eng.n_lanes):
            f, nb = eng.log_drain_async(l, self.buf.data_ptr(), int(eng.cfg.log_ring_bytes))
            eng.log_drain_wait()
            eng.log_release(l, f + nb)
            assert f + nb == eng.log_head(l), f"{what}: lane {l} host {f + nb} != device {eng.log_head(l)}"
            heads.append(f + nb)
        return heads


def device_round(cuda_lib, eng, fn, reqs, pay):
    import torch
    from gigapaxos_b200.abi import DevRoundBufs
    dev = torch.device("cuda", 0)
    n = len(reqs)
    d_reqs = torch.from_numpy(reqs.view(np.uint8).copy()).to(dev)
    d_pay = torch.from_numpy(np.concatenate([pay, np.zeros(16, np.uint8)])).to(dev)
    d_status = torch.zeros(max(n, 1), dtype=torch.int32, device=dev)
    d_exec = torch.zeros(max(n, 1) * eng.n_lanes * 24, dtype=torch.uint8, device=dev)
    bufs = DevRoundBufs(d_reqs.data_ptr(), d_pay.data_ptr(), len(pay), n, d_status.data_ptr(), d_exec.data_ptr())
    torch.cuda.synchronize()
    try:
        cuda_lib.check(cuda_lib.fn(fn)(eng.handle, C.byref(bufs), None))
    finally:
        torch.cuda.synchronize()


def test_heads_agree_after_every_logging_call(cuda_lib):
    G = 16  # one pass over the entry points stays inside the 64 KiB ring: each is checked before and after a wrap
    eng = Engine(cuda_lib, make_config(cuda_lib, max_groups=G, max_batch_recs=4 * G, max_batch_payload=1 << 16,
                                       log_ring_bytes=RING))
    eng.create_groups(group_descs(G))
    hd = Heads(eng)
    gids = np.arange(G)
    r = 0

    def batch():
        nonlocal r
        r += 1
        return make_requests(np.repeat(gids, 1 + r % 2), payload_len=1 + r % 23, seed=3, round_no=r, entry_lane=r % 3)

    def accepts_then_decisions():
        acc, blob, _ = eng.propose(*batch())
        replies, _ = eng.handle_accepts(acc, blob)
        hd.check("gpx_handle_accepts")
        eng.handle_decisions(eng.handle_accept_replies(replies))

    def accepts_fused():
        acc, blob, _ = eng.propose(*batch())
        eng.handle_accepts_fused(acc, blob)

    def prepares():  # ballot (0, 0) is below every group's: VOID images, but a segment all the same
        p = np.zeros(G, dtype=abi.decision_dtype)
        p["gid"] = gids
        eng.handle_prepares(p)

    def submit():
        eng.round_wait(eng.round_submit(*batch()))

    calls = [("gpx_handle_decisions", accepts_then_decisions), ("gpx_handle_accepts_fused", accepts_fused),
             ("gpx_handle_prepares", prepares), ("gpx_round", lambda: eng.round(*batch())),
             ("gpx_round_phases", lambda: eng.round_phases(*batch())), ("gpx_round_submit", submit)]
    calls += [(fn, lambda fn=fn: device_round(cuda_lib, eng, fn, *batch()))
              for fn in ("round_device", "round_device_compact", "round_device_phases")]
    unwrapped, wrapped = set(), set()
    for _ in range(40):
        for what, call in calls:
            before = hd.check("before " + what)
            call()
            after = hd.check(what)
            assert all(a > b for a, b in zip(after, before)), f"{what} logged nothing"
            (unwrapped if max(after) <= RING else wrapped if min(before) > RING else set()).add(what)
        if min(after) > 3 * RING:
            break
    names = {what for what, _ in calls}
    assert unwrapped == names and wrapped == names
    eng.close()


@pytest.mark.parametrize("graph", [False, True])
def test_heads_agree_after_spread_rounds(cuda_lib, graph):
    import torch
    from test_spread_c_gpu import NODE0, Cluster
    N, G, R, P = 3, 24, 3, 8
    ring = 1 << 17
    cl = Cluster(cuda_lib, N, G, R, P, graph=graph, log_ring_bytes=ring)
    hds = [Heads(e) for e in cl.engines]
    fixed = None
    if graph:  # equal io blocks from round to round: the captured graph is replayed
        fixed = {i: (torch.zeros(4 * G * 32, dtype=torch.uint8, device=cl.dev),
                     torch.zeros(4 * G * 64 + 64, dtype=torch.uint8, device=cl.dev)) for i in range(N)}
    gids = np.arange(G)
    for r in range(200):
        reqs, pay = make_requests(gids, payload_len=P, seed=7, round_no=r)
        reqs["flags"] = (cl.coord[gids].astype(np.uint32) << 8)
        reqs["entry_node"] = NODE0 + cl.coord[gids]
        cl.round(reqs, pay, fixed)
        heads = [hd.check(f"spread round {r} node {k}")[0] for k, hd in enumerate(hds)]
        if min(heads) > 2 * ring:
            break
    assert min(heads) > 2 * ring
    cl.close()


def test_device_round_larger_than_the_ring_is_refused(cuda_lib):
    G = 1024  # 1024 requests: 80 B of images each plus payload -- more than a 64 KiB ring holds
    eng = Engine(cuda_lib, make_config(cuda_lib, max_groups=G, max_batch_recs=G, log_ring_bytes=RING))
    eng.create_groups(group_descs(G))
    hd = Heads(eng)
    device_round(cuda_lib, eng, "round_device", *make_requests(np.arange(64), seed=2))
    before = hd.check("round_device")
    for fn in ("round_device", "round_device_compact", "round_device_phases"):
        with pytest.raises(GpxErrorT) as ex:
            device_round(cuda_lib, eng, fn, *make_requests(np.arange(G), seed=2, round_no=1))
        assert ex.value.code == abi.GPX_ERANGE
        assert hd.check(fn) == before
        assert [eng.log_head(l) for l in range(eng.n_lanes)] == before
    eng.close()


def test_device_round_waits_for_release_under_backpressure(cuda_lib):
    import torch
    G = 64
    eng = Engine(cuda_lib, make_config(cuda_lib, max_groups=G, max_batch_recs=G, log_ring_bytes=RING,
                                       log_backpressure=1))
    eng.create_groups(group_descs(G))
    buf = torch.zeros(RING, dtype=torch.uint8).pin_memory()
    refused = None
    for r in range(100):
        heads = [eng.log_head(l) for l in range(eng.n_lanes)]
        try:
            device_round(cuda_lib, eng, "round_device", *make_requests(np.arange(G), payload_len=40, seed=4, round_no=r))
        except GpxErrorT as ex:
            assert ex.code == abi.GPX_EAGAIN
            assert [eng.log_head(l) for l in range(eng.n_lanes)] == heads, "a refused call logged"
            refused = r
            break
    assert refused is not None and refused > 0, "nothing was released: the ring must fill up"
    for l in range(eng.n_lanes):
        f, nb = eng.log_drain_async(l, buf.data_ptr(), RING)
        eng.log_drain_wait()
        assert f + nb == eng.log_head(l)
        eng.log_release(l, f + nb)
    device_round(cuda_lib, eng, "round_device", *make_requests(np.arange(G), payload_len=40, seed=4, round_no=refused))
    assert all(eng.log_head(l) > heads[l] for l in range(eng.n_lanes))
    eng.close()
