"""The host-side mirror of the reference interface (PaxosManager / Replicable) driven like the
reference's own integration test (testing/TESTPaxosMain.java:154-176 + TESTPaxosClient): create
groups, send requests through every entry replica, check every request got its response and the
RSM invariant of testing/TESTPaxosApp.java (seqnum == slot; identical state on every replica).
Runs against the oracle on CPU and, marked gpu, against the CUDA engine."""
import numpy as np
import pytest

from gigapaxos_b200.paxos_manager import HashChainApp, NoopPaxosApp, PaxosManager
from helpers import Engine, abi, make_config

NODES = [100, 101, 102]


def make_pm(lib, app_cls, p1b=False, **kw):
    eng = Engine(lib, make_config(lib, max_groups=64, max_batch_recs=4096, max_batch_payload=1 << 20, **kw))
    return PaxosManager(eng, [app_cls() for _ in NODES], NODES, device_phase1b=p1b, device_log_find=p1b)


def drive(lib):
    pm = make_pm(lib, HashChainApp, checkpoint_interval=5)
    names = [f"TESTPaxosApp{i}" for i in range(10)]
    assert pm.createPaxosInstanceBatch({n: None for n in names}, NODES)
    assert not pm.createPaxosInstance(names[0], 0, NODES)  # already exists (PaxosManager.java:646-652)
    responses = []
    rng = np.random.default_rng(1)
    sent = 0
    for r in range(12):
        for n in names:
            for _ in range(int(rng.integers(1, 4))):
                val = bytes(rng.integers(97, 123, size=int(rng.integers(1, 20))).astype(np.uint8))
                rid = pm.propose(n, val, callback=lambda req, ok: responses.append(req.request_id),
                                 entry_node=NODES[int(rng.integers(0, 3))])
                assert rid is not None
                sent += 1
        pm.run_round()
    assert pm.propose("nonexistent", b"x") is None
    assert sorted(responses) == list(range(1, sent + 1))  # every client got its response exactly once
    assert not pm.outstanding
    s0 = pm.apps[0].state
    assert all(a.state == s0 for a in pm.apps) and len(s0) == 10  # RSMInvariant: replicas agree
    assert all(a.seqnum == pm.apps[0].seqnum for a in pm.apps)
    cps = [c for c in pm.checkpoints if c[1] == 0]
    assert cps and all(c[2] % 5 == 0 for c in cps)  # shouldCheckpoint: slot % CPI == 0
    # reconfiguration churn (BASELINE config 4): stop at epoch 0, re-create at epoch 1
    assert pm.proposeStop(names[3], 1, b"stop") is None  # wrong version: dropped (PISM :441-447)
    assert pm.proposeStop(names[3], 0, b"stop") is not None
    pm.run_round()
    assert pm.isStopped(names[3]) and not pm.isStopped(names[4])
    pm.propose(names[3], b"late")
    pm.run_round()
    assert any(sp[0] == names[3] and sp[2] == abi.RS_DROPPED for sp in pm.slow_path)  # stopped: dropped
    assert not pm.createPaxosInstance(names[3], 0, NODES)
    assert pm.createPaxosInstance(names[3], 1, NODES, initialState=None)
    assert pm.getVersion(names[3]) == 1
    for a in pm.apps:
        a.seqnum[names[3]] = 1
    got = []
    pm.propose(names[3], b"fresh", callback=lambda req, ok: got.append(req.slot))
    pm.run_round()
    assert got == [1]  # the new epoch starts at slot 1 again (HotRestoreInfo.createHRI)
    assert pm.kill(names[5]) and pm.propose(names[5], b"x") is None
    return pm


def test_paxos_manager_mirror_cpu(oracle_lib):
    drive(oracle_lib)


def test_noop_app_and_stop_batch_quirk(oracle_lib):
    """NoopPaxosApp echoes; a batch that contains a STOP executes only its first request because the
    acceptor is already STOPPED when the batch runs (PISM.execute :1813-1815)."""
    pm = make_pm(oracle_lib, NoopPaxosApp)
    pm.createPaxosInstance("NoopPaxosApp0", 0, NODES)
    out = []
    pm.propose("NoopPaxosApp0", b"a", callback=lambda r, ok: out.append(r.response_value))
    pm.run_round()
    assert out == [b"echoing [a]"]
    pm.propose("NoopPaxosApp0", b"x", stop=True, callback=lambda r, ok: out.append(r.response_value))
    pm.propose("NoopPaxosApp0", b"y", callback=lambda r, ok: out.append(r.response_value))
    pm.run_round()
    assert out == [b"echoing [a]", b"echoing [x]"] and pm.isStopped("NoopPaxosApp0")
    assert all(a.executed == 2 for a in pm.apps)


@pytest.mark.gpu
def test_paxos_manager_mirror_gpu(cuda_lib, oracle_lib):
    pg = drive(cuda_lib)
    po = drive(oracle_lib)
    assert pg.apps[0].state == po.apps[0].state and pg.checkpoints == po.checkpoints
    assert pg.num_decisions == po.num_decisions


# ---- pause / unpause (PaxosManager.pause :2284, unpause :2370; HotRestoreInfo) ---------------------------------
def test_hot_restore_info_string_is_the_reference_format():
    """the one literal-valued JUnit test near this path: paxosutil/HotRestoreInfo.java:159-175"""
    from gigapaxos_b200.paxos_manager import HotRestoreInfo
    h = HotRestoreInfo("paxos0", 2, [1, 4, 67], 5, (3, 4), 3, (45, 67), 34, [1, 3, 5])
    s = str(h)
    assert s == "paxos0|2|[1,4,67]|5|3:4|3|45:67|34|[1,3,5]"
    assert str(HotRestoreInfo.parse(s)) == s
    n = HotRestoreInfo("g", 0, [100, 101, 102], 1, (0, 101), -1, None, -1, None)
    assert str(n) == "g|0|[100,101,102]|1|0:101|-1|null|-1|null" and HotRestoreInfo.parse(str(n)) == n


def drive_pausing(lib, pause: bool):
    """the same request schedule with and without pausing idle instances in between: the replicated state
    machines must end in the same state, paused instances come back on demand (propose -> unpause)"""
    import ctypes as C
    pm = make_pm(lib, HashChainApp, checkpoint_interval=4)
    names = [f"TESTPaxosApp{i}" for i in range(12)]
    pm.createPaxosInstanceBatch({n: None for n in names}, NODES)
    rng = np.random.default_rng(3)
    hri_seen = []
    for r in range(10):
        active = [n for n in names if rng.random() < 0.6]
        for n in active:
            pm.propose(n, f"{n}:{r}".encode(), entry_node=NODES[int(rng.integers(0, 3))])
        if r == 4:
            pm.propose(names[0], b"queued")
            if pause:
                assert not pm.pause(names[0])  # a request is queued: not idle
        pm.run_round()
        if pause and r % 3 == 0:
            for n in names[::2]:
                if n in pm.instances:
                    gid = pm.instances[n].gid
                    row = pm.engine.dump_rows(np.array([gid], dtype=np.uint32), 1)
                    assert pm.pause(n) and pm.isPaused(n) and n not in pm.instances
                    hri_seen.append((pm.paused[n][1], row))
    if pause:
        assert hri_seen and pm.paused  # some instances are still paused at the end
        if lib.has("hri_from_row"):  # cross-check the string against the oracle's C++ formatter
            for s, row in hri_seen:
                out = C.create_string_buffer(512)
                name = s.split("|")[0].encode()
                assert lib.fn("hri_from_row")(name, row.ctypes.data_as(C.c_void_p), out, C.c_size_t(512)) == 0
                assert out.value.decode() == s
        for n in list(pm.paused):
            assert pm.unpause(n)
    return pm


def test_pause_unpause_cpu(oracle_lib):
    a, b = drive_pausing(oracle_lib, True), drive_pausing(oracle_lib, False)
    assert a.apps[0].state == b.apps[0].state and all(x.state == a.apps[0].state for x in a.apps)
    assert a.num_decisions == b.num_decisions
    names = sorted(a.instances)
    ra = {n: a.engine.dump_rows(np.array([a.instances[n].gid], dtype=np.uint32), 0)[0] for n in names}
    rb = {n: b.engine.dump_rows(np.array([b.instances[n].gid], dtype=np.uint32), 0)[0] for n in names}
    for n in names:
        for f in ("acc_slot", "acc_bnum", "acc_bcoord", "acc_gc_slot", "next_proposal_slot", "coord_active"):
            assert ra[n][f] == rb[n][f], (n, f)


@pytest.mark.gpu
def test_pause_unpause_gpu(cuda_lib, oracle_lib):
    g, o = drive_pausing(cuda_lib, True), drive_pausing(oracle_lib, True)
    assert g.apps[0].state == o.apps[0].state and g.num_decisions == o.num_decisions
    assert g.checkpoints == o.checkpoints


# ---- view change: host half of phase 1 over the device's phase 1a (PISM.checkRunForCoordinator :2090,
#      handlePrepareReply :957, PCS.combinePValuesOntoProposals :393) ------------------------------------------------
def drive_view_change(lib, p1b=False):
    from helpers import make_requests
    pm = make_pm(lib, HashChainApp, checkpoint_interval=100, p1b=p1b)
    eng = pm.engine
    names = [f"TESTPaxosApp{i}" for i in range(9)]
    pm.createPaxosInstanceBatch({n: None for n in names}, NODES)
    for r in range(3):
        for n in names:
            pm.propose(n, f"{n}:{r}".encode())
        pm.run_round()
    gids = np.array([pm.instances[n].gid for n in names], dtype=np.uint32)
    rows0 = eng.dump_rows(gids, 0)
    old_coord = {n: NODES.index(int(rows0[i]["acc_bcoord"])) for i, n in enumerate(names)}
    # the old coordinators get two more slots ACCEPTed at a majority / a minority of the lanes and then "die": no
    # replies are tallied, nothing is decided
    for k, reach in enumerate((0b011, 0b101, 0b100)):  # third slot: only one acceptor ever sees it
        reqs, pay = make_requests(gids, payload_len=9 + k, seed=5, round_no=k)
        reqs["flags"] = [old_coord[n] << 8 for n in names]
        reqs["entry_node"] = [NODES[old_coord[n]] for n in names]
        acc, blob, st = eng.propose(reqs, pay)
        assert np.all(st > 0)
        acc["dst_mask"] = reach
        eng.handle_accepts(acc, blob)
    before = pm.apps[0].seqnum.copy() if hasattr(pm.apps[0].seqnum, "copy") else dict(pm.apps[0].seqnum)
    # the next node in line runs for coordinator in every group
    won = []
    for n in names:
        new_lane = (old_coord[n] + 1) % 3
        assert pm.runForCoordinator(n, new_lane)
        won.append(new_lane)
    rows = [eng.dump_rows(gids, l) for l in range(3)]
    for i, n in enumerate(names):
        nl = won[i]
        assert rows[nl][i]["coord_exists"] and rows[nl][i]["coord_active"]
        assert rows[nl][i]["coord_bcoord"] == NODES[nl] and rows[nl][i]["coord_bnum"] == rows0[i]["acc_bnum"] + 1
        assert all(not rows[l][i]["coord_exists"] for l in range(3) if l != nl)
        # every replica executed the carried-over slots: at least the two slots a majority had accepted
        assert all(rows[l][i]["acc_slot"] >= rows0[i]["acc_slot"] + 2 for l in range(3))
        assert len({int(rows[l][i]["acc_slot"]) for l in range(3)}) == 1
    s0 = pm.apps[0].state
    assert all(a.state == s0 for a in pm.apps)  # the carried-over values were executed identically everywhere
    assert all(pm.apps[0].seqnum[n] > before[n] for n in names)
    # a stale candidate is preempted: some acceptor has promised a higher ballot
    g0 = int(gids[0])
    cand = (won[0] + 2) % 3
    p = np.zeros(2, dtype=abi.patch_dtype)
    for k, l in enumerate(x for x in range(3) if x != cand):  # a majority has promised ballot 50 to someone else
        p[k]["gid"], p[k]["lane"], p[k]["op"], p[k]["a"], p[k]["b"] = g0, l, abi.PATCH_SET_BALLOT, 50, NODES[won[0]]
    eng.patch(p)
    assert not pm.runForCoordinator(names[0], cand)
    # business as usual under the new coordinators
    got = []
    for r in range(2):
        for n in names[1:]:
            pm.propose(n, f"{n}:after{r}".encode(), entry_node=NODES[won[names.index(n)]],
                       callback=lambda req, ok: got.append(req.slot))
        pm.run_round()
    assert len(got) == 2 * (len(names) - 1) and all(a.state == pm.apps[0].state for a in pm.apps)
    return pm


def test_view_change_cpu(oracle_lib):
    drive_view_change(oracle_lib)


def _same_end_state(a, b):
    assert a.apps[0].state == b.apps[0].state and a.num_decisions == b.num_decisions
    names = sorted(a.instances)
    for lane in range(3):
        ra = a.engine.dump_rows(np.array([a.instances[n].gid for n in names], dtype=np.uint32), lane)
        rb = b.engine.dump_rows(np.array([b.instances[n].gid for n in names], dtype=np.uint32), lane)
        for f in ra.dtype.names:
            assert np.array_equal(ra[f], rb[f]), (lane, f)


def test_phase1b_in_the_engine_equals_the_host_twin_cpu(oracle_lib):
    """gpx_handle_prepare_replies (here: the oracle's restatement of PCS phase 1b) against the host-language twin
    (tally_prepare_replies / combine_carryover + gpx_patch) through whole view changes: same rows, same executions"""
    _same_end_state(drive_view_change(oracle_lib, p1b=True), drive_view_change(oracle_lib))
    _same_end_state(drive_auto_election(oracle_lib, p1b=True), drive_auto_election(oracle_lib))
    _same_end_state(drive_lagging_election(oracle_lib, p1b=True), drive_lagging_election(oracle_lib))


@pytest.mark.gpu
def test_view_change_gpu(cuda_lib, oracle_lib):
    g, o = drive_view_change(cuda_lib), drive_view_change(oracle_lib)
    assert g.apps[0].state == o.apps[0].state and g.num_decisions == o.num_decisions
    names = sorted(g.instances)
    for lane in range(3):
        rg = g.engine.dump_rows(np.array([g.instances[n].gid for n in names], dtype=np.uint32), lane)
        ro = o.engine.dump_rows(np.array([o.instances[n].gid for n in names], dtype=np.uint32), lane)
        for f in rg.dtype.names:
            assert np.array_equal(rg[f], ro[f]), (lane, f)


def _reply(acc_idx, ballot, accepted=(), gc_slot=-1, flags=0):
    """a PREPARE_REPLY record as gpx_handle_prepares writes it: accepted = [(slot, bnum, bcoord, stop)]"""
    r = np.zeros(1, dtype=abi.prepare_reply_dtype)[0]
    r["bnum"], r["bcoord"], r["first_slot"] = ballot[0], ballot[1], gc_slot
    r["who"] = abi.who(acc_idx, 0, flags)
    for k, (slot, bn, bc, stop) in enumerate(sorted(accepted)):
        a = r["accepted"][k]
        a["slot"], a["bnum"], a["bcoord"], a["req_id"], a["flags"] = slot, bn, bc, 1000 + slot, (2 if stop else 0) | (1 << 16)
    r["n_accepted"] = len(accepted)
    return r


def test_prepare_reply_tally_follows_the_reference_code():
    """The scenario of PaxosCoordinatorState.main's phase-1 half (PaxosCoordinatorState.java:1008-1178): 43 members, my
    ballot (2, 21); carry-overs at slots 2 (two ballots), 6, 7, 8, 9 reported by members[2], members[0], members[4];
    then the even members answer with nothing -- evaluated by the CODE the scenario runs through, where it and the
    scenario's own assertions disagree:
      * recordSlotNumber :786-807 records PrepareReplyPacket.getMinSlot() :151-164, which STARTS at firstSlot (gcSlot + 1
        = 0 for these replies) -- so every heard member records 0, the view change fills from slot 0, and main()'s
        `assert (slot >= maxMinSlot)` with maxMinSlot = 7 (:1165) cannot hold at this revision (it matches the static
        getMinSlot(int, Map) :166-177 the packet stores in its unused minSlot field).  Filling from firstSlot is what
        keeps a group live: slots 0, 1, 3, 4, 5 were accepted by nobody that answered and get no-ops;
      * processStop :478-554 compares ballots that ProposalStateAtCoordinator's constructor :153-157 has re-stamped with
        the new ballot, so it converts nothing; a regular request behind a STOP is its assert(false) branch."""
    from gigapaxos_b200.paxos_manager import PaxosManager
    R, my = 43, (2, 21)
    T = PaxosManager.tally_prepare_replies
    assert T([_reply(0xFF, (29, 42), flags=abi.F_VOID)], R, my)[0] == "waiting"      # not a member: ignored
    assert T([_reply(3, (1, 21))], R, my) == ("waiting", [-1] * R, {})              # lower ballot: ignored
    assert T([_reply(3, (2, 20))], R, my)[0] == "waiting"
    assert T([_reply(3, (2, 22))], R, my)[0] == "preempted"                         # isPreemptable
    rs = [_reply(2, my, [(2, 1, 20, False)]),                                        # members[2]
          _reply(2, my, [(2, 1, 20, False)]),                                        # duplicate: ignored
          _reply(0, my, [(2, 1, 21, False), (6, 1, 21, False)]),                     # members[0]
          _reply(4, my, [(7, 1, 21, False), (8, 1, 22, False), (9, 1, 20, False)])]  # members[4]
    rs += [_reply(i, my) for i in range(0, R, 2)]                                    # members 0, 2, 4, ... with nothing
    for cut in (len(rs) - 1, len(rs)):
        verdict, ns, carry = T(rs[:cut], R, my)
        assert verdict == ("majority" if cut == len(rs) else "waiting")            # 22 of 43 heard only at the end
    assert ns[2] == 0 and ns[0] == 0 and ns[4] == 0 and ns[6] == 0 and ns[1] == -1   # getMinSlot() = firstSlot here
    assert sorted(carry) == [2, 6, 7, 8, 9] and int(carry[2][0]["bcoord"]) == 21    # the higher ballot wins slot 2
    plan, nxt, fl = PaxosManager.combine_carryover(carry, ns, acc_slot=0)
    assert nxt == 0 and fl == 0 and [e[0] for e in plan] == list(range(10))
    assert [e[1] for e in plan] == [abi.CO_NOOP, abi.CO_NOOP, abi.CO_PVALUE, abi.CO_NOOP, abi.CO_NOOP, abi.CO_NOOP,
                                    abi.CO_PVALUE, abi.CO_PVALUE, abi.CO_PVALUE, abi.CO_PVALUE]
    # acceptors that have garbage-collected through slot 6 answer firstSlot = 7: the fill starts there
    rs7 = [_reply(2, my, [(7, 1, 20, False)], gc_slot=6), _reply(0, my, [(9, 1, 21, False)], gc_slot=6)]
    rs7 += [_reply(i, my, gc_slot=6) for i in range(4, R, 2)]
    verdict, ns, carry = T(rs7, R, my)
    assert verdict == "majority" and ns[2] == ns[0] == ns[4] == 7
    plan, nxt, _ = PaxosManager.combine_carryover(carry, ns, 0)
    assert nxt == 7 and [(e[0], e[1]) for e in plan] == [(7, abi.CO_PVALUE), (8, abi.CO_NOOP), (9, abi.CO_PVALUE)]
    # processStop: no conversion (same ballot everywhere after re-stamping); a request behind a STOP is flagged, and
    # since the last proposal is not a STOP a fresh one follows (:538-542)
    rs[3] = _reply(4, my, [(7, 1, 21, False), (8, 1, 22, True), (9, 1, 20, False)])
    _, ns, carry = T(rs, R, my)
    plan, _, fl = PaxosManager.combine_carryover(carry, ns, 0)
    assert fl == abi.ELF_STOP_ORDER and [e[1] for e in plan[7:]] == [abi.CO_PVALUE] * 3 + [abi.CO_STOP_NEW]
    assert plan[-1][0] == 10 and bool(int(plan[8][2]["flags"]) & 2) and not (int(plan[9][2]["flags"]) & 2)
    # a STOP in the last carried-over slot: nothing to add
    rs[3] = _reply(4, my, [(7, 1, 21, False), (8, 1, 19, False), (9, 1, 20, True)])
    _, ns, carry = T(rs, R, my)
    plan, _, fl = PaxosManager.combine_carryover(carry, ns, 0)
    assert fl == 0 and len(plan) == 10 and bool(int(plan[-1][2]["flags"]) & 2)
    # a reply whose lowest accepted slot lies below its firstSlot (accepts added from the journal) records that slot
    verdict, ns, carry = T([_reply(0, my, [(3, 1, 20, False)], gc_slot=5)] + [_reply(i, my, gc_slot=5) for i in range(2, R, 2)],
                           R, my)
    assert verdict == "majority" and ns[0] == 3 and ns[2] == 6
    # device rules: more than GPX_MAX_PLAN slots to fill -> refused
    verdict, ns, carry = T([_reply(0, my, [(40, 1, 20, False)])] + [_reply(i, my) for i in range(2, R, 2)], R, my)
    assert verdict == "majority" and PaxosManager.combine_carryover(carry, ns, 0) is None


# ---- catching up a lagging replica (PISM.syncLongDecisionGaps :1550 / handleSyncDecisionsPacket :2426 / checkpoint
#      transfer :1852) ------------------------------------------------------------------------------------------------
def drive_sync(lib, p1b=False):
    from gigapaxos_b200.paxos_manager import RequestPacket
    from helpers import make_requests
    pm = make_pm(lib, HashChainApp, checkpoint_interval=100, p1b=p1b)
    eng = pm.engine
    names = [f"TESTPaxosApp{i}" for i in range(6)]
    pm.createPaxosInstanceBatch({n: None for n in names}, NODES)
    for r in range(2):
        for n in names:
            pm.propose(n, f"{n}:{r}".encode())
        pm.run_round()
    gids = np.array([pm.instances[n].gid for n in names], dtype=np.uint32)
    rows0 = eng.dump_rows(gids, 0)
    coord = [NODES.index(int(rows0[i]["acc_bcoord"])) for i in range(len(names))]

    def rounds_without_lane2(k0, k1):
        """lane 2 is partitioned away: lanes 0 and 1 keep deciding (a majority) and executing"""
        for k in range(k0, k1):
            reqs, pay = make_requests(gids, payload_len=5 + k % 7, seed=9, round_no=k)
            reqs["flags"] = [c << 8 for c in coord]
            reqs["entry_node"] = [NODES[c] for c in coord]
            acc, blob, st = eng.propose(reqs, pay)
            assert np.all(st > 0)
            acc["dst_mask"] = 0b011
            rep, _ = eng.handle_accepts(acc, blob)
            dec = eng.handle_accept_replies(rep)
            assert len(dec) == len(names)
            dec["dst_mask"] = 0b011
            ex, extra = eng.handle_decisions(dec)
            batches = {int(r["req_id"]): [RequestPacket(names[i], int(r["req_id"]),
                                                        bytes(pay[int(r["payload_off"]): int(r["payload_off"]) + int(r["payload_len"])]),
                                                        entry_replica=NODES[coord[i]])]
                       for i, r in enumerate(reqs)}
            pm._apply(np.concatenate([ex, extra]), batches)

    rounds_without_lane2(0, 11)  # 11 slots: more than the window W = 8
    assert pm.apps[2].state != pm.apps[0].state and pm.apps[1].state == pm.apps[0].state
    for n in names:  # getLoggedDecisions + getActualDecisions from the donor's journal, W slots at a time
        assert pm.syncDecisions(n, 2) == 11
        assert pm.syncDecisions(n, 2) == 0
    assert pm.apps[2].state == pm.apps[0].state and pm.apps[2].seqnum == pm.apps[0].seqnum
    r2, r0 = eng.dump_rows(gids, 2), eng.dump_rows(gids, 0)
    assert np.array_equal(r2["acc_slot"], r0["acc_slot"])
    # the lane falls behind again, but now it has promised a higher ballot to someone: the old accepts are refused,
    # so it catches up by checkpoint transfer (handleCheckpoint -> jumpSlot)
    # (groups whose coordinator sits on lane 2 are left alone: bumping its acceptor's ballot would depose it)
    bump = [i for i in range(len(names)) if coord[i] != 2]
    assert bump
    p = np.zeros(len(bump), dtype=abi.patch_dtype)
    p["gid"], p["lane"], p["op"], p["a"], p["b"] = gids[bump], 2, abi.PATCH_SET_BALLOT, 9, NODES[2]
    eng.patch(p)
    rounds_without_lane2(11, 14)
    for i, n in enumerate(names):
        assert pm.syncDecisions(n, 2) == (1 if i in bump else 3)  # one checkpoint / three replayed slots
    assert pm.apps[2].state == pm.apps[0].state
    r2, r0 = eng.dump_rows(gids, 2), eng.dump_rows(gids, 0)
    assert np.array_equal(r2["acc_slot"], r0["acc_slot"]) and np.all(r2["acc_bnum"][bump] == 9)
    return pm


def test_sync_decisions_cpu(oracle_lib):
    a = drive_sync(oracle_lib)
    b = drive_sync(oracle_lib, p1b=True)  # the donor's journal looked up by gpx_log_find instead of a host walk of the ring
    assert a.apps[2].state == b.apps[2].state and a.num_decisions == b.num_decisions


@pytest.mark.gpu
def test_sync_decisions_gpu(cuda_lib, oracle_lib):
    g, o = drive_sync(cuda_lib), drive_sync(oracle_lib)
    assert g.apps[2].state == o.apps[2].state and g.apps[0].state == o.apps[0].state
    names = sorted(g.instances)
    for lane in range(3):
        rg = g.engine.dump_rows(np.array([g.instances[n].gid for n in names], dtype=np.uint32), lane)
        ro = o.engine.dump_rows(np.array([o.instances[n].gid for n in names], dtype=np.uint32), lane)
        for f in rg.dtype.names:
            assert np.array_equal(rg[f], ro[f]), (lane, f)


def drive_auto_election(lib, p1b=False):
    """a proposal that finds no coordinator makes its entry replica run for coordinator (PISM.handleProposal :862-885
    -> checkRunForCoordinator(true)); the request is decided by the new coordinator in the next round"""
    pm = make_pm(lib, HashChainApp, p1b=p1b)
    names = [f"TESTPaxosApp{i}" for i in range(5)]
    pm.createPaxosInstanceBatch({n: None for n in names}, NODES)
    for n in names:
        pm.propose(n, b"first")
    pm.run_round()
    gids = np.array([pm.instances[n].gid for n in names], dtype=np.uint32)
    rows = pm.engine.dump_rows(gids, 0)
    # every coordinator crashes: its row is gone (the acceptors keep their ballots)
    p = np.zeros(3 * len(names), dtype=abi.patch_dtype)
    for k in range(len(p)):
        p[k]["gid"], p[k]["lane"], p[k]["op"] = gids[k // 3], k % 3, abi.PATCH_RESIGN_COORD
    pm.engine.patch(p)
    got = []
    for i, n in enumerate(names):
        entry = (NODES.index(int(rows[i]["acc_bcoord"])) + 1) % 3  # a surviving replica receives the request
        pm.propose(n, b"second", entry_node=NODES[entry], callback=lambda req, ok: got.append((req.paxos_id, req.slot)))
    assert pm.run_round() == 0 and not got   # nobody could propose; elections ran instead
    assert pm.run_round() == 3 * len(names)  # the new coordinators decide the waiting requests
    assert sorted(got) == sorted((n, 2) for n in names)
    rows2 = pm.engine.dump_rows(gids, 0)
    assert np.all(rows2["acc_bnum"] == rows["acc_bnum"] + 1) and all(a.state == pm.apps[0].state for a in pm.apps)
    return pm


def test_auto_election_cpu(oracle_lib):
    drive_auto_election(oracle_lib)


@pytest.mark.gpu
def test_auto_election_gpu(cuda_lib, oracle_lib):
    g, o = drive_auto_election(cuda_lib), drive_auto_election(oracle_lib)
    assert g.apps[0].state == o.apps[0].state and g.num_decisions == o.num_decisions


# ---- a LAGGING replica runs for coordinator (ADVICE r1, high): with journaling the executed accepts have left the
#      acceptors' memory; the preparer must still learn them (PISM.handlePrepare -> getLoggedAccepts,
#      GET_ACCEPTED_PVALUES_FROM_DISK) or it would re-decide a decided slot with a new value ------------------------------
def drive_lagging_election(lib, p1b=False):
    from gigapaxos_b200.paxos_manager import RequestPacket
    from helpers import make_requests
    pm = make_pm(lib, HashChainApp, checkpoint_interval=100, p1b=p1b)
    eng = pm.engine
    names = [f"TESTPaxosApp{i}" for i in range(5)]
    pm.createPaxosInstanceBatch({n: None for n in names}, NODES)
    for n in names:
        pm.propose(n, f"{n}:first".encode())
    pm.run_round()
    gids = np.array([pm.instances[n].gid for n in names], dtype=np.uint32)
    rows0 = eng.dump_rows(gids, 0)
    coord = [NODES.index(int(rows0[i]["acc_bcoord"])) for i in range(len(names))]
    # lane 0 is partitioned away for three slots: lanes 1 and 2 decide and execute them (only groups they coordinate)
    lagging = [i for i in range(len(names)) if coord[i] != 0]
    assert lagging
    g2 = gids[lagging]
    for k in range(3):
        reqs, pay = make_requests(g2, payload_len=6, seed=4, round_no=k)
        reqs["flags"] = [coord[i] << 8 for i in lagging]
        reqs["entry_node"] = [NODES[coord[i]] for i in lagging]
        acc, blob, st = eng.propose(reqs, pay)
        assert np.all(st > 0)
        acc["dst_mask"] = 0b110
        rep, _ = eng.handle_accepts(acc, blob)
        dec = eng.handle_accept_replies(rep)
        dec["dst_mask"] = 0b110
        ex, extra = eng.handle_decisions(dec)
        batches = {int(r["req_id"]): [RequestPacket(names[lagging[j]], int(r["req_id"]),
                                                    bytes(pay[int(r["payload_off"]): int(r["payload_off"]) + int(r["payload_len"])]),
                                                    entry_replica=NODES[coord[lagging[j]]])]
                   for j, r in enumerate(reqs)}
        pm._apply(np.concatenate([ex, extra]), batches)
    assert np.all(eng.dump_rows(g2, 0)["acc_slot"] == 2) and np.all(eng.dump_rows(g2, 1)["acc_slot"] == 5)
    # the lagging lane 0 runs for coordinator of those groups and then proposes a NEW value
    for i in lagging:
        assert pm.runForCoordinator(names[i], 0)
        pm.propose(names[i], b"NEWVALUE", entry_node=NODES[0])
    pm.run_round()
    # every replica executed the same sequence: the old slots 2..4 kept their values, NEWVALUE landed behind them
    assert pm.apps[0].state == pm.apps[1].state == pm.apps[2].state
    assert pm.apps[0].seqnum == pm.apps[1].seqnum == pm.apps[2].seqnum
    for l in range(3):
        assert np.all(eng.dump_rows(g2, l)["acc_slot"] == 6)
    return pm


def test_lagging_lane_election_cpu(oracle_lib):
    drive_lagging_election(oracle_lib)


@pytest.mark.gpu
def test_lagging_lane_election_gpu(cuda_lib, oracle_lib):
    a, b = drive_lagging_election(cuda_lib), drive_lagging_election(oracle_lib)
    assert a.apps[0].state == b.apps[0].state


def test_create_and_kill_respect_the_pause_table(oracle_lib):
    """ADVICE r1 (medium): createPaxosInstance of a PAUSED name must unpause it and answer 'already exists' (it goes
    through PaxosManager.getInstance :2453), not wipe its state; kill must drop the pause-table entry."""
    pm = make_pm(oracle_lib, HashChainApp)
    pm.createPaxosInstance("p0", 0, NODES)
    pm.propose("p0", b"x")
    pm.run_round()
    state = pm.apps[0].state.get("p0") if isinstance(pm.apps[0].state, dict) else pm.apps[0].state
    assert pm.pause("p0") and pm.isPaused("p0")
    assert pm.createPaxosInstance("p0", 0, NODES) is False  # exists (paused): not re-created
    assert not pm.isPaused("p0") and "p0" in pm.instances
    after = pm.apps[0].state.get("p0") if isinstance(pm.apps[0].state, dict) else pm.apps[0].state
    assert after == state
    rows = pm.engine.dump_rows(np.array([pm.instances["p0"].gid], dtype=np.uint32), 0)
    assert int(rows[0]["acc_slot"]) == 2  # the restored row, not a fresh one
    assert pm.pause("p0") and pm.kill("p0") and not pm.isPaused("p0")
    assert pm.propose("p0", b"y") is None  # gone for good



def drive_failover_after_wrap(lib, overwritten):
    """40 groups decide rounds until every lane's 64 KiB log ring has wrapped twice; then the last ACCEPT of groups
    0..9 reaches only lanes 0 and 1 and is never decided; when `overwritten`, the other groups decide rounds for more
    than one lap after it.  The next node then runs for coordinator of groups 0..9 (one batch per old coordinator):
    the carried-over requests' bodies are in the acceptors' rings as long as the ring has not lapped them.  Returns
    (manager, names, the ten request bodies, the takeover as a callable)."""
    from helpers import group_descs, make_requests
    ring = 1 << 16
    eng = Engine(lib, make_config(lib, max_groups=64, max_batch_recs=4096, max_batch_payload=1 << 20,
                                  log_ring_bytes=ring))
    pm = PaxosManager(eng, [HashChainApp() for _ in NODES], NODES, device_phase1b=lib.has("handle_prepare_replies"))
    names = [f"TESTPaxosApp{i}" for i in range(40)]
    assert pm.createPaxosInstanceBatch({n: None for n in names}, NODES)
    r = 0
    while min(eng.log_head(l) for l in range(3)) < 2 * ring:
        for n in names:
            pm.propose(n, b"%s:%d" % (n.encode(), r))
        pm.run_round()
        r += 1
    gids = np.array([pm.instances[n].gid for n in names[:10]], dtype=np.uint32)
    coord = np.array([NODES.index(int(x)) for x in eng.dump_rows(gids, 0)["acc_bcoord"]])
    reqs, pay = make_requests(gids, payload_len=9, seed=5)
    reqs["flags"] = coord << 8
    reqs["entry_node"] = np.array(NODES)[coord]
    acc, blob, _ = eng.propose(reqs, pay)
    acc["dst_mask"] = 0b011
    eng.handle_accepts(acc, blob)
    bodies = [bytes(pay[int(o): int(o) + 9]) for o in reqs["payload_off"]]
    if overwritten:
        h0 = [eng.log_head(l) for l in range(3)]
        while min(eng.log_head(l) - h0[l] for l in range(3)) <= ring:
            for n in names[10:]:
                pm.propose(n, b"%s:%d" % (n.encode(), r))
            pm.run_round()
            r += 1

    def takeover():
        for c in range(3):
            won = pm.runForCoordinators([names[i] for i in range(10) if coord[i] == c], (c + 1) % 3)
            assert all(won.values())
        pm.run_round()
    return pm, names, bodies, takeover


@pytest.mark.parametrize("overwritten", [False, True])
def test_failover_after_the_ring_wrapped_cpu(oracle_lib, overwritten):
    pm, names, bodies, takeover = drive_failover_after_wrap(oracle_lib, overwritten)
    if overwritten:
        with pytest.raises(abi.GpxError, match="overwritten"):
            takeover()
        return
    takeover()
    for n, b in zip(names, bodies):  # the carried-over request executed with its own body on every replica
        assert all(a.state[n][: len(b)] == b for a in pm.apps)


@pytest.mark.gpu
@pytest.mark.parametrize("overwritten", [False, True])
def test_failover_after_the_ring_wrapped_gpu(cuda_lib, oracle_lib, overwritten):
    (g, names, bodies, tg), (o, _, _, to) = drive_failover_after_wrap(cuda_lib, overwritten), \
        drive_failover_after_wrap(oracle_lib, overwritten)
    if overwritten:
        for t in (tg, to):
            with pytest.raises(abi.GpxError, match="overwritten"):
                t()
        return
    tg()
    to()
    for n, b in zip(names, bodies):
        assert all(a.state[n][: len(b)] == b for a in g.apps)
    assert all(a.state == o.apps[0].state and a.seqnum == o.apps[0].seqnum for a in g.apps)
