"""Host-side mirror of the reference's interface for the hot path.

`PaxosManager` mirrors the calls of gigapaxos/PaxosManager.java that feed and drain the
phase-2 path -- createPaxosInstance (:632, batch form :664-691), propose (:1214) /
proposeStop, executed (:311-330), kill (:2162) -- on top of the engine's C ABI, and
`Replicable` / `NoopPaxosApp` mirror gigapaxos/interfaces/Replicable.java and
gigapaxos/examples/noop/NoopPaxosApp.java:19-72.  The reference's host language is Java; no
JVM exists in this image, so this mirror is Python (INTEGRATION.md shows the JNI binding).

One manager serves all co-located replicas ("lanes") of its groups, the way the reference's
TESTPaxosMain runs several PaxosManagers in one JVM (testing/TESTPaxosMain.java:51-64).
Requests are queued per call like RequestBatcher.enqueue (RequestBatcher.java:112) and one
`run_round()` is one pass of the hot path: batch + propose, then accept -> tally -> commit on
the device; the EXEC records come back in per-group slot order and are applied to the app of
every replica (PISM.execute :1755-1842).
"""
from __future__ import annotations

import hashlib
import time
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from . import abi
from .abi import Engine


class Replicable:
    """gigapaxos/interfaces/Replicable.java: execute / checkpoint / restore."""

    def execute(self, name: str, request: "RequestPacket", do_not_reply_to_client: bool) -> bool:
        raise NotImplementedError

    def checkpoint(self, name: str) -> Optional[str]:
        return None

    def restore(self, name: str, state: Optional[str]) -> bool:
        return True


class NoopPaxosApp(Replicable):
    """gigapaxos/examples/noop/NoopPaxosApp.java:19-72: echoes the request, null checkpoints."""

    def __init__(self):
        self.executed = 0

    def execute(self, name, request, do_not_reply_to_client):
        request.response_value = b"echoing [" + request.request_value + b"]"  # :26-28
        self.executed += 1
        return True


class HashChainApp(Replicable):
    """The invariant app of the reference's tests (testing/TESTPaxosApp.java:143-232):
    state = requestValue + SHA(state) and seqnum == slot (in-order, gap-free execution)."""

    def __init__(self):
        self.state: Dict[str, bytes] = {}
        self.seqnum: Dict[str, int] = {}

    def execute(self, name, request, do_not_reply_to_client):
        cur = self.state.get(name, b"")
        self.state[name] = request.request_value + hashlib.sha1(cur).digest()  # TESTPaxosApp.java:179-180
        expect = self.seqnum.get(name, 1)
        if request.slot is not None and request.batch_index == 0:
            assert request.slot == expect, f"{name}: executing slot {request.slot}, expected {expect}"  # :190
            self.seqnum[name] = expect + 1
        request.response_value = b"ok"
        return True

    def checkpoint(self, name):
        return self.state.get(name, b"").hex()

    def restore(self, name, state):
        self.state[name] = bytes.fromhex(state) if state else b""
        return True


@dataclass
class RequestPacket:
    """paxospackets/RequestPacket.java essentials."""
    paxos_id: str
    request_id: int
    request_value: bytes
    stop: bool = False
    entry_replica: int = -1
    entry_time: float = 0.0
    response_value: Optional[bytes] = None
    slot: Optional[int] = None
    batch_index: int = 0
    callback: Optional[Callable[["RequestPacket", bool], None]] = field(default=None, repr=False)


@dataclass
class HotRestoreInfo:
    """paxosutil/HotRestoreInfo.java:40-120: the state a paused instance is rebuilt from, and its '|'-separated
    string form (the value of the pause table, SQLPaxosLogger.pause)."""
    paxosID: str
    version: int
    members: List[int]
    accSlot: int
    accBallot: tuple  # (ballotNumber, coordinatorID)
    accGCSlot: int
    coordBallot: Optional[tuple]  # None unless this node is an ACTIVE coordinator (getBallotIfActive :400)
    nextProposalSlot: int  # -1 unless active (getNextProposalSlotIfActive :375)
    nodeSlots: Optional[List[int]]

    @staticmethod
    def _ints(a) -> str:  # Util.arrayOfIntToString :241-248
        return "[" + ",".join(str(int(x)) for x in a) + "]"

    def __str__(self) -> str:  # HotRestoreInfo.toString :88-107
        b = lambda t: f"{t[0]}:{t[1]}"  # Ballot.toString :105
        return "|".join([self.paxosID, str(self.version), self._ints(self.members), str(self.accSlot),
                         b(self.accBallot), str(self.accGCSlot), b(self.coordBallot) if self.coordBallot else "null",
                         str(self.nextProposalSlot), self._ints(self.nodeSlots) if self.nodeSlots is not None else "null"])

    @classmethod
    def parse(cls, ser: str) -> "HotRestoreInfo":  # HotRestoreInfo(String) :71-85
        t = ser.split("|")
        ints = lambda x: [int(v) for v in x.replace("[", "").replace("]", "").replace(" ", "").split(",")]
        bal = lambda x: tuple(int(v) for v in x.split(":"))
        return cls(t[0], int(t[1]), ints(t[2]), int(t[3]), bal(t[4]), int(t[5]), bal(t[6]) if t[6] != "null" else None,
                   int(t[7]), ints(t[8]) if t[8] != "null" else None)

    @classmethod
    def from_row(cls, paxosID: str, row) -> "HotRestoreInfo":
        """PISM.tryPause :2004-2025 from one dumped engine row (gpx_row)"""
        n = int(row["n_members"])
        active = bool(row["coord_exists"]) and bool(row["coord_active"])
        return cls(paxosID, int(row["version"]), [int(x) for x in row["members"][:n]], int(row["acc_slot"]),
                   (int(row["acc_bnum"]), int(row["acc_bcoord"])), int(row["acc_gc_slot"]),
                   (int(row["coord_bnum"]), int(row["coord_bcoord"])) if active else None,
                   int(row["next_proposal_slot"]) if active else -1,
                   [int(x) for x in row["node_slots"][:n]] if active else None)

    def to_row(self, gid: int, lane: int, my_node: int) -> np.ndarray:
        """PISM.hotRestore :677-690: the acceptor comes back ACTIVE; the coordinator only at the node it names"""
        r = np.zeros(1, dtype=abi.row_dtype)
        n = len(self.members)
        r["gid"], r["lane"], r["version"] = gid, lane, self.version
        r["name_hash"] = abi.java_string_hash(self.paxosID)  # getCPI :2694-2697 is a function of the paxosID
        r["acc_slot"], r["acc_bnum"], r["acc_bcoord"], r["acc_gc_slot"] = (self.accSlot, self.accBallot[0],
                                                                            self.accBallot[1], self.accGCSlot)
        r["state"] = abi.ST_ACTIVE_1  # paxosState.setActive(): no recovery
        r["n_members"] = n
        r["members"][0, :n] = self.members
        if self.coordBallot is not None and self.coordBallot[1] == my_node:
            r["coord_exists"], r["coord_active"] = 1, 1
            r["coord_bnum"], r["coord_bcoord"] = self.coordBallot
            r["next_proposal_slot"] = self.nextProposalSlot
            r["node_slots"][0, :n] = self.nodeSlots
        return r


NO_OP = b"NO_OP"  # RequestPacket.NO_OP: fills the slot gaps a new coordinator finds (PCS.makeNoopPValue :886-897)


def _jsub(a: int, b: int) -> int:
    """Java's wrap-around int subtraction"""
    d = (a - b) & 0xFFFFFFFF
    return d - (1 << 32) if d & 0x80000000 else d


def _jadd(a: int, b: int) -> int:
    """Java's wrap-around int addition"""
    return _jsub(a, -b)


@dataclass
class _Instance:
    gid: int
    version: int
    members: Sequence[int]
    stopped: bool = False


class PaxosManager:
    """Mirror of the PaxosManager calls on the hot path, for co-located replicas."""

    def __init__(self, engine: Engine, apps: Sequence[Replicable], nodes: Sequence[int],
                 device_phase1b: Optional[bool] = None, device_log_find: Optional[bool] = None):
        if len(apps) != engine.n_lanes or len(nodes) != engine.n_lanes:
            raise ValueError("one app and one node id per lane")
        self.engine = engine
        self.apps = list(apps)
        self.nodes = list(nodes)
        self.instances: Dict[str, _Instance] = {}
        self.gid_name: Dict[int, str] = {}
        self.free_gids: List[int] = []
        self.next_gid = 0
        self.queue: Dict[str, List[RequestPacket]] = {}  # RequestBatcher.batched :49
        self.outstanding: Dict[int, RequestPacket] = {}  # PaxosManager.outstanding
        self.next_request_id = 1
        self.checkpoints: List[tuple] = []
        self.num_decisions = 0
        self.slow_path: List[tuple] = []
        self.auto_elect = True  # run for coordinator when a proposal finds none (PISM.handleProposal :862-885)
        self._elect: Dict[str, int] = {}
        self.paused: Dict[str, List[str]] = {}  # paxosID -> HotRestoreInfo string per lane (the pause table)
        # phase 1b (tally of PREPARE_REPLYs, carry-over, no-op fill, install): inside the engine
        # (gpx_handle_prepare_replies, the default when the library has it) or by the host-language twin below + gpx_patch
        self.device_phase1b = engine.L.has("handle_prepare_replies") if device_phase1b is None else device_phase1b
        # logged decisions / accepts for a lagging replica: a scan of the donor's ring on the device (gpx_log_find) or a
        # walk of the whole ring on the host
        self.device_log_find = engine.L.has("log_find") if device_log_find is None else device_log_find

    # ---- instance management ------------------------------------------------------------
    def _alloc_gid(self) -> int:
        if self.free_gids:
            return self.free_gids.pop()
        g = self.next_gid
        if g >= int(self.engine.cfg.max_groups):
            raise RuntimeError("PINSTANCES_CAPACITY exceeded")
        self.next_gid += 1
        return g

    def createPaxosInstance(self, paxosID: str, version: int, gms: Sequence[int], initialState: Optional[str] = None,
                            batch: bool = False) -> bool:
        """PaxosManager.createPaxosInstance :632-662: refuses an existing (paxosID, version' >= version);
        a higher version replaces a stopped lower one (reconfiguration: stop at e, create at e+1)."""
        return self.createPaxosInstanceBatch({paxosID: initialState}, gms, version=version, batch=batch)

    def createPaxosInstanceBatch(self, nameStates: Dict[str, Optional[str]], gms: Sequence[int], version: int = 0,
                                 batch: bool = True) -> bool:
        """PaxosManager.createPaxosInstance(Map, Set) :664-691 (HotRestoreInfo.createHRI initial rows)."""
        descs = np.zeros(len(nameStates), dtype=abi.group_desc_dtype)
        created = True
        k = 0
        for name, state in nameStates.items():
            if name in self.paused:  # createPaxosInstance goes through getInstance :2453, which unpauses first: a paused
                self.unpause(name)   # instance exists -- creating it again must not wipe its state
            old = self.instances.get(name)
            if old is not None:
                if old.version >= version or not old.stopped:
                    created = False  # :646-652 "paxos instance already exists"
                    continue
                self._release(name)
            gid = self._alloc_gid()
            self.instances[name] = _Instance(gid, version, sorted(gms))
            self.gid_name[gid] = name
            d = descs[k]
            d["gid"], d["version"], d["name_hash"], d["n_members"] = gid, version, abi.java_string_hash(name), len(gms)
            d["members"][: len(gms)] = sorted(gms)
            d["init_mode"] = abi.INIT_BATCH if batch else abi.INIT_DEFAULT
            k += 1
            for app in self.apps:
                app.restore(name, state)  # PISM ctor :213-217 / putInitialState :692
        if k:
            self.engine.create_groups(descs[:k])
        return created

    def _release(self, name: str):
        inst = self.instances.pop(name)
        self.gid_name.pop(inst.gid, None)
        self.engine.destroy_groups([inst.gid])
        self.free_gids.append(inst.gid)

    def kill(self, paxosID: str) -> bool:
        """PaxosManager.kill :2162."""
        was_paused = self.paused.pop(paxosID, None) is not None  # a killed instance leaves no pause-table entry behind
        if paxosID not in self.instances:
            return was_paused
        self._release(paxosID)
        return True

    # ---- view change: the host half of phase 1 over the device's phase 1a -----------------------------------
    def runForCoordinator(self, paxosID: str, lane: int) -> bool:
        """PISM.checkRunForCoordinator(forceRun) :2090-2150 at the node of `lane`, then PISM.handlePrepareReply
        :1017-1068 / PCS.isPrepareAcceptedByMajority :326-391, combinePValuesOntoProposals :393-444, processStop
        :478-554 and spawnCommandersForProposals :556-575 for the PREPARE_REPLYs of the local lanes.

        The acceptors answer on the device (gpx_handle_prepares); the replies are tallied, the carry-over is laid out
        and the new coordinator installed by gpx_handle_prepare_replies (or, device_phase1b = False, by the
        host-language twin and gpx_patch records); the carried-over pvalues are then re-proposed in slot order under
        the new ballot, their request bodies read from the log ring of the acceptor that reported them.  Returns False
        when the election was preempted or found no majority."""
        inst = self.instances.get(paxosID)
        if inst is None or inst.stopped:
            return False
        eng, L = self.engine, self.engine.n_lanes
        gids = np.array([inst.gid], dtype=np.uint32)
        members = list(inst.members)
        R = len(members)
        me = self.nodes[lane]
        cur = eng.dump_rows(gids, lane)[0]
        new_ballot = (int(cur["acc_bnum"]) + 1, me)  # new Ballot(curBallot.ballotNumber + 1, myID) :2143
        prep = np.zeros(1, dtype=abi.decision_dtype)
        prep["gid"], prep["slot"] = inst.gid, int(cur["acc_slot"])  # PreparePacket(newBallot, paxosState.getSlot())
        prep["bnum"], prep["bcoord"] = new_ballot
        prep["flags"], prep["dst_mask"] = abi.F_PREPARE, (1 << L) - 1
        # A preparer that is BEHIND some acceptor must hear about the accepts of [my slot, acceptor's slot) as well.
        # With journaling they have left the acceptor's memory (executed accepts are served from the journal:
        # PISM.handlePrepare -> getLoggedAccepts, GET_ACCEPTED_PVALUES_FROM_DISK); the acceptor flags its reply
        # GPX_F_FROM_LOG and the host adds them from the acceptor's log.  When the ring no longer holds them the lane
        # catches up first (PISM.syncLongDecisionGaps) -- electing it with a stale first slot would let it re-decide a
        # decided slot with a new value.
        rows_before = [eng.dump_rows(gids, l)[0] for l in range(L)]
        logged = {}
        if any(_jsub(int(r["acc_slot"]), int(cur["acc_slot"])) > 0 for l, r in enumerate(rows_before) if l != lane):
            logged = self._logged_accepts(inst.gid, int(cur["acc_slot"]), [l for l in range(L) if l != lane])
            if logged is None:
                self.syncDecisions(paxosID, lane)
                cur = eng.dump_rows(gids, lane)[0]
                if any(_jsub(int(eng.dump_rows(gids, l)[0]["acc_slot"]), int(cur["acc_slot"])) > 0
                       for l in range(L) if l != lane):
                    return False  # still behind: no election from here
                logged = {}
                new_ballot = (int(cur["acc_bnum"]) + 1, me)
                prep["slot"], prep["bnum"] = int(cur["acc_slot"]), new_ballot[0]
        replies = eng.handle_prepares(prep)
        # (reply index == lane: gpx_handle_prepares answers at index i * n_lanes + lane and there is one PREPARE)
        if self.device_phase1b:
            res = self._phase1b_engine(inst.gid, lane, new_ballot, int(cur["acc_slot"]), replies, logged)
        else:
            res = self._phase1b_host(inst.gid, lane, R, new_ballot, int(cur["acc_slot"]), replies, logged)
        if res is None:
            return False
        plan = res
        # spawnCommandersForProposals :556-575: one ACCEPT per carried-over slot, in slot order, under my ballot
        for sl, kind, pv, src in plan:
            if kind == abi.CO_NOOP:
                reqs = [RequestPacket(paxosID, 0, NO_OP, entry_replica=me)]
            elif kind == abi.CO_STOP_NEW:
                reqs = [RequestPacket(paxosID, 0, b"STOP", stop=True, entry_replica=me)]  # PCS :541
            else:
                reqs = self._requests_of(paxosID, pv, src, me)
            self._submit(reqs, carryover=True)
        return True

    def runForCoordinators(self, paxosIDs: Sequence[str], lane: int) -> Dict[str, bool]:
        """The mass case: the node that coordinated these groups is gone and the node of `lane` runs for coordinator of
        all of them at once (the failure detector's sweep fires PISM.checkRunForCoordinator :2090-2150 per instance).
        ONE gpx_handle_prepares call, ONE gpx_handle_prepare_replies call (k_prepare_tally: one thread per election),
        then plan entry j of every elected group in round j (spawnCommandersForProposals :556-575) -- at most
        GPX_MAX_PLAN + 1 rounds however many groups elect.  A group whose candidate is behind one of its acceptors takes
        the single-group path (it needs the acceptors' logged accepts, or a sync, first)."""
        eng, L, me = self.engine, self.engine.n_lanes, self.nodes[lane]
        res: Dict[str, bool] = {}
        names = []
        for n in paxosIDs:
            inst = self.instances.get(n)
            if inst is None or inst.stopped:
                res[n] = False
            elif n not in res and n not in names:
                names.append(n)
        if not self.device_phase1b or not names:
            for n in names:
                res[n] = self.runForCoordinator(n, lane)
            return res
        gids = np.array([self.instances[n].gid for n in names], dtype=np.uint32)
        rows = [eng.dump_rows(gids, l) for l in range(L)]
        cur = rows[lane]
        behind = np.zeros(len(names), dtype=bool)
        for l in range(L):
            if l != lane:
                behind |= (rows[l]["acc_slot"].astype(np.int64) - cur["acc_slot"].astype(np.int64)).astype(np.int32) > 0
        batch = [i for i in range(len(names)) if not behind[i]]
        if batch:
            b = np.array(batch)
            prep = np.zeros(len(b), dtype=abi.decision_dtype)
            prep["gid"], prep["slot"] = gids[b], cur["acc_slot"][b]  # PreparePacket(newBallot, paxosState.getSlot())
            prep["bnum"], prep["bcoord"] = cur["acc_bnum"][b] + 1, me  # new Ballot(curBallot.ballotNumber + 1, myID)
            prep["flags"], prep["dst_mask"] = abi.F_PREPARE, (1 << L) - 1
            replies = eng.handle_prepares(prep)  # reply of PREPARE i at lane l: index i * L + l
            els = np.zeros(len(b), dtype=abi.election_dtype)
            els["gid"], els["lane"], els["bnum"], els["bcoord"] = prep["gid"], lane, prep["bnum"], me
            els["slot"], els["first_reply"], els["n_replies"] = prep["slot"], np.arange(len(b)) * L, L
            outs = eng.handle_prepare_replies(els, replies)
            plans = {}
            for k, i in enumerate(batch):
                o = outs[k]
                res[names[i]] = int(o["verdict"]) == abi.EL_MAJORITY
                if res[names[i]] and int(o["n_plan"]):
                    plans[names[i]] = o["plan"][: int(o["n_plan"])]
            # the request bodies of every carried-over pvalue, one gpx_log_gather per acceptor lane that holds some
            # (reply record index i * L + l: the acceptor at lane l reported the pvalue and has its body in its ring)
            body_of = {}
            if eng.L.has("log_gather"):
                per_lane: Dict[int, list] = {}
                for n, plan in plans.items():
                    for j, c in enumerate(plan):
                        if int(c["kind"]) == abi.CO_PVALUE and int(c["pv"]["payload_len"]):
                            per_lane.setdefault(int(c["src_reply"]) % L, []).append((n, j, c["pv"]))
                for l, items in per_lane.items():
                    pos = self._blob_positions(l, [(self.instances[n].gid, pv) for n, _, pv in items])
                    got = eng.log_gather(l, pos, [int(pv["payload_len"]) for _, _, pv in items])
                    for (n, j, _), b in zip(items, got):
                        body_of[(n, j)] = b
            for j in range(max((len(p) for p in plans.values()), default=0)):
                reqs: List[RequestPacket] = []
                for n in sorted(plans, key=lambda x: self.instances[x].gid):
                    if j >= len(plans[n]):
                        continue
                    c = plans[n][j]
                    if int(c["kind"]) == abi.CO_NOOP:
                        reqs.append(RequestPacket(n, 0, NO_OP, entry_replica=me))
                    elif int(c["kind"]) == abi.CO_STOP_NEW:
                        reqs.append(RequestPacket(n, 0, b"STOP", stop=True, entry_replica=me))  # PCS :541
                    elif (n, j) in body_of or not int(c["pv"]["payload_len"]):
                        reqs.extend(self._requests_from_blob(n, c["pv"], body_of.get((n, j), b""), me))
                    else:
                        reqs.extend(self._requests_of(n, c["pv"], int(c["src_reply"]) % L, me))
                self._submit(reqs, carryover=True)
        for i in range(len(names)):
            if behind[i]:
                res[names[i]] = self.runForCoordinator(names[i], lane)
        return res

    def _phase1b_host(self, gid, lane, R, new_ballot, acc_slot, replies, logged):
        """phase 1b in the host language (tally_prepare_replies / combine_carryover), its result installed with
        gpx_patch records.  Returns the plan [(slot, kind, pvalue, source lane)] or None."""
        eng, L = self.engine, self.engine.n_lanes
        gids = np.array([gid], dtype=np.uint32)
        verdict, node_slots, carry = self.tally_prepare_replies(replies, R, new_ballot, logged)
        if verdict != "majority":
            return None
        comb = self.combine_carryover(carry, node_slots, acc_slot)
        if comb is None:
            return None
        plan, next_slot, _ = comb
        # coordinators of a LOWER ballot resign (PISM.handlePrepare -> nullifyCoordinatorIfPreempted); the new one starts
        # ACTIVE at the first slot it has to fill
        pts = []
        for l in range(L):
            r = eng.dump_rows(gids, l)[0]
            if l != lane and bool(r["coord_exists"]) and (
                    _jsub(int(r["coord_bnum"]), new_ballot[0]) or _jsub(int(r["coord_bcoord"]), new_ballot[1])) > 0:
                continue  # a coordinator with a higher ballot is not ours to remove
            pts.append((gid, l, abi.PATCH_RESIGN_COORD, 0, 0, 0, 0))
        pts.append((gid, lane, abi.PATCH_INSTALL_COORD, new_ballot[0], new_ballot[1], next_slot, 1))
        for i, v in enumerate(node_slots):
            pts.append((gid, lane, abi.PATCH_SET_NODE_SLOT, i, v, 0, 0))
        p = np.zeros(len(pts), dtype=abi.patch_dtype)
        for i, t in enumerate(pts):
            p[i]["gid"], p[i]["lane"], p[i]["op"], p[i]["a"], p[i]["b"], p[i]["c"], p[i]["d"] = t
        eng.patch(p)
        return plan

    def _phase1b_engine(self, gid, lane, new_ballot, acc_slot, replies, logged):
        """phase 1b inside the engine (gpx_handle_prepare_replies: one kernel tallies, carries over, fills, installs).
        A reply that grew beyond GPX_MAX_WINDOW pvalues by its logged accepts travels as GPX_F_MORE continuation
        records.  Returns the plan [(slot, kind, pvalue, source lane)] or None."""
        recs, rec_lane = [], []
        for l, rep in enumerate(replies):
            acc = list(rep["accepted"][: int(rep["n_accepted"])])
            if logged and logged.get(l):
                have = {int(pv["slot"]) for pv in acc}
                acc = sorted(acc + [pv for pv in logged[l] if int(pv["slot"]) not in have], key=lambda pv: int(pv["slot"]))
            chunks = [acc[k: k + abi.GPX_MAX_WINDOW] for k in range(0, len(acc), abi.GPX_MAX_WINDOW)] or [[]]
            for ci, ch in enumerate(chunks):
                r = rep.copy()
                r["n_accepted"] = len(ch)
                r["accepted"][:] = 0
                for k, pv in enumerate(ch):
                    r["accepted"][k] = pv
                if ci + 1 < len(chunks):
                    r["who"] = int(r["who"]) | (abi.F_MORE << 16)
                recs.append(r)
                rec_lane.append(l)
        el = np.zeros(1, dtype=abi.election_dtype)
        el["gid"], el["lane"], el["bnum"], el["bcoord"], el["slot"] = gid, lane, new_ballot[0], new_ballot[1], acc_slot
        el["first_reply"], el["n_replies"] = 0, len(recs)
        out = self.engine.handle_prepare_replies(el, np.array(recs, dtype=abi.prepare_reply_dtype))[0]
        if int(out["verdict"]) != abi.EL_MAJORITY:
            return None
        return [(int(c["slot"]), int(c["kind"]), c["pv"].copy() if int(c["kind"]) == abi.CO_PVALUE else None,
                 rec_lane[int(c["src_reply"])] if int(c["kind"]) == abi.CO_PVALUE else 0)
                for c in out["plan"][: int(out["n_plan"])]]

    def _logged_accepts(self, gid: int, first_slot: int, lanes: Sequence[int]):
        """AbstractPaxosLogger.getLoggedAccepts for the PREPARE path (PISM.handlePrepare :896-955 with
        GET_ACCEPTED_PVALUES_FROM_DISK): per lane of `lanes`, the logged ACCEPTs of `gid` with slot >= first_slot found
        in its log ring (the highest ballot per slot), as {lane: [accepted pvalue records in slot order]} -- what that
        acceptor's PREPARE_REPLY would carry had the accepts still been in memory.  None when a ring has wrapped past
        what would be needed (the caller then syncs instead)."""
        out = {}
        ring = int(self.engine.cfg.log_ring_bytes)
        for l in lanes:
            head = self.engine.log_head(l)
            if head > ring:
                return None
            best = {}
            if self.device_log_find:  # getLoggedAccepts as a scan of the acceptor's ring on the device (gpx_log_find)
                top = _jadd(int(self.engine.dump_rows(np.array([gid], dtype=np.uint32), l)[0]["acc_slot"]),
                            int(self.engine.cfg.window))
                sl = first_slot
                while _jsub(sl, top) < 0:
                    w = np.zeros(1, dtype=abi.log_want_dtype)
                    w["gid"], w["min_slot"], w["n_slots"] = gid, sl, min(abi.GPX_LOG_SPAN, _jsub(top, sl))
                    for h in self.engine.log_find(l, w)[0][: int(w["n_slots"][0])]:
                        a = h["accept"]
                        if int(a["flags"]) & abi.F_VOID:
                            continue
                        pv = np.zeros(1, dtype=abi.accepted_pvalue_dtype)[0]
                        pv["slot"], pv["bnum"], pv["bcoord"] = int(a["slot"]), int(a["bnum"]), int(a["bcoord"])
                        pv["frame_ref"] = int(h["blob_pos"]) // 16
                        pv["req_id"], pv["payload_len"] = int(a["req_id"]), int(a["payload_len"])
                        pv["flags"] = (2 if int(a["flags"]) & abi.F_STOP else 0) | (int(a["nreq"]) << 16)
                        best[int(a["slot"])] = pv
                    sl = _jadd(sl, abi.GPX_LOG_SPAN)
                out[l] = [best[k] for k in sorted(best)]
                continue
            buf = self.engine.log_read(l, 0, head)
            for hdr, imgs, payload, pay_off in abi.parse_log(buf):
                if int(hdr["rec_bytes"]) != 48:
                    continue
                sel = imgs[(imgs["gid"] == gid) & ((imgs["flags"] & abi.F_VOID) == 0)]
                for a in sel:
                    sl = int(a["slot"])
                    if _jsub(sl, first_slot) < 0:
                        continue
                    pv = np.zeros(1, dtype=abi.accepted_pvalue_dtype)[0]
                    pv["slot"], pv["bnum"], pv["bcoord"] = sl, int(a["bnum"]), int(a["bcoord"])
                    pv["frame_ref"] = (pay_off + int(a["payload_off"])) // 16
                    pv["req_id"], pv["payload_len"] = int(a["req_id"]), int(a["payload_len"])
                    pv["flags"] = (2 if int(a["flags"]) & abi.F_STOP else 0) | (int(a["nreq"]) << 16)
                    ex = best.get(sl)
                    if ex is None or (_jsub(int(pv["bnum"]), int(ex["bnum"])) or
                                      _jsub(int(pv["bcoord"]), int(ex["bcoord"]))) > 0:
                        best[sl] = pv
            out[l] = [best[k] for k in sorted(best)]
        return out

    @staticmethod
    def tally_prepare_replies(replies, R: int, new_ballot: tuple, logged=None):
        """PISM.handlePrepareReply :1017-1068 over a sequence of gpx_prepare_reply records, in order: returns
        ("preempted" | "majority" | "waiting" | "overflow", nodeSlotNumbers, carryover {slot: (pvalue, reply index)}).
        logged[l]: accepted pvalues the acceptor behind reply l serves from its journal (GPX_F_FROM_LOG: with
        journaling the executed accepts have left its memory) -- part of its reply as far as the tally goes.
        The host-language twin of gpx_handle_prepare_replies (include/gpx.h), kept for engines without it and as a
        second restatement the CPU tests hold against the oracle's."""
        node_slots = [-1] * R  # PCS ctor :169-171
        heard, carry = set(), {}
        for l, rep in enumerate(replies):
            fl = abi.who_flags(int(rep["who"]))
            if fl & abi.F_VOID:
                continue
            rb = (int(rep["bnum"]), int(rep["bcoord"]))
            c = _jsub(rb[0], new_ballot[0]) or _jsub(rb[1], new_ballot[1])
            if c > 0:  # isPreemptable :271-278 -> getPreActivesIfPreempted: the election is lost
                return "preempted", node_slots, carry
            idx = abi.who_acc(int(rep["who"]))
            if c < 0 or idx in heard or idx >= R:  # canIgnorePrepareReply :287-316
                continue
            acc = list(rep["accepted"][: int(rep["n_accepted"])])
            if logged and logged.get(l):
                have = {int(pv["slot"]) for pv in acc}
                acc = sorted(acc + [pv for pv in logged[l] if int(pv["slot"]) not in have], key=lambda pv: int(pv["slot"]))
            # recordSlotNumber :786-807 with PrepareReplyPacket.getMinSlot() :151-164: it starts at firstSlot (= gcSlot + 1;
            # the record holds gcSlot) and takes the wrap-aware minimum with the accepted slots
            min_slot = _jadd(int(rep["first_slot"]), 1)
            for pv in acc:
                if _jsub(int(pv["slot"]), min_slot) < 0:
                    min_slot = int(pv["slot"])
            if _jsub(node_slots[idx], min_slot) < 0:
                node_slots[idx] = min_slot
            for pv in acc:  # the pvalue of the highest ballot per slot is carried over :347-366
                ex = carry.get(int(pv["slot"]))
                if ex is None or (_jsub(int(pv["bnum"]), int(ex[0]["bnum"])) or
                                  _jsub(int(pv["bcoord"]), int(ex[0]["bcoord"]))) > 0:
                    carry[int(pv["slot"])] = (pv.copy(), l)
                    if len(carry) > abi.GPX_MAX_CARRY:  # device rule
                        return "overflow", node_slots, carry
            heard.add(idx)
            if len(heard) > R // 2:  # WaitforUtility.heardFromMajority
                return "majority", node_slots, carry
        return "waiting", node_slots, carry

    @staticmethod
    def combine_carryover(carry: dict, node_slots: List[int], acc_slot: int):
        """PCS.combinePValuesOntoProposals :393-444 (this mirror keeps no pre-active proposals: requests wait in
        its queue): the slots from getMaxMinCarryoverSlot :921 to getMaxPValueSlot :903, carried-over pvalue or
        no-op, then processStop :478-554.  Returns (plan [(slot, kind, pvalue | None, reply index)], the first slot
        the new coordinator proposes, flags) or None when the range exceeds GPX_MAX_PLAN (device rule)."""
        if not carry:
            return [], acc_slot, 0  # PCS ctor: nextProposalSlotNumber = paxosState.getSlot()
        max_carry = max_min = None
        for sl in carry:
            max_carry = sl if max_carry is None or _jsub(sl, max_carry) > 0 else max_carry
        for v in node_slots:
            max_min = v if max_min is None or _jsub(v, max_min) > 0 else max_min
        span = _jsub(max_carry, max_min)
        if span >= abi.GPX_MAX_PLAN:
            return None
        plan: List[tuple] = []
        for d in range(span + 1):  # (span < 0: every carried-over slot lies below the slots to fill)
            sl = _jadd(max_min, d)
            plan.append((sl, abi.CO_PVALUE) + carry[sl] if sl in carry else (sl, abi.CO_NOOP, None, 0))
        plan, flags = PaxosManager._process_stop(plan, _jadd(max_carry, 1))
        return plan, (plan[0][0] if plan else _jadd(max_carry, 1)), flags

    @staticmethod
    def _process_stop(plan: List[tuple], next_slot: int):
        """PCS.processStop :478-554.  Every proposal carries the NEW coordinator's ballot here (the constructor of
        ProposalStateAtCoordinator :153-157 re-stamps it), so neither of its two conversions (request behind a
        higher-ballot STOP -> STOP :495-509, STOP before a higher-ballot request -> no-op :510-523) can be taken: a
        regular request behind a STOP is the reference's assert(false) :524, reported as ELF_STOP_ORDER.  What remains
        is the tail :538-542: a STOP was carried over but the last proposal is not one -> a fresh STOP behind it."""
        is_stop = lambda e: e[1] == abi.CO_STOP_NEW or (e[1] == abi.CO_PVALUE and bool(int(e[2]["flags"]) & 2))
        flags = 0
        for e1 in plan:
            if not is_stop(e1):
                continue
            for e2 in plan:
                if not is_stop(e2) and e2[1] != abi.CO_NOOP and _jsub(e1[0], e2[0]) < 0:
                    flags |= abi.ELF_STOP_ORDER
        if plan and any(is_stop(e) for e in plan) and not is_stop(plan[-1]):
            plan = plan + [(next_slot, abi.CO_STOP_NEW, None, 0)]
        return plan, flags

    def _blob_positions(self, lane: int, items) -> List[int]:
        """the log positions (for gpx_log_read / gpx_log_gather) of the request blobs of carried-over pvalues, given as
        [(gid, accepted pvalue)] reported by the acceptor at `lane`.  frame_ref * 16 is the blob's offset in the lane's
        ring of log_ring_bytes: until the ring has wrapped that is its position.  After that the offset does not say
        which lap wrote it, so the ACCEPT that logged the pvalue is looked up among the bytes still in the ring
        (gpx_log_find from the oldest intact segment boundary) and its blob position taken.  A pvalue whose ACCEPT is
        no longer there raises GPX_ERANGE: its body was overwritten."""
        eng = self.engine
        head, ring = eng.log_head(lane), int(eng.cfg.log_ring_bytes)
        if head <= ring:
            return [int(pv["frame_ref"]) * 16 for _, pv in items]
        start = self._oldest_segment(lane, head, ring)
        todo: Dict[int, List[int]] = {}
        for gid, pv in items:
            todo.setdefault(int(gid), []).append(int(pv["slot"]))
        for g, sl in todo.items():
            todo[g] = sorted(set(sl), key=lambda s, s0=sl[0]: _jsub(s, s0))
        hits = {}
        while todo:  # one want per group and call, GPX_LOG_SPAN slots from its lowest slot still to find
            gids = sorted(todo)
            w = np.zeros(len(gids), dtype=abi.log_want_dtype)
            w["gid"], w["min_slot"], w["n_slots"] = gids, [todo[g][0] for g in gids], abi.GPX_LOG_SPAN
            found = eng.log_find(lane, w, start)
            for i, g in enumerate(gids):
                s0 = todo[g][0]
                for s in todo[g]:
                    if _jsub(s, s0) < abi.GPX_LOG_SPAN:
                        hits[(g, s)] = found[i, _jsub(s, s0)]
                todo[g] = [s for s in todo[g] if _jsub(s, s0) >= abi.GPX_LOG_SPAN]
                if not todo[g]:
                    del todo[g]
        out = []
        for gid, pv in items:
            h = hits[(int(gid), int(pv["slot"]))]
            a = h["accept"]
            same = all(int(a[f]) == int(pv[f]) for f in ("bnum", "bcoord", "req_id", "payload_len"))
            if int(a["flags"]) & abi.F_VOID or not same:
                raise abi.GpxError(abi.GPX_ERANGE, f"the request body of group {int(gid)} slot {int(pv['slot'])} "
                                                   f"at lane {lane} was overwritten in the log ring")
            out.append(int(h["blob_pos"]))
        return out

    def _oldest_segment(self, lane: int, head: int, ring: int) -> int:
        """the first segment boundary among the last `ring` bytes before the head of a lane's log: a segment header
        names its own absolute position (ring_off), and the walk from the boundary over the headers (to the next lap
        where a launch skipped the ring end, as k_log_dir walks) ends at the head"""
        buf = self.engine.log_read(lane, head - ring, ring)
        n = ring // 32 - 1
        hdr = np.lib.stride_tricks.as_strided(buf, shape=(n, 64), strides=(32, 1)).copy().view(abi.seg_hdr_dtype)[:, 0]
        pos = head - ring + 32 * np.arange(n, dtype=np.int64)
        ok = (hdr["magic"] == abi.SEG_MAGIC) & (hdr["ring_off"] == pos.astype(np.uint64)) & (pos % ring + 64 <= ring)
        for k in np.nonzero(ok)[0]:
            p = int(pos[k])
            while p + 64 <= head:
                i = (p - (head - ring)) // 32
                if i < n and ok[i]:
                    h = hdr[i]
                    body = int(h["n_slots"]) * int(h["rec_bytes"]) + ((int(h["payload_bytes"]) + 15) & ~15)
                    p = (p + 64 + body + 31) & ~31
                else:  # the tail a launch skipped at the ring end
                    p = (p // ring + 1) * ring
            if p == head:
                return int(pos[k])
        raise abi.GpxError(abi.GPX_ERANGE, f"no intact segment boundary in the log ring of lane {lane}")

    def _requests_of(self, paxosID: str, pv, src_lane: int, entry: int) -> List[RequestPacket]:
        """the request(s) of an accepted pvalue, read back from the log ring of the acceptor lane that reported it"""
        n = int(pv["payload_len"])
        pos = self._blob_positions(src_lane, [(self.instances[paxosID].gid, pv)])[0] if n else 0
        blob = bytes(self.engine.log_read(src_lane, pos, n)) if n else b""
        return self._requests_from_blob(paxosID, pv, blob, entry)

    # ---- catching up a replica that fell behind (PISM.syncLongDecisionGaps :1550, checkpoint transfer :1852) ----
    def syncDecisions(self, paxosID: str, lane: int) -> int:
        """PISM.requestMissingDecisions :2292-2316 at `lane` and handleSyncDecisionsPacket :2426-2500 at the replica
        that is furthest ahead: the missing slots [my slot, donor's slot) are served from the donor's journal (its log
        ring): getLoggedDecisions plus getActualDecisions -- the decision images name slot and ballot, the ACCEPT images
        of that ballot carry the request.  They are replayed at the lagging lane W slots at a time (accept, then
        commit) and its application executes them.  When that cannot close the gap (the lane has promised a higher
        ballot, or the donor's ring no longer holds the slots) the replica takes a checkpoint instead
        (handleCheckpoint :1852-1879: restore the app state, jumpSlot).  Returns the number of slots executed."""
        inst = self.instances.get(paxosID)
        if inst is None:
            return 0
        eng, L, gid = self.engine, self.engine.n_lanes, inst.gid
        gids = np.array([gid], dtype=np.uint32)
        rows = [eng.dump_rows(gids, l)[0] for l in range(L)]
        donor = max(range(L), key=lambda l: _jsub(int(rows[l]["acc_slot"]), int(rows[lane]["acc_slot"])))
        lo, hi = int(rows[lane]["acc_slot"]), int(rows[donor]["acc_slot"])
        if donor == lane or _jsub(hi, lo) <= 0:
            return 0
        want = lambda sl: _jsub(sl, lo) >= 0 and _jsub(sl, hi) < 0
        accepts, decisions = {}, {}
        if self.device_log_find:
            # getLoggedDecisions + getActualDecisions (PISM :2463-2502, :2539-2583) as scans of the donor's log ring on the
            # device (gpx_log_find): per slot the decision and the accept logged last; only the found bodies cross PCIe
            sl = lo
            while _jsub(sl, hi) < 0:
                w = np.zeros(1, dtype=abi.log_want_dtype)
                w["gid"], w["min_slot"], w["n_slots"] = gid, sl, min(abi.GPX_LOG_SPAN, _jsub(hi, sl))
                good = []
                for h in eng.log_find(donor, w)[0][: int(w["n_slots"][0])]:
                    d, a = h["decision"], h["accept"]
                    if int(d["flags"]) & abi.F_VOID or int(a["flags"]) & abi.F_VOID:
                        continue
                    if (_jsub(int(a["bnum"]), int(d["bnum"])) or _jsub(int(a["bcoord"]), int(d["bcoord"]))) < 0:
                        continue  # the accept on record is older than the decision: no body for it here
                    good.append(h)
                if eng.L.has("log_gather"):  # all bodies of the chunk in one device->host copy
                    bodies = eng.log_gather(donor, [int(h["blob_pos"]) for h in good], [int(h["accept"]["payload_len"]) for h in good])
                else:
                    bodies = [bytes(eng.log_read(donor, int(h["blob_pos"]), int(h["accept"]["payload_len"])))
                              if int(h["accept"]["payload_len"]) else b"" for h in good]
                for h, body in zip(good, bodies):
                    d, a = h["decision"], h["accept"]
                    decisions[int(d["slot"])] = d.copy()
                    accepts[(int(d["slot"]), int(d["bnum"]), int(d["bcoord"]))] = (a.copy(), body)
                sl = _jadd(sl, abi.GPX_LOG_SPAN)
        else:
            for hdr, imgs, payload, _ in abi.parse_log(eng.log_read(donor)):
                for a in imgs:
                    if (int(a["flags"]) & abi.F_VOID) or int(a["gid"]) != gid or not want(int(a["slot"])):
                        continue
                    if int(hdr["rec_bytes"]) == 48:
                        o, n = int(a["payload_off"]), int(a["payload_len"])
                        accepts[(int(a["slot"]), int(a["bnum"]), int(a["bcoord"]))] = (a.copy(), bytes(payload[o: o + n]))
                    elif int(a["flags"]) & abi.F_DECISION:
                        decisions[int(a["slot"])] = a.copy()
        executed, W, sl = 0, int(eng.cfg.window), lo
        while _jsub(sl, hi) < 0:
            chunk = []
            while len(chunk) < W and _jsub(sl, hi) < 0:
                d = decisions.get(sl)
                a = accepts.get((sl, int(d["bnum"]), int(d["bcoord"]))) if d is not None else None
                if a is None:
                    break  # the donor's journal no longer has this slot
                chunk.append((d, a))
                sl += 1
            if not chunk:
                break
            acc = np.zeros(len(chunk), dtype=abi.accept_dtype)
            dec = np.zeros(len(chunk), dtype=abi.decision_dtype)
            blob, batches = bytearray(), {}
            for k, (d, (a, body)) in enumerate(chunk):
                for f in abi.accept_dtype.names:
                    acc[k][f] = a[f]
                acc[k]["flags"], acc[k]["dst_mask"], acc[k]["payload_off"] = int(a["flags"]) & ~0x40, 1 << lane, len(blob)
                blob += body + bytes(-len(body) % 16)
                for f in ("gid", "slot", "bnum", "bcoord", "req_id"):
                    dec[k][f] = a[f]
                dec[k]["median_cp"] = max(int(d["median_cp"]), -1)
                dec[k]["flags"] = abi.F_DECISION | (int(a["flags"]) & abi.F_STOP)
                dec[k]["dst_mask"] = 1 << lane
                pv = {"req_id": int(a["req_id"]), "flags": (2 if int(a["flags"]) & abi.F_STOP else 0) | (int(a["nreq"]) << 16)}
                batches[int(a["req_id"])] = self._requests_from_blob(paxosID, pv, body, self.nodes[donor])
            eng.handle_accepts(acc, np.frombuffer(bytes(blob), dtype=np.uint8))
            ex, extra = eng.handle_decisions(dec)
            n = self._apply(np.concatenate([ex, extra]), batches)
            executed += n
            if n == 0:
                break  # e.g. the lane has promised a higher ballot: the accepts were refused
        now = int(eng.dump_rows(gids, lane)[0]["acc_slot"])
        if _jsub(hi, now) > 0:
            executed += self._transfer_checkpoint(paxosID, donor, lane, hi)
        return executed

    def _transfer_checkpoint(self, paxosID: str, donor: int, lane: int, slot: int) -> int:
        """PISM.handleCheckpoint :1852-1879: the app state of a replica that is ahead replaces mine and the acceptor
        jumps to the slot after the checkpoint (PaxosAcceptor.jumpSlot :564-578)."""
        inst = self.instances[paxosID]
        self.apps[lane].restore(paxosID, self.apps[donor].checkpoint(paxosID))
        p = np.zeros(1, dtype=abi.patch_dtype)
        p["gid"], p["lane"], p["op"], p["a"] = inst.gid, lane, abi.PATCH_JUMP_SLOT, slot
        self.engine.patch(p)
        return 1

    def _requests_from_blob(self, paxosID: str, pv, blob: bytes, entry: int) -> List[RequestPacket]:
        nreq, stop = int(pv["flags"]) >> 16, bool(int(pv["flags"]) & 2)
        if nreq <= 1:
            known = self.outstanding.get(int(pv["req_id"]))
            return [RequestPacket(paxosID, int(pv["req_id"]), blob, stop=stop,
                                  entry_replica=known.entry_replica if known else entry,
                                  callback=known.callback if known else None)]
        ents = np.frombuffer(blob[: 16 * nreq], dtype=abi.batch_ent_dtype)
        out, off = [], 16 * nreq
        for e in ents:
            known = self.outstanding.get(int(e["req_id"]))
            out.append(RequestPacket(paxosID, int(e["req_id"]), blob[off: off + int(e["len"])],
                                     stop=bool(int(e["flags"]) & abi.F_STOP),
                                     entry_replica=known.entry_replica if known else entry,
                                     callback=known.callback if known else None))
            off += int(e["len"])
        return out

    # ---- pause / unpause (PaxosManager.pause :2284-2330, unpause :2370-2437) ------------------------------
    def pause(self, paxosID: str) -> bool:
        """Move an idle instance out of the engine: PISM.tryPause :2004-2035 succeeds only when every replica is
        caught up (nothing committed-but-unexecuted, no outstanding proposal); the rows are kept as
        HotRestoreInfo strings (the pause table) and the gid is freed."""
        inst = self.instances.get(paxosID)
        if inst is None or inst.stopped or self.queue.get(paxosID):
            return False
        gids = np.array([inst.gid], dtype=np.uint32)
        for lane in range(self.engine.n_lanes):
            if int(self.engine.group_flags(gids, lane)[0]) & abi.GF_NOT_CAUGHT_UP:
                return False
        hris = [str(HotRestoreInfo.from_row(paxosID, self.engine.dump_rows(gids, lane)[0]))
                for lane in range(self.engine.n_lanes)]
        self.paused[paxosID] = hris
        self._release(paxosID)  # forceStop + removal from pinstances
        return True

    def pauseBatch(self, paxosIDs: Sequence[str]) -> List[str]:
        """PaxosManager.pause(Map, dequeue) :2327-2366, the body of the Deactivator's sweep (syncAndDeactivate :2806-2900):
        ONE gpx_pause_groups call tries every candidate (PISM.tryPause at every replica), returns the HotRestoreInfo rows of
        those that were caught up and frees their gids; the rows go into the pause table as the strings
        SQLPaxosLogger.pause writes.  Returns the names that were paused."""
        cand = [n for n in dict.fromkeys(paxosIDs)
                if n in self.instances and not self.instances[n].stopped and not self.queue.get(n)]
        if not cand:
            return []
        if not self.engine.L.has("pause_groups"):
            return [n for n in cand if self.pause(n)]
        gids = np.array([self.instances[n].gid for n in cand], dtype=np.uint32)
        rows, ok = self.engine.pause_groups(gids)
        done = []
        for i, n in enumerate(cand):
            if not ok[i]:
                continue
            self.paused[n] = [str(HotRestoreInfo.from_row(n, rows[i, lane])) for lane in range(self.engine.n_lanes)]
            inst = self.instances.pop(n)  # the engine has already freed the gid (forceStop + softCrash)
            self.gid_name.pop(inst.gid, None)
            self.free_gids.append(inst.gid)
            done.append(n)
        return done

    def syncAndDeactivate(self, pause: bool = True) -> Dict[str, int]:
        """PaxosManager.syncAndDeactivate :2806-2900, the body of the Deactivator thread: every instance that is behind
        catches up (syncPaxosInstance -> PISM.syncLongDecisionGaps :1550), every idle one is paused in batches.  The
        reference tests each of pinstances in turn; here the engine names the groups (gpx_select_groups: one launch per
        lane over all gids) -- those flagged NEEDS_SYNC, then those that are caught up on every lane -- and one
        gpx_pause_groups call takes the idle ones out.  Returns {"synced": slots executed by catching up, "paused": n}."""
        eng, L = self.engine, self.engine.n_lanes
        if not (eng.L.has("select_groups") and eng.L.has("pause_groups")):
            raise RuntimeError("the engine library has no gpx_select_groups / gpx_pause_groups")
        synced = 0
        for lane in range(L):
            listed = eng.select_groups(lane, abi.GF_NEEDS_SYNC, abi.GF_NEEDS_SYNC)
            for gid in listed:
                name = self.gid_name.get(int(gid))
                if name is not None:
                    synced += self.syncDecisions(name, lane)
            if len(listed) and eng.L.has("clear_group_flags"):  # dealt with: out of the slow-path list
                eng.clear_group_flags(lane, listed, abi.GF_NEEDS_SYNC | abi.GF_OVERFLOW)
        paused: List[str] = []
        if pause:
            idle = None
            for lane in range(L):
                g = set(int(x) for x in eng.select_groups(lane, abi.GF_NOT_CAUGHT_UP, 0))
                idle = g if idle is None else idle & g
            names = [self.gid_name[g] for g in sorted(idle or ()) if g in self.gid_name]
            paused = self.pauseBatch(names)
        return {"synced": synced, "paused": len(paused)}

    def unpause(self, paxosID: str) -> bool:
        """PaxosManager.unpause :2370: rebuild the instance from its HotRestoreInfo (PISM.hotRestore :677-690)."""
        hris = self.paused.pop(paxosID, None)
        if hris is None or paxosID in self.instances:
            return False
        infos = [HotRestoreInfo.parse(h) for h in hris]
        gid = self._alloc_gid()
        self.instances[paxosID] = _Instance(gid, infos[0].version, list(infos[0].members))
        self.gid_name[gid] = paxosID
        rows = np.concatenate([h.to_row(gid, lane, self.nodes[lane]) for lane, h in enumerate(infos)])
        self.engine.load_rows(rows)
        return True

    def unpauseBatch(self, paxosIDs: Sequence[str]) -> List[str]:
        """PaxosManager.unpause :2370 for many instances at once (a burst of requests for groups the sweep has moved out):
        ONE gpx_load_rows call rebuilds all of them from their HotRestoreInfo strings (PISM.hotRestore :677-690)."""
        rows, done = [], []
        for n in dict.fromkeys(paxosIDs):
            hris = self.paused.get(n)
            if hris is None or n in self.instances:
                continue
            infos = [HotRestoreInfo.parse(h) for h in hris]
            gid = self._alloc_gid()
            self.instances[n] = _Instance(gid, infos[0].version, list(infos[0].members))
            self.gid_name[gid] = n
            rows += [h.to_row(gid, lane, self.nodes[lane]) for lane, h in enumerate(infos)]
            del self.paused[n]
            done.append(n)
        if rows:
            self.engine.load_rows(np.concatenate(rows))
        return done

    def isPaused(self, paxosID: str) -> bool:
        return paxosID in self.paused

    def isStopped(self, paxosID: str) -> bool:
        inst = self.instances.get(paxosID)
        return inst is None or inst.stopped

    def getVersion(self, paxosID: str) -> Optional[int]:
        inst = self.instances.get(paxosID)
        return None if inst is None else inst.version

    # ---- proposing ----------------------------------------------------------------------------
    def propose(self, paxosID: str, requestValue: bytes, callback=None, entry_node: Optional[int] = None,
                stop: bool = False, version: Optional[int] = None) -> Optional[int]:
        """PaxosManager.propose :1214-1243: returns the request id, or None when the instance does not
        exist (or the version does not match, PISM :441-447)."""
        inst = self.instances.get(paxosID)
        if inst is None and paxosID in self.paused and self.unpause(paxosID):  # PaxosManager.getInstance :2453 -> unpause
            inst = self.instances.get(paxosID)
        if inst is None or (version is not None and version != inst.version):
            return None
        rid = self.next_request_id
        self.next_request_id += 1
        req = RequestPacket(paxosID, rid, bytes(requestValue), stop=stop,
                            entry_replica=self.nodes[0] if entry_node is None else entry_node,
                            entry_time=time.time(), callback=callback)
        self.queue.setdefault(paxosID, []).append(req)  # RequestBatcher.enqueueImpl :112-129
        self.outstanding[rid] = req
        return rid

    def proposeStop(self, paxosID: str, version: int, requestValue: bytes, callback=None) -> Optional[int]:
        """PaxosManager.proposeStop: a STOP request for epoch `version`."""
        return self.propose(paxosID, requestValue, callback, stop=True, version=version)

    # ---- one pass of the hot path -----------------------------------------------------------------
    def run_round(self) -> int:
        """Drain the request queues through the engine; returns the number of executed slots."""
        names = [n for n in self.queue if self.queue[n]]
        if not names:
            return 0
        reqs_l: List[RequestPacket] = []
        for n in sorted(names, key=lambda x: self.instances[x].gid if x in self.instances else -1):
            if n not in self.instances:
                for r in self.queue[n]:
                    self.outstanding.pop(r.request_id, None)
                continue
            reqs_l.extend(self.queue[n])
        self.queue = {}
        return self._submit(reqs_l)

    def _submit(self, reqs_l: List[RequestPacket], carryover: bool = False) -> int:
        """one engine round over a list of requests already grouped by paxos instance.  carryover: the re-proposal of a
        carried-over pvalue by a new coordinator -- it must take exactly its slot, so a refusal is an error (requeueing
        it would shift every later carried-over slot)"""
        if not reqs_l:
            return 0
        n = len(reqs_l)
        reqs = np.zeros(n, dtype=abi.request_dtype)
        offs, off = [], 0
        for r in reqs_l:
            offs.append(off)
            off += (len(r.request_value) + 15) // 16 * 16
        payload = np.zeros(off, dtype=np.uint8)
        for i, r in enumerate(reqs_l):
            inst = self.instances[r.paxos_id]
            lane = self.nodes.index(r.entry_replica) if r.entry_replica in self.nodes else 0
            reqs[i]["gid"] = inst.gid
            reqs[i]["flags"] = (abi.F_STOP if r.stop else 0) | (lane << 8)
            reqs[i]["req_id"] = r.request_id
            reqs[i]["payload_off"], reqs[i]["payload_len"] = offs[i], len(r.request_value)
            reqs[i]["entry_node"] = r.entry_replica
            payload[offs[i]: offs[i] + len(r.request_value)] = np.frombuffer(r.request_value, dtype=np.uint8)
        status, ex, extra = self.engine.round(reqs, payload)
        if carryover and any(int(st) <= 0 and int(st) != abi.RS_BATCHED for st in status):
            raise RuntimeError(f"carried-over pvalue could not be re-proposed: status {[int(x) for x in status]}")
        # requests the engine could not propose go back to the host slow path (retry / forward / prepare)
        elect: Dict[str, int] = {}
        for i, st in enumerate(status):
            if st in (abi.RS_BACKPRESSURE,):
                self.queue.setdefault(reqs_l[i].paxos_id, []).append(reqs_l[i])
            elif st == abi.RS_NOCOORD and self.auto_elect:
                # PISM.handleProposal :862-885: no coordinator for my acceptor's ballot -> checkRunForCoordinator(true)
                # at the entry replica; the request waits in the queue and is proposed by the new coordinator
                r = reqs_l[i]
                elect.setdefault(r.paxos_id, self.nodes.index(r.entry_replica) if r.entry_replica in self.nodes else 0)
                self.queue.setdefault(r.paxos_id, []).append(r)
            elif st < 0 and st != abi.RS_BATCHED:
                self.slow_path.append((reqs_l[i].paxos_id, reqs_l[i].request_id, int(st)))
                self.outstanding.pop(reqs_l[i].request_id, None)
        self._elect = elect
        # batches: a positive status starts a slot, RS_BATCHED entries follow it (RequestPacket.batched)
        batches: Dict[int, List[RequestPacket]] = {}
        cur = None
        for i, st in enumerate(status):
            if st > 0:
                cur = reqs_l[i].request_id
                batches[cur] = [reqs_l[i]]
            elif st == abi.RS_BATCHED and cur is not None:
                batches[cur].append(reqs_l[i])
        done = self._apply(np.concatenate([ex, extra]), batches)
        by_lane: Dict[int, List[str]] = {}
        for name, lane in self._elect.items():
            by_lane.setdefault(lane, []).append(name)
        self._elect = {}
        for lane, names in by_lane.items():
            for name, won in self.runForCoordinators(names, lane).items():
                if not won:  # preempted / no majority: give the requests back
                    for r in self.queue.pop(name, []):
                        self.slow_path.append((name, r.request_id, abi.RS_NOCOORD))
                        self.outstanding.pop(r.request_id, None)
        return done

    def _apply(self, ex: np.ndarray, batches: Dict[int, List[RequestPacket]]) -> int:
        """PISM.execute :1755-1842 + PaxosManager.executed :311-330 for every EXEC record, per group in
        slot order (primary and extra records of one call interleave)."""
        ex = ex[(ex["flags"] & abi.F_VOID) == 0]
        if len(ex) == 0:
            return 0
        lanes = (ex["flags"] >> 12) & 0xF
        ex = ex[np.lexsort((ex["slot"], ex["gid"], lanes))]
        executed = 0
        for x in ex:
            lane = int((x["flags"] >> 12) & 0xF)
            name = self.gid_name.get(int(x["gid"]))
            if name is None:
                continue
            batch = batches.get(int(x["req_id"]))
            if batch is None:  # decided elsewhere / earlier round: only the id is known here
                first = self.outstanding.get(int(x["req_id"]))
                batch = [first] if first is not None else []
            is_stop = bool(x["flags"] & abi.F_STOP)
            for bi, req in enumerate(batch):
                if req.request_id == 0 and req.request_value == NO_OP:  # PISM.execute skips no-ops :1786-1790
                    continue
                view = RequestPacket(req.paxos_id, req.request_id, req.request_value, req.stop, req.entry_replica,
                                     req.entry_time, slot=int(x["slot"]), batch_index=bi, callback=req.callback)
                entry = req.entry_replica == self.nodes[lane]
                self.apps[lane].execute(name, view, do_not_reply_to_client=not entry)  # :1802-1806
                if entry:  # PaxosManager.executed: callback / response from the entry replica only
                    req.response_value, req.slot = view.response_value, view.slot
                    self.outstanding.pop(req.request_id, None)
                    if req.callback is not None:
                        req.callback(req, True)
                # PISM.execute :1813-1815: the acceptor is already STOPPED when a stop batch executes,
                # so only the first request of a stop batch is executed
                if is_stop:
                    break
            if x["flags"] & abi.F_CKPT:  # PISM.shouldCheckpoint :2037 -> consistentCheckpoint :1711-1723
                self.checkpoints.append((name, lane, int(x["slot"]), self.apps[lane].checkpoint(name)))
            if is_stop:
                self.instances[name].stopped = True
            if lane == 0:
                self.num_decisions += 1
            executed += 1
        return executed

    def flush(self, max_rounds: int = 64) -> int:
        total = 0
        for _ in range(max_rounds):
            if not any(self.queue.values()):
                break
            total += self.run_round()
        return total
