"""Synthetic watch-event churn for the resident tick (``lwse_resident_tick``).

A controller sees events, not tables.  A *churn plan* is a list of patch sets; one set is what
one reconcile pass of the work queue has to digest:

* pod status updates — ``frac_pods`` of the pod state bytes get a new value (phase flips
  Pending <-> Running, restart counts move, a few deletions start);
* scheduling events — ``frac_reqs`` of the placement requests change sides: unpinned leaders
  get bound to the node the previous placement round chose for them, as many bound ones go
  back to unscheduled (pod recreated); the group rows carry the same ``leader_node``.

Set 2j+1 undoes the scheduling events of set 2j, so a long run stays at the profile's 5 %
unscheduled leaders.  Both bench arms consume the same plan: the GPU engine as row patches,
the CPU arm as (apply patches, reconcile the dirty objects) — ``dirty_*`` are the row numbers
the event source hands a controller for free.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from . import records as R


@dataclass
class PatchSet:
    pod_rows: np.ndarray
    pod_vals: np.ndarray
    req_rows: np.ndarray = field(default_factory=lambda: np.zeros(0, np.uint32))
    req_vals: np.ndarray = field(default_factory=lambda: R.aligned_empty(0, R.PLACE_REQ))
    grp_rows: np.ndarray = field(default_factory=lambda: np.zeros(0, np.uint32))
    grp_vals: np.ndarray = field(default_factory=lambda: R.aligned_empty(0, R.GROUP_REC))
    dirty_groups: np.ndarray = field(default_factory=lambda: np.zeros(0, np.uint32))
    dirty_lws: np.ndarray = field(default_factory=lambda: np.zeros(0, np.uint32))

    def h2d_bytes(self) -> int:
        return int(self.pod_rows.nbytes + self.pod_vals.nbytes + self.req_rows.nbytes + self.req_vals.nbytes
                   + self.grp_rows.nbytes + self.grp_vals.nbytes)


def _toggle_states(vals: np.ndarray, rng) -> np.ndarray:
    v = vals.astype(np.uint8).copy()
    r = rng.random(len(v))
    phase = v & R.POD_PHASE_MASK
    flip = (r < 0.60) & ((phase == R.POD_PHASE_PENDING) | (phase == R.POD_PHASE_RUNNING))
    v[flip] ^= np.uint8(3)  # Pending <-> Running
    v[(r >= 0.60) & (r < 0.80)] ^= np.uint8(R.POD_ANY_RESTART)
    v[(r >= 0.80) & (r < 0.85)] ^= np.uint8(R.POD_DELETING)
    return v


def make_plan(t, reqs: np.ndarray | None, place_out: np.ndarray | None, frac_pods: float, frac_reqs: float = 0.0,
              n_sets: int = 4, seed: int = 7, patch_groups: bool = True) -> list[PatchSet]:
    """Patch sets for tables ``t`` (a ``synth.Tables``).  Applied in order, cyclically, they keep
    mirror tables on the host consistent: every set's values are computed from the state the
    previous sets leave behind (the plan simulates the run once).
    ``patch_groups=False``: the request table is sharded differently from the group table (strong
    scaling: placement by namespace owner, sweep by UID hash) — a scheduling event then patches the
    request row here and the group row on the rank that sweeps the group (not generated)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n_pods = len(t.pod_state)
    state = t.pod_state.copy()
    groups = t.groups.copy()
    cur_reqs = None if reqs is None else reqs.copy()
    pod_group = np.repeat(np.arange(len(groups), dtype=np.uint32), groups["pod_count"].astype(np.int64))
    # only valid when the pod table is laid out group after group (synth tables are)
    laid_out = len(pod_group) == n_pods and bool(
        np.all(groups["pod_base"].astype(np.int64) == np.concatenate([[0], np.cumsum(groups["pod_count"].astype(np.int64))[:-1]])))
    sets: list[PatchSet] = []
    n_p = int(round(n_pods * frac_pods))
    swap = None
    for k in range(n_sets):
        rows = np.sort(rng.choice(n_pods, size=n_p, replace=False)).astype(np.uint32) if 0 < n_p < n_pods else (
            np.arange(n_pods, dtype=np.uint32) if n_p >= n_pods else np.zeros(0, np.uint32))
        vals = R.aligned_empty(len(rows), R.POD_STATE)
        vals[:] = _toggle_states(state[rows], rng)
        state[rows] = vals
        ps = PatchSet(pod_rows=rows, pod_vals=vals)
        dg = pod_group[rows] if laid_out else np.zeros(0, np.uint32)
        dl = np.zeros(0, np.uint32)
        if laid_out and len(rows):
            leader = rows.astype(np.int64) == groups["pod_base"][dg].astype(np.int64)
            dl = groups["lws_index"][dg[leader]]
        if cur_reqs is not None and frac_reqs > 0 and len(cur_reqs):
            if k % 2 == 0:
                n_s = max(1, int(round(len(cur_reqs) * frac_reqs / 2)))
                unp = np.flatnonzero((cur_reqs["leader_node"] == R.NONE) & (cur_reqs["size"] >= 1))
                if place_out is not None:  # only those the round placed: bind them where it put them
                    unp = unp[(place_out["flags"][unp] & R.PLACE_PLACED) != 0]
                pin = np.flatnonzero(cur_reqs["leader_node"] < R.NODE_NOT_FOUND)
                a = rng.choice(unp, size=min(n_s, len(unp)), replace=False) if len(unp) else np.zeros(0, np.int64)
                b = rng.choice(pin, size=min(n_s, len(pin)), replace=False) if len(pin) else np.zeros(0, np.int64)
                new_nodes = np.concatenate([place_out["leader_node"][a] if place_out is not None
                                            else np.zeros(len(a), np.uint32), np.full(len(b), R.NONE, np.uint32)])
                rr = np.concatenate([a, b]).astype(np.uint32)
                old_nodes = cur_reqs["leader_node"][rr].copy()
                swap = (rr, old_nodes)
            else:
                rr, new_nodes = swap  # undo the previous set's scheduling events
            order = np.argsort(rr, kind="stable")
            rr, new_nodes = rr[order], new_nodes[order]
            cur_reqs["leader_node"][rr] = new_nodes
            rv = R.aligned_empty(len(rr), R.PLACE_REQ)
            rv[:] = cur_reqs[rr]
            ps.req_rows, ps.req_vals = rr, rv
            if patch_groups:
                gr = cur_reqs["group"][rr].astype(np.uint32)
                groups["leader_node"][gr] = new_nodes
                gv = R.aligned_empty(len(gr), R.GROUP_REC)
                gv[:] = groups[gr]
                ps.grp_rows, ps.grp_vals = gr, gv
                dg = np.concatenate([dg, gr])
                dl = np.concatenate([dl, groups["lws_index"][gr]])
        ps.dirty_groups = np.unique(dg).astype(np.uint32)
        ps.dirty_lws = np.unique(dl).astype(np.uint32)
        sets.append(ps)
    return sets


def apply_to_mirror(ps: PatchSet, pod_state: np.ndarray, groups: np.ndarray, reqs: np.ndarray | None) -> None:
    """The host-side mirror of one tick's patches (plain numpy; the CPU arm uses the oracle's C loop)."""
    pod_state[ps.pod_rows] = ps.pod_vals
    if len(ps.grp_rows):
        groups[ps.grp_rows] = ps.grp_vals
    if reqs is not None and len(ps.req_rows):
        reqs[ps.req_rows] = ps.req_vals


class ArenaPlan:
    """A churn plan laid out in an engine's patch arena: the rows / values the tick descriptors
    point at are views of pinned, mapped memory the GPU reads in place."""

    def __init__(self, engine, sets: list[PatchSet], flags: int, range_threshold: float = 0.2):
        need = 4096
        for ps in sets:
            need += sum(((a.nbytes + 255) // 256 + 1) * 256 for a in
                        (ps.pod_rows, ps.pod_vals, ps.req_rows, ps.req_vals, ps.grp_rows, ps.grp_vals))
        self.arena = engine.resident_arena(need)
        self._cursor = 0
        self.ticks = []
        self.h2d_bytes = []
        n_pods = engine._resident_pods
        for ps in sets:
            segs = []
            if len(ps.pod_rows) >= range_threshold * n_pods and len(ps.pod_rows) == n_pods:
                # the whole column changed: one contiguous DMA copy instead of a scatter
                segs.append((R.TABLE_POD_STATE, 0, self._put(ps.pod_vals), True))
                nbytes = ps.pod_vals.nbytes
            else:
                if len(ps.pod_rows):
                    segs.append((R.TABLE_POD_STATE, self._put(ps.pod_rows), self._put(ps.pod_vals)))
                nbytes = ps.pod_rows.nbytes + ps.pod_vals.nbytes
            if len(ps.grp_rows):
                segs.append((R.TABLE_GROUPS, self._put(ps.grp_rows), self._put(ps.grp_vals)))
                nbytes += ps.grp_rows.nbytes + ps.grp_vals.nbytes
            if len(ps.req_rows):
                segs.append((R.TABLE_PLACE_REQS, self._put(ps.req_rows), self._put(ps.req_vals)))
                nbytes += ps.req_rows.nbytes + ps.req_vals.nbytes
            self.ticks.append(engine.make_tick(segs, flags))
            self.h2d_bytes.append(int(nbytes))

    def _put(self, a: np.ndarray) -> np.ndarray:
        off = (self._cursor + 255) // 256 * 256
        view = self.arena[off: off + a.nbytes].view(a.dtype)
        view[...] = a.reshape(-1) if a.dtype.fields is None else a
        self._cursor = off + a.nbytes
        return view


# --------------------------------------------------------------------------- #
# DisaggregatedSet tables (lwse_ds_resident_tick)
# --------------------------------------------------------------------------- #
@dataclass
class DsPatchSet:
    """One reconcile pass of the DS controller's work queue, as row patches (rows sorted, distinct)."""

    rr_rows: np.ndarray
    rr_vals: np.ndarray
    role_rows: np.ndarray = field(default_factory=lambda: np.zeros(0, np.uint32))
    role_vals: np.ndarray = field(default_factory=lambda: R.aligned_empty(0, R.DS_ROLE_REC))

    def h2d_bytes(self) -> int:
        return int(self.rr_rows.nbytes + self.rr_vals.nbytes + self.role_rows.nbytes + self.role_vals.nbytes)


def make_ds_plan(t, sweep_ds, frac_revroles: float, n_sets: int = 4, frac_target: float = 0.001,
                 seed: int = 11) -> list[DsPatchSet]:
    """Patch sets for DS tables ``t`` (a ``synth.DsTables``), simulated once from its state:
    in every set a fraction ``frac_revroles`` of the (revision, role) rows where an LWS exists
    applies the previous sweep's decision (``replicas ← revrole_out``: the controller scaled the
    child) and half of those become ready (``ready_replicas ← replicas``); about ``frac_target``
    of the spec roles get a new ``target_replicas``.  ``sweep_ds(ds, roles, revroles)`` is the
    sweep the decisions come from (the oracle).  The layout never changes: no row moves, no
    child LWS appears or goes, so every set is valid for the resident tables of ``t``."""
    rng = np.random.Generator(np.random.PCG64(seed))
    roles, rr = t.roles.copy(), t.revroles.copy()
    exists = np.flatnonzero((rr["flags"] & R.RR_EXISTS) != 0)
    in_spec = np.flatnonzero((roles["flags"] & R.ROLE_IN_SPEC) != 0)
    n_rr = int(round(len(exists) * frac_revroles))
    n_ro = int(round(len(in_spec) * frac_target))
    sets = []
    for _ in range(n_sets):
        _, _, rr_out = sweep_ds(t.ds, roles, rr)
        rows = np.sort(rng.choice(exists, size=min(n_rr, len(exists)), replace=False)).astype(np.uint32)
        want = rr_out[rows]
        scaled = want >= 0
        rr["replicas"][rows[scaled]] = want[scaled]
        rr["flags"][rows[scaled]] &= np.uint32(~R.RR_REPLICAS_NIL & 0xFFFFFFFF)
        ready = rows[rng.random(len(rows)) < 0.5]
        rr["ready_replicas"][ready] = rr["replicas"][ready]
        rv = R.aligned_empty(len(rows), R.DS_REVROLE_REC)
        rv[:] = rr[rows]
        ps = DsPatchSet(rows, rv)
        if n_ro:
            ro = np.sort(rng.choice(in_spec, size=min(n_ro, len(in_spec)), replace=False)).astype(np.uint32)
            roles["target_replicas"][ro] = np.maximum(roles["target_replicas"][ro] + rng.choice(np.array([-1, 1]), len(ro)), 0)
            vals = R.aligned_empty(len(ro), R.DS_ROLE_REC)
            vals[:] = roles[ro]
            ps.role_rows, ps.role_vals = ro, vals
        sets.append(ps)
    return sets


def apply_ds_to_mirror(ps: DsPatchSet, roles: np.ndarray, revroles: np.ndarray) -> None:
    """The host-side mirror of one DS tick's patches."""
    revroles[ps.rr_rows] = ps.rr_vals
    if len(ps.role_rows):
        roles[ps.role_rows] = ps.role_vals


# --------------------------------------------------------------------------- #
# Joint LWS + DS ticks (lwse_joint_tick_submit)
# --------------------------------------------------------------------------- #
def _arena_bytes(arrays) -> int:
    return sum((a.nbytes + 255) // 256 * 256 for a in arrays)


class JointArenaPlan:
    """The joint counterpart of ``ArenaPlan``: pass k's LWS ``PatchSet`` and ``DsPatchSet`` are
    written into region k % 2 of the engine's patch arena, so that two joint ticks can be in flight.
    Pass k+2 reuses the region of pass k: submit it only after pass k's wait returned (the engine
    allows two ticks in flight, so a pipelined caller has waited for it by then).  ``lws_sets``
    None: DS-only ticks.  Every array starts on a 256-byte boundary of its region."""

    def __init__(self, engine, lws_sets, ds_sets, flags: int = 0):
        self.engine, self.lws_sets, self.ds_sets, self.flags = engine, lws_sets, ds_sets, flags
        self.n_passes = len(ds_sets)
        assert lws_sets is None or len(lws_sets) == self.n_passes
        need = max((_arena_bytes(self._arrays(k)) for k in range(self.n_passes)), default=0)
        self.region_bytes = (need + 4095) // 4096 * 4096
        self.arena = engine.resident_arena(2 * self.region_bytes)
        self.spans = []  # (pass, byte offset, bytes) of every array tick() wrote, in order

    def _arrays(self, k):
        out = []
        if self.lws_sets is not None:
            ps = self.lws_sets[k]
            out += [a for pair in ((ps.pod_rows, ps.pod_vals), (ps.grp_rows, ps.grp_vals), (ps.req_rows, ps.req_vals))
                    if len(pair[0]) for a in pair]
        d = self.ds_sets[k]
        out += [a for pair in ((d.rr_rows, d.rr_vals), (d.role_rows, d.role_vals)) if len(pair[0]) for a in pair]
        return out

    def tick(self, k: int):
        """Write pass k % n_passes into its region → (Tick or None, DsTick) descriptors pointing there."""
        p = k % self.n_passes
        cursor = (k % 2) * self.region_bytes

        def put(a):
            nonlocal cursor
            view = self.arena[cursor: cursor + a.nbytes].view(a.dtype)
            view[...] = a.reshape(-1) if a.dtype.fields is None else a
            self.spans.append((k, cursor, a.nbytes))
            cursor += (a.nbytes + 255) // 256 * 256
            return view

        lws_tick = None
        if self.lws_sets is not None:
            ps, segs = self.lws_sets[p], []
            for table, rows, vals in ((R.TABLE_POD_STATE, ps.pod_rows, ps.pod_vals), (R.TABLE_GROUPS, ps.grp_rows, ps.grp_vals),
                                      (R.TABLE_PLACE_REQS, ps.req_rows, ps.req_vals)):
                if len(rows):
                    segs.append((table, put(rows), put(vals)))
            lws_tick = self.engine.make_tick(segs, self.flags)
        d, segs = self.ds_sets[p], []
        for table, rows, vals in ((R.TABLE_DS_REVROLES, d.rr_rows, d.rr_vals), (R.TABLE_DS_ROLES, d.role_rows, d.role_vals)):
            if len(rows):
                segs.append((table, put(rows), put(vals)))
        assert cursor <= (k % 2 + 1) * self.region_bytes
        return lws_tick, self.engine.make_ds_tick(segs)
