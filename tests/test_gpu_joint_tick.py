"""The joint LWS + DS tick (lwse_joint_tick / _submit / _wait) on the GPU: its six change lists against
the two separate ticks and the oracles, two ticks in flight, DS-only ticks in flight, a ring shared with
LWS-only ticks, the refusals, both scatter paths, BAD_TABLE, the two incremental encoders, and a DS tick
that drains the ring."""
import ctypes as C

import numpy as np
import pytest

import oracle
from lws_b200 import churn, encoder, informer, synth
from lws_b200 import records as R
from lws_b200.engine import Engine, LwseError, lib
from test_gpu_ds_tick import Model

pytestmark = pytest.mark.gpu

LISTS = (("lws", "n_lws"), ("group", "n_groups"), ("place", "n_place"))
DS_LISTS = (("ds", "n_ds"), ("role", "n_roles"), ("revrole", "n_revroles"))


@pytest.fixture(scope="module")
def engines():
    oracle.build()
    a, b = Engine(0), Engine(0)
    yield a, b
    a.close()
    b.close()


class Lws:
    """Resident LWS tables + placement on an engine, their host mirrors and the oracle."""

    def __init__(self, t, reqs, engines):
        self.t, self.reqs = t, reqs
        self.flags = t.flags | R.TICK_PLACE
        self.occ = R.occupancy_of(t.pod_ident, len(t.nodes))
        for e in engines:
            e.upload_nodes(t.nodes, t.n_domains)
            e.resident_load(t.lws, t.groups, t.pod_state, t.pod_ident)
            e.resident_place_load(reqs, t.n_namespaces)
        self.pst, self.grp, self.req = t.pod_state.copy(), t.groups.copy(), reqs.copy()

    def apply(self, ps):
        churn.apply_to_mirror(ps, self.pst, self.grp, self.req)

    def check(self, engine):
        t = self.t
        lo, go, _ = oracle.sweep_lws(t.lws, self.grp, self.pst, t.pod_ident, t.nodes, flags=t.flags)
        got = engine.resident_outputs()
        assert got[0].tobytes() == lo.tobytes() and got[1].tobytes() == go.tobytes()
        want_p = oracle.place(t.nodes, self.occ, t.n_domains, t.n_namespaces, self.req)
        assert engine.resident_place_outputs().tobytes() == want_p.tobytes()


def _lws(engines, scale=0.5, seed=43, name="fuzz"):
    t = synth.make(synth.profile(name, scale), seed=seed)
    return Lws(t, t.place_requests(), engines)


def _ds(engines, t):
    for e in engines:
        e.ds_resident_load(t.ds, t.roles, t.revroles)
    return t.roles.copy(), t.revroles.copy()


def _ds_segs(ps):
    return [(R.TABLE_DS_REVROLES, ps.rr_rows, ps.rr_vals)] + (
        [(R.TABLE_DS_ROLES, ps.role_rows, ps.role_vals)] if len(ps.role_rows) else [])


def _copy(lres, dres):
    """A tick's six lists as {name: (rows, row bytes)} copies (the views are reused two submits later)."""
    out = {}
    for res, lists in ((lres, LISTS), (dres, DS_LISTS)):
        for name, n in lists:
            assert len(res[f"{name}_rows"]) == res[n], name
            rows, vals = res[f"{name}_rows"].copy(), res[f"{name}_out"].copy()
            out[name] = (rows, vals)
    return out


def _same_sets(a, b):
    for name in a:
        ra, va = a[name]
        rb, vb = b[name]
        assert len(ra) == len(rb), name
        oa, ob = np.argsort(ra, kind="stable"), np.argsort(rb, kind="stable")
        assert np.array_equal(ra[oa], rb[ob]), name
        if len(ra):
            assert va[oa].tobytes() == vb[ob].tobytes(), name


def _zero_mirror(engine, ticks, lws_shape, ds_shape):
    """A zero mirror with every tick's lists applied in order equals the committed outputs."""
    m = [R.aligned_empty(n, dt) for n, dt in zip(lws_shape, (R.LWS_OUT, R.GROUP_OUT))]
    d = [R.aligned_empty(n, dt) for n, dt in zip(ds_shape, (R.DS_OUT, R.DS_ROLE_OUT, R.DS_REVROLE_OUT))]
    for lists in ticks:
        for k, name in enumerate(("lws", "group")):
            m[k][lists[name][0]] = lists[name][1]
        for k, name in enumerate(("ds", "role", "revrole")):
            d[k][lists[name][0]] = lists[name][1]
    got = engine.resident_outputs()
    assert got[0].tobytes() == m[0].tobytes() and got[1].tobytes() == m[1].tobytes()
    got = engine.ds_resident_outputs()
    for g, w in zip(got, d):
        assert g.tobytes() == w.tobytes()


def _empty(engine, lws=True, flags=0):
    return engine.joint_tick(engine.make_tick((), flags) if lws else None, engine.make_ds_tick())


def _nothing_listed(res):
    lres, dres = res
    assert (lres["n_lws"], lres["n_groups"], lres["n_place"]) == (0, 0, 0)
    assert (dres["n_ds"], dres["n_roles"], dres["n_revroles"]) == (0, 0, 0)


# --------------------------------------------------------------------------- 1. joint == separate
# ("reduced": the size compute-sanitizer runs)
@pytest.mark.parametrize("scale,n_ds", [(0.5, 20_000), (0.1, 3_000)], ids=["full", "reduced"])
def test_joint_equals_separate(engines, scale, n_ds):
    e1, e2 = engines
    L = _lws(engines, scale)
    t = synth.make_ds(n_ds, n_roles_choices=(2, 3, 4), fuzz=0.1, seed=31)
    roles, rr = _ds(engines, t)
    model = Model(len(t.ds), len(t.roles), len(t.revroles))
    lplan = churn.make_plan(L.t, L.reqs, oracle.place(L.t.nodes, L.occ, L.t.n_domains, L.t.n_namespaces, L.reqs),
                            0.03, 0.05, n_sets=6, seed=5)
    dplan = churn.make_ds_plan(t, oracle.sweep_ds, 0.02, n_sets=6, frac_target=0.002, seed=6)
    jp = churn.JointArenaPlan(e1, lplan, dplan, L.flags)
    for k in range(-1, 6):
        if k < 0:  # the first tick after the loads: every row
            lt, dt = e1.make_tick((), L.flags), e1.make_ds_tick()
            segs, dsegs = (), []
        else:
            L.apply(lplan[k])
            churn.apply_ds_to_mirror(dplan[k], roles, rr)
            lt, dt = jp.tick(k)
            ps = lplan[k]
            segs = [(R.TABLE_POD_STATE, ps.pod_rows, ps.pod_vals), (R.TABLE_GROUPS, ps.grp_rows, ps.grp_vals),
                    (R.TABLE_PLACE_REQS, ps.req_rows, ps.req_vals)]
            dsegs = _ds_segs(dplan[k])
        joint = _copy(*e1.joint_tick(lt, dt))
        sep = _copy(e2.resident_tick(e2.make_tick(segs, L.flags)), e2.ds_resident_tick(e2.make_ds_tick(dsegs)))
        _same_sets(joint, sep)
        model.check_tick({f"{n}_rows": joint[n][0] for n, _ in DS_LISTS} | {f"{n}_out": joint[n][1] for n, _ in DS_LISTS}
                         | {c: len(joint[n][0]) for n, c in DS_LISTS}, t.ds, roles, rr)
        if k in (-1, 5):
            L.check(e1)
            L.check(e2)


# --------------------------------------------------------------------------- 2. pipelined, full size
def _pipelined(engine, jp, n):
    """Two joint ticks in flight throughout → every tick's lists in order."""
    out = []
    for k in range(n):
        if k >= 2:
            out.append(_copy(*engine.joint_tick_wait()))
        engine.joint_tick_submit(*jp.tick(k))
    while len(out) < n:
        out.append(_copy(*engine.joint_tick_wait()))
    return out


def test_pipelined_full_c3_c4(engines):
    e1, e2 = engines
    L = _lws(engines, 1.0, seed=3, name="C3")
    t = synth.make_ds(50_000, seed=23)
    roles, rr = _ds(engines, t)
    first = [_copy(*_empty(e, flags=L.flags)) for e in engines]
    _same_sets(*first)
    lplan = churn.make_plan(L.t, L.reqs, e1.resident_place_outputs(), 0.01, 0.01, n_sets=4, seed=7)
    dplan = churn.make_ds_plan(t, oracle.sweep_ds, 0.01, n_sets=4, frac_target=0.0, seed=8)
    n = 8
    piped = _pipelined(e1, churn.JointArenaPlan(e1, lplan, dplan, L.flags), n)
    jp2 = churn.JointArenaPlan(e2, lplan, dplan, L.flags)
    serial = [_copy(*e2.joint_tick(*jp2.tick(k))) for k in range(n)]
    for a, b in zip(piped, serial):
        _same_sets(a, b)
    shapes = (len(L.t.lws), len(L.t.groups)), (len(t.ds), len(t.roles), len(t.revroles))
    for e, ticks in ((e1, first[:1] + piped), (e2, first[1:] + serial)):
        _zero_mirror(e, ticks, *shapes)
    for k in range(n):
        L.apply(lplan[k % 4])
        churn.apply_ds_to_mirror(dplan[k % 4], roles, rr)
    ds_o, ro_o, rr_o = oracle.sweep_ds(t.ds, roles, rr)
    for e in engines:
        L.check(e)
        got = e.ds_resident_outputs()
        assert got[0].tobytes() == ds_o.tobytes() and got[1].tobytes() == ro_o.tobytes() and np.array_equal(got[2], rr_o)


# --------------------------------------------------------------------------- 3. DS-only ticks in flight
@pytest.mark.parametrize("n_ds", [50_000, 5_000], ids=["full", "reduced"])
def test_ds_only_ticks_in_flight_follow_the_model(n_ds):
    """On a fresh engine that holds DS tables only (lwse_resident_load never called)."""
    oracle.build()
    e1 = Engine(0)
    try:
        _ds_only_ticks(e1, n_ds)
    finally:
        e1.close()


def _ds_only_ticks(e1, n_ds):
    t = synth.make_ds(n_ds, n_roles_choices=(2, 3, 5, 10), fuzz=0.1, seed=23)
    roles, rr = _ds([e1], t)
    with pytest.raises(LwseError) as ei:  # an LWS part needs the LWS tables
        e1.joint_tick(e1.make_tick(()), e1.make_ds_tick())
    assert ei.value.status == -6
    model = Model(len(t.ds), len(t.roles), len(t.revroles))
    plan = churn.make_ds_plan(t, oracle.sweep_ds, 0.01, n_sets=6, frac_target=0.002, seed=4)
    jp = churn.JointArenaPlan(e1, None, plan)
    snaps = []

    def check(res):
        lres, dres = res
        assert lres is None  # (no LWS tables on this engine)
        model.check_tick(dres, t.ds, *snaps.pop(0))

    snaps.append((roles.copy(), rr.copy()))
    e1.joint_tick_submit(None, e1.make_ds_tick())
    for k in range(12):
        churn.apply_ds_to_mirror(plan[k % 6], roles, rr)
        snaps.append((roles.copy(), rr.copy()))
        e1.joint_tick_submit(*jp.tick(k))
        check(e1.joint_tick_wait())
    check(e1.joint_tick_wait())
    assert not snaps
    model.check_outputs(e1, model.check_tick(_empty(e1, lws=False)[1], t.ds, roles, rr))


# --------------------------------------------------------------------------- 4. one ring, both kinds
@pytest.mark.parametrize("graph", [None, "2"])
def test_mixed_ring(monkeypatch, graph):
    if graph is not None:
        monkeypatch.setenv("LWSE_TICK_GRAPH", graph)
    oracle.build()
    e = Engine(0)
    try:
        L = _lws([e])
        t = synth.make_ds(8000, n_roles_choices=(2, 3), fuzz=0.1, seed=9)
        roles, rr = _ds([e], t)
        model = Model(len(t.ds), len(t.roles), len(t.revroles))
        model.check_tick(_empty(e, flags=L.flags)[1], t.ds, roles, rr)
        lplan = churn.make_plan(L.t, L.reqs, e.resident_place_outputs(), 0.02, 0.04, n_sets=4, seed=2)
        dplan = churn.make_ds_plan(t, oracle.sweep_ds, 0.02, n_sets=4, seed=3)
        jp = churn.JointArenaPlan(e, lplan, dplan, L.flags)
        # an LWS tick, then a joint tick; a resident_tick_wait refuses the joint tick at the head of the ring
        L.apply(lplan[0])
        e.resident_tick_submit(jp.tick(0)[0])
        L.apply(lplan[1])
        churn.apply_ds_to_mirror(dplan[1], roles, rr)
        e.joint_tick_submit(*jp.tick(1))
        lres, dres = e.joint_tick_wait()  # the LWS-only tick
        assert lres["n_groups"] > 0 and (dres["n_ds"], dres["n_roles"], dres["n_revroles"]) == (0, 0, 0)
        with pytest.raises(LwseError) as ei:
            e.resident_tick_wait()
        assert ei.value.status == -1
        lres, dres = e.joint_tick_wait()  # still in flight, with its DS lists
        model.check_tick(dres, t.ds, roles, rr)
        # joint and LWS-only ticks alternate with two in flight (an LWS tick behind a joint one may be
        # replayed as a graph); every DS list in order, then the outputs
        in_flight = []  # per tick: the DS mirrors it saw, or None for an LWS-only tick
        replayed_behind_joint = 0

        def wait_oldest():
            snap = in_flight.pop(0)
            lres, dres = e.joint_tick_wait()
            if snap is None:
                assert (dres["n_ds"], dres["n_roles"], dres["n_revroles"]) == (0, 0, 0)
            else:
                model.check_tick(dres, t.ds, *snap)

        for k in range(2, 12):
            if len(in_flight) == 2:
                wait_oldest()
            L.apply(lplan[k % 4])
            lt, dt = jp.tick(k)
            if k % 2 == 0:
                churn.apply_ds_to_mirror(dplan[k % 4], roles, rr)
                in_flight.append((roles.copy(), rr.copy()))
                e.joint_tick_submit(lt, dt)
            else:
                behind_joint = in_flight[-1] is not None
                in_flight.append(None)
                before = e.graph_tick_count
                e.resident_tick_submit(lt)
                replayed_behind_joint += behind_joint and e.graph_tick_count == before + 1
        while in_flight:
            wait_oldest()
        # (the first LWS-only tick of its shape runs eagerly, the four after it are replayed)
        assert replayed_behind_joint >= 3
        L.check(e)
        model.check_outputs(e, model.check_tick(_empty(e, flags=L.flags)[1], t.ds, roles, rr))
    finally:
        e.close()


# --------------------------------------------------------------------------- 5. refusals
def test_refusals_change_nothing():
    oracle.build()
    e = Engine(0)
    try:
        L = _lws([e], 0.2, seed=11)
        t = synth.make_ds(3000, n_roles_choices=(2, 3), fuzz=0.1, seed=12)
        lt = e.make_tick((), L.flags)
        with pytest.raises(LwseError) as ei:  # the DS tables are not loaded
            e.joint_tick(lt, e.make_ds_tick())
        assert ei.value.status == -6
        _ds([e], t)
        _empty(e, flags=L.flags)
        _nothing_listed(_empty(e, flags=L.flags))
        # segments that would change rows if any of them were applied
        pst = L.pst.copy()
        rows = np.arange(0, 64, dtype=np.uint32)
        vals = R.aligned_empty(64, R.POD_STATE)
        vals[:] = pst[rows] ^ np.uint8(3)
        rr_rows = np.flatnonzero((t.revroles["flags"] & R.RR_EXISTS) != 0)[:8].astype(np.uint32)
        rr_vals = R.aligned_empty(len(rr_rows), R.DS_REVROLE_REC)
        rr_vals[:] = t.revroles[rr_rows]
        rr_vals["ready_replicas"] += 5
        good_l = [(R.TABLE_POD_STATE, rows, vals)]
        good_d = [(R.TABLE_DS_REVROLES, rr_rows, rr_vals)]
        cases = [
            ("DS id in the LWS part", good_l + [(R.TABLE_DS, np.array([0], np.uint32), t.ds[:1].copy())], good_d, L.flags, 0),
            ("LWS id in the DS part", good_l, good_d + [(R.TABLE_LWS, np.array([0], np.uint32), L.t.lws[:1].copy())], L.flags, 0),
            ("9 LWS segments", [(R.TABLE_POD_STATE, rows[i::9].copy(), vals[i::9].copy()) for i in range(9)], good_d, L.flags, 0),
            ("9 DS segments", good_l, [(R.TABLE_DS_REVROLES, rr_rows[i:i + 1].copy(), rr_vals[i:i + 1].copy()) for i in range(8)]
             + [(R.TABLE_DS_ROLES, np.array([0], np.uint32), t.roles[:1].copy())], L.flags, 0),
            ("shared occupancy", good_l, good_d, L.flags | R.TICK_SHARED_OCCUPANCY, 0),
            ("DS flags", good_l, good_d, L.flags, 1),
        ]
        for name, lsegs, dsegs, flags, ds_flags in cases:
            dt = e.make_ds_tick(dsegs)
            dt.flags = ds_flags
            with pytest.raises(LwseError) as ei:
                e.joint_tick(e.make_tick(lsegs, flags), dt)
            assert ei.value.status == -1, name
            _nothing_listed(_empty(e, flags=L.flags))
        rc = lib().lwse_joint_tick(e._h, C.byref(e.make_tick(good_l, L.flags)), None)  # ds = NULL
        assert rc == -1
        _nothing_listed(_empty(e, flags=L.flags))
        # a third submit
        e.joint_tick_submit(e.make_tick((), L.flags), e.make_ds_tick())
        e.joint_tick_submit(e.make_tick((), L.flags), e.make_ds_tick())
        with pytest.raises(LwseError) as ei:
            e.joint_tick_submit(e.make_tick(good_l, L.flags), e.make_ds_tick(good_d))
        assert ei.value.status == -6
        with pytest.raises(LwseError) as ei:  # the one-call form with ticks in flight
            e.joint_tick(e.make_tick(good_l, L.flags), e.make_ds_tick(good_d))
        assert ei.value.status == -6
        _nothing_listed(e.joint_tick_wait())
        _nothing_listed(e.joint_tick_wait())
        _nothing_listed(_empty(e, flags=L.flags))
        L.check(e)
    finally:
        e.close()


# --------------------------------------------------------------------------- 6. one scatter or two
@pytest.mark.parametrize("split", [1, 6])
def test_one_and_two_scatter_launches(engines, split):
    e, _ = engines
    L = _lws([e], 0.3, seed=17)
    t = synth.make_ds(6000, n_roles_choices=(2, 4), fuzz=0.1, seed=18)
    roles, rr = _ds([e], t)
    ds = t.ds.copy()
    model = Model(len(t.ds), len(t.roles), len(t.revroles))
    model.check_tick(_empty(e, flags=L.flags)[1], ds, roles, rr)
    lplan = churn.make_plan(L.t, L.reqs, e.resident_place_outputs(), 0.05, 0.05, n_sets=2, seed=19)
    dplan = churn.make_ds_plan(t, oracle.sweep_ds, 0.05, n_sets=2, frac_target=0.01, seed=20)
    for k in range(2):
        ps, dp = lplan[k], dplan[k]
        L.apply(ps)
        churn.apply_ds_to_mirror(dp, roles, rr)
        lsegs = [(R.TABLE_POD_STATE, ps.pod_rows[i::split].copy(), ps.pod_vals[i::split].copy()) for i in range(split)]
        lsegs.append((R.TABLE_GROUPS, ps.grp_rows, ps.grp_vals))
        dsegs = _ds_segs(dp)
        if split > 1:  # three DS segments: 6 + 1 + 3 = 10 engine-stream segments, two scatter launches
            d_rows = np.arange(0, 40, 3, dtype=np.uint32)
            dsegs.append((R.TABLE_DS, d_rows, ds[d_rows].copy()))
            assert len(dsegs) == 3
        lsegs.append((R.TABLE_PLACE_REQS, ps.req_rows, ps.req_vals))  # (side stream)
        assert (split + 1 + len(dsegs) > 8) == (split > 1)
        lres, dres = e.joint_tick(e.make_tick(lsegs, L.flags), e.make_ds_tick(dsegs))
        assert lres["n_groups"] > 0
        model.check_outputs(e, model.check_tick(dres, ds, roles, rr))
        L.check(e)


# --------------------------------------------------------------------------- 7. BAD_TABLE
def test_bad_table_in_a_joint_tick(engines):
    e, _ = engines
    L = _lws([e], 0.1, seed=21)
    t = synth.make_ds(4000, n_roles_choices=(2, 3), fuzz=0.1, seed=8)
    ds, roles, rr = t.ds.copy(), t.roles.copy(), t.revroles.copy()
    _ds([e], t)
    model = Model(len(ds), len(roles), len(rr))
    model.check_tick(_empty(e, flags=L.flags)[1], ds, roles, rr)
    ok = np.flatnonzero((oracle.sweep_ds(ds, roles, rr)[0]["flags"] & R.DOUT_BAD_TABLE) == 0)
    d = int(ok[len(ok) // 2])
    good = ds[d:d + 1].copy()
    bad = good.copy()
    bad["rev_base"] = len(rr) - 1
    ds[d] = bad[0]
    lres, dres = e.joint_tick(e.make_tick((), L.flags), e.make_ds_tick([(R.TABLE_DS, np.array([d], np.uint32), bad)]))
    assert (dres["n_ds"], dres["n_roles"], dres["n_revroles"]) == (1, 0, 0)
    assert int(dres["ds_rows"][0]) == d and int(dres["ds_out"][0]["flags"]) == R.DOUT_BAD_TABLE
    model.check_outputs(e, model.check_tick(dres, ds, roles, rr))
    row = int(good["rev_base"][0])
    v = rr[row:row + 1].copy()
    v["replicas"] += 3
    v["flags"] |= R.RR_EXISTS
    rr[row] = v[0]
    ds[d] = good[0]
    _, dres = e.joint_tick(e.make_tick((), L.flags), e.make_ds_tick([(R.TABLE_DS, np.array([d], np.uint32), good),
                                                                      (R.TABLE_DS_REVROLES, np.array([row], np.uint32), v)]))
    assert d in dres["ds_rows"].tolist()
    model.check_outputs(e, model.check_tick(dres, ds, roles, rr))
    L.check(e)


# --------------------------------------------------------------------------- 8. through both encoders
def test_both_incremental_encoders_into_joint_ticks(engines):
    import dataclasses

    from informer_world import World, make_world, outputs_by_name
    from test_oracle_ds_flows import abc

    e, _ = engines
    items, cluster = make_world(5, n_lws=20, n_nodes=40)
    world = World(items, cluster, 6)
    enc = informer.IncrementalEncoder(list(world.items.values()), world.cluster(), "zone")
    lws, groups, pst, pid, reqs = enc.full_tables()
    e.upload_nodes(enc.node_rec, len(enc.domain_values))
    e.resident_load(lws, groups, pst, pid)
    e.resident_place_load(reqs, enc.n_namespaces)
    ds_item, children = abc((2, 4), (1, 2), (1, 2), (1, 1), ("A", "B"))
    key = (ds_item.namespace, ds_item.name)
    denc = informer.DsIncrementalEncoder([encoder.DsItem(ds_item, "C", children)], spare=4.0)
    e.ds_resident_load(*denc.full_tables())
    flags = R.SWEEP_GANG | R.TICK_PLACE
    _empty(e, flags=flags)
    names = {sl.lws_row: k for k, sl in enc.slots.items()}
    rng = np.random.Generator(np.random.PCG64(9))
    for step in range(15):
        for _ in range(int(world.rng.integers(1, 6))):
            world.step(enc)
        for c in list(denc.items[key].children):  # child LWS status events
            if rng.random() < 0.5:
                ready = int(rng.integers(0, 1 + (c.replicas or 1)))
                denc.child_event("MODIFIED", key, dataclasses.replace(c, readyReplicas=ready))
        p, dp = enc.flush(), denc.flush()
        assert not enc.needs_reload and not denc.needs_reload
        e.joint_tick(e.make_tick(p.segments, flags), e.make_ds_tick(dp.segments))
        g_lo, g_go = e.resident_outputs()
        got = outputs_by_name(enc.lws[: enc.n_lws], enc.groups, g_lo, g_go, names)
        fresh = list(world.items.values())
        ft = encoder.encode_lws(fresh, world.cluster(), "zone")
        w_lo, w_go, _ = oracle.sweep_lws(ft.lws, ft.groups, ft.pod_state, ft.pod_ident, ft.nodes, flags=R.SWEEP_GANG)
        want = outputs_by_name(ft.lws, ft.groups, w_lo, w_go, {i: (it.lws.namespace, it.lws.name) for i, it in enumerate(fresh)})
        assert got == want, f"step {step}"
        # the DS results against the oracle on a fresh encode of the same object
        fds = encoder.encode_ds([denc.items[key]])
        w_ds, w_ro, w_rr = oracle.sweep_ds(fds.ds, fds.roles, fds.revroles)
        g_ds, g_ro, g_rr = e.ds_resident_outputs()
        sl = denc.slots[key]
        n = int(fds.ds["n_roles"][0])
        n_rr = (int(fds.ds["n_old_revs"][0]) + 1) * n
        assert g_ds[sl.ds_row: sl.ds_row + 1].tobytes() == w_ds[:1].tobytes(), f"step {step}"
        assert g_ro[sl.role_base: sl.role_base + n].tobytes() == w_ro[:n].tobytes(), f"step {step}"
        assert np.array_equal(g_rr[sl.rev_base: sl.rev_base + n_rr], w_rr[:n_rr]), f"step {step}"


# --------------------------------------------------------------------------- 9. a drain in the middle
def test_ds_tick_drains_a_joint_tick_in_flight(engines):
    e, _ = engines
    L = _lws([e], 0.2, seed=33)
    t = synth.make_ds(5000, n_roles_choices=(2, 3), fuzz=0.1, seed=34)
    roles, rr = _ds([e], t)
    _empty(e, flags=L.flags)
    lplan = churn.make_plan(L.t, L.reqs, e.resident_place_outputs(), 0.03, 0.05, n_sets=2, seed=35)
    dplan = churn.make_ds_plan(t, oracle.sweep_ds, 0.03, n_sets=2, seed=36)
    jp = churn.JointArenaPlan(e, lplan, dplan, L.flags)
    L.apply(lplan[0])
    churn.apply_ds_to_mirror(dplan[0], roles, rr)
    e.joint_tick_submit(*jp.tick(0))
    churn.apply_ds_to_mirror(dplan[1], roles, rr)
    e.ds_resident_tick(e.make_ds_tick(_ds_segs(dplan[1])))  # waits for the joint tick, drops its lists
    with pytest.raises(LwseError):
        e.joint_tick_wait()  # nothing in flight any more
    ds_o, ro_o, rr_o = oracle.sweep_ds(t.ds, roles, rr)
    got = e.ds_resident_outputs()
    assert got[0].tobytes() == ds_o.tobytes() and got[1].tobytes() == ro_o.tobytes() and np.array_equal(got[2], rr_o)
    L.check(e)
