"""The resident DisaggregatedSet tick (lwse_ds_resident_tick) on the GPU: every tick's three change
lists against the committed-value model of include/lwse.h, computed on the host from consecutive
oracle runs on mirror tables; the committed outputs against the oracle and against a zero mirror
with every tick's lists applied."""
import dataclasses

import numpy as np
import pytest

import oracle
from lws_b200 import api, churn, encoder, informer, synth
from lws_b200 import records as R
from lws_b200.engine import LwseError

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from lws_b200.engine import Engine

    oracle.build()
    e = Engine(0)
    yield e
    e.close()


def _ranges(base, count):
    base, count = base.astype(np.int64), count.astype(np.int64)
    total = int(count.sum())
    start = np.concatenate([[0], np.cumsum(count)[:-1]])
    return np.repeat(base - start, count) + np.arange(total)


def _differ(a, b):
    return np.any(a.view(np.uint8).reshape(len(a), -1) != b.view(np.uint8).reshape(len(b), -1), axis=1)


class Model:
    """The committed values and the listing rules of the header, on the host."""

    def __init__(self, n_ds, n_roles, n_rr):
        self.committed = (R.aligned_empty(n_ds, R.DS_OUT), R.aligned_empty(n_roles, R.DS_ROLE_OUT),
                          R.aligned_empty(n_rr, R.DS_REVROLE_OUT))
        self.mirror = tuple(x.copy() for x in self.committed)  # zero + every tick's lists
        self.first = True

    def check_tick(self, res, ds, roles, revroles):
        ds_o, ro_o, rr_o = oracle.sweep_ds(ds, roles, revroles)
        ds_c, ro_c, rr_c = self.committed
        valid = np.flatnonzero((ds_o["flags"] & R.DOUT_BAD_TABLE) == 0)
        n = ds["n_roles"][valid].astype(np.int64)
        role_rows = _ranges(ds["role_base"][valid], n)
        rr_rows = _ranges(ds["rev_base"][valid], (ds["n_old_revs"][valid].astype(np.int64) + 1) * n)
        role_chg = self.first | _differ(ro_o[role_rows], ro_c[role_rows])
        rr_chg = self.first | (rr_o[rr_rows] != rr_c[rr_rows])
        owner_ro, owner_rr = np.repeat(valid, n), np.repeat(valid, (ds["n_old_revs"][valid].astype(np.int64) + 1) * n)
        ds_chg = self.first | _differ(ds_o, ds_c)
        ds_chg[owner_ro[role_chg]] = True
        ds_chg[owner_rr[rr_chg]] = True
        want = {"ds": (np.flatnonzero(ds_chg), ds_o), "role": (np.sort(role_rows[role_chg]), ro_o),
                "revrole": (np.sort(rr_rows[rr_chg]), rr_o)}
        for name, (rows, new) in want.items():
            got_rows, got_out = res[f"{name}_rows"], res[f"{name}_out"]
            assert res["n_" + {"ds": "ds", "role": "roles", "revrole": "revroles"}[name]] == len(rows), name
            o = np.argsort(got_rows, kind="stable")
            assert np.array_equal(got_rows[o], rows), name
            assert got_out[o].tobytes() == new[rows].tobytes(), name
        for k, name in enumerate(("ds", "role", "revrole")):
            rows, new = want[name]
            self.committed[k][rows] = new[rows]
            self.mirror[k][res[f"{name}_rows"]] = res[f"{name}_out"]
        self.first = False
        return ds_o, ro_o, rr_o, role_rows, rr_rows

    def check_outputs(self, engine, tick_result):
        ds_o, ro_o, rr_o, role_rows, rr_rows = tick_result
        got = engine.ds_resident_outputs()
        for g, m in zip(got, self.mirror):
            assert g.tobytes() == m.tobytes(), "outputs differ from the zero mirror plus every tick's lists"
        assert got[0].tobytes() == ds_o.tobytes()
        assert got[1][role_rows].tobytes() == ro_o[role_rows].tobytes()
        assert np.array_equal(got[2][rr_rows], rr_o[rr_rows])


def _full_c4():
    return synth.make_ds(50_000, n_roles_choices=(2, 3, 5, 10), fuzz=0.1, seed=23)


def test_c4_ticks_follow_the_committed_value_model(engine):
    t = _full_c4()
    roles, rr = t.roles.copy(), t.revroles.copy()
    engine.ds_resident_load(t.ds, t.roles, t.revroles)
    model = Model(len(t.ds), len(t.roles), len(t.revroles))
    first = engine.ds_resident_tick(engine.make_ds_tick())
    assert first["n_ds"] == len(t.ds)
    model.check_outputs(engine, model.check_tick(first, t.ds, roles, rr))
    again = engine.ds_resident_tick(engine.make_ds_tick())
    assert (again["n_ds"], again["n_roles"], again["n_revroles"]) == (0, 0, 0)

    plan = churn.make_ds_plan(t, oracle.sweep_ds, 0.01, n_sets=12, frac_target=0.002, seed=4)
    need = sum(ps.h2d_bytes() + 1024 for ps in plan) + 4096
    arena = engine.resident_arena(need)
    cursor = 0

    def put(a):
        nonlocal cursor
        off = (cursor + 255) // 256 * 256
        view = arena[off: off + a.nbytes].view(a.dtype)
        view[...] = a
        cursor = off + a.nbytes
        return view

    n_in_arena = 0
    for k, ps in enumerate(plan):
        segs = [(R.TABLE_DS_REVROLES, ps.rr_rows, ps.rr_vals)]
        if len(ps.role_rows):
            segs.append((R.TABLE_DS_ROLES, ps.role_rows, ps.role_vals))
        if k % 2 == 0:  # in the arena: consumed in place
            segs = [(tb, put(rows), put(vals)) for tb, rows, vals in segs]
            n_in_arena += 1
        churn.apply_ds_to_mirror(ps, roles, rr)
        res = engine.ds_resident_tick(engine.make_ds_tick(segs))
        assert res["n_revroles"] > 0
        model.check_outputs(engine, model.check_tick(res, t.ds, roles, rr))
    assert n_in_arena == 6


def test_bad_table_is_listed_alone_and_recovers(engine):
    t = synth.make_ds(4000, n_roles_choices=(2, 3), fuzz=0.1, seed=8)
    ds, roles, rr = t.ds.copy(), t.roles.copy(), t.revroles.copy()
    engine.ds_resident_load(ds, roles, rr)
    model = Model(len(ds), len(roles), len(rr))
    model.check_tick(engine.ds_resident_tick(engine.make_ds_tick()), ds, roles, rr)
    ok = np.flatnonzero((oracle.sweep_ds(ds, roles, rr)[0]["flags"] & R.DOUT_BAD_TABLE) == 0)
    d = int(ok[len(ok) // 2])
    good = ds[d:d + 1].copy()
    bad = good.copy()
    bad["rev_base"] = len(rr) - 1  # the revision range runs out of the table
    ds[d] = bad[0]
    res = engine.ds_resident_tick(engine.make_ds_tick([(R.TABLE_DS, np.array([d], np.uint32), bad)]))
    assert (res["n_ds"], res["n_roles"], res["n_revroles"]) == (1, 0, 0)
    assert int(res["ds_rows"][0]) == d and int(res["ds_out"][0]["flags"]) == R.DOUT_BAD_TABLE
    model.check_outputs(engine, model.check_tick(res, ds, roles, rr))
    # while it is bad, one of its rows changes; patched back, it is listed against its committed value
    row = int(good["rev_base"][0])
    v = rr[row:row + 1].copy()
    v["replicas"] += 3
    v["flags"] |= R.RR_EXISTS
    rr[row] = v[0]
    ds[d] = good[0]
    res = engine.ds_resident_tick(engine.make_ds_tick([(R.TABLE_DS, np.array([d], np.uint32), good),
                                                       (R.TABLE_DS_REVROLES, np.array([row], np.uint32), v)]))
    assert d in res["ds_rows"].tolist()
    model.check_outputs(engine, model.check_tick(res, ds, roles, rr))


# --------------------------------------------------------------------------- reference flows
def _run_flow_on_engine(engine, target, a, b, surge, order, check_orphans=False):
    from test_oracle_ds_flows import abc

    ds, children = abc(target, a, b, surge, order)
    key = (ds.namespace, ds.name)
    enc = informer.DsIncrementalEncoder([encoder.DsItem(ds, "C", children)], spare=4.0)
    engine.ds_resident_load(*enc.full_tables())
    mirror = [np.zeros(len(x), dtype) for x, dtype in zip(enc.full_tables(), (R.DS_OUT, R.DS_ROLE_OUT, R.DS_REVROLE_OUT))]
    clock = 100.0

    def kid(role, rev):
        return next((c for c in enc.items[key].children if c.role == role and c.revision == rev), None)

    def replicas(role, rev):
        c = kid(role, rev)
        return -1 if c is None else c.replicas

    for step in range(20):
        res = engine.ds_resident_tick(engine.make_ds_tick(enc.flush().segments))
        for k, name in enumerate(("ds", "role", "revrole")):
            mirror[k][res[f"{name}_rows"]] = res[f"{name}_out"]
        sl, names, olds = enc.slots[key], enc.role_names(key), enc.old_revisions(key)
        out = mirror[0][sl.ds_row]
        n = len(names)
        rr_out = mirror[2][sl.rev_base: sl.rev_base + (len(olds) + 1) * n]
        # the reconcile's decisions come back as watch events of the child LWS objects (ds_sim.DsSim)
        for r, rev in enumerate(olds):
            if int(out["drained_revs"]) >> r & 1:
                for c in [c for c in enc.items[key].children if c.revision == rev]:
                    enc.child_event("DELETED", key, c)
        if int(out["flags"]) & R.DOUT_INIT:
            for c in list(enc.items[key].children):
                if c.revision != "C":
                    ann = dict(c.annotations)
                    ann[api.DSInitialReplicasAnnotationKey] = str(1 if c.replicas is None else c.replicas)
                    enc.child_event("MODIFIED", key, dataclasses.replace(c, annotations=ann))
        for r, rev in enumerate(olds + ["C"]):
            for i, role in enumerate(names):
                want = int(rr_out[r * n + i])
                c = kid(role, rev)
                if c is None:
                    if want >= 0 and rev == "C":
                        clock += 1
                        enc.child_event("ADDED", key, api.ChildLWS(role, rev, want, 0, clock))
                elif want >= 0 and c.replicas != want:
                    enc.child_event("MODIFIED", key, dataclasses.replace(c, replicas=want))
        for c in list(enc.items[key].children):  # simulateAllReady
            if c.replicas is not None and c.readyReplicas != c.replicas:
                enc.child_event("MODIFIED", key, dataclasses.replace(c, readyReplicas=c.replicas))
        assert not enc.needs_reload
        if check_orphans:
            norm = lambda v: 0 if v == -1 else v
            for rev in ("A", "B"):
                p, d = norm(replicas("prefill", rev)), norm(replicas("decode", rev))
                assert (p == 0) == (d == 0), f"step {step}: {rev} orphaned prefill={p} decode={d}"
    for rev in ("A", "B"):
        for role in ("prefill", "decode"):
            assert replicas(role, rev) in (0, -1), f"{rev}/{role} not drained"
    assert (replicas("prefill", "C"), replicas("decode", "C")) == tuple(target)


@pytest.mark.parametrize("order", [("A", "B"), ("B", "A")])
def test_mid_rollout_abc_through_the_tick(engine, order):
    _run_flow_on_engine(engine, (2, 4), (1, 2), (1, 2), (1, 1), order)


@pytest.mark.parametrize("order", [("A", "B"), ("B", "A")])
def test_asymmetric_sizes_coordinated_drain_through_the_tick(engine, order):
    _run_flow_on_engine(engine, (4, 3), (1, 2), (3, 1), (1, 2), order, check_orphans=True)


# --------------------------------------------------------------------------- one engine, both controllers
def test_lws_and_ds_ticks_coexist(engine):
    tl = synth.make(synth.profile("fuzz", 0.5), seed=43)
    reqs = tl.place_requests()
    engine.upload_nodes(tl.nodes, tl.n_domains)
    engine.resident_load(tl.lws, tl.groups, tl.pod_state, tl.pod_ident)
    engine.resident_place_load(reqs, tl.n_namespaces)
    occ = R.occupancy_of(tl.pod_ident, len(tl.nodes))
    flags = tl.flags | R.TICK_PLACE
    t = synth.make_ds(20_000, n_roles_choices=(2, 4), fuzz=0.1, seed=31)
    roles, rr = t.roles.copy(), t.revroles.copy()
    engine.ds_resident_load(t.ds, t.roles, t.revroles)
    model = Model(len(t.ds), len(t.roles), len(t.revroles))
    m_pst, m_grp, m_req = tl.pod_state.copy(), tl.groups.copy(), reqs.copy()

    def check_lws():
        lo, go, _ = oracle.sweep_lws(tl.lws, m_grp, m_pst, tl.pod_ident, tl.nodes, flags=tl.flags)
        got = engine.resident_outputs()
        assert got[0].tobytes() == lo.tobytes() and got[1].tobytes() == go.tobytes()
        assert engine.resident_place_outputs().tobytes() == oracle.place(tl.nodes, occ, tl.n_domains, tl.n_namespaces,
                                                                         m_req).tobytes()

    engine.resident_tick(engine.make_tick((), flags))
    check_lws()
    model.check_tick(engine.ds_resident_tick(engine.make_ds_tick()), t.ds, roles, rr)
    lplan = churn.make_plan(tl, reqs, engine.resident_place_outputs(), 0.03, 0.05, n_sets=4, seed=5)
    ticks = churn.ArenaPlan(engine, lplan, flags).ticks
    dplan = churn.make_ds_plan(t, oracle.sweep_ds, 0.02, n_sets=4, seed=6)
    for k in range(4):  # LWS and DS ticks alternate
        churn.apply_to_mirror(lplan[k], m_pst, m_grp, m_req)
        engine.resident_tick(ticks[k])
        check_lws()
        ps = dplan[k]
        churn.apply_ds_to_mirror(ps, roles, rr)
        segs = [(R.TABLE_DS_REVROLES, ps.rr_rows, ps.rr_vals)] + (
            [(R.TABLE_DS_ROLES, ps.role_rows, ps.role_vals)] if len(ps.role_rows) else [])
        model.check_outputs(engine, model.check_tick(engine.ds_resident_tick(engine.make_ds_tick(segs)), t.ds, roles, rr))
    # a stateless DS sweep in between leaves the resident DS state alone
    engine.sweep_ds_host(*synth.make_ds(3000, seed=2).__dict__.values())
    res = engine.ds_resident_tick(engine.make_ds_tick())
    assert (res["n_ds"], res["n_roles"], res["n_revroles"]) == (0, 0, 0)
    # a DS tick while an LWS tick is in flight: the LWS tick completes, the DS results are right
    churn.apply_to_mirror(lplan[0], m_pst, m_grp, m_req)
    engine.resident_tick_submit(ticks[0])
    ps = dplan[0]
    v = ps.rr_vals.copy()
    v["ready_replicas"] += 1
    rr[ps.rr_rows] = v
    res = engine.ds_resident_tick(engine.make_ds_tick([(R.TABLE_DS_REVROLES, ps.rr_rows, v)]))
    model.check_outputs(engine, model.check_tick(res, t.ds, roles, rr))
    check_lws()
    # the LWS tick does not take the DS tables, and a refused tick changes nothing
    row = np.array([0], np.uint32)
    with pytest.raises(LwseError):
        engine.resident_tick(engine.make_tick([(R.TABLE_DS, row, t.ds[:1].copy())], flags))
    with pytest.raises(LwseError):
        engine.resident_tick(engine.make_tick([(R.TABLE_LWS, row, tl.lws[:1].copy()),
                                               (R.TABLE_DS_REVROLES, row, rr[:1].copy())], flags))
    res = engine.ds_resident_tick(engine.make_ds_tick())
    assert (res["n_ds"], res["n_roles"], res["n_revroles"]) == (0, 0, 0)
    again = engine.resident_tick(engine.make_tick((), flags))
    assert (again["n_lws"], again["n_groups"]) == (0, 0)
    check_lws()
