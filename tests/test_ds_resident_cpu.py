"""CPU checks of the resident DisaggregatedSet tick's host side: the C ABI of ``lwse_ds_tick``, the
watch-event encoder (``informer.DsIncrementalEncoder``) and the DS churn plan (``churn.make_ds_plan``)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle
from lws_b200 import api, churn, encoder, informer, synth
from lws_b200 import records as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def _oracle():
    oracle.build()


def test_ds_tick_layout_matches_header():
    fields = [f for f, _ in R.DsTick._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{ROOT}/include/lwse.h"', "int main(){",
             'printf("size %zu\\n", sizeof(lwse_ds_tick));']
    lines += [f'printf("{f} %zu\\n", offsetof(lwse_ds_tick, {f}));' for f in fields]
    lines += [f'printf("{n} %d\\n", (int){n});' for n in ("LWSE_TABLE_DS", "LWSE_TABLE_DS_ROLES", "LWSE_TABLE_DS_REVROLES")]
    lines.append("return 0;}")
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "p.c"), os.path.join(d, "p")
        open(src, "w").write("\n".join(lines))
        subprocess.run(["gcc", "-o", exe, src], check=True)
        got = dict(l.split() for l in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split("\n") if l)
    assert int(got["size"]) == C.sizeof(R.DsTick)
    for f in fields:
        assert int(got[f]) == getattr(R.DsTick, f).offset, f
    assert (int(got["LWSE_TABLE_DS"]), int(got["LWSE_TABLE_DS_ROLES"]), int(got["LWSE_TABLE_DS_REVROLES"])) == (
        R.TABLE_DS, R.TABLE_DS_ROLES, R.TABLE_DS_REVROLES)


# --------------------------------------------------------------------------- encoder
ROLES = ["prefill", "decode", "router"]


def make_item(rng, name, n_roles=2, rev="r0"):
    cfg = api.RollingUpdateConfiguration(maxSurge=int(rng.integers(1, 3)), maxUnavailable=0)
    ds = api.DisaggregatedSet(name, roles=[api.DisaggregatedRoleSpec(ROLES[i], int(rng.integers(1, 6)), cfg)
                                           for i in range(n_roles)])
    kids = [api.ChildLWS(ROLES[i], rev, int(rng.integers(0, 5)), 0, 1.0) for i in range(n_roles)]
    return encoder.DsItem(ds, rev, kids)


def compare_with_fresh_encode(enc):
    """The oracle on the incremental tables equals the oracle on a fresh encode of the same cache,
    per (DS, role, revision)."""
    ds_o, ro_o, rr_o = oracle.sweep_ds(*enc.full_tables())
    keys = sorted(enc.items)
    fresh = encoder.encode_ds([enc.items[k] for k in keys])
    f_ds, f_ro, f_rr = oracle.sweep_ds(fresh.ds, fresh.roles, fresh.revroles)
    for j, k in enumerate(keys):
        sl, names, olds = enc.slots[k], enc.role_names(k), enc.old_revisions(k)
        assert names == fresh.role_names[j] and olds == fresh.old_revisions[j], k
        assert ds_o[sl.ds_row].tobytes() == f_ds[j].tobytes(), k
        n, fb = len(names), fresh.ds[j]
        for i in range(n):
            assert ro_o[sl.role_base + i].tobytes() == f_ro[int(fb["role_base"]) + i].tobytes(), (k, names[i])
        for r in range(len(olds) + 1):
            for i in range(n):
                assert rr_o[sl.rev_base + r * n + i] == f_rr[int(fb["rev_base"]) + r * n + i], (k, r, names[i])


def apply_patches(mirror, patches):
    index = {R.TABLE_DS: 0, R.TABLE_DS_ROLES: 1, R.TABLE_DS_REVROLES: 2}
    for table, rows, vals in patches.segments:
        assert np.all(np.diff(rows.astype(np.int64)) > 0)
        mirror[index[table]][rows] = vals


def random_event(rng, enc, clock):
    """One watch event of the kinds a DS controller sees (returns a label for the failure message)."""
    keys = sorted(enc.items)
    key = keys[int(rng.integers(len(keys)))]
    it = enc.items[key]
    kind = int(rng.integers(5))
    if kind == 0:  # a new target revision appears: spec change, then the controller creates its children
        rev = f"r{clock}"
        enc.ds_event("MODIFIED", encoder.DsItem(it.ds, rev))
        for role in it.ds.roles[: int(rng.integers(0, len(it.ds.roles) + 1))]:
            enc.child_event("ADDED", key, api.ChildLWS(role.name, rev, 0, 0, float(clock)))
        return "new revision"
    if kind == 1:  # a drained old revision is deleted
        olds = sorted({c.revision for c in it.children if c.revision != it.revision})
        if olds:
            rev = olds[int(rng.integers(len(olds)))]
            for c in [c for c in it.children if c.revision == rev]:
                enc.child_event("DELETED", key, c)
        return "revision deleted"
    if kind == 2:  # a role is removed from the spec (its old children become a removed role)
        if len(it.ds.roles) > 1:
            ds = api.DisaggregatedSet(it.ds.name, it.ds.namespace, it.ds.uid, it.ds.roles[:-1])
            enc.ds_event("MODIFIED", encoder.DsItem(ds, f"r{clock}"))
        return "role removed"
    if kind == 3:  # readiness / replicas of a child change
        if it.children:
            c = it.children[int(rng.integers(len(it.children)))]
            nc = api.ChildLWS(c.role, c.revision, c.replicas, int(rng.integers(0, 6)), c.creationTimestamp,
                              dict(c.annotations))
            if rng.random() < 0.5:
                nc.replicas = int(rng.integers(0, 6))
                nc.annotations[api.DSInitialReplicasAnnotationKey] = str(int(rng.integers(0, 6)))
            enc.child_event("MODIFIED", key, nc)
        return "child modified"
    # a child of the target revision is created
    missing = [r.name for r in it.ds.roles if not any(c.role == r.name and c.revision == it.revision for c in it.children)]
    if missing:
        enc.child_event("ADDED", key, api.ChildLWS(missing[0], it.revision, 1, 0, float(clock)))
    return "child added"


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_incremental_encoder_matches_fresh_encode(seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    items = [make_item(rng, f"ds-{i}", n_roles=int(rng.integers(1, 4))) for i in range(12)]
    enc = informer.DsIncrementalEncoder(items, spare=4.0)
    mirror = [x.copy() for x in enc.full_tables()]
    compare_with_fresh_encode(enc)
    seen = set()
    for step in range(60):
        for _ in range(int(rng.integers(1, 4))):
            seen.add(random_event(rng, enc, 10 + step))
        slots_before = {k: (s.role_base, s.rev_base) for k, s in enc.slots.items()}
        patches = enc.flush()
        assert not enc.needs_reload
        if any((s.role_base, s.rev_base) != slots_before[k] for k, s in enc.slots.items()):
            seen.add("relocated")
        apply_patches(mirror, patches)
        for m, t in zip(mirror, enc.full_tables()):
            assert m.tobytes() == t.tobytes(), f"step {step}: patched mirror differs from the encoder's tables"
        compare_with_fresh_encode(enc)
    assert seen >= {"new revision", "revision deleted", "role removed", "child modified", "relocated"}, seen


def test_incremental_encoder_relocates_then_needs_reload():
    rng = np.random.Generator(np.random.PCG64(9))
    enc = informer.DsIncrementalEncoder([make_item(rng, f"ds-{i}") for i in range(4)], spare=0.0)
    key = ("default", "ds-0")
    mirror = [x.copy() for x in enc.full_tables()]
    base0 = enc.slots[key].rev_base
    relocated = False
    for k in range(40):  # every new target revision keeps the old ones: the DS grows until nothing fits
        it = enc.items[key]
        rev = f"grow-{k}"
        enc.ds_event("MODIFIED", encoder.DsItem(it.ds, rev))
        for role in it.ds.roles:
            enc.child_event("ADDED", key, api.ChildLWS(role.name, rev, 1, 1, float(100 + k)))
        patches = enc.flush()
        if enc.needs_reload:
            break
        relocated |= enc.slots[key].rev_base != base0
        apply_patches(mirror, patches)
        assert all(m.tobytes() == t.tobytes() for m, t in zip(mirror, enc.full_tables()))
        compare_with_fresh_encode(enc)
    assert relocated and enc.needs_reload
    enc2 = informer.DsIncrementalEncoder([make_item(rng, "x")])
    enc2.ds_event("ADDED", make_item(rng, "y"))
    assert enc2.needs_reload


# --------------------------------------------------------------------------- churn
def test_ds_plan_keeps_the_mirror_consistent():
    t = synth.make_ds(3000, n_roles_choices=(2, 3, 10), fuzz=0.1, seed=5)
    sets = churn.make_ds_plan(t, oracle.sweep_ds, 0.05, n_sets=6, frac_target=0.01)
    roles, rr = t.roles.copy(), t.revroles.copy()
    exists = rr["flags"] & R.RR_EXISTS
    for ps in sets:
        assert len(ps.rr_rows) and np.all(np.diff(ps.rr_rows.astype(np.int64)) > 0)
        _, _, want = oracle.sweep_ds(t.ds, roles, rr)  # the decisions this set applies
        churn.apply_ds_to_mirror(ps, roles, rr)
        scaled = want[ps.rr_rows] >= 0
        assert np.array_equal(rr["replicas"][ps.rr_rows[scaled]], want[ps.rr_rows[scaled]])
        assert np.all(exists[ps.rr_rows])
        assert ps.h2d_bytes() == ps.rr_rows.nbytes + ps.rr_vals.nbytes + ps.role_rows.nbytes + ps.role_vals.nbytes
    assert np.array_equal(rr["flags"] & R.RR_EXISTS, exists), "the layout never changes"
    assert any(len(ps.role_rows) for ps in sets)
    # the plan simulated the same run: replaying it from the start reproduces its values
    again = churn.make_ds_plan(t, oracle.sweep_ds, 0.05, n_sets=6, frac_target=0.01)
    assert all(a.rr_vals.tobytes() == b.rr_vals.tobytes() for a, b in zip(sets, again))
