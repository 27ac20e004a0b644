"""The arena layout of joint ticks (churn.JointArenaPlan), on the CPU: every array 256-byte aligned
inside its pass's region, regions alternating so that the two ticks in flight never share a byte,
and the tick descriptors pointing at what was written."""
import numpy as np
import pytest

import oracle
from lws_b200 import churn
from lws_b200 import records as R
from lws_b200 import synth


class FakeEngine:
    """The three engine calls the plan makes; the arena is ordinary page-aligned host memory."""

    def __init__(self):
        self.buf = None

    def resident_arena(self, min_bytes):
        raw = np.zeros(min_bytes + 8192, np.uint8)
        off = (-raw.ctypes.data) % 4096
        self.buf = raw[off: off + min_bytes + 4096]
        return self.buf

    def make_tick(self, segs, flags):
        return ("lws", segs, flags)

    def make_ds_tick(self, segs):
        return ("ds", segs)


def _plans(with_lws):
    t = synth.make(synth.profile("fuzz", 0.2), seed=12)
    reqs = t.place_requests()
    occ = R.occupancy_of(t.pod_ident, len(t.nodes))
    place = oracle.place(t.nodes, occ, t.n_domains, t.n_namespaces, reqs)
    lplan = churn.make_plan(t, reqs, place, 0.02, 0.05, n_sets=4, seed=3) if with_lws else None
    d = synth.make_ds(3000, n_roles_choices=(2, 4), fuzz=0.1, seed=5)
    dplan = churn.make_ds_plan(d, oracle.sweep_ds, 0.02, n_sets=4, frac_target=0.01, seed=6)
    return lplan, dplan


@pytest.mark.parametrize("with_lws", [True, False])
def test_regions_alternate_aligned_and_in_bounds(with_lws):
    lplan, dplan = _plans(with_lws)
    eng = FakeEngine()
    plan = churn.JointArenaPlan(eng, lplan, dplan, flags=R.TICK_PLACE)
    rb = plan.region_bytes
    assert rb % 4096 == 0 and len(plan.arena) >= 2 * rb
    per_pass = {}
    for k in range(10):
        lws_tick, ds_tick = plan.tick(k)
        spans = [(o, n) for kk, o, n in plan.spans if kk == k]
        per_pass[k] = spans
        for o, n in spans:
            assert o % 256 == 0
            assert (k % 2) * rb <= o and o + n <= (k % 2 + 1) * rb
        # the descriptors' arrays are views of the arena holding the pass's patches
        p = k % len(dplan)
        segs = (lws_tick[1] if lws_tick is not None else []) + ds_tick[1]
        assert (lws_tick is not None) == with_lws
        for _, rows, vals in segs:
            assert np.shares_memory(rows, plan.arena) and np.shares_memory(vals, plan.arena)
        ds_tables = [tb for tb, _, _ in ds_tick[1]]
        assert set(ds_tables) <= {R.TABLE_DS_REVROLES, R.TABLE_DS_ROLES}
        assert np.array_equal(ds_tick[1][0][1], dplan[p].rr_rows)
        assert ds_tick[1][0][2].tobytes() == dplan[p].rr_vals.tobytes()
        if with_lws:
            assert lws_tick[2] == R.TICK_PLACE and lws_tick[1][0][0] == R.TABLE_POD_STATE
            assert np.array_equal(lws_tick[1][0][1], lplan[p].pod_rows)
            assert np.array_equal(lws_tick[1][0][2], lplan[p].pod_vals)
        if k:  # the tick before is still in flight: no byte in common
            prev = per_pass[k - 1]
            for o, n in spans:
                assert all(o + n <= po or po + pn <= o for po, pn in prev)
