"""The joint LWS + DS tick (lwse_joint_tick) at C3 + C4 against the two separate ticks.

    python profiles/joint_tick.py OUT_DIR [--blocks 4] [--seconds 1.0] [--label NAME]

C3: synth profile "C3" at scale 1.0 with placement; each pass patches 1 % of the pod rows and 1 % of the
placement requests (churn.make_plan).  C4: 50 000 DisaggregatedSets (synth.make_ds); each pass patches 1 %
of the revision-role rows (churn.make_ds_plan, as profiles/ds_tick.py).  Every pass's patches lie in the
engine's patch arena.  In alternating blocks of at least ``--seconds`` each, per pass of both work queues:
  * separate:        lwse_resident_tick, then lwse_ds_resident_tick;
  * joint_serial:    one lwse_joint_tick;
  * joint_pipelined: lwse_joint_tick_submit / _wait with two ticks in flight.
The times are host clock over whole blocks; every call returns only after its sequence word (for the
pipelined form the block ends with the last wait).  Every shape is warmed first.  After the timed blocks
the resident outputs of both controllers are checked against the oracle on host mirrors.  Prints one JSON
line and writes it to OUT_DIR/joint_tick_<label>.json with the card's name and power limit, read in the
same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import oracle  # noqa: E402
from lws_b200 import churn, synth  # noqa: E402
from lws_b200 import records as R  # noqa: E402
from lws_b200.engine import Engine  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--blocks", type=int, default=4)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--n-ds", type=int, default=50_000)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--label", default="joint")
    a = ap.parse_args()
    os.makedirs(a.out_dir, exist_ok=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]

    oracle.build()
    tl = synth.make(synth.profile("C3", a.scale), seed=3)
    reqs = tl.place_requests()
    flags = tl.flags | R.TICK_PLACE
    td = synth.make_ds(a.n_ds)
    eng = Engine(0)
    eng.upload_nodes(tl.nodes, tl.n_domains)
    eng.resident_load(tl.lws, tl.groups, tl.pod_state, tl.pod_ident)
    eng.resident_place_load(reqs, tl.n_namespaces)
    eng.ds_resident_load(td.ds, td.roles, td.revroles)
    eng.joint_tick(eng.make_tick((), flags), eng.make_ds_tick())
    lplan = churn.make_plan(tl, reqs, eng.resident_place_outputs(), 0.01, 0.01, n_sets=8, seed=7)
    dplan = churn.make_ds_plan(td, oracle.sweep_ds, 0.01, n_sets=8, frac_target=0.0)
    # every pass in its own arena region: descriptors built once, nothing copied inside the timed blocks
    need = sum(ps.h2d_bytes() + dp.h2d_bytes() + 8 * 256 for ps, dp in zip(lplan, dplan)) + 4096
    arena = eng.resident_arena(need)
    cursor = 0

    def put(x):
        nonlocal cursor
        off = (cursor + 255) // 256 * 256
        view = arena[off: off + x.nbytes].view(x.dtype)
        view[...] = x
        cursor = off + x.nbytes
        return view

    lticks, dticks = [], []
    for ps, dp in zip(lplan, dplan):
        segs = [(tb, put(r), put(v)) for tb, r, v in ((R.TABLE_POD_STATE, ps.pod_rows, ps.pod_vals),
                                                      (R.TABLE_GROUPS, ps.grp_rows, ps.grp_vals),
                                                      (R.TABLE_PLACE_REQS, ps.req_rows, ps.req_vals)) if len(r)]
        lticks.append(eng.make_tick(segs, flags))
        dticks.append(eng.make_ds_tick([(R.TABLE_DS_REVROLES, put(dp.rr_rows), put(dp.rr_vals))]))
    n_pass = len(lticks)
    applied = 0
    rows_out = {"separate": [], "joint_serial": [], "joint_pipelined": []}

    def rows(lres, dres):
        return lres["n_lws"] + lres["n_groups"] + lres["n_place"] + dres["n_ds"] + dres["n_roles"] + dres["n_revroles"]

    def separate(k):
        return rows(eng.resident_tick(lticks[k]), eng.ds_resident_tick(dticks[k]))

    def joint_serial(k):
        return rows(*eng.joint_tick(lticks[k], dticks[k]))

    def block(mode, seconds, record):
        """Whole cycles of the plan until `seconds` passed → µs per pass."""
        nonlocal applied
        n, t0 = 0, time.perf_counter()
        while True:
            if mode == "joint_pipelined":
                out = []
                eng.joint_tick_submit(lticks[0], dticks[0])
                for k in range(1, n_pass):
                    eng.joint_tick_submit(lticks[k], dticks[k])
                    out.append(rows(*eng.joint_tick_wait()))
                out.append(rows(*eng.joint_tick_wait()))
            else:
                fn = separate if mode == "separate" else joint_serial
                out = [fn(k) for k in range(n_pass)]
            if record:
                rows_out[mode].extend(out)
            n += n_pass
            applied += n_pass
            dt = time.perf_counter() - t0
            if dt >= seconds:
                return dt / n * 1e6

    modes = ("separate", "joint_serial", "joint_pipelined")
    for m in modes:  # warm every shape
        block(m, 0.3, False)
    us = {m: [] for m in modes}
    for _ in range(a.blocks):
        for m in modes:
            us[m].append(block(m, a.seconds, True))

    # every block runs whole cycles of the plan: the final state is one cycle applied to the loaded tables
    assert applied % n_pass == 0 and applied >= n_pass
    pst, grp, rq = tl.pod_state.copy(), tl.groups.copy(), reqs.copy()
    roles, rr = td.roles.copy(), td.revroles.copy()
    for ps, dp in zip(lplan, dplan):
        churn.apply_to_mirror(ps, pst, grp, rq)
        churn.apply_ds_to_mirror(dp, roles, rr)
    lo, go, _ = oracle.sweep_lws(tl.lws, grp, pst, tl.pod_ident, tl.nodes, flags=tl.flags)
    got_l = eng.resident_outputs()
    occ = R.occupancy_of(tl.pod_ident, len(tl.nodes))
    want_p = oracle.place(tl.nodes, occ, tl.n_domains, tl.n_namespaces, rq)
    ok_lws = got_l[0].tobytes() == lo.tobytes() and got_l[1].tobytes() == go.tobytes()
    ok_place = eng.resident_place_outputs().tobytes() == want_p.tobytes()
    got_d = eng.ds_resident_outputs()
    ok_ds = all(g.tobytes() == w.tobytes() for g, w in zip(got_d, oracle.sweep_ds(td.ds, roles, rr)))
    eng.close()
    line = {
        "workload": f"C3 x {a.scale} ({len(tl.lws)} LWS, {len(tl.groups)} groups, {len(tl.pod_state)} pods, {len(reqs)} requests, "
                    f"placement on) + C4 ({a.n_ds} DS, {len(td.revroles)} revision-role rows)",
        "ds_sweep_placement": a.label,
        "card": card,
        **{f"{m}_us_per_pass_blocks": [round(x, 2) for x in us[m]] for m in modes},
        **{f"{m}_us_per_pass_median": round(statistics.median(us[m]), 2) for m in modes},
        "patch_bytes_per_pass": int(np.mean([ps.h2d_bytes() + dp.h2d_bytes() for ps, dp in zip(lplan, dplan)])),
        **{f"{m}_changed_rows_per_pass": round(float(np.mean(rows_out[m])), 1) for m in modes},
        "passes_timed": {m: len(rows_out[m]) for m in modes},
        "outputs_equal_oracle": {"lws": ok_lws, "place": ok_place, "ds": ok_ds},
    }
    s = json.dumps(line)
    print(s)
    with open(os.path.join(a.out_dir, f"joint_tick_{a.label}.json"), "w") as f:
        f.write(s + "\n")
    if not (ok_lws and ok_place and ok_ds):
        sys.exit(1)


if __name__ == "__main__":
    main()
