"""Resident DisaggregatedSet tick (lwse_ds_resident_tick) at C4 against the stateless sweep.

    python profiles/ds_tick.py OUT_DIR [--blocks 4] [--seconds 1.0]

C4: 50 000 DisaggregatedSets of 2 roles (synth.make_ds).  Each tick carries the patches of one set of
a DS churn plan: 1 % of the (revision, role) rows apply the previous decisions / become ready, laid out
in the engine's patch arena.  In alternating blocks of at least ``--seconds`` each:
  * tick:  e2e time per ``lwse_ds_resident_tick`` (host clock; a tick returns when its lists are in
           pinned memory, so the clock covers the whole tick);
  * sweep: e2e time per ``lwse_sweep_ds_host`` on the same tables (upload of the three tables, sweep,
           download of every result row, stream synchronize).
Every shape is warmed first.  The last tick's committed outputs are checked against the oracle on
host mirrors.  Prints one JSON line and writes it to OUT_DIR/ds_tick.json, with the card's name and
power limit read in the same run.
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
    a = ap.parse_args()
    os.makedirs(a.out_dir, exist_ok=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]

    oracle.build()
    t = synth.make_ds(a.n_ds)
    eng = Engine(0)
    eng.ds_resident_load(t.ds, t.roles, t.revroles)
    eng.ds_resident_tick(eng.make_ds_tick())
    plan = churn.make_ds_plan(t, oracle.sweep_ds, 0.01, n_sets=8, frac_target=0.0)
    arena = eng.resident_arena(sum(ps.h2d_bytes() + 1024 for ps in plan) + 4096)
    cursor = 0

    def put(x):
        nonlocal cursor
        off = (cursor + 255) // 256 * 256
        view = arena[off: off + x.nbytes].view(x.dtype)
        view[...] = x
        cursor = off + x.nbytes
        return view

    ticks = [eng.make_ds_tick([(R.TABLE_DS_REVROLES, put(ps.rr_rows), put(ps.rr_vals))]) for ps in plan]
    outs = (R.aligned_empty(len(t.ds), R.DS_OUT), R.aligned_empty(len(t.roles), R.DS_ROLE_OUT),
            R.aligned_empty(len(t.revroles), R.DS_REVROLE_OUT))
    applied = 0
    rows_out = []

    def tick_block(seconds, record):
        nonlocal applied
        n, t0 = 0, time.perf_counter()
        while True:
            for tk in ticks:
                res = eng.ds_resident_tick(tk)
                if record:
                    rows_out.append(res["n_ds"] + res["n_roles"] + res["n_revroles"])
            n += len(ticks)
            applied += len(ticks)
            dt = time.perf_counter() - t0
            if dt >= seconds:
                return dt / n * 1e6

    def sweep_block(seconds):
        n, t0 = 0, time.perf_counter()
        while True:
            for _ in range(8):
                eng.sweep_ds_host(t.ds, t.roles, t.revroles, out=outs)
            n += 8
            dt = time.perf_counter() - t0
            if dt >= seconds:
                return dt / n * 1e6

    tick_block(0.2, False)  # warm both shapes
    sweep_block(0.2)
    tick_us, sweep_us = [], []
    for _ in range(a.blocks):
        tick_us.append(tick_block(a.seconds, True))
        sweep_us.append(sweep_block(a.seconds))

    # the last tick's state: the plan's sets applied cyclically, `applied` ticks in all
    roles, rr = t.roles.copy(), t.revroles.copy()
    for k in range(applied):
        churn.apply_ds_to_mirror(plan[k % len(plan)], roles, rr)
    want = oracle.sweep_ds(t.ds, roles, rr)
    got = eng.ds_resident_outputs()
    ok = all(g.tobytes() == w.tobytes() for g, w in zip(got, want))
    eng.close()
    line = {
        "workload": f"C4 resident DS tick ({a.n_ds} DS, 2 roles, {len(t.revroles)} revision-role rows)",
        "card": card,
        "tick_us_per_call_blocks": [round(x, 2) for x in tick_us],
        "sweep_ds_host_us_per_call_blocks": [round(x, 2) for x in sweep_us],
        "tick_us_median": round(statistics.median(tick_us), 2),
        "sweep_ds_host_us_median": round(statistics.median(sweep_us), 2),
        "patch_bytes_per_tick": int(np.mean([ps.h2d_bytes() for ps in plan])),
        "patched_revrole_rows_per_tick": int(np.mean([len(ps.rr_rows) for ps in plan])),
        "changed_rows_out_per_tick": round(float(np.mean(rows_out)), 1),
        "ticks_timed": len(rows_out),
        "sweep_ds_host_input_bytes": int(t.ds.nbytes + t.roles.nbytes + t.revroles.nbytes),
        "outputs_equal_oracle": ok,
    }
    s = json.dumps(line)
    print(s)
    with open(os.path.join(a.out_dir, "ds_tick.json"), "w") as f:
        f.write(s + "\n")
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
