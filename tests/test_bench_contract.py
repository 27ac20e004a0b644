"""The bench.py JSON line: the committed N=1 line of this round (profiles/r2_bench_line_n1.json) has
every key the contract names, and the reference arm — which runs on CPU — still prints its line.
--dump-outputs writes what the timed path computed in its last step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                       timeout=timeout)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])


def columns(records):
    """A record table as --dump-outputs writes it: float64, one column per field."""
    return np.stack([records[f] for f in records.dtype.names], axis=1).astype(np.float64)


def test_committed_bench_line_has_the_contract_keys():
    d = json.load(open(os.path.join(ROOT, "profiles", "r2_bench_line_n1.json")))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
        assert k in d, k
    assert d["config"]["workload"] == "C3" and d["n_gpus"] == 1 and d["higher_is_better"] is True
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert d["gpu_launches"] >= 3 * d["steps"]  # a device tick is four launches (fused, LWS pass, condense, namespace kernel)
    # the headline e2e is the pipelined resident tick; its latency (one tick at a time) and the churn variants are stated
    e = d["e2e"]
    assert e["ms_per_step"] > 0 and e["latency_ms_per_step"] >= e["ms_per_step"]
    assert abs(e["value"] - d["config"]["groups"] / (e["ms_per_step"] * 1e-3)) / e["value"] < 1e-6
    assert {"churn_1pct", "churn_10pct", "churn_100pct", "no_churn"} <= set(e["variants"])
    assert e["oracle_check"]["sweep_equals_oracle"] is True and e["oracle_check"]["placement_equals_spec_oracle"] is True
    assert d["oracle_check"]["sweep_equals_oracle"] is True
    assert d["roofline"]["traffic"] and d["roofline"]["traffic"] >= d["roofline"]["bytes_per_launch"]
    ref = json.load(open(os.path.join(ROOT, "profiles", "r2_bench_line_reference.json")))
    assert ref["impl"] == "reference" and ref["metric"] == d["metric"] and ref["unit"] == d["unit"]
    assert ref["config"]["groups"] == d["config"]["groups"] and ref["e2e"]["h2d_bytes_per_step"] == 0
    assert abs(d["value"] - d["config"]["groups"] / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6


def test_reference_arm_prints_its_line_on_cpu():
    line = run_bench("--impl", "reference", "--workload", "C2", "--steps", "2", "--warmup", "1")
    assert line["impl"] == "reference" and line["unit"] == "groups/s" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] in ("port", "reference")


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--dump-outputs writes the result tables of the last timed step, one float64 column per record
    field; the inputs are seeded, so a second run writes the same arrays."""
    from lws_b200 import records as R

    args = ("--impl", "reference", "--workload", "C2", "--steps", "2", "--warmup", "1", "--dump-outputs")
    line = run_bench(*args, str(tmp_path / "a"))
    run_bench(*args, str(tmp_path / "b"))
    for name, dt, rows in (("lws_out", R.LWS_OUT, line["config"]["lws"]), ("group_out", R.GROUP_OUT, line["config"]["groups"])):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float64 and a.shape == (rows, len(dt.names)), name
        assert np.array_equal(a, b), name


@pytest.mark.gpu
def test_dumped_outputs_are_the_tick_results(tmp_path):
    """--dump-outputs on the engine: the tables of the last timed tick equal the CPU oracle's on the
    same seeded cluster."""
    import oracle
    from lws_b200 import records as R
    from lws_b200 import synth

    run_bench("--workload", "C3", "--scale", "0.1", "--steps", "3", "--warmup", "1", "--e2e-steps", "10",
              "--dump-outputs", str(tmp_path), timeout=900)
    t = synth.make("C3", 0.1, seed=synth.SEED)
    reqs = t.place_requests()
    assert len(reqs) > 0
    lo, go, _ = oracle.sweep_lws(t.lws, t.groups, t.pod_state, t.pod_ident, t.nodes, flags=t.flags)
    po = oracle.place(t.nodes, R.occupancy_of(t.pod_ident, len(t.nodes)), t.n_domains, t.n_namespaces, reqs)
    for name, want in (("lws_out", lo), ("group_out", go), ("place_out", po)):
        assert np.array_equal(np.load(tmp_path / f"{name}.npy"), columns(want)), name
