#!/usr/bin/env python
"""Benchmark of the reconcile tick — BASELINE.json's metric on its config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C3|C3-steady|C2|C5|C4]
                    [--dump-outputs DIR]

metric   pod-group reconciles/sec: pod groups brought up to date / time of one tick (fused pod
         scan + group pass, LWS pass; the placement round when the workload has
         exclusive-topology groups).
workload BASELINE.json configs[2] ("C3"): 100k LWS x size 64 (100k groups, 6.3M pod rows), 10k
         nodes, topology-aware gang placement on for every group (200 namespaces, 5 % of the
         leaders unscheduled).  It fits one GPU, so N=1 runs exactly it; N>1 is weak scaling by
         default — every rank holds its own C3-sized shard of an N-times larger cluster (objects
         shard by LWS UID hash, no data-path collective for the sweep) — and `--scaling strong`
         shards the ONE C3 cluster over the ranks.
value    whole-job groups/s with the tables resident in HBM (CUDA events on the launching
         stream, max over ranks).  Inputs rotate through copies whose total size exceeds L2.
e2e      the same metric through the product path a controller uses, lwse_resident_tick():
         watch-event churn in (1 % of the pod state rows + scheduling events per tick, written
         into the engine's pinned arena), changed result rows out (pinned change lists), the
         full sweep and the placement round inside, HOST wall clock around the call.
         e2e.full_handover is the stateless path (lwse_reconcile_host: every table handed over
         every step).
roofline the dominant kernel alone: algorithmic bytes / its CUDA-event duration, against
         MEASURED_PEAKS.json's HBM copy bandwidth.
cpu_baseline  the CPU oracle (a port of the reference's Go arithmetic — the reference itself
         needs a Go toolchain, absent here) on one host core, full sweep.

--impl reference times that same oracle on the host threads as an event-driven controller: per
step it applies the same churn to its host tables and reconciles the dirty objects (rank 0 only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "pod-group reconciles/sec on 100k-group x 10k-node synthetic cluster"
UNIT = "groups/s"
L2_BYTES = 126 * 1024 * 1024
CHURN = 0.01        # share of the pod state rows that change per tick (the e2e workload)
CHURN_REQS = 0.01   # share of the placement requests that change sides per tick


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--e2e-steps", type=int, default=200)
    ap.add_argument("--exchange", default="lagged", choices=["lagged", "instep"],
                    help="multi-GPU occupancy exchange: 'lagged' = the round of tick s reads the snapshot every rank pushed "
                         "at tick s-1 (no rank waits for the slowest launch), 'instep' = it waits for this tick's pushes")
    ap.add_argument("--graph", action="store_true",
                    help="replay CUDA graphs instead of eager launches (measured slower: programmatic "
                         "dependent launch does not span graph replays)")
    ap.add_argument("--no-check", action="store_true", help="skip the oracle comparison of the outputs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result tables of the last one (rank 0's) as DIR/<table>.npy; "
                         "the inputs are seeded, so two builds run with the same arguments can be compared table by table")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


DUMP_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, tables):
    """Write each result table as <out_dir>/<name>.npy: float64, one row per record, one column per
    field in record order (every field is a 32-bit integer, so float64 holds it exactly).  Should the
    tables exceed DUMP_BYTES in all, each keeps the same share of its rows, drawn with a fixed seed,
    and <name>_rows.npy lists which."""
    arrays = {name: (np.stack([a[f] for f in a.dtype.names], axis=1) if a.dtype.names else a).astype(np.float64)
              for name, a in tables.items()}
    total = sum(a.nbytes for a in arrays.values())
    share = 1.0 if total <= DUMP_BYTES else DUMP_BYTES / (2 * total)  # the row indices cost at most as much again
    rng = np.random.default_rng(0)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if share < 1.0:
            rows = np.sort(rng.choice(len(a), int(len(a) * share), replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def make_tables(args, rank, world=1):
    """The rank's tables.  weak scaling: every rank its own cluster shard (own seed, own
    namespaces), all on the same nodes; strong scaling: the ONE cluster of seed 0 — its sweep
    sharded by LWS UID hash, its placement requests by namespace owner (exclusivity is per
    namespace, so whole namespaces are the unit of placement work)."""
    from lws_b200 import synth

    if args.scaling == "strong" and world > 1:
        from lws_b200 import distributed as D

        t = synth.make(args.workload, args.scale, seed=synth.SEED)
        s_lws, s_grp, s_pst, s_pid, lrows, _ = D.shard_lws_tables(t.lws, t.groups, t.pod_state, t.pod_ident, world)[rank]
        reqs, n_ns, _ = D.requests_of_rank(t.place_requests(), world, rank)
        shard = synth.Tables(profile=t.profile, lws=s_lws, groups=s_grp, pod_state=s_pst, pod_ident=s_pid, nodes=t.nodes,
                             n_domains=t.n_domains, flags=t.flags, ns_of_lws=t.ns_of_lws[lrows], n_namespaces=n_ns)
        shard.requests = reqs
        return shard
    t = synth.make(args.workload, args.scale, seed=synth.SEED + rank)
    t.requests = t.place_requests()
    return t


# --------------------------------------------------------------------------- #
# the CPU arm
# --------------------------------------------------------------------------- #
class CpuArm:
    """The reference's arithmetic (oracle port) as a controller would run it: host tables, the
    placement spec round, and — for the churn workload — event-driven reconciles of the dirty objects."""

    def __init__(self, t, threads):
        import oracle
        from lws_b200 import records as R

        self.o, self.R, self.t, self.threads = oracle, R, t, threads
        self.lws, self.groups = t.lws.copy(), t.groups.copy()
        self.pst, self.pid = t.pod_state.copy(), t.pod_ident
        self.reqs = getattr(t, "requests", None)
        if self.reqs is None:
            self.reqs = t.place_requests()
        self.reqs = self.reqs.copy()
        self.occ = R.occupancy_of(t.pod_ident, len(t.nodes))
        self.lws_out = R.aligned_empty(len(t.lws), R.LWS_OUT)
        self.group_out = R.aligned_empty(len(t.groups), R.GROUP_OUT)
        self.place_out = None

    def place(self):
        if len(self.reqs):
            self.place_out = self.o.place(self.t.nodes, self.occ, self.t.n_domains, self.t.n_namespaces, self.reqs,
                                          threads=self.threads)

    def full_step(self):
        lo, go, _ = self.o.sweep_lws(self.lws, self.groups, self.pst, self.pid, self.t.nodes, flags=self.t.flags,
                                     threads=self.threads)
        self.lws_out, self.group_out = lo, go
        self.place()

    def churn_step(self, ps):
        o, R = self.o, self.R
        o.apply_patch(self.pst, ps.pod_rows, ps.pod_vals)
        if len(ps.grp_rows):
            o.apply_patch(self.groups, ps.grp_rows, ps.grp_vals)
        if len(ps.req_rows):
            o.apply_patch(self.reqs, ps.req_rows, ps.req_vals)
        o.sweep_dirty(self.lws, self.groups, self.pst, self.pid, self.t.nodes, self.lws_out, self.group_out,
                      ps.dirty_groups, ps.dirty_lws, flags=self.t.flags, threads=self.threads)
        self.place()  # the placement spec has no incremental form: the round is solved again


def cpu_oracle_rate(t, threads, min_seconds=1.0, max_reps=50):
    """groups/s of the CPU oracle over the whole workload (full sweep + placement spec round)."""
    arm = CpuArm(t, threads)
    arm.full_step()  # warm
    reps, t0 = 0, time.perf_counter()
    while True:
        arm.full_step()
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds or reps >= max_reps:
            break
    return len(t.groups) * reps / dt, dt / reps, reps


def churn_plan(t, reqs, place_out, frac_pods=CHURN, frac_reqs=CHURN_REQS, n_sets=4, patch_groups=True):
    """The tick-by-tick event stream both arms digest (same seed: same events)."""
    from lws_b200 import churn
    from lws_b200 import records as R

    if frac_pods <= 0:
        return [churn.PatchSet(np.zeros(0, np.uint32), R.aligned_empty(0, R.POD_STATE))]
    return churn.make_plan(t, reqs if len(reqs) else None, place_out if len(reqs) else None, frac_pods,
                           frac_reqs if len(reqs) else 0.0, n_sets=n_sets, seed=11, patch_groups=patch_groups)


def run_reference(args):
    """The reference arm: the reference's CPU arithmetic (oracle port) on the host threads, driven
    by the same churn plan as the engine's e2e leg."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    if args.workload == "C4":
        return run_reference_ds(args)
    t = make_tables(args, 0, world)
    # the port spawns its worker threads per step; pick the thread count that is fastest on this
    # box (more threads than the memory system can feed only add spawn cost) — the baseline gets
    # the best configuration available to it
    probe = CpuArm(t, 1)
    probe.full_step()
    plan = churn_plan(t, probe.reqs, probe.place_out)
    best = None
    for cand in sorted({c for c in (1, 4, 8, 16, 32, 64, 128, host_threads()) if c <= host_threads()}):
        arm = CpuArm(t, cand)
        arm.full_step()
        arm.churn_step(plan[0])
        t0 = time.perf_counter()
        for k in range(4):
            arm.churn_step(plan[(k + 1) % len(plan)])
        dt = (time.perf_counter() - t0) / 4
        if best is None or dt < best[0]:
            best = (dt, cand)
    threads = best[1]
    arm = CpuArm(t, threads)
    arm.full_step()
    i = 0
    for _ in range(max(args.warmup, 1)):
        arm.churn_step(plan[i % len(plan)])
        i += 1
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arm.churn_step(plan[i % len(plan)])
        i += 1
    dt = time.perf_counter() - t0
    value = len(t.groups) * args.steps / dt
    if args.dump_outputs:
        outs = {"lws_out": arm.lws_out, "group_out": arm.group_out}
        if arm.place_out is not None:
            outs["place_out"] = arm.place_out
        dump_outputs(args.dump_outputs, outs)
    # the same arm sweeping everything every step (no event source): reported beside it
    full = CpuArm(t, threads)
    full.full_step()
    t1 = time.perf_counter()
    n_full = max(3, min(args.steps, 10))
    for _ in range(n_full):
        full.full_step()
    full_dt = (time.perf_counter() - t1) / n_full
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u8/int32/u64 (integer compare)",
        "data": "synthetic", "config": {**t.describe(), "churn": {"pod_state_rows": CHURN, "placement_requests": CHURN_REQS}},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"full {t.profile.name} cluster per step as an event-driven controller: apply the step's "
                                   f"{len(plan[0].pod_rows)} pod-status / {len(plan[0].req_rows)} scheduling events to the host "
                                   f"tables, reconcile the {len(plan[0].dirty_groups)} dirty groups / {len(plan[0].dirty_lws)} "
                                   f"dirty objects on {threads} of {host_threads()} host threads (the fastest count on this "
                                   f"box), solve the placement spec round; {args.steps} steps"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "full_sweep": {"value": len(t.groups) / full_dt, "unit": UNIT, "ms_per_step": full_dt * 1e3, "cores": threads,
                       "note": "the same port sweeping every object every step (no event source)"},
        "note": "CPU port of the reference's Go arithmetic (no Go toolchain here); excludes the "
                "informer-cache List/DeepCopy and API round-trips that dominate the real reconciler",
    }
    print(json.dumps(line), flush=True)


def run_reference_ds(args):
    import oracle
    from lws_b200 import synth

    n_ds = max(1, int(round(50_000 * args.scale)))
    d = synth.make_ds(n_ds, (2,))
    oracle.sweep_ds(d.ds, d.roles, d.revroles)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        outs = oracle.sweep_ds(d.ds, d.roles, d.revroles)
    dt = time.perf_counter() - t0
    value = n_ds * args.steps / dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("ds_out", "ds_role_out", "ds_revrole_out"), outs)))
    print(json.dumps({
        "impl": "reference", "metric": "DisaggregatedSet reconciles/sec (2-role rollout partition calc)", "value": value,
        "unit": "sets/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "int32 (float64 planner in the port)", "data": "synthetic",
        "config": {"workload": "C4", "sets": n_ds, "roles": 2},
        "cpu_baseline": {"value": value, "unit": "sets/s", "cores": 1, "kind": "port", "sample": f"{n_ds} sets per step"},
        "e2e": {"value": value, "unit": "sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


# --------------------------------------------------------------------------- #
# C4: DisaggregatedSet sweep
# --------------------------------------------------------------------------- #
def run_ours_ds(args):
    import torch
    import torch.distributed as dist

    import oracle
    from lws_b200 import records as R
    from lws_b200 import synth
    from lws_b200.engine import Engine

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_total = max(world, int(round(50_000 * args.scale)))
    # a DS and its child LWS rows shard together by hash(DS.UID): rank r sweeps its share
    n_ds = n_total // world if args.scaling == "strong" else n_total
    d = synth.make_ds(n_ds, (2,), seed=synth.SEED + rank)
    eng = Engine(local_rank)

    def up(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)

    copies = 8
    sets = [dict(ds=up(d.ds), ro=up(d.roles), rr=up(d.revroles),
                 o1=torch.empty(len(d.ds) * R.DS_OUT.itemsize, dtype=torch.uint8, device=dev),
                 o2=torch.empty(len(d.roles) * R.DS_ROLE_OUT.itemsize, dtype=torch.uint8, device=dev),
                 o3=torch.empty(len(d.revroles) * 4, dtype=torch.uint8, device=dev)) for _ in range(copies)]
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)

    def step(i):
        s = sets[i % copies]
        eng.sweep_ds_device(s["ds"], len(d.ds), s["ro"], len(d.roles), s["rr"], len(d.revroles), s["o1"], s["o2"], s["o3"],
                            stream=eng.stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    W = max(args.warmup, 3)
    for i in range(W):
        step(i)
    barrier()
    with ClockSampler(local_rank) as clk:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.launch_count
        with torch.cuda.stream(stream):
            e0.record(stream)
            for i in range(args.steps):
                step(i)
            e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1) / args.steps
        launches = eng.launch_count - l0
        if args.dump_outputs and rank == 0:
            last = sets[(args.steps - 1) % copies]
            dump_outputs(args.dump_outputs, {"ds_out": last["o1"].cpu().numpy().view(R.DS_OUT),
                                             "ds_role_out": last["o2"].cpu().numpy().view(R.DS_ROLE_OUT),
                                             "ds_revrole_out": last["o3"].cpu().numpy().view(R.DS_REVROLE_OUT)})
        for i in range(20000):
            step(i)
        torch.cuda.synchronize()
    # e2e: host tables in, host results out — page-locked on both sides, as the contract asks
    def pinned(a, dtype=None, n=None):
        dtype = a.dtype if dtype is None else dtype
        n = len(a) if n is None else n
        ten = torch.empty(max(n * dtype.itemsize, 16), dtype=torch.uint8).pin_memory()
        view = ten.numpy()[: n * dtype.itemsize].view(dtype)
        if a is not None:
            view[...] = a
        return ten, view

    keep = [pinned(d.ds), pinned(d.roles), pinned(d.revroles), pinned(None, R.DS_OUT, len(d.ds)),
            pinned(None, R.DS_ROLE_OUT, len(d.roles)), pinned(None, R.DS_REVROLE_OUT, len(d.revroles))]
    h_ds, h_ro, h_rr, h_o1, h_o2, h_o3 = [v for _, v in keep]

    def e2e():
        return eng.sweep_ds_host(h_ds, h_ro, h_rr, out=(h_o1, h_o2, h_o3))

    got = e2e()
    barrier()
    t0 = time.perf_counter()
    n_e2e = 20
    for _ in range(n_e2e):
        e2e()
    e2e_s = (time.perf_counter() - t0) / n_e2e
    want = oracle.sweep_ds(d.ds, d.roles, d.revroles)
    ok = all(a.tobytes() == b.tobytes() for a, b in zip(got, want))
    if not ok:
        raise SystemExit("bench.py: DS sweep differs from the oracle")
    stats = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(n_ds)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms, e2e_ms = [float(x) for x in stats.tolist()]
    if rank == 0:
        peak, peak_src = measured_peak()
        algo = d.algorithmic_bytes()
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 1.0:
            oracle.sweep_ds(d.ds, d.roles, d.revroles)
            reps += 1
        cpu = n_ds * reps / (time.perf_counter() - t0)
        print(json.dumps({
            "metric": "DisaggregatedSet reconciles/sec (2-role rollout partition calc)", "value": float(tot.item()) / (ms * 1e-3),
            "unit": "sets/s", "n_gpus": world, "steps": args.steps, "warmup": W, "ms_per_step": ms,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int32/int64", "data": "synthetic",
            "config": {"workload": "C4", "sets_per_rank": n_ds, "roles": 2, "revision_role_rows": int(len(d.revroles)),
                       "parallelism": f"shard-by-ds-uid x{world}", "l2": f"{copies} rotating copies (tables are {algo / 1e6:.1f} MB: L2-resident by size — launch-bound)"},
            "e2e": {"value": float(tot.item()) / (e2e_ms * 1e-3), "unit": "sets/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(d.ds.nbytes + d.roles.nbytes + d.revroles.nbytes),
                    "d2h_bytes_per_step": int(len(d.ds) * 16 + len(d.roles) * 8 + len(d.revroles) * 4),
                    "api": "lwse_sweep_ds_host, page-locked host tables and result rows"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "ds_sweep_kernel", "achieved": algo / (ms * 1e-3) / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": algo / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                         "bytes_per_launch": int(algo), "peak_source": peak_src,
                         "note": "7 MB per launch: the kernel is launch / latency bound, not HBM bound"},
            "cpu_baseline": {"value": cpu, "unit": "sets/s", "cores": 1, "kind": "port", "sample": f"{n_ds} sets x{reps}"},
            "oracle_check": {"outputs_equal_oracle": True},
            "clocks": clk.summary()}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------- #
# the engine
# --------------------------------------------------------------------------- #
def run_ours(args):
    import torch
    import torch.distributed as dist

    from lws_b200 import churn
    from lws_b200 import records as R
    from lws_b200.engine import Engine

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU path to benchmark")
    if args.workload == "C4":
        return run_ours_ds(args)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    t = make_tables(args, rank, world)
    eng = Engine(local_rank)
    eng.upload_nodes(t.nodes, t.n_domains)
    n_lws, n_grp, n_pod, n_nodes = len(t.lws), len(t.groups), len(t.pod_state), len(t.nodes)
    n_ns = t.n_namespaces
    algo_bytes = t.algorithmic_bytes()
    # placement: one request per group of an exclusive-topology object; the per-node occupancy of
    # this shard's pods is a resident input column (the resident engine maintains it itself)
    reqs = t.requests
    n_req = len(reqs)
    place_on = n_req > 0
    occ_host = R.occupancy_of(t.pod_ident, n_nodes)  # this rank's pods
    # the encoder lays the requests out grouped by namespace: the engine then gives every namespace its own CTA
    grouped = n_req > 0 and bool(np.all(np.diff(reqs["ns"].astype(np.int64)) >= 0))
    place_flags = R.SWEEP_PLACE_GROUPED if (grouped and world == 1) else 0
    occ_sum = occ_host
    if world > 1:  # every rank's pods load the same nodes: the rounds see the sum (exchanged on the device per tick)
        tot = torch.from_numpy(occ_host.astype(np.int64)).to(dev)
        dist.all_reduce(tot)
        occ_sum = tot.cpu().numpy().astype(np.uint32)
        anyreq = torch.tensor([n_req], dtype=torch.int64, device=dev)
        dist.all_reduce(anyreq, op=dist.ReduceOp.MAX)
        place_on = int(anyreq.item()) > 0

    # ---- resident copies, rotated so that the working set exceeds L2 ----
    copies = max(2, int(np.ceil(2.5 * L2_BYTES / algo_bytes)) + 1)  # bytes a sweep touches x copies > 2.5 x L2

    def up(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)

    sets = []
    for _ in range(copies):
        sets.append(dict(
            lws=up(t.lws), grp=up(t.groups), pst=up(t.pod_state), pid=up(t.pod_ident),
            lo=torch.empty(n_lws * R.LWS_OUT.itemsize, dtype=torch.uint8, device=dev),
            go=torch.empty(n_grp * R.GROUP_OUT.itemsize, dtype=torch.uint8, device=dev)))
    from lws_b200 import distributed as D

    d_occ = torch.from_numpy(D.padded_occupancy(occ_host).view(np.int32)).to(dev)
    d_reqs = up(reqs) if n_req else torch.zeros(32, dtype=torch.uint8, device=dev)
    d_pout = torch.empty(max(n_req, 1) * R.PLACE_OUT.itemsize, dtype=torch.uint8, device=dev)
    xflags = 0
    if world > 1 and place_on:
        # multi-GPU: requests are local to the rank (own namespaces), the per-node occupancy is shared —
        # each tick the rank's counters go to every peer with NVLink peer stores + flags (no collective
        # library on the data path), lagged by one tick so that no rank waits for the slowest launch
        D.connect_exchange(eng, 0, world, rank, device=dev)
        xflags = R.EXCHANGE_LAGGED if args.exchange == "lagged" else 0

    # time on the stream the kernels are launched on: the engine's own stream
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)
    sptr = eng.stream

    def sweep(i, flags):
        s = sets[i % copies]
        eng.sweep_lws_device(s["lws"], n_lws, s["grp"], n_grp, s["pst"], s["pid"], n_pod, s["lo"], s["go"], None,
                             flags=flags, stream=sptr)

    descs = {}

    def desc(i, flags):
        k = (i % copies, flags)
        if k not in descs:
            s = sets[i % copies]
            descs[k] = eng.device_tables(s["lws"], n_lws, s["grp"], n_grp, s["pst"], s["pid"], n_pod, s["lo"],
                                         s["go"], None, flags=flags)
        return descs[k]

    def step(i, flags):
        """One C call per tick: sweep on the engine's stream, the placement branch on its side stream."""
        if world == 1:
            eng.reconcile_device(desc(i, flags), d_reqs, n_req if place_on else 0, d_occ, n_ns, d_pout, stream=sptr)
        elif place_on:
            eng.reconcile_shared_device(desc(i, flags), d_reqs, n_req, d_occ, n_ns, d_pout, flags=xflags, stream=sptr)
        else:
            sweep(i, flags)

    def place_alone():
        if world == 1:
            if grouped:
                eng.place_grouped_device(d_reqs, n_req, d_occ, n_ns, d_pout, stream=sptr)
            else:
                eng.place_device(d_reqs, n_req, d_occ, n_ns, d_pout, stream=sptr)
        else:
            eng.reconcile_shared_device(None, d_reqs, n_req, d_occ, n_ns, d_pout, flags=xflags, stream=sptr)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    use_graph = args.graph and world == 1

    def timed(fn, steps, warmup):
        """ms per call of fn(i) over `steps` calls, CUDA events on the launching stream."""
        for i in range(warmup):
            fn(i)
        barrier()
        graphs = None
        if use_graph:
            ok = 1
            try:
                graphs = []
                for k in range(copies):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=stream, capture_error_mode="thread_local"):
                        fn(k)
                    graphs.append(g)
            except Exception as exc:  # pragma: no cover
                print(f"bench.py[{rank}]: graph capture failed ({exc}); timing eager launches", file=sys.stderr)
                ok = 0
            if world > 1:
                flag = torch.tensor([ok], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                ok = int(flag.item())
            if not ok:
                graphs = None
            torch.cuda.synchronize()
        run = (lambda i: graphs[i % copies].replay()) if graphs else fn
        with torch.cuda.stream(stream):
            for i in range(3):
                run(i)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = eng.launch_count
            e0.record(stream)
            h0 = time.perf_counter()
            for i in range(steps):
                run(i)
            timed.host_ms = (time.perf_counter() - h0) * 1e3 / steps
            e1.record(stream)
        barrier()
        launched = eng.launch_count - l0
        if graphs:
            launched = timed.per_call.get(fn, 0) * steps
        return e0.elapsed_time(e1) / steps, launched

    timed.per_call = {}

    def count_launches(fn):
        l0 = eng.launch_count
        fn(0)
        torch.cuda.synchronize()
        timed.per_call[fn] = eng.launch_count - l0

    SCAN_ONLY = R.SWEEP_SKIP_GROUP_PASS | R.SWEEP_SKIP_LWS_PASS
    GROUP_ONLY = R.SWEEP_SKIP_POD_SCAN | R.SWEEP_SKIP_LWS_PASS
    LWS_ONLY = R.SWEEP_SKIP_POD_SCAN | R.SWEEP_SKIP_GROUP_PASS
    W = max(args.warmup, 3)
    full_step = lambda i: step(i, t.flags | place_flags)  # noqa: E731
    count_launches(full_step)
    with ClockSampler(local_rank) as clk:
        ms_step, launches = timed(full_step, args.steps, W)
        host_ms_step = getattr(timed, "host_ms", None)
        if args.dump_outputs and rank == 0:  # before the passes below write into the same buffers
            last = sets[(args.steps - 1) % copies]
            outs = {"lws_out": last["lo"].cpu().numpy().view(R.LWS_OUT),
                    "group_out": last["go"].cpu().numpy().view(R.GROUP_OUT)}
            if place_on and n_req:
                outs["place_out"] = d_pout.cpu().numpy()[: n_req * R.PLACE_OUT.itemsize].view(R.PLACE_OUT)
            dump_outputs(args.dump_outputs, outs)
        # each pass alone (same rotating inputs), for the per-kernel roofline
        ms_sweep, _ = timed(lambda i: sweep(i, t.flags), args.steps, 3)
        ms_fused, _ = timed(lambda i: sweep(i, t.flags | R.SWEEP_SKIP_LWS_PASS), args.steps, 3)
        ms_lws, _ = timed(lambda i: sweep(i, t.flags | LWS_ONLY), args.steps, 3)
        ms_scan, _ = timed(lambda i: sweep(i, t.flags | SCAN_ONLY), args.steps, 3)
        ms_group, _ = timed(lambda i: sweep(i, t.flags | GROUP_ONLY), args.steps, 3)
        ms_place = timed(lambda i: place_alone(), args.steps, 3)[0] if place_on else 0.0
        # keep the GPU under the same load long enough for nvidia-smi to sample clocks
        n_load = torch.tensor([ms_step], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(n_load, op=dist.ReduceOp.MAX)
        n_load = int(min(max(1000.0 / max(float(n_load.item()), 1e-3), 2000), 60000)) // 100
        i = 0
        for _ in range(n_load):
            for _ in range(100):
                step(i, t.flags | place_flags)
                i += 1
            torch.cuda.synchronize()
        # the placement round alone, in each of its forms (same rows; checked against the oracle below)
        forms = {}
        if place_on and world == 1:
            d_pout2 = torch.empty_like(d_pout)

            def form_fn(kind):
                if kind == "general":
                    return lambda i: eng.place_device(d_reqs, n_req, d_occ, n_ns, d_pout2, stream=sptr)
                fl = R.SWEEP_PLACE_SCAN if kind == "scan" else 0
                return lambda i: eng.place_grouped_device(d_reqs, n_req, d_occ, n_ns, d_pout2, flags=fl, stream=sptr)

            for kind in (("general", "grouped", "scan") if grouped else ("general",)):
                ms_k, _ = timed(form_fn(kind), max(10, args.steps // 2), 3)
                forms[kind] = {"ms": ms_k}
                if kind != "general":
                    r_k, scans = eng.place_grouped_device(d_reqs, n_req, d_occ, n_ns, d_pout2, stream=sptr, want_rounds=True,
                                                          flags=R.SWEEP_PLACE_SCAN if kind == "scan" else 0)
                    forms[kind].update({"rounds": int(r_k), "request_scans": int(scans)})
    clocks = clk.summary()
    torch.cuda.synchronize()
    if place_on and world == 1:
        rounds = (eng.place_grouped_device(d_reqs, n_req, d_occ, n_ns, d_pout, stream=sptr, want_rounds=True)[0] if grouped
                  else eng.place_device(d_reqs, n_req, d_occ, n_ns, d_pout, stream=sptr, want_rounds=True))
    else:
        rounds = None
    torch.cuda.synchronize()

    # ---- outputs of the device-resident tick against the oracle (outside the timed region) ----
    check = {"done": False}
    if not args.no_check:
        import oracle

        want_lo, want_go, _ = oracle.sweep_lws(t.lws, t.groups, t.pod_state, t.pod_ident, t.nodes, flags=t.flags,
                                               threads=min(host_threads(), 32))
        step(0, t.flags | place_flags)
        torch.cuda.synchronize()
        ok = (sets[0]["lo"].cpu().numpy().tobytes() == want_lo.tobytes()
              and sets[0]["go"].cpu().numpy().tobytes() == want_go.tobytes())
        place_ok = None
        if place_on:
            if world == 1:
                want_po = oracle.place(t.nodes, occ_host, t.n_domains, n_ns, reqs, threads=min(host_threads(), 32))
                place_ok = d_pout.cpu().numpy()[: n_req * R.PLACE_OUT.itemsize].tobytes() == want_po.tobytes()
                for kind in forms:  # every form of the round gives the same rows
                    form_fn(kind)(0)
                    torch.cuda.synchronize()
                    forms[kind]["equals_spec_oracle"] = bool(
                        d_pout2.cpu().numpy()[: n_req * R.PLACE_OUT.itemsize].tobytes() == want_po.tobytes())
                    place_ok = place_ok and forms[kind]["equals_spec_oracle"]
            else:  # this rank's requests against the occupancy of every rank's pods (static here: lag or not, the same sum)
                want_po = oracle.place(t.nodes, occ_sum, t.n_domains, n_ns, reqs, threads=min(host_threads(), 32))
                place_ok = d_pout.cpu().numpy()[: n_req * R.PLACE_OUT.itemsize].tobytes() == want_po.tobytes()
        check = {"done": True, "sweep_equals_oracle": bool(ok), "placement_equals_spec_oracle": place_ok}
        if not ok or place_ok is False:
            raise SystemExit(f"bench.py[{rank}]: device-resident tick differs from the oracle: {check}")

    # ---- end to end (1): the resident tick, the product path ----
    def pinned(a):
        ten = torch.empty(max(a.nbytes, 16), dtype=torch.uint8).pin_memory()
        view = ten.numpy()[: a.nbytes].view(a.dtype)
        view[...] = a
        return ten, view

    def wall(fn, reps, warm=3):
        for _ in range(warm):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        return (time.perf_counter() - t0) / reps, r

    eng.resident_load(t.lws, t.groups, t.pod_state, t.pod_ident)
    tick_flags = t.flags
    if n_req:
        eng.resident_place_load(reqs, n_ns)
        tick_flags |= R.TICK_PLACE
        if world > 1:
            tick_flags |= R.TICK_SHARED_OCCUPANCY | xflags
    first = eng.resident_tick(eng.make_tick((), tick_flags))  # every row is reported once
    base_place = eng.resident_place_outputs() if n_req else None
    e2e_variants = {}
    mirror = None
    for name, frac_p, frac_r in (("churn_1pct", CHURN, CHURN_REQS), ("churn_10pct", 0.10, CHURN_REQS),
                                 ("churn_100pct", 1.0, CHURN_REQS), ("no_churn", 0.0, 0.0)):
        if name != "churn_1pct" and world > 1:
            continue
        plan = churn_plan(t, reqs, base_place, frac_p, frac_r, patch_groups=not (args.scaling == "strong" and world > 1))
        # every variant starts from the loaded tables
        eng.resident_load(t.lws, t.groups, t.pod_state, t.pod_ident)
        if n_req:
            eng.resident_place_load(reqs, n_ns)
        ap = churn.ArenaPlan(eng, plan, tick_flags)
        eng.resident_tick(eng.make_tick((), tick_flags))
        state = {"i": 0, "d2h": 0, "rows": (0, 0, 0)}

        def tick_step(ap=ap, state=state):
            r = eng.resident_tick(ap.ticks[state["i"] % len(ap.ticks)])
            state["i"] += 1
            state["rows"] = (r["n_lws"], r["n_groups"], r["n_place"])
            return r

        reps = args.e2e_steps if frac_p < 0.5 else max(20, args.e2e_steps // 5)
        reps = (reps + len(plan) - 1) // len(plan) * len(plan)  # whole cycles: every rank ends on the same set
        sec, last = wall(tick_step, reps, warm=len(plan))
        changed = state["rows"]

        def pipelined(n_ticks, ap=ap, state=state):
            """The same ticks through lwse_resident_tick_submit / _wait, two in flight: while the GPU
            sweeps tick k the copy engine moves the patches of tick k+1; every tick's results are
            waited for and read inside the timed region."""
            barrier()
            t0 = time.perf_counter()
            eng.resident_tick_submit(ap.ticks[state["i"] % len(ap.ticks)])
            state["i"] += 1
            for _ in range(n_ticks - 1):
                eng.resident_tick_submit(ap.ticks[state["i"] % len(ap.ticks)])
                state["i"] += 1
                r = eng.resident_tick_wait()
            r = eng.resident_tick_wait()
            state["rows_pipelined"] = (r["n_lws"], r["n_groups"], r["n_place"])
            return (time.perf_counter() - t0) / n_ticks

        pipelined(len(plan))  # warm-up
        sec_pipe = pipelined(reps)
        d2h = changed[0] * (4 + R.LWS_OUT.itemsize) + changed[1] * (4 + R.GROUP_OUT.itemsize) + changed[2] * (4 + R.PLACE_OUT.itemsize) + 28
        e2e_variants[name] = {"ms_per_step": sec * 1e3, "pipelined_ms_per_step": sec_pipe * 1e3, "h2d_bytes_per_step": int(np.mean(ap.h2d_bytes)),
                              "d2h_bytes_per_step": int(d2h), "changed_rows_last_step": {"lws": changed[0], "groups": changed[1], "placement": changed[2]},
                              "pod_rows_per_step": int(len(plan[0].pod_rows)), "request_rows_per_step": int(len(plan[0].req_rows)),
                              "placement_rounds": int(last["rounds"])}
        if name == "churn_1pct" and not args.no_check:
            # replay the same ticks on host mirrors, run the oracle on them, compare every row
            import oracle

            m_pst, m_grp, m_req = t.pod_state.copy(), t.groups.copy(), (reqs.copy() if n_req else None)
            for k in range(state["i"]):
                churn.apply_to_mirror(plan[k % len(plan)], m_pst, m_grp, m_req)
            w_lo, w_go, _ = oracle.sweep_lws(t.lws, m_grp, m_pst, t.pod_ident, t.nodes, flags=t.flags,
                                             threads=min(host_threads(), 32))
            g_lo, g_go = eng.resident_outputs()
            ok = g_lo.tobytes() == w_lo.tobytes() and g_go.tobytes() == w_go.tobytes()
            pl_ok = None
            if n_req:
                w_po = oracle.place(t.nodes, occ_sum, t.n_domains, n_ns, m_req, threads=min(host_threads(), 32))
                pl_ok = eng.resident_place_outputs().tobytes() == w_po.tobytes()
            mirror = {"ticks_replayed": state["i"], "sweep_equals_oracle": bool(ok), "placement_equals_spec_oracle": pl_ok}
            if not ok or pl_ok is False:
                raise SystemExit(f"bench.py[{rank}]: resident tick differs from the oracle after {state['i']} ticks: {mirror}")
    e2e_tick_s = e2e_variants["churn_1pct"]["pipelined_ms_per_step"] * 1e-3  # the headline: two ticks in flight
    e2e_serial_s = e2e_variants["churn_1pct"]["ms_per_step"] * 1e-3           # one tick at a time (its latency)

    # ---- end to end (2): full handover through the stateless host entry point ----
    full = None
    if world == 1:
        keep, h = [], {}
        for name, arr in (("lws", t.lws), ("groups", t.groups), ("pst", t.pod_state), ("pid", t.pod_ident),
                          ("lo", R.aligned_empty(n_lws, R.LWS_OUT)), ("go", R.aligned_empty(n_grp, R.GROUP_OUT)),
                          ("reqs", reqs), ("occ", occ_host), ("po", R.aligned_empty(max(n_req, 1), R.PLACE_OUT))):
            ten, view = pinned(arr)
            keep.append(ten)
            h[name] = view

        def handover():
            if n_req:
                # (the encoder emits the request table grouped by namespace: promised, checked on the device)
                return eng.reconcile_host(h["lws"], h["groups"], h["pst"], h["pid"], h["reqs"], h["occ"], n_ns,
                                          flags=t.flags | (R.SWEEP_PLACE_GROUPED if grouped else 0), out=(h["lo"], h["go"]),
                                          place_out=h["po"])[2]
            eng.sweep_lws_host(h["lws"], h["groups"], h["pst"], h["pid"], flags=t.flags, out=(h["lo"], h["go"]))

        sec, _ = wall(handover, max(10, args.e2e_steps // 10))
        ev = t.event_pods()
        full = {"value": n_grp / sec, "unit": UNIT, "ms_per_step": sec * 1e3,
                "h2d_bytes_per_step": int(t.lws.nbytes + t.groups.nbytes + t.pod_state.nbytes + ev * R.POD_IDENT.itemsize
                                          + reqs.nbytes + occ_host.nbytes),
                "d2h_bytes_per_step": int(n_lws * R.LWS_OUT.itemsize + n_grp * R.GROUP_OUT.itemsize + n_req * R.PLACE_OUT.itemsize),
                "api": "lwse_reconcile_host: every table handed over every step (pinned host tables); state bytes, group and "
                       f"LWS rows uploaded, identity rows of the {ev} event pods read in place over PCIe"}

    if world > 1 and place_on:  # a timed-out wait (a rank fell behind by more than 2 s or is gone) invalidates the run
        xerr = torch.tensor([eng.exchange_status()], device=dev)
        dist.all_reduce(xerr, op=dist.ReduceOp.MAX)
        if int(xerr.item()) != 0:
            raise SystemExit(f"bench.py[{rank}]: a peer-exchange wait timed out")
    # ---- max over ranks ----
    stats = torch.tensor([ms_step, ms_group, e2e_tick_s * 1e3, ms_scan, ms_lws, ms_place, ms_sweep, ms_fused, e2e_serial_s * 1e3],
                         dtype=torch.float64, device=dev)
    groups = torch.tensor([float(n_grp)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(groups, op=dist.ReduceOp.SUM)
    ms_step, ms_group, e2e_ms, ms_scan, ms_lws, ms_place, ms_sweep, ms_fused, e2e_serial_ms = [float(x) for x in stats.tolist()]
    total_groups = float(groups.item())

    if rank == 0:
        peak, peak_src = measured_peak()
        ev = t.event_pods()
        words = (n_pod + 31) // 32
        group_rows = n_grp * (R.GROUP_REC.itemsize + R.GROUP_OUT.itemsize + 1) + n_lws * 16
        avg_pods = (n_pod + max(n_grp, 1) - 1) // max(n_grp, 1)
        fused_on = 16 <= avg_pods <= 256  # the engine's rule (lwse_lws_kernels.cu launch_lws_sweep)
        passes = {
            # algorithmic bytes per launch: rows read once + rows written once.  A sweep is the fused
            # scan + group kernel followed by the LWS pass (small groups); the three-kernel form
            # (large groups) is timed beside it.
            "group_fused_kernel": (n_pod * 1 + group_rows + ev * (1 + R.POD_IDENT.itemsize), ms_fused),
            "lws_sweep_kernel": (n_lws * (R.LWS_REC.itemsize + R.LWS_OUT.itemsize) + n_grp * 1, ms_lws),
            "pod_scan_kernel": (n_pod * 1 + 2 * words * 4, ms_scan),
            "group_sweep_kernel": (group_rows + 2 * words * 4 + ev * (1 + R.POD_IDENT.itemsize), ms_group),
        }
        in_step = ("group_fused_kernel", "lws_sweep_kernel") if fused_on else (
            "pod_scan_kernel", "group_sweep_kernel", "lws_sweep_kernel")
        traffic = None
        try:  # per-launch DRAM bytes of the committed ncu capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            if t.profile.name == tj.get("workload", "C3") and args.scale == 1.0:
                traffic = tj["dram_bytes_per_launch"]
        except Exception:
            pass
        dom = max(in_step, key=lambda k: passes[k][1])
        dom_bytes, dom_ms = passes[dom]
        achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
        cpu_rate, cpu_s, cpu_reps = cpu_oracle_rate(t, 1)
        tick = e2e_variants["churn_1pct"]
        pair_evals = None
        if place_on and world == 1 and "scan" in forms:
            unp = int((reqs["leader_node"] == R.NONE).sum())
            sc = forms["scan"]
            pairs = sc["request_scans"] * n_nodes
            pair_evals = {"form": "scan (lwse_place_grouped_device, LWSE_SWEEP_PLACE_SCAN): every (request, node) pair scored "
                                  "from the TMA-staged node table", "unpinned_requests": unp, "nodes": n_nodes,
                          "request_scans": sc["request_scans"], "pairs_per_call": int(pairs), "ms_per_call": sc["ms"],
                          "pair_evals_per_s": pairs / (sc["ms"] * 1e-3),
                          "note": "ms includes the condense kernel and the 93k pinned claims of the same call"}
        line = {
            "metric": METRIC, "value": total_groups / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": W, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u8/int32/u64 (integer compare)", "data": "synthetic",
            "config": {**t.describe(), "parallelism": f"shard-by-uid x{world} ({args.scaling})",
                       "placement": {"requests_per_rank": int(n_req), "unpinned": int((reqs['leader_node'] == R.NONE).sum()) if n_req else 0,
                                     "namespaces": int(n_ns), "rounds": rounds, "grouped_by_namespace": bool(grouped),
                                     "forms": forms, "pair_evals": pair_evals,
                                     "exchange": (f"per tick the rank's occupancy counters ({n_nodes * 4} B) to every peer with NVLink peer stores + "
                                                  f"flags (lwse_reconcile_shared_device, {args.exchange}); requests are rank-local (ranks own "
                                                  "namespaces); no collective library on the data path") if (world > 1 and place_on) else "none"},
                       "launch": ("CUDA graph replay") if use_graph else "eager launches, programmatic dependent launch",
                       "step": ("one lwse_reconcile_device call per tick: fused pod scan + group pass, LWS pass, placement round concurrently on the engine's side stream" if world == 1 else
                                "one lwse_reconcile_shared_device call per tick and rank: sweep of the shard ∥ (occupancy push, placement round over the rank's namespaces)"),
                       "l2": f"inputs rotate over {copies} resident copies ({copies * algo_bytes / 1e6:.0f} MB > L2)"},
            "e2e": {"value": total_groups / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                    "latency_ms_per_step": e2e_serial_ms,
                    "h2d_bytes_per_step": tick["h2d_bytes_per_step"], "d2h_bytes_per_step": tick["d2h_bytes_per_step"],
                    "api": "lwse_resident_tick_submit / _wait, two ticks in flight (the work queue keeps flowing: while the GPU "
                           "sweeps tick k the copy engine moves the patches of tick k+1).  Per step, all inside the timed region: "
                           "the watch-event churn (row patches in the engine's pinned arena) copied host->device and scattered, "
                           "full sweep + placement round, the changed result rows copied by the publish kernel into pinned change "
                           "lists, the host waits for every tick's sequence word and reads its counts.  latency_ms_per_step = the "
                           "same ticks one at a time through lwse_resident_tick (submit + wait)",
                    "churn": {"pod_state_rows": CHURN, "placement_requests": CHURN_REQS},
                    "timing": "host wall clock (time.perf_counter) around the calls, max over ranks",
                    "variants": e2e_variants, "full_handover": full, "oracle_check": mirror},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": (traffic or {}).get(dom),
                         "bytes_per_launch": int(dom_bytes), "ms_per_launch": dom_ms, "peak_source": peak_src,
                         "timing": "back-to-back launches of the kernel alone (programmatic dependent launch lets "
                                   "consecutive launches overlap their prologues), CUDA events",
                         "passes": {k: {"bytes": int(v[0]), "ms": v[1], "gbs": v[0] / (v[1] * 1e-3) / 1e9,
                                        "frac": v[0] / (v[1] * 1e-3) / 1e9 / peak, "in_step": k in in_step}
                                    for k, v in passes.items()}},
            "ms_sweep_only": ms_sweep, "ms_placement_only": ms_place, "host_enqueue_ms_per_step": host_ms_step,
            "cpu_baseline": {"value": cpu_rate, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": f"full {t.profile.name} step x{cpu_reps} ({cpu_s * 1e3:.1f} ms per step: full sweep + placement spec round)"},
            "oracle_check": check,
            "clocks": clocks,
            "algorithmic_bytes_per_step": int(algo_bytes),
            "sweep_gbs": algo_bytes / (ms_sweep * 1e-3) / 1e9,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()  # no rank frees its exchange buffer while a peer may still push into it
        eng.close()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
