#!/usr/bin/env python
"""bench.py — rows/s of the Q3-shaped filter -> join -> group-by (BASELINE.json configs[3], "C4")
on N B200s, with the roofline of its dominant kernel, the other SURVEY 8(d) configurations
(C1, C2 uniform / Zipf, C3 materialising / fused, C5 one GPU's share) measured in the same run,
and the reference's CPU path timed on the same box.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's CPU path (pandas restatement)
    python bench.py ... --dump-outputs DIR    # also write the last timed step's result as DIR/grp.npy, DIR/rev.npy

Headline workload (SURVEY 8d, seed 4): fact(fk int64, x int64, val float64) with --rows rows in
total (default 1e9, strong scaling: rows/N per GPU, 8 partitions spread over the GPUs),
dim(pk, flag, grp) 10M rows, 1M groups;
    SELECT d.grp, SUM(f.val) AS rev FROM fact f JOIN dim d ON f.fk = d.pk
    WHERE f.x > 0 AND d.flag < 5 GROUP BY d.grp

value : fact/dim resident in HBM, step = Context.sql(Q) (plan + plugins) + execution, result left
        on the device (N>1: every rank keeps the groups of its key range); timed with CUDA events,
        barrier + synchronize on both sides, max over ranks.  Inputs (24 GB) are far larger than
        L2 (126 MB), so no explicit L2 flush.
e2e   : same query through the public API on HOST (pinned) tables: every step copies the referenced
        fact/dim columns host->device and the result device->host (pandas).  PCIe-bound.
verified_full_size (every N): the full-size result checked through size-independent properties --
        sum of the group sums == masked sum of val (1e-9 relative), the set size of the groups,
        key uniqueness -- with the invariants all-reduced over the ranks.
exchange (N>1): where a step's time goes (build / bcast / scan / presence / reduce_scatter / compact).
configs (N=1): C1, C2 (uniform f64, uniform int64, Zipf 1.1), C3 (materialising, fused SUM(v*w)),
        C4 with a sparse primary key (hash lookup), C5 (one GPU's 500M-row share): ms, rows/s, roofline
        of the dominant kernel from live CUDA events, each verified against plain torch fp64/int64.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

QUERY = ("SELECT d.grp, SUM(f.val) AS rev FROM fact f JOIN dim d ON f.fk = d.pk "
         "WHERE f.x > 0 AND d.flag < 5 GROUP BY d.grp")
DIM_ROWS = 10_000_000
N_GROUPS = 1_000_000
BYTES_PER_FACT_ROW = 24       # fk + x + val, each read once (SURVEY 8d, BASELINE.md §3)
TOTAL_PARTITIONS = 8          # BASELINE configs: "8 partitions"; spread over the GPUs of the run


def parts_per_gpu(world):
    return max(1, TOTAL_PARTITIONS // world)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=float, default=float(os.environ.get("B200SQL_BENCH_ROWS", 1e9)))
    ap.add_argument("--cpu-sample-rows", type=float,
                    default=float(os.environ.get("B200SQL_CPU_SAMPLE_ROWS", 128e6)))
    ap.add_argument("--cpu-budget-s", type=float, default=float(os.environ.get("B200SQL_CPU_BUDGET_S", 150)))
    ap.add_argument("--dim-dist", default=os.environ.get("B200SQL_BENCH_DIM", "replicated"), choices=["replicated", "root"],
                    help="N>1: 'replicated' = every GPU holds the 10M-row dim table (registered once, before the timed "
                         "region) and builds its own lookup every step; 'root' = rows on rank 0 only, the finished "
                         "lookup is broadcast every step (NCCL)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--configs", default=os.environ.get("B200SQL_BENCH_CONFIGS", "all"),
                    help="comma list of C1,C2,C2i,C2z,C3,C3f,C4s,C5 (default all)")
    ap.add_argument("--config-scale", type=float, default=float(os.environ.get("B200SQL_CONFIG_SCALE", 1.0)),
                    help="scale the row counts of the extra configs (smoke runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the result of the last one as DIR/<column>.npy (float64, "
                         "rows ordered by the group key), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU arm's result; it does not apply to --impl reference")
    return args


# ---------------------------------------------------------------------------------------------
# CPU arm: the reference's path (oracle = pandas restatement; the only place bench.py runs it)
# ---------------------------------------------------------------------------------------------
def cpu_tables(rows, seed=4, threads=None):
    """The C4 tables as pandas frames.  The fact columns are generated in parallel chunks (numpy's
    generators release the GIL) so that a 128M-row sample does not take a minute to make."""
    import numpy as np
    import pandas as pd
    from concurrent.futures import ThreadPoolExecutor
    rows = int(rows)
    rng = np.random.default_rng(seed)
    dim = pd.DataFrame({"pk": rng.permutation(DIM_ROWS).astype(np.int64),
                        "flag": rng.integers(0, 10, DIM_ROWS), "grp": rng.integers(0, N_GROUPS, DIM_ROWS)})
    threads = threads or min(32, os.cpu_count() or 1)
    nchunk = max(1, min(threads, rows // 1_000_000 or 1))
    bounds = [(rows * i // nchunk, rows * (i + 1) // nchunk) for i in range(nchunk)]
    fk = np.empty(rows, np.int64)
    x = np.empty(rows, np.int64)
    val = np.empty(rows, np.float64)

    def fill(i):
        lo, hi = bounds[i]
        r = np.random.default_rng([seed, i])
        fk[lo:hi] = r.integers(0, DIM_ROWS, hi - lo)
        x[lo:hi] = r.integers(-2**31, 2**31, hi - lo)
        val[lo:hi] = r.random(hi - lo)

    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(fill, range(nchunk)))
    return pd.DataFrame({"fk": fk, "x": x, "val": val}, copy=False), dim


def cpu_step(fact_parts, dim, workers):
    from oracle import pandas_oracle as O
    t0 = time.perf_counter()
    out = O.c4_q3(fact_parts, dim, workers=workers)
    return time.perf_counter() - t0, len(out)


def run_cpu_baseline(sample_rows, steps=1, warmup=0, budget_s=150.0):
    """The reference's Dask-threads path on this box's host cores: the C4 query on a bounded sample of
    the fact table against the FULL 10M-row dim table.  Partitioning: the configuration's 8 partitions
    (8 pandas tasks at a time, like dask's threaded scheduler on an 8-partition frame) and, when the box
    has more cores, a 32-partition layout of the same rows; both are tried on a 1/4 sub-sample and the
    faster one is used and reported.  The sample shrinks only if steps x (sample time) would exceed
    `budget_s`; it never goes below 32M rows (below that, hashing the dim table once per partition
    dominates and the number says nothing about the 1B-row workload)."""
    from oracle import pandas_oracle as O
    cores = os.cpu_count() or 1
    sample_rows = int(sample_rows)
    fact, dim = cpu_tables(sample_rows)
    layouts = [TOTAL_PARTITIONS] + ([32] if cores >= 32 else [])
    cal_rows = max(8_000_000, sample_rows // 4)
    cal = fact.iloc[:cal_rows]
    trials = {}
    for p in layouts:
        parts = O.split(cal, p)
        trials[p] = cal_rows / cpu_step(parts, dim, min(p, cores))[0]
    best_p = max(trials, key=trials.get)
    rate = trials[best_p]
    n_runs = max(1, steps) + max(0, warmup)
    fit = int(rate * budget_s / n_runs)
    if fit < sample_rows:
        sample_rows = max(32_000_000, min(sample_rows, fit))
        fact = fact.iloc[:sample_rows]
    parts = O.split(fact, best_p)
    workers = min(best_p, cores)
    for _ in range(warmup):
        cpu_step(parts, dim, workers)
    ts, groups = [], 0
    for _ in range(max(1, steps)):
        t, groups = cpu_step(parts, dim, workers)
        ts.append(t)
    t = sorted(ts)[len(ts) // 2]
    return {"value": sample_rows / t, "unit": "rows/s", "cores": cores, "threads_used": workers, "kind": "port",
            "partitions": best_p, "sample_rows": sample_rows, "dim_rows": DIM_ROWS, "groups_out": groups,
            "scale_factor_vs_1e9_rows": sample_rows / 1e9,
            "layout_trials_rows_per_s": {str(k): v for k, v in trials.items()},
            "sample": f"{sample_rows} fact rows of the same workload x the full {DIM_ROWS}-row dim, "
                      f"{best_p} partitions on {workers} threads ({cores} cores), pandas restatement of "
                      "table_scan.py/join.py/aggregate.py with a broadcast build side and the split_every tree "
                      "(oracle/pandas_oracle.py c4_q3); dask and the Rust planner are not installable here",
            "seconds_per_step": t}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base = run_cpu_baseline(args.cpu_sample_rows, steps=args.steps, warmup=args.warmup, budget_s=args.cpu_budget_s)
    keep = ("value", "unit", "cores", "threads_used", "kind", "partitions", "sample_rows", "dim_rows", "sample",
            "scale_factor_vs_1e9_rows", "layout_trials_rows_per_s")
    line = {
        "impl": "reference", "metric": "rows/s on Q3-shaped filter->join->groupby", "value": base["value"],
        "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": base["seconds_per_step"] * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {k: base[k] for k in keep},
        "e2e": {"value": base["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, n):
    return {"workload": "C4: TPC-H-Q3-shaped filter->join->groupby (BASELINE.json configs[3])",
            "fact_rows_total": int(args.rows), "fact_rows_per_gpu": int(args.rows) // n, "dim_rows": DIM_ROWS,
            "groups": N_GROUPS, "partitions_per_gpu": parts_per_gpu(n), "query": QUERY,
            "l2": "inputs (24 B/row x rows) >> 126 MB L2, no flush needed",
            "planning": "Context.sql() is called every step; its plan (not its result) is served from the "
                        "prepared-statement cache after the first call; build side, lookup and group table "
                        "are rebuilt every step",
            "parallelism": (f"fact sharded over {n} GPU(s); " +
                            ("dim replicated (registered on every GPU before the timed region, as a broadcast-join "
                             "engine keeps small dimension tables), every GPU builds its pk->slot lookup every step; "
                             if args.dim_dist == "replicated" else
                             "dim on rank 0, its pk->slot lookup broadcast every step (NCCL); ") +
                            "dense partial aggregates merged by key range (b2_peer_merge over NVLink peer memory, "
                            "ncclReduceScatter where symmetric memory is unavailable: the line's `merge` key says "
                            "which ran), every rank compacts and keeps the groups of its range")
            if n > 1 else "single GPU"}


def merge_kind():
    """How the ranks' partial group tables were merged in this process (decided by the executor)."""
    try:
        from dask_sql_b200 import executor
        if executor.stats.get("peer_merge_plans", 0) > 0:
            return ("b2_peer_merge: one kernel per GPU over NVLink peer memory (in-kernel barrier, rank-ordered "
                    "reduction of its slot range, existence merged in the same pass)")
    except Exception:
        pass
    return "ncclReduceScatter per accumulator array + presence bytes"


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi-equivalent clock / throttle-reason samples (NVML) taken only while `active`:
    the thread and NVML are brought up before the warm-up so that the first sample falls inside
    the timed region, which is only tens of milliseconds long."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.active = False
        self.nv = self.h = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def run(self):
        nv, h = self.nv, self.h
        if nv is None:
            return
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown"}
        try:
            while not self.stop_flag:
                if self.active:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                time.sleep(0.004)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def load_peaks():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    return peak_gbs, src


def load_traffic():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


def kernel_roofline(kev, kernel, bytes_per_row, peak_gbs, peak_src, traffic, step_s=None, steps=1):
    """roofline of `kernel` from the live CUDA events the executor recorded around its launches."""
    durs = [(rows, a.elapsed_time(b) * 1e-3) for name, rows, a, b in kev if name == kernel]
    if not durs:
        return None
    rows_l = sum(r for r, _ in durs) / len(durs)
    avg = sum(d for _, d in durs) / len(durs)
    achieved = rows_l * bytes_per_row / avg / 1e9
    tr = traffic.get(kernel, {}).get("dram_bytes_per_row")
    out = {"kernel": kernel, "bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
           "frac": achieved / peak_gbs, "traffic": tr * rows_l if tr is not None else None,
           "peak_source": peak_src, "algorithmic_bytes_per_launch": rows_l * bytes_per_row,
           "algorithmic_bytes_per_row": bytes_per_row, "avg_launch_ms": avg * 1e3, "launches_timed": len(durs)}
    if step_s:
        out["kernel_share_of_step"] = sum(d for _, d in durs) / steps / step_s
    return out


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        return reference_arm(args)

    # stdout carries exactly ONE JSON line: libraries that write to fd 1 (NCCL prints its version
    # banner there) are pointed at stderr for the whole run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from dask_sql_b200 import Context, executor

    n_total = int(args.rows)
    n_local = n_total // world
    # fit the shard into this GPU (and, for e2e, pinned host memory): shrink, loudly, if needed
    free_b, total_b = torch.cuda.mem_get_info()
    need = n_local * BYTES_PER_FACT_ROW * 1.15 + DIM_ROWS * 24 * 4
    if need > free_b:
        if args.dump_outputs:   # the inputs, and so the dumped result, would depend on the free memory
            raise SystemExit(f"[bench] {n_total} fact rows do not fit this GPU's free HBM; pass a smaller --rows "
                             "to --dump-outputs")
        n_local = int((free_b - DIM_ROWS * 96) / (BYTES_PER_FACT_ROW * 1.15))
        n_total = n_local * world
        print(f"[bench] shrinking to {n_total} fact rows to fit HBM", file=sys.stderr)
    args.rows = n_total

    g = torch.Generator(device=dev)
    g.manual_seed(4 + rank)
    fk = torch.randint(0, DIM_ROWS, (n_local,), dtype=torch.int64, device=dev, generator=g)
    x = torch.randint(-2**31, 2**31, (n_local,), dtype=torch.int64, device=dev, generator=g)
    val = torch.rand(n_local, dtype=torch.float64, device=dev, generator=g)
    gd = torch.Generator(device=dev)
    gd.manual_seed(4)
    # every rank generates the (seed-identical) dim columns -- the verification needs them -- but only
    # rank 0 registers rows: the table is 'root' and reaches the others through the join's broadcast
    pk = torch.randperm(DIM_ROWS, device=dev, generator=gd)
    flag = torch.randint(0, 10, (DIM_ROWS,), dtype=torch.int64, device=dev, generator=gd)
    grp = torch.randint(0, N_GROUPS, (DIM_ROWS,), dtype=torch.int64, device=dev, generator=gd)
    dim_dist = "local" if world == 1 else args.dim_dist
    nd = DIM_ROWS if (rank == 0 or dim_dist != "root") else 0

    c = Context()
    fact_dist = "sharded" if world > 1 else "local"
    c.create_table("fact", {"fk": fk, "x": x, "val": val}, persist=True, npartitions=parts_per_gpu(world),
                   distribution=fact_dist)
    c.create_table("dim", {"pk": pk[:nd], "flag": flag[:nd], "grp": grp[:nd]}, persist=True, distribution=dim_dist)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step_resident():
        lazy = c.sql(QUERY)
        return executor.execute(lazy, top=True)

    # ---- value: device-resident inputs
    sampler = ClockSampler(local)
    if os.environ.get("B200SQL_NO_SAMPLER") != "1":
        sampler.start()
    for _ in range(args.warmup):
        parts = step_resident()
    barrier()
    sampler.active = True
    launches0 = executor.stats["launches"]
    executor.prefill_timing_events(args.steps * (2 * parts_per_gpu(world) + 24) + 64)
    executor.kernel_events = []
    executor.phase_events = [] if (world > 1 and os.environ.get("B200SQL_NO_PHASES") != "1") else None
    if os.environ.get("B200SQL_CALL_TIMES") == "1":
        executor.D.trace = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prof = None
    if os.environ.get("B200SQL_BENCH_PROFILE") == "1" and rank == 0:     # host-side profile of the timed loop
        import cProfile
        prof = cProfile.Profile()
    w0 = time.perf_counter()
    e0.record()
    if prof is not None:
        prof.enable()
    for _ in range(args.steps):
        parts = step_resident()
    if prof is not None:
        prof.disable()
    e1.record()
    host_issue = time.perf_counter() - w0
    if rank == 0 and os.environ.get("B200SQL_CALL_TIMES") == "1":
        torch.cuda.synchronize()
        tr = executor.D.trace
        seg = {}
        for (la, ea), (lb, eb) in zip(tr, tr[1:]):
            if la != "select:written":
                seg[la + "->" + lb] = seg.get(la + "->" + lb, 0.0) + ea.elapsed_time(eb)
        print("[select_launch GPU ms per step] " + json.dumps({k: round(v / args.steps, 4) for k, v in seg.items()}),
              file=sys.stderr)
        from dask_sql_b200 import _lib as _L, parallel as _P
        print("[collective host ms: calls, total] " + json.dumps({k: [v[0], round(v[1] * 1e3, 3)] for k, v in (_P.coll_times or {}).items()}),
              file=sys.stderr)
        print("[call times over the timed loop + warm-up] " + json.dumps(
            {k: [v[0], round(v[1] * 1e3, 3)] for k, v in sorted(_L.call_times.items(), key=lambda kv: -kv[1][1])}),
            file=sys.stderr)
    if prof is not None:
        import io
        import pstats
        buf = io.StringIO()
        pstats.Stats(prof, stream=buf).sort_stats("cumulative").print_stats(45)
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        open(os.path.join(ROOT, "gpurun_out", f"host_profile_n{world}.txt"), "w").write(buf.getvalue())
    barrier()
    sampler.active = False
    wall = time.perf_counter() - w0
    dev_s = e0.elapsed_time(e1) * 1e-3
    t_step = max_over_ranks(max(dev_s, 0.0)) / args.steps
    launches = executor.stats["launches"] - launches0
    kev, pev = executor.kernel_events, executor.phase_events
    executor.kernel_events = executor.phase_events = None
    sampler.stop_flag = True
    if sampler.is_alive():
        sampler.join(timeout=2)
    n_groups_local = parts[0].n
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, parts, rank)

    peak_gbs, peak_src = load_peaks()
    traffic = load_traffic()
    roofline = kernel_roofline(kev, "b2_star_agg_kernel", BYTES_PER_FACT_ROW, peak_gbs, peak_src, traffic,
                               dev_s / args.steps, args.steps)

    exchange = None
    if pev:
        tot = {}
        for name, a, b in pev:
            tot[name] = tot.get(name, 0.0) + a.elapsed_time(b)
        exchange = {k + "_ms": v / args.steps for k, v in tot.items()}
        exchange["host_issue_ms"] = host_issue / args.steps * 1e3
        exchange["step_ms_this_rank"] = dev_s / args.steps * 1e3
        exchange["note"] = ("CUDA-event time per step on rank 0's stream; a phase includes the wait for slower "
                            "ranks inside its collective")

    # ---- full-size parity through size-independent properties, at every N
    try:
        verified = verify_full_size(torch, dist, world, parts, fk, x, val, pk, flag, grp)
    except Exception as e:  # the check must never take the measurement down with it
        verified = {"ok": False, "error": f"{type(e).__name__}: {e}"}
    n_groups_out = verified.get("groups", n_groups_local)

    # ---- e2e: host-resident (pinned) tables through the public API, pandas result
    e2e = None
    if not args.no_e2e:
        try:
            e2e = run_e2e(args, torch, dist, dev, world, rank, fk, x, val, pk[:nd], flag[:nd], grp[:nd], fact_dist,
                          dim_dist, barrier, max_over_ranks)
        except Exception as e:  # e.g. not enough pinnable host memory
            e2e = {"error": f"{type(e).__name__}: {e}"}

    c = None
    del fk, x, val, parts
    torch.cuda.empty_cache()

    configs = None
    if world == 1 and not args.no_configs:
        configs = run_configs(args, torch, dev, peak_gbs, peak_src, traffic)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = run_cpu_baseline(args.cpu_sample_rows, budget_s=args.cpu_budget_s)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "threads_used", "kind", "partitions", "sample_rows",
                                   "dim_rows", "sample", "layout_trials_rows_per_s")}

    if rank == 0:
        line = {
            "metric": "rows/s on Q3-shaped filter->join->groupby", "value": n_total / t_step, "unit": "rows/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_step * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(args, world), "clocks": sampler.summary(),
            "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "groups_out": n_groups_out, "verified_full_size": verified, "exchange": exchange,
            "wall_ms_per_step": wall / args.steps * 1e3,
            "fused_star_pipeline": executor.stats["star_fused"] > 0, "configs": configs,
            "merge": merge_kind() if world > 1 else None,
        }
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def verify_full_size(torch, dist, world, parts, fk, x, val, pk, flag, grp):
    """The oracle cannot run 1e9 rows in the bench, so the full-size result is checked through
    properties that do not depend on size (plain torch ops on the resident inputs, fp64), with every
    invariant summed / OR-ed over the ranks so that the check holds at any N:
      * checksum of checksums: the sum over groups of SUM(val) equals the sum of val over the fact
        rows that pass both predicates (1e-9 relative, BASELINE.json north_star tolerance);
      * the number of groups equals the number of distinct grp among dim rows with flag < 5 that at
        least one passing fact row (on ANY rank) references; group keys are unique, also across ranks
        (the ranks' key ranges must not overlap)."""
    res = parts[0]
    keys, rev = res["grp"].data, res["rev"].data
    nd, dev = pk.numel(), pk.device
    ok_dim = torch.zeros(nd, dtype=torch.bool, device=dev)
    ok_dim[pk] = flag < 5                                   # indexed by key value: pk is a permutation of 0..nd-1
    grp_by_pk = torch.empty_like(grp)
    grp_by_pk[pk] = grp
    hit = torch.zeros(nd, dtype=torch.int32, device=dev)
    total = torch.zeros(1, dtype=torch.float64, device=dev)
    rows = torch.zeros(1, dtype=torch.int64, device=dev)
    chunk = 1 << 26
    for lo in range(0, fk.numel(), chunk):
        f = fk[lo:lo + chunk]
        m = (x[lo:lo + chunk] > 0) & ok_dim[f]
        total += val[lo:lo + chunk][m].sum()
        hit[f[m]] = 1
        rows += m.sum()
    got = rev.sum().reshape(1)
    ngroups = torch.tensor([keys.numel()], dtype=torch.int64, device=dev)
    unique = int(torch.unique(keys).numel()) == int(keys.numel())
    disjoint = True
    if world > 1:
        dist.all_reduce(total)
        dist.all_reduce(rows)
        dist.all_reduce(got)
        dist.all_reduce(ngroups)
        dist.all_reduce(hit, op=dist.ReduceOp.MAX)
        big = 1 << 62
        span = torch.tensor([int(keys.min()) if keys.numel() else big, int(keys.max()) if keys.numel() else -big],
                            dtype=torch.int64, device=dev)
        spans = [torch.empty_like(span) for _ in range(world)]
        dist.all_gather(spans, span)
        last = -big
        for s in spans:
            lo_k, hi_k = int(s[0]), int(s[1])
            if lo_k == big:
                continue
            disjoint &= lo_k > last
            last = hi_k
        u = torch.tensor([1 if unique else 0], dtype=torch.int64, device=dev)
        dist.all_reduce(u, op=dist.ReduceOp.MIN)
        unique = bool(int(u))
    groups_expected = int(torch.unique(grp_by_pk[hit.bool()]).numel())
    got_f, exp_f = float(got.item()), float(total.item())
    rel = abs(got_f - exp_f) / max(abs(exp_f), 1e-300)
    groups = int(ngroups.item())
    return {"sum_of_group_sums_rel_err": rel, "tolerance": 1e-9, "groups": groups,
            "groups_expected": groups_expected, "keys_unique": bool(unique and disjoint),
            "rows_contributing": int(rows.item()), "ranks": world,
            "ok": bool(rel <= 1e-9 and groups == groups_expected and unique and disjoint)}


RESULT_COLUMNS = ("grp", "rev")      # QUERY's output columns, group key first
DUMP_ARRAY_BYTES = 63 * 10**6        # the .npy files stay under 64 MB in all, headers included


def dump_outputs(out_dir, parts, rank):
    """Write the result of the timed query, the columns a caller of Context.sql(QUERY) receives, as
    out_dir/<column>.npy in float64 (the int64 group keys are far below 2**53, so exactly).  SQL leaves
    the order of GROUP BY output open and two builds may emit it differently, so rows are ordered by the
    group key.  A result larger than DUMP_ARRAY_BYTES is written as a fixed, seeded sample of its rows.
    N>1: the ranks' key ranges are gathered (a collective, every rank calls it) and rank 0 writes."""
    import numpy as np
    import pandas as pd
    from dask_sql_b200 import device as D, executor
    parts = [executor.gather_keyrange(p) for p in parts]
    if rank != 0:
        return
    frame = pd.concat([pd.DataFrame({c: D.column_to_host(p[c]) for c in RESULT_COLUMNS}) for p in parts],
                      ignore_index=True)
    cols = {c: frame[c].to_numpy(dtype=np.float64, na_value=np.nan) for c in RESULT_COLUMNS}
    order = np.argsort(cols[RESULT_COLUMNS[0]], kind="stable")
    keep = DUMP_ARRAY_BYTES // (8 * len(cols))
    if len(order) > keep:
        order = order[np.sort(np.random.default_rng(0).choice(len(order), keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for c, v in cols.items():
        np.save(os.path.join(out_dir, c + ".npy"), v[order])


def run_e2e(args, torch, dist, dev, world, rank, fk, x, val, pk, flag, grp, fact_dist, dim_dist, barrier,
            max_over_ranks):
    from dask_sql_b200 import Context, executor

    host = {}
    for name, t in (("fk", fk), ("x", x), ("val", val), ("pk", pk), ("flag", flag), ("grp", grp)):
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t)
        host[name] = h
    torch.cuda.synchronize()
    c = Context()
    c.create_table("fact", {k: host[k] for k in ("fk", "x", "val")}, persist=False, npartitions=parts_per_gpu(world),
                   distribution=fact_dist)
    c.create_table("dim", {k: host[k] for k in ("pk", "flag", "grp")}, persist=False, distribution=dim_dist)
    steps = max(2, min(args.steps, 5))
    for _ in range(1):
        c.sql(QUERY, return_futures=False)
    barrier()
    h0, d0 = executor.stats["h2d_bytes"], executor.stats["d2h_bytes"]
    t0 = time.perf_counter()
    for _ in range(steps):
        out = c.sql(QUERY, return_futures=False)
    barrier()
    t = max_over_ranks(time.perf_counter() - t0) / steps
    n_total = int(args.rows)
    h2d = (executor.stats["h2d_bytes"] - h0) // steps
    return {"value": n_total / t, "unit": "rows/s", "ms_per_step": t * 1e3, "steps": steps,
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": (executor.stats["d2h_bytes"] - d0) // steps,
            "result_rows": len(out), "h2d_gbs_per_gpu": h2d / t / 1e9,
            "bound": "PCIe host->device copy of the referenced columns (24 B per fact row); the kernels add ~1 %",
            "api": "Context.create_table(host pinned columns, persist=False); Context.sql(Q, return_futures=False)"}


# ---------------------------------------------------------------------------------------------
# the other SURVEY 8(d) configurations, one GPU
# ---------------------------------------------------------------------------------------------
def _time_query(torch, executor, c, sql, steps, warmup, kernel_names):
    """(ms per step, kernel events, parts of the last step) of c.sql(sql) executed on the device."""
    # The warm-up runs exactly like the timed loop -- results are NOT resolved between steps, so a step
    # allocates while the previous step's outputs are still alive -- or the caching allocator meets a new
    # pattern inside the timed region and stalls the stream behind cudaMalloc / cudaFree (seen as a 1-19 ms
    # hole in a phase that otherwise takes 0.04-2.4 ms).
    parts = None
    for _ in range(2):
        for _ in range(max(warmup, steps)):
            parts = executor.execute(c.sql(sql), top=True)
        torch.cuda.synchronize()
        for p in parts:
            p.resolve()
    torch.cuda.synchronize()
    executor.kernel_events = []
    executor.phase_events = []
    l0 = executor.stats["launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        parts = executor.execute(c.sql(sql), top=True)
    e1.record()
    torch.cuda.synchronize()
    for p in parts:
        p.resolve()
    kev, pev = executor.kernel_events, executor.phase_events
    executor.kernel_events = executor.phase_events = None
    breakdown = {}
    for name, _, a, b in kev:
        breakdown[name] = breakdown.get(name, 0.0) + a.elapsed_time(b) / steps
    for name, a, b in pev:
        breakdown["phase:" + name] = breakdown.get("phase:" + name, 0.0) + a.elapsed_time(b) / steps
    _time_query.breakdown = {k: round(v, 4) for k, v in breakdown.items()}
    return e0.elapsed_time(e1) / steps, kev, parts, (executor.stats["launches"] - l0) // steps


def _zipf_keys(torch, n, nkeys, s, dev, gen):
    """n draws from Zipf(s) over nkeys ranks (inverse CDF by binary search), ranks mapped to keys
    by a random permutation so that hot keys are scattered over the key range."""
    w = torch.arange(1, nkeys + 1, dtype=torch.float64, device=dev).pow_(-s)
    cdf = torch.cumsum(w, 0)
    cdf /= cdf[-1].clone()
    out = torch.empty(n, dtype=torch.int64, device=dev)
    chunk = 1 << 25
    for lo in range(0, n, chunk):
        u = torch.rand(min(chunk, n - lo), dtype=torch.float64, device=dev, generator=gen)
        out[lo:lo + chunk] = torch.searchsorted(cdf, u).clamp_(max=nkeys - 1)
    perm = torch.randperm(nkeys, device=dev, generator=gen)
    return perm[out]


def run_configs(args, torch, dev, peak_gbs, peak_src, traffic):
    from dask_sql_b200 import Context, executor
    want = {w.strip() for w in args.configs.split(",")} if args.configs != "all" else None
    sc = args.config_scale
    steps, warmup = max(3, min(args.steps, 5)), max(3, min(args.warmup, 3))
    out = {}

    # the L2 serves ~200 G REDG (reduction atomics without return value) per second on this part
    # (scripts/microbench/redg.cu "red_spread f64_1red", L2-resident table; profiles/r02_redg.jsonl): the
    # second roofline of the group-by stage, which issues one per row (SURVEY 8d: "random 32 B-sector
    # throughput ... report it").  Plain random LOADS are served faster than that (C3f sustains 287 G/s), so
    # the figure is attached to the REDG kernels only.
    L2_REQ_PEAK = 200.7

    def entry(name, rows, ms, kev, kernel, bytes_per_row, launches, query, verified, extra=None, random_per_row=None,
              has_capture=True):
        # has_capture=False: profiles/traffic.json holds no ncu capture of THIS variant of the kernel
        tr = traffic if has_capture else {}
        e = {"rows": rows, "ms": ms, "rows_per_s": rows / (ms * 1e-3), "query": query,
             "breakdown_ms_per_step": getattr(_time_query, "breakdown", None),
             "algorithmic_gbs_whole_query": rows * bytes_per_row / (ms * 1e-3) / 1e9,
             "frac_of_peak_whole_query": rows * bytes_per_row / (ms * 1e-3) / 1e9 / peak_gbs,
             "roofline": kernel_roofline(kev, kernel, bytes_per_row, peak_gbs, peak_src, tr, ms * 1e-3, steps),
             "gpu_launches_per_step": launches, "verified": verified, "steps": steps, "warmup": warmup}
        if extra:
            e.update(extra)
        if random_per_row and e["roofline"]:
            r = e["roofline"]
            rows_l = r["algorithmic_bytes_per_launch"] / r["algorithmic_bytes_per_row"]
            ach = rows_l * random_per_row / (r["avg_launch_ms"] * 1e-3) / 1e9
            e["roofline_l2_requests"] = {"kernel": kernel, "bound": "L2 reduction-atomic (REDG) rate", "unit": "G requests/s",
                                         "random_requests_per_row": random_per_row, "achieved": ach, "peak": L2_REQ_PEAK,
                                         "frac": ach / L2_REQ_PEAK,
                                         "peak_source": "measured: scripts/microbench/redg.cu, one REDG.F64 per row into "
                                                        "an 8 MB table (profiles/r02_redg.jsonl)",
                                         "note": "streamed columns add ~0.25-0.5 sector requests per row on top"}
        out[name] = e

    def guarded(name, fn):
        if want is not None and name not in want:
            return
        try:
            fn()
        except Exception as ex:  # one configuration must not take the others down
            out[name] = {"error": f"{type(ex).__name__}: {ex}"}
        torch.cuda.empty_cache()

    g = torch.Generator(device=dev)

    # ---- C1: SELECT SUM(x) FROM t WHERE x > 0 -- 1B rows (the 10M-row nominal size fits L2 and measures
    # launch latency; both are reported)
    def c1():
        for label, n, nparts in (("C1", int(1e9 * sc), 8), ("C1_nominal_10M", int(1e7 * sc), 1)):
            g.manual_seed(1)
            xx = torch.randint(-2**31, 2**31, (n,), dtype=torch.int64, device=dev, generator=g)
            c = Context()
            c.create_table("t", {"x": xx}, persist=True, npartitions=nparts)
            q = "SELECT SUM(x) AS s FROM t WHERE x > 0"
            ms, kev, parts, nl = _time_query(torch, executor, c, q, steps, warmup, ())
            got = int(parts[0]["s"].data[0].item())
            exp = int(xx[xx > 0].sum().item())
            entry(label, n, ms, kev, "b2_scan_agg_kernel", 8, nl, q, {"ok": got == exp, "sum": got, "expected": exp},
                  {"partitions": nparts, "l2": "8 GB >> L2" if n > 5e7 else "80 MB fits L2: launch-latency bound"},
                  has_capture=n > 5e7)
            del xx, c

    # ---- C2: GROUP BY key SUM(val), 200M rows, 1M keys, 8 partitions
    def c2(name, kind):
        n, nkeys = int(2e8 * sc), 1_000_000
        g.manual_seed(2)
        if kind == "zipf":
            key = _zipf_keys(torch, n, nkeys, 1.1, dev, g)
        else:
            key = torch.randint(0, nkeys, (n,), dtype=torch.int64, device=dev, generator=g)
        if kind == "int":
            v = torch.randint(-1000, 1001, (n,), dtype=torch.int64, device=dev, generator=g)
        else:
            v = torch.rand(n, dtype=torch.float64, device=dev, generator=g)
        c = Context()
        c.create_table("t", {"key": key, "val": v}, persist=True, npartitions=8)
        q = "SELECT key, SUM(val) AS s FROM t GROUP BY key"
        ms, kev, parts, nl = _time_query(torch, executor, c, q, steps, warmup, ())
        res = parts[0]
        k_out, s_out = res["key"].data, res["s"].data
        exp = torch.zeros(nkeys, dtype=v.dtype, device=dev)
        exp.index_add_(0, key, v)
        cnt = torch.bincount(key, minlength=nkeys)
        present = cnt > 0
        ok_keys = bool(torch.equal(k_out, torch.nonzero(present).reshape(-1)))
        if kind == "int":
            ok_vals = ok_keys and bool(torch.equal(s_out, exp[present]))
            err = 0.0
        else:
            e = exp[present]
            err = float(((s_out - e).abs() / e.abs().clamp_min(1e-300)).max().item()) if ok_keys else float("inf")
            ok_vals = err <= 1e-9
        top = float(cnt.max().item()) / n
        entry(name, n, ms, kev, "b2_groupby_dense_kernel", 16, nl, q,
              {"ok": bool(ok_keys and ok_vals), "groups": int(k_out.numel()), "max_rel_err": err,
               "checked": "every group against torch index_add_ (fp64 / int64)"},
              {"keys": nkeys, "distribution": "Zipf(1.1), ranks scattered by a permutation" if kind == "zipf"
               else "uniform", "hottest_key_share": top, "val": "int64" if kind == "int" else "float64",
               "partitions": 8, "grouped_kernel": executor.stats.get("grouped_groupby", 0) > 0},
              random_per_row=None if kind == "zipf" else 1.0, has_capture=kind != "zipf")

    # ---- C3: INNER JOIN 1B-row fact x 10M-row dim, 80 % match; materialising and fused SUM(v*w)
    def c3(name, fused):
        n, ndim = int(1e9 * sc), int(1e7 * sc) or 1
        g.manual_seed(3)
        pkk = torch.randperm(ndim, device=dev, generator=g)
        w = torch.randint(0, 1000, (ndim,), dtype=torch.int64, device=dev, generator=g)
        fkk = torch.randint(0, int(ndim * 1.25), (n,), dtype=torch.int64, device=dev, generator=g)
        v = torch.rand(n, dtype=torch.float64, device=dev, generator=g)
        c = Context()
        c.create_table("fact", {"fk": fkk, "v": v}, persist=True, npartitions=8)
        c.create_table("dim", {"pk": pkk, "w": w}, persist=True)
        w_by_pk = torch.empty_like(w)
        w_by_pk[pkk] = w
        m = fkk < ndim
        n_match = int(m.sum().item())
        if fused:
            q = "SELECT SUM(f.v * d.w) AS s FROM fact f JOIN dim d ON f.fk = d.pk"
            ms, kev, parts, nl = _time_query(torch, executor, c, q, steps, warmup, ())
            got = float(parts[0]["s"].data[0].item())
            exp = 0.0
            ch = 1 << 26
            for lo in range(0, n, ch):
                mm = m[lo:lo + ch]
                exp += float((v[lo:lo + ch][mm] * w_by_pk[fkk[lo:lo + ch][mm]].double()).sum().item())
            rel = abs(got - exp) / max(abs(exp), 1e-300)
            entry(name, n, ms, kev, "b2_join_agg_kernel", 16, nl, q, {"ok": rel <= 1e-9, "rel_err": rel},
                  {"match_rate": n_match / n, "dim_rows": ndim, "partitions": 8,
                   "algorithmic_bytes": "16 B per fact row (fk, v) + 16 B per dim row"})
        else:
            q = "SELECT f.fk, f.v, d.w FROM fact f JOIN dim d ON f.fk = d.pk"
            ms, kev, parts, nl = _time_query(torch, executor, c, q, steps, warmup, ())
            rows_out, s_fk, s_v, s_w, order_ok = 0, 0, 0.0, 0, True
            for p in parts:
                p.resolve()
                rows_out += p.n
                s_fk += int(p["fk"].data.sum().item())
                s_v += float(p["v"].data.sum().item())
                s_w += int(p["w"].data.sum().item())
            # first partition row by row.  The streaming probe emits warp batches in the order they reserve
            # their output range (SQL leaves join order unspecified), so both sides are put in the order of
            # (v, fk) first: the multiset of output rows must equal the multiset of matching input rows.
            p0 = parts[0]
            k0 = p0.n
            idx = torch.nonzero(m[: fkk.numel() // 8 + 64]).reshape(-1)[:k0]

            def canon(fk_c, v_c, w_c):
                o = torch.argsort(v_c, stable=True)
                o = o[torch.argsort(fk_c[o], stable=True)]
                return fk_c[o], v_c[o], w_c[o]

            got3 = canon(p0["fk"].data, p0["v"].data, p0["w"].data)
            exp3 = canon(fkk[idx], v[idx], w_by_pk[fkk[idx]])
            order_ok = all(bool(torch.equal(a, b)) for a, b in zip(got3, exp3))
            del got3, exp3
            e_fk = int(fkk[m].sum().item())
            e_w = 0
            e_v = 0.0
            ch = 1 << 26
            for lo in range(0, n, ch):
                mm = m[lo:lo + ch]
                e_w += int(w_by_pk[fkk[lo:lo + ch][mm]].sum().item())
                e_v += float(v[lo:lo + ch][mm].sum().item())
            rel = abs(s_v - e_v) / max(abs(e_v), 1e-300)
            ok = rows_out == n_match and s_fk == e_fk and s_w == e_w and rel <= 1e-9 and order_ok
            bpr = 16 + 24 * n_match / n       # read fk, v; write (fk, v, w) per matching row
            entry(name, n, ms, kev, "b2_join_onepass", bpr, nl, q,
                  {"ok": bool(ok), "rows_out": rows_out, "rows_expected": n_match, "sum_v_rel_err": rel,
                   "first_partition_rows_exact": order_ok,
                   "checked": "row count, integer column checksums exact, float checksum 1e-9, partition 0's rows "
                              "one by one as a multiset"},
                  {"match_rate": n_match / n, "dim_rows": ndim, "partitions": 8,
                   "algorithmic_bytes": "16 B read per fact row + 24 B written per output row (+16 B per dim row)"})

    # ---- C4 with a sparse primary key: the pk -> slot lookup is a hash table, not a direct-address array
    def c4s():
        n, ndim = int(5e8 * sc), int(1e7 * sc) or 1
        g.manual_seed(44)
        pk0 = torch.randperm(ndim, device=dev, generator=g)
        mult = 1_000_003
        pks = pk0 * mult - 7                                   # key range 1e13: no direct-address lookup possible
        fl = torch.randint(0, 10, (ndim,), dtype=torch.int64, device=dev, generator=g)
        gr = torch.randint(0, N_GROUPS, (ndim,), dtype=torch.int64, device=dev, generator=g)
        fk0 = torch.randint(0, ndim, (n,), dtype=torch.int64, device=dev, generator=g)
        xx = torch.randint(-2**31, 2**31, (n,), dtype=torch.int64, device=dev, generator=g)
        vv = torch.rand(n, dtype=torch.float64, device=dev, generator=g)
        c = Context()
        c.create_table("fact", {"fk": fk0 * mult - 7, "x": xx, "val": vv}, persist=True, npartitions=4)
        c.create_table("dim", {"pk": pks, "flag": fl, "grp": gr}, persist=True)
        ms, kev, parts, nl = _time_query(torch, executor, c, QUERY, steps, warmup, ())
        res = parts[0]
        ok_dim = torch.zeros(ndim, dtype=torch.bool, device=dev)
        ok_dim[pk0] = fl < 5
        g_by = torch.empty_like(gr)
        g_by[pk0] = gr
        m = (xx > 0) & ok_dim[fk0]
        exp = torch.zeros(N_GROUPS, dtype=torch.float64, device=dev)
        exp.index_add_(0, g_by[fk0[m]], vv[m])
        hitg = torch.zeros(N_GROUPS, dtype=torch.bool, device=dev)
        hitg[g_by[fk0[m]]] = True
        order = torch.argsort(res["grp"].data)
        k_sorted, s_sorted = res["grp"].data[order], res["rev"].data[order]
        ok_keys = bool(torch.equal(k_sorted, torch.nonzero(hitg).reshape(-1)))
        err = float(((s_sorted - exp[hitg]).abs() / exp[hitg].abs().clamp_min(1e-300)).max().item()) if ok_keys \
            else float("inf")
        entry("C4_sparse_pk", n, ms, kev, "b2_star_agg_kernel", 24, nl, QUERY,
              {"ok": bool(ok_keys and err <= 1e-9), "groups": int(k_sorted.numel()), "max_rel_err": err,
               "checked": "every group against torch index_add_"},
              {"lookup": "open-addressing hash table (b2_star_build_hash): int64 keys + int32 slots, 12 B/slot",
               "dim_rows": ndim, "partitions": 4}, has_capture=False)

    # ---- C5: one GPU's share (500M rows) of GROUP BY over 100M keys, SUM + AVG
    def c5():
        n, nkeys = int(5e8 * sc), int(1e8 * sc) or 1
        g.manual_seed(5)
        key = torch.randint(0, nkeys, (n,), dtype=torch.int64, device=dev, generator=g)
        v = torch.rand(n, dtype=torch.float64, device=dev, generator=g)
        c = Context()
        c.create_table("t", {"key": key, "val": v}, persist=True, npartitions=8)
        q = "SELECT key, SUM(val) AS s, AVG(val) AS a FROM t GROUP BY key"
        ms, kev, parts, nl = _time_query(torch, executor, c, q, steps, warmup, ())
        res = parts[0]
        k_out, s_out, a_out = res["key"].data, res["s"].data, res["a"].data
        cnt = torch.bincount(key, minlength=nkeys)
        present = cnt > 0
        ok_keys = bool(torch.equal(k_out, torch.nonzero(present).reshape(-1)))
        exp = torch.zeros(nkeys, dtype=torch.float64, device=dev)
        exp.index_add_(0, key, v)
        if ok_keys:
            e = exp[present]
            err_s = float(((s_out - e).abs() / e.abs().clamp_min(1e-300)).max().item())
            ea = e / cnt[present].double()
            err_a = float(((a_out - ea).abs() / ea.abs().clamp_min(1e-300)).max().item())
        else:
            err_s = err_a = float("inf")
        entry("C5_one_gpu_share", n, ms, kev, "b2_part_scatter_kernel", 32, nl, q,
              {"ok": bool(ok_keys and err_s <= 1e-9 and err_a <= 1e-9), "groups": int(k_out.numel()),
               "max_rel_err_sum": err_s, "max_rel_err_avg": err_a,
               "checked": "every group against torch index_add_ / bincount"},
              {"keys": nkeys, "partitions": 8, "partitioned_groupby": executor.stats["partitioned_groupby"] > 0,
               "algorithmic_bytes_whole_query": "16 B per row in (+ 24 B per group out)",
               "note": "whole-query fractions use 16 B/row; the roofline entry is the scatter kernel's own "
                       "32 B/row (16 read + 16 written)"})
        # whole-query figure on the compulsory 16 B/row
        out["C5_one_gpu_share"]["algorithmic_gbs_whole_query"] = n * 16 / (ms * 1e-3) / 1e9
        out["C5_one_gpu_share"]["frac_of_peak_whole_query"] = n * 16 / (ms * 1e-3) / 1e9 / peak_gbs

    guarded("C1", c1)
    guarded("C2", lambda: c2("C2", "float"))
    guarded("C2i", lambda: c2("C2i", "int"))
    guarded("C2z", lambda: c2("C2z", "zipf"))
    guarded("C3", lambda: c3("C3", False))
    guarded("C3f", lambda: c3("C3f", True))
    guarded("C4s", c4s)
    guarded("C5", c5)
    return out


if __name__ == "__main__":
    main()
