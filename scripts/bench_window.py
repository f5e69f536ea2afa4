"""Window-function benchmark on one GPU: a 200M-row HBM-resident table w(k, t, v) with k uniform over
1M / 100 / 1 partitions, t a unique order key and v float64 with 1 % NULL, running

    SELECT k, t, v,
           ROW_NUMBER() OVER (PARTITION BY k ORDER BY t)                                        AS rn,
           SUM(v)       OVER (PARTITION BY k ORDER BY t)                                        AS run,
           AVG(v)       OVER (PARTITION BY k ORDER BY t ROWS BETWEEN 7 PRECEDING AND CURRENT ROW) AS ma8,
           LAG(v)       OVER (PARTITION BY k ORDER BY t)                                        AS prev
    FROM w

through Context.sql() (results stay on the device).  Prints one JSON line: card and power limit, per-phase
CUDA-event times (sort, gather, segments, each window kernel), algorithmic bytes/row and share of the HBM
peak per window kernel, whole-query rows/s, full-size verification with torch ops, and a pandas arm on a
10M-row sample.  Usage: python scripts/bench_window.py [--rows N] [--steps K] [--warmup W] [--out FILE]"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

QUERY = """SELECT k, t, v,
       ROW_NUMBER() OVER (PARTITION BY k ORDER BY t) AS rn,
       SUM(v) OVER (PARTITION BY k ORDER BY t) AS run,
       AVG(v) OVER (PARTITION BY k ORDER BY t ROWS BETWEEN 7 PRECEDING AND CURRENT ROW) AS ma8,
       LAG(v) OVER (PARTITION BY k ORDER BY t) AS prev
FROM w"""

# algorithmic bytes per row of each window kernel: the values it must read and write, plus the int32
# segment arrays it reads (partition / peer bounds)
BYTES_PER_ROW = {
    "window_segments": 8 * 2 + 5 * 4,          # partition key + order key in; 5 int32 segment arrays out
    "window_row_number": 4 + 8,                # part_start in; int64 out
    "window_sum": 8 + 4 + 4 + 8,               # v, part_start, peer_end in; float64 out
    "window_avg": 8 + 4 + 4 + 8,               # v, part_start, part_end in; float64 out
    "window_lag": 8 + 4 + 4 + 8,               # v, part_start, part_end in; float64 out
}


def card():
    out = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        out["power_limit_w"] = nv.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception as e:  # pragma: no cover
        out["power_limit_error"] = type(e).__name__
    return out


def make_table(n, parts, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    k = torch.randint(0, parts, (n,), device="cuda", generator=g, dtype=torch.int64)
    t = torch.randperm(n, device="cuda", generator=g).to(torch.int64)
    v = torch.randn(n, device="cuda", generator=g, dtype=torch.float64) * 100.0
    v[torch.rand(n, device="cuda", generator=g) < 0.01] = float("nan")
    return {"k": k, "t": t, "v": v}


def verify(cols, parts):
    """size-independent properties of the full result, with torch ops"""
    k, rn, run, v, prev = cols["k"], cols["rn"], cols["run"], cols["v"], cols["prev"]
    n = k.numel()
    cnt = torch.bincount(k, minlength=parts)
    mx = torch.zeros(parts, dtype=torch.int64, device="cuda").scatter_reduce(0, k, rn, reduce="amax")
    ok_rn = bool(torch.equal(mx, cnt)) and int(rn.sum()) == int((cnt * (cnt + 1) // 2).sum())
    last = torch.ones(n, dtype=torch.bool, device="cuda")
    last[:-1] = k[1:] != k[:-1]
    nansum = torch.zeros(parts, dtype=torch.float64, device="cuda").index_add_(0, k, torch.nan_to_num(v, nan=0.0))
    exp = nansum[k[last]]
    got = run[last]
    rel = ((got - exp).abs() / exp.abs().clamp_min(1.0)).max().item()
    same = torch.zeros(n, dtype=torch.bool, device="cuda")
    same[1:] = k[1:] == k[:-1]
    pv, vv = prev[1:][same[1:]], v[:-1][same[1:]]
    ok_prev = bool(torch.equal(torch.isnan(pv), torch.isnan(vv))) and \
        bool(torch.equal(pv[~torch.isnan(pv)], vv[~torch.isnan(vv)])) and bool(torch.isnan(prev[~same]).all())
    return {"rn": ok_rn, "run_rel_err": rel, "run": rel <= 1e-9, "prev": ok_prev}


def cpu_arm(rows, parts, seed):
    import pandas as pd
    rng = np.random.default_rng(seed)
    v = rng.normal(0, 100, rows)
    v[rng.random(rows) < 0.01] = np.nan
    df = pd.DataFrame({"k": rng.integers(0, parts, rows), "t": rng.permutation(rows), "v": v})
    t0 = time.perf_counter()
    s = df.sort_values(["k", "t"], kind="stable")
    g = s.groupby("k", sort=False)["v"]
    s = s.assign(rn=g.cumcount() + 1, run=g.cumsum(), ma8=g.rolling(8, min_periods=1).mean().reset_index(level=0, drop=True),
                 prev=g.shift())
    dt = time.perf_counter() - t0
    return {"rows": rows, "seconds": dt, "rows_per_s": rows / dt, "impl": "pandas sort + groupby cumsum/rolling(8)/shift"}


def run_config(rows, parts, steps, warmup, peak_gbs):
    from dask_sql_b200 import Context, executor as X
    c = Context()
    c.create_table("w", make_table(rows, parts, seed=parts), persist=True)
    lf = c.sql(QUERY)
    for _ in range(warmup):
        X.execute(lf)
        torch.cuda.synchronize()
    X.prefill_timing_events(64 * steps)
    X.kernel_events = []
    times, out = [], None
    try:
        for _ in range(steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = X.execute(lf)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) * 1e-3)
        kev = X.kernel_events
    finally:
        X.kernel_events = None
    phases = {}
    for name, nrows, a, b in kev:
        phases.setdefault(name, []).append(a.elapsed_time(b) * 1e-3)
    # per query: median launch time x launches per query (medians, like the query time: the GPU is shared)
    phases = {k: sorted(v)[len(v) // 2] * (len(v) / steps) for k, v in phases.items()}
    step = sorted(times)[len(times) // 2]
    kernels = {}
    for name, bpr in BYTES_PER_ROW.items():
        if name in phases:
            gbs = rows * bpr / phases[name] / 1e9
            kernels[name] = {"ms": phases[name] * 1e3, "bytes_per_row": bpr, "gb_s": gbs, "hbm_share": gbs / peak_gbs}
    part = out[0]
    cols = {name: part[name].data for name in ("k", "t", "v", "rn", "run", "prev")}
    ver = verify(cols, parts)
    ver["ok"] = ver["rn"] and ver["run"] and ver["prev"]
    del out, part, cols, lf
    c.drop_table("w")
    torch.cuda.empty_cache()
    return {"partitions": parts, "rows": rows, "query_ms": step * 1e3, "rows_per_s": rows / step,
            "phase_ms": {k: v * 1e3 for k, v in phases.items()},
            "sort_share": phases.get("window_sort", 0.0) / step, "kernels": kernels, "verify": ver}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=200_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--cpu-rows", type=int, default=10_000_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    from bench import load_peaks
    peak_gbs, peak_src = load_peaks()
    res = {"bench": "window", "card": card(), "hbm_peak_gbs": peak_gbs, "hbm_peak_src": peak_src,
           "query": " ".join(QUERY.split()), "configs": []}
    for parts in (1_000_000, 100, 1):
        res["configs"].append(run_config(a.rows, parts, a.steps, a.warmup, peak_gbs))
    res["cpu"] = cpu_arm(a.cpu_rows, 1_000_000 * a.cpu_rows // a.rows or 1, seed=1)
    res["verify"] = "ok" if all(c["verify"]["ok"] for c in res["configs"]) else "FAILED"
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0 if res["verify"] == "ok" else 1


if __name__ == "__main__":
    sys.exit(main())
