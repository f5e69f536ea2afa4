"""bench.py's own checking code, on CPU: the full-size verifier must accept the right answer and reject the
failures it exists for (round 1's N=8 run returned phantom groups and nothing noticed), the roofline
arithmetic must be what DESIGN.md says it is, and both arms must describe the same workload."""
import importlib.util
import os
import sys

import numpy as np
import pandas as pd
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec = importlib.util.spec_from_file_location("b200_bench", os.path.join(ROOT, "bench.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    finally:
        sys.argv = argv


class _Col:
    def __init__(self, t):
        self.data = t


def _q3(nf=20_000, nd=500, ngroups=60, seed=3):
    rng = np.random.default_rng(seed)
    pk = rng.permutation(nd).astype(np.int64)
    flag = rng.integers(0, 10, nd)
    grp = rng.integers(0, ngroups, nd)
    fk = rng.integers(0, nd, nf)
    x = rng.integers(-100, 100, nf)
    val = rng.random(nf)
    fact = pd.DataFrame({"fk": fk, "x": x, "val": val})
    dim = pd.DataFrame({"pk": pk, "flag": flag, "grp": grp})
    e = fact[fact.x > 0].merge(dim[dim.flag < 5], left_on="fk", right_on="pk")
    exp = e.groupby("grp").agg(rev=("val", "sum")).reset_index()
    t = lambda a: torch.from_numpy(np.asarray(a))
    return (t(fk), t(x), t(val), t(pk), t(flag), t(grp)), exp


def _parts(keys, rev):
    return [{"grp": _Col(torch.tensor(np.array(keys, dtype=np.int64))),
             "rev": _Col(torch.tensor(np.array(rev, dtype=np.float64)))}]


def test_full_size_verifier_accepts_the_right_answer_and_rejects_wrong_ones(bench):
    cols, exp = _q3()
    assert len(exp) < 60, "the data must leave some groups without any row"
    ok = bench.verify_full_size(torch, None, 1, _parts(exp.grp, exp.rev), *cols)
    assert ok["ok"] and ok["groups"] == ok["groups_expected"] == len(exp) and ok["keys_unique"]
    assert ok["rows_contributing"] > 0 and ok["sum_of_group_sums_rel_err"] <= 1e-9

    # a phantom group with sum 0.0 (what a lost -0.0 existence mark produces): the checksum still matches,
    # the group count does not
    missing = sorted(set(range(60)) - set(exp.grp.tolist()))[0]
    bad = bench.verify_full_size(torch, None, 1, _parts(list(exp.grp) + [missing], list(exp.rev) + [0.0]), *cols)
    assert not bad["ok"] and bad["groups"] == bad["groups_expected"] + 1 and bad["sum_of_group_sums_rel_err"] <= 1e-9

    # a lost group, a wrong sum, a duplicated key
    assert not bench.verify_full_size(torch, None, 1, _parts(exp.grp[1:], exp.rev[1:]), *cols)["ok"]
    rev = exp.rev.to_numpy().copy()
    rev[0] *= 1.0 + 1e-6
    assert not bench.verify_full_size(torch, None, 1, _parts(exp.grp, rev), *cols)["ok"]
    dup_keys = exp.grp.to_numpy().copy()
    dup_keys[1] = dup_keys[0]
    assert not bench.verify_full_size(torch, None, 1, _parts(dup_keys, exp.rev), *cols)["ok"]


def test_roofline_arithmetic(bench):
    class Ev:
        def __init__(self, t):
            self.t = t

        def elapsed_time(self, other):
            return other.t - self.t

    kev = [["k", 125_000_000, Ev(0.0), Ev(0.5)], ["k", 125_000_000, Ev(1.0), Ev(1.7)], ["other", 1, Ev(0), Ev(9)]]
    r = bench.kernel_roofline(kev, "k", 24, 6564.2, "measured", {"k": {"dram_bytes_per_row": 26.0}}, 0.005, 1)
    assert r["launches_timed"] == 2 and abs(r["avg_launch_ms"] - 0.6) < 1e-12
    assert abs(r["achieved"] - 125e6 * 24 / 0.6e-3 / 1e9) < 1e-6            # algorithmic bytes / mean launch time
    assert abs(r["frac"] - r["achieved"] / 6564.2) < 1e-12
    assert r["traffic"] == 26.0 * 125_000_000 and r["algorithmic_bytes_per_launch"] == 24 * 125_000_000
    assert abs(r["kernel_share_of_step"] - 1.2e-3 / 0.005) < 1e-9
    assert bench.kernel_roofline(kev, "absent", 24, 6564.2, "m", {}) is None
    assert bench.kernel_roofline(kev, "k", 24, 6564.2, "m", {})["traffic"] is None


def test_both_arms_describe_the_same_workload(bench, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    args = bench.parse_args()
    for n in (1, 2, 4, 8):
        a, b = bench.workload_config(args, n), bench.workload_config(args, n)
        assert a == b and a["fact_rows_per_gpu"] * n == a["fact_rows_total"]
        assert a["partitions_per_gpu"] == max(1, 8 // n) and a["query"] == bench.QUERY
    # nothing in the description may depend on what ran in THIS process (the reference arm never loads the kernels)
    import dask_sql_b200.executor as X
    before = dict(X.stats)
    try:
        X.stats["peer_merge_plans"] = 3
        assert bench.workload_config(args, 8) == a
        assert "b2_peer_merge" in bench.merge_kind()
        X.stats["peer_merge_plans"] = 0
        assert "ncclReduceScatter" in bench.merge_kind()
    finally:
        X.stats.clear()
        X.stats.update(before)


def test_arguments_that_cannot_be_honoured_are_refused(bench, monkeypatch):
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
        with pytest.raises(SystemExit):
            bench.parse_args()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--dump-outputs", "out"])
    args = bench.parse_args()
    assert args.steps == 7 and args.dump_outputs == "out"


def test_dump_outputs_writes_the_result_in_key_order(bench, tmp_path, monkeypatch):
    from dask_sql_b200 import device as D
    rng = np.random.default_rng(7)
    keys = rng.permutation(1000).astype(np.int64) * 3 + 5
    rev = rng.random(1000)

    def part(lo, hi):
        return {"grp": D.DeviceColumn(torch.from_numpy(keys[lo:hi].copy()), None, D.I64),
                "rev": D.DeviceColumn(torch.from_numpy(rev[lo:hi].copy()), None, D.F64)}

    parts = [part(0, 400), part(400, 1000)]
    bench.dump_outputs(str(tmp_path / "all"), parts, 0)
    order = np.argsort(keys)
    for name, exp in (("grp", keys[order].astype(np.float64)), ("rev", rev[order])):
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == np.float64
        np.testing.assert_array_equal(got, exp)

    # a result above the size limit: the same seeded sample of rows every time, still in key order
    monkeypatch.setattr(bench, "DUMP_ARRAY_BYTES", 16 * 100)
    bench.dump_outputs(str(tmp_path / "a"), parts, 0)
    bench.dump_outputs(str(tmp_path / "b"), parts[::-1], 0)
    ga, ra = np.load(tmp_path / "a" / "grp.npy"), np.load(tmp_path / "a" / "rev.npy")
    assert len(ga) == len(ra) == 100 and np.all(np.diff(ga) > 0)
    np.testing.assert_array_equal(ga, np.load(tmp_path / "b" / "grp.npy"))
    by_key = dict(zip(keys.astype(np.float64), rev))
    assert [by_key[k] for k in ga] == ra.tolist()

    bench.dump_outputs(str(tmp_path / "other"), parts, 1)      # only rank 0 writes
    assert not (tmp_path / "other").exists()


def test_cpu_arm_runs_the_configured_partitioning(bench, monkeypatch):
    """The reference arm on a tiny sample: 8 partitions (the configuration's), the full dim table, the
    fields VERDICT r01 asked for."""
    monkeypatch.setattr(bench, "DIM_ROWS", 2_000)
    monkeypatch.setattr(bench, "N_GROUPS", 100)
    monkeypatch.setattr(os, "cpu_count", lambda: 4)
    out = bench.run_cpu_baseline(64_000, steps=1, warmup=0, budget_s=60.0)
    assert out["partitions"] == 8 and out["threads_used"] == 4 and out["kind"] == "port"
    assert out["dim_rows"] == 2_000 and out["sample_rows"] >= 64_000 - 1 and out["value"] > 0
    assert set(out["layout_trials_rows_per_s"]) == {"8"} and 0 < out["groups_out"] <= 100


# ---- the same verifier over two gloo ranks: fact rows split by row range, result split by key range ----------
def _verify_worker(rank, size, port, case, out_q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=size)
    try:
        argv, sys.argv = sys.argv, ["bench.py"]
        spec = importlib.util.spec_from_file_location("b200_bench", os.path.join(ROOT, "bench.py"))
        bench = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(bench)
        sys.argv = argv
        (fk, x, val, pk, flag, grp), exp = _q3()
        n = fk.numel()
        lo, hi = n * rank // size, n * (rank + 1) // size            # this rank's fact shard
        missing = sorted(set(range(60)) - set(exp.grp.tolist()))[-1]   # the largest group id that no row reaches
        cut = missing                                                  # key ranges: [0, cut) and [cut, 60)
        assert 0 < cut < 59
        mine = exp[(exp.grp < cut) == (rank == 0)]
        keys, rev = list(mine.grp), list(mine.rev)
        if case == "phantom" and rank == 1:                            # a group nobody saw, on one rank only
            keys, rev = [missing] + keys, [0.0] + rev
        if case == "overlap" and rank == 1:                            # a key of rank 0's range shows up on rank 1 too
            k0 = int(exp.grp[exp.grp < cut].iloc[-1])
            keys, rev = [k0] + keys, [0.0] + rev
        out = bench.verify_full_size(torch, dist, size, _parts(keys, rev), fk[lo:hi], x[lo:hi], val[lo:hi], pk, flag, grp)
        out_q.put((rank, case, out["ok"], out["groups"], out["groups_expected"], out["keys_unique"]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("case", ["good", "phantom", "overlap"])
def test_full_size_verifier_over_two_ranks(case):
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_verify_worker, args=(r, 2, port, case, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, _, ok, groups, expected, unique in results:           # every rank reaches the same verdict
        if case == "good":
            assert ok and groups == expected and unique
        elif case == "phantom":
            assert not ok and groups == expected + 1
        else:
            assert not ok and not unique
