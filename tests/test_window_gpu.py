"""Window functions on the GPU: the reference's known answers (tests/golden/window_vectors.py), a sqlite3
differential through Context.sql(), and the C-ABI kernels (b2_window_segments / _rank / _offset / _agg)
against numpy at sizes that reach every carry path."""
import ctypes as C
import sqlite3

import numpy as np
import pandas as pd
import pytest

from tests.golden import window_vectors as W

pytestmark = pytest.mark.gpu


def _norm(df):
    out = pd.DataFrame({str(c): pd.to_numeric(df[c]).to_numpy(dtype=float, na_value=np.nan) for c in df.columns})
    if len(out):
        out = out.sort_values(list(out.columns), na_position="last").reset_index(drop=True)
    return out


def assert_same(got, exp, rtol=1e-9, check_names=True, atol=0.0):
    assert len(got.columns) == len(exp.columns), f"{list(got.columns)} vs {list(exp.columns)}"
    if check_names:
        assert [str(c) for c in got.columns] == [str(c) for c in exp.columns]
    g, e = _norm(got), _norm(exp)
    e.columns = g.columns
    assert len(g) == len(e), f"{len(g)} rows vs {len(e)}"
    for c in g.columns:
        np.testing.assert_allclose(g[c].to_numpy(), e[c].to_numpy(), rtol=rtol, atol=atol, equal_nan=True, err_msg=c)


@pytest.fixture()
def c():
    from dask_sql_b200 import Context
    return Context()


@pytest.mark.parametrize("case", W.CASES, ids=[c["name"] for c in W.CASES])
@pytest.mark.parametrize("npartitions", [1, 3])
def test_reference_window_answers(c, case, npartitions):
    for name, df in W.tables_of(case).items():
        c.create_table(name, df, npartitions=npartitions)
    got = c.sql(case["sql"]).compute()
    assert_same(got, case["expected"], rtol=0)


# ---- sqlite3 differential -------------------------------------------------------------------------
def _data(n=400, seed=7):
    rng = np.random.default_rng(seed)
    k1 = rng.integers(0, 6, n).astype(float)
    k1[rng.random(n) < 0.08] = np.nan                      # NULL partition keys form one partition
    k2 = rng.integers(0, 2, n)
    v = rng.normal(0, 10, n).round(3)
    v[rng.random(n) < 0.1] = np.nan
    iv = rng.integers(-50, 50, n).astype(float)
    iv[rng.random(n) < 0.1] = np.nan
    tie = rng.integers(0, 5, n).astype(float)               # ties: only for tie-invariant functions
    tie[rng.random(n) < 0.05] = np.nan
    df = pd.DataFrame({"k1": pd.array(np.where(np.isnan(k1), None, k1), dtype="Int64"), "k2": k2,
                       "t": rng.permutation(n), "v": v, "iv": pd.array(np.where(np.isnan(iv), None, iv), dtype="Int64"),
                       "tie": tie, "flag": rng.random(n) < 0.5})
    return df


def _sqlite_eq(c, sql, df, rtol=1e-9):
    c.create_table("w", df, npartitions=2)
    con = sqlite3.connect(":memory:")
    df.astype({"flag": int}).to_sql("w", con, index=False)
    got = c.sql(sql).compute()
    exp = pd.read_sql(sql, con)
    assert_same(got, exp, rtol=rtol, check_names=False, atol=1e-9)


_SQLITE_QUERIES = [
    # total order inside each partition: (k1, k2) partitions, t unique
    """SELECT k1, k2, t, ROW_NUMBER() OVER (PARTITION BY k1, k2 ORDER BY t) AS rn,
              LAG(v) OVER (PARTITION BY k1, k2 ORDER BY t) AS lg, LEAD(iv, 2, -1) OVER (PARTITION BY k1 ORDER BY t DESC NULLS LAST) AS ld,
              FIRST_VALUE(v) OVER (PARTITION BY k1 ORDER BY t ROWS BETWEEN 2 PRECEDING AND 1 FOLLOWING) AS fv,
              LAST_VALUE(iv) OVER (PARTITION BY k1 ORDER BY t ROWS BETWEEN 1 FOLLOWING AND 4 FOLLOWING) AS lv
       FROM w""",
    """SELECT k1, t, SUM(v) OVER (PARTITION BY k1 ORDER BY t ROWS BETWEEN 3 PRECEDING AND 2 FOLLOWING) AS s,
              AVG(iv) OVER (PARTITION BY k1 ORDER BY t ROWS BETWEEN UNBOUNDED PRECEDING AND 1 PRECEDING) AS a,
              COUNT(v) OVER (PARTITION BY k1 ORDER BY t ROWS BETWEEN 40 PRECEDING AND 35 FOLLOWING) AS cn,
              SUM(iv) OVER (PARTITION BY k1 ORDER BY t ROWS BETWEEN 40 PRECEDING AND 35 FOLLOWING) AS si,
              MIN(v) OVER (PARTITION BY k1 ORDER BY t ROWS BETWEEN 2 FOLLOWING AND UNBOUNDED FOLLOWING) AS mn,
              MAX(iv) OVER (PARTITION BY k1 ORDER BY t ROWS BETWEEN 5 PRECEDING AND 2 PRECEDING) AS mx,
              SUM(flag) OVER (PARTITION BY k1 ORDER BY t) AS sf, COUNT(*) OVER (PARTITION BY k2) AS cs
       FROM w""",
    # ties: RANK / DENSE_RANK and RANGE frames (peer-based) are tie-invariant
    """SELECT k1, t, RANK() OVER (PARTITION BY k1 ORDER BY tie NULLS FIRST) AS r,
              DENSE_RANK() OVER (PARTITION BY k1 ORDER BY tie DESC NULLS LAST) AS dr,
              SUM(iv) OVER (PARTITION BY k1 ORDER BY tie NULLS LAST) AS rs,
              COUNT(*) OVER (PARTITION BY k2 ORDER BY tie NULLS FIRST RANGE BETWEEN CURRENT ROW AND UNBOUNDED FOLLOWING) AS rc,
              MAX(v) OVER (ORDER BY tie NULLS LAST, k2 RANGE BETWEEN CURRENT ROW AND CURRENT ROW) AS pm,
              AVG(v) OVER (PARTITION BY k2, k1) AS pa
       FROM w""",
]


@pytest.mark.parametrize("qi", range(len(_SQLITE_QUERIES)))
def test_window_matches_sqlite(c, qi):
    _sqlite_eq(c, _SQLITE_QUERIES[qi], _data())


def test_grouped_window_and_top_n(c):
    df = _data(2000, seed=3)
    _sqlite_eq(c, """SELECT k2, SUM(iv) AS s, RANK() OVER (ORDER BY SUM(iv) DESC NULLS LAST) AS r,
                            SUM(SUM(iv)) OVER () AS tot
                     FROM w GROUP BY k2""", df)
    _sqlite_eq(c, """SELECT k1, t, rn FROM (SELECT k1, t, ROW_NUMBER() OVER (PARTITION BY k1 ORDER BY v DESC NULLS LAST, t) AS rn
                                           FROM w) s WHERE rn <= 3""", df)
    got = c.sql("""SELECT k1, t, ROW_NUMBER() OVER (PARTITION BY k1 ORDER BY t) AS rn FROM w
                   ORDER BY rn DESC, t LIMIT 5""").compute()
    con = sqlite3.connect(":memory:")
    df.astype({"flag": int}).to_sql("w", con, index=False)
    exp = pd.read_sql("""SELECT k1, t, ROW_NUMBER() OVER (PARTITION BY k1 ORDER BY t) AS rn FROM w
                         ORDER BY rn DESC, t LIMIT 5""", con)
    np.testing.assert_array_equal(got["t"].to_numpy(), exp["t"].to_numpy())
    np.testing.assert_array_equal(got["rn"].to_numpy(), exp["rn"].to_numpy())


def test_default_frame_includes_peers(c):
    """DESIGN section 6: with ORDER BY the default frame is RANGE ... CURRENT ROW (ties share a running
    sum), where the reference's expanding() gives tied rows different sums."""
    c.create_table("p", pd.DataFrame({"k": [1, 1, 1, 1], "o": [1, 2, 2, 3], "v": [1, 10, 100, 1000]}))
    got = c.sql("SELECT o, SUM(v) OVER (PARTITION BY k ORDER BY o) AS s FROM p").compute()
    assert sorted(zip(got["o"], got["s"])) == [(1, 1), (2, 111), (2, 111), (3, 1111)]


# ---- C-ABI ----------------------------------------------------------------------------------------
def _cols(arrays):
    import torch
    from dask_sql_b200 import device as D
    return [D.column_from_host(a, torch.device("cuda")) for a in arrays]


def _segments(keys, npart):
    import torch
    from dask_sql_b200 import _lib as L, device as D
    n = len(keys[0]) if keys else 0
    seg = torch.empty((5, max(n, 1)), dtype=torch.int32, device="cuda")
    segs = L.WSegs(*[seg[i].data_ptr() for i in range(5)])
    ws = torch.empty(L.window_ws_bytes(n), dtype=torch.uint8, device="cuda")
    cols = _cols(keys)
    kc = (L.Col * max(1, len(cols)))(*[x.as_struct() for x in cols])
    L.window_segments(kc, npart, len(cols), n, C.byref(segs), D.ptr(ws), D.stream_ptr())
    return seg[:, :n], segs, ws


def _np_segments(keys, npart):
    n = len(keys[0])

    def diff(a):
        a = np.asarray(a, dtype=float)
        a = np.where(a == 0, 0.0, a)                                 # -0.0 == 0.0
        na = np.isnan(a)
        d = np.ones(n, bool)
        d[1:] = ~((a[1:] == a[:-1]) | (na[1:] & na[:-1]))
        return d

    pf = np.zeros(n, bool)
    pf[0] = True
    for k in keys[:npart]:
        pf |= diff(k)
    qf = pf.copy()
    for k in keys[npart:]:
        qf |= diff(k)
    idx = np.arange(n)
    ps = np.maximum.accumulate(np.where(pf, idx, 0))
    qs = np.maximum.accumulate(np.where(qf, idx, 0))
    nxt = lambda f: np.minimum.accumulate(np.where(np.r_[f[1:], True], np.r_[idx[1:], n], n)[::-1])[::-1]  # noqa: E731
    return ps, nxt(pf), qs, nxt(qf), np.cumsum(qf)


@pytest.mark.parametrize("n", [1, 2, 7, 2048, 2049, 3 * 2048 * 148 + 5, 3_000_001])
def test_segments_match_numpy(n):
    rng = np.random.default_rng(n)
    part = np.sort(rng.integers(0, max(1, n // 700), n)).astype(np.int64)     # partitions spanning tiles
    single = np.arange(n) // 1                                                 # a 1-row partition per row
    order = rng.integers(0, 3, n).astype(float)
    order[rng.random(n) < 0.1] = np.nan
    order[rng.random(n) < 0.1] = -0.0
    order = np.concatenate([np.sort(order[part == p]) for p in np.unique(part)]) if n else order
    for keys, npart in [([part, order], 1), ([part], 1), ([order], 0), ([single], 1)]:
        seg, _, _ = _segments(keys, npart)
        exp = _np_segments(keys, npart)
        got = seg.cpu().numpy()
        for i in range(5):
            np.testing.assert_array_equal(got[i], exp[i], err_msg=f"array {i}, npart={npart}")


def test_segments_of_zero_rows_and_one_partition_of_50m_rows():
    import torch
    _segments([np.zeros(0, np.int64)], 1)
    torch.cuda.synchronize()
    n = 50_000_000
    seg, segs, ws = _segments([np.zeros(n, np.int64)], 1)
    assert int(seg[0].max()) == 0 and int(seg[1].min()) == n and int(seg[4][-1]) == 1
    _check_agg_running_sum_int(n, segs, ws, np.zeros(n, np.int64))


def _agg(val, op, frame, segs, ws, n, dtype):
    import torch
    from dask_sql_b200 import _lib as L, device as D
    vs = val.as_struct() if val is not None else L.Col()
    out = torch.empty(n, dtype=dtype, device="cuda")
    valid = torch.empty(max(1, (n + 31) // 32), dtype=torch.int32, device="cuda")
    L.window_agg(C.byref(vs), op, C.byref(frame), n, C.byref(segs), D.ptr(out),
                 D.ptr(valid) if op != L.WIN_COUNT else None, D.ptr(ws), D.stream_ptr())
    mask = np.unpackbits(valid.cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool)
    return out.cpu().numpy(), mask


def _check_agg_running_sum_int(n, segs, ws, part):
    import torch
    from dask_sql_b200 import _lib as L
    rng = np.random.default_rng(1)
    v = rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)       # wraps
    (col,) = _cols([v])
    fr = L.WFrame(0, L.WB_UNBOUNDED, L.WB_OFFSET, 0, 0, 0)
    got, ok = _agg(col, L.WIN_SUM, fr, segs, ws, n, torch.int64)
    exp = pd.Series(v).groupby(part).cumsum().to_numpy()
    assert ok.all()
    np.testing.assert_array_equal(got, exp)


def _np_frame_sum(v, part_start, part_end, lo, hi):
    """int64 wrapping SUM over ROWS BETWEEN lo AND hi (signed offsets) via exact prefix differences."""
    n = len(v)
    cs = np.concatenate([[0], np.cumsum(v)])
    i = np.arange(n)
    fs = np.maximum(i + lo, part_start)
    fe = np.minimum(i + hi, part_end - 1)
    empty = fs > fe
    fs, fe = np.clip(fs, 0, n - 1), np.clip(fe, 0, n - 1)
    return cs[fe + 1] - cs[fs], empty


@pytest.mark.parametrize("lo,hi", [(-5, 3), (-100, 40), (2, 7), (-7, -1), (-3000, 3000)])
def test_framed_int_sum_matches_prefix_differences(lo, hi):
    import torch
    from dask_sql_b200 import _lib as L
    n = 2_000_003
    rng = np.random.default_rng(abs(lo))
    part = np.sort(rng.integers(0, 3000, n)).astype(np.int64)
    part[: 5000] = np.arange(5000)                                   # 1-row partitions at the start
    part = np.sort(part)
    v = rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)
    seg, segs, ws = _segments([part], 1)
    ps, pe = seg[0].cpu().numpy(), seg[1].cpu().numpy()
    (col,) = _cols([v])
    fr = L.WFrame(0, L.WB_OFFSET, L.WB_OFFSET, 0, lo, hi)
    got, ok = _agg(col, L.WIN_SUM, fr, segs, ws, n, torch.int64)
    exp, empty = _np_frame_sum(v, ps, pe, lo, hi)
    np.testing.assert_array_equal(ok, ~empty)
    np.testing.assert_array_equal(got[~empty], exp[~empty])
    cnt, _ = _agg(col, L.WIN_COUNT, fr, segs, ws, n, torch.int64)
    np.testing.assert_array_equal(cnt, np.where(empty, 0, np.minimum(np.arange(n) + hi, pe - 1)
                                                - np.maximum(np.arange(n) + lo, ps) + 1))


def test_float_sum_and_avg_are_bit_identical_between_runs():
    import torch
    from dask_sql_b200 import _lib as L
    n = 10_000_000
    rng = np.random.default_rng(5)
    v = rng.normal(0, 1e6, n)
    v[rng.random(n) < 0.01] = np.nan
    part = np.sort(rng.integers(0, 3, n)).astype(np.int64)
    _, segs, ws = _segments([part], 1)
    (col,) = _cols([v])
    for fr in (L.WFrame(0, L.WB_UNBOUNDED, L.WB_OFFSET, 0, 0, 0), L.WFrame(0, L.WB_OFFSET, L.WB_UNBOUNDED, 0, -3, 0)):
        for op in (L.WIN_SUM, L.WIN_AVG):
            a, ma = _agg(col, op, fr, segs, ws, n, torch.float64)
            b, mb = _agg(col, op, fr, segs, ws, n, torch.float64)
            assert a.tobytes() == b.tobytes() and (ma == mb).all()
    run, ok = _agg(col, L.WIN_SUM, L.WFrame(0, L.WB_UNBOUNDED, L.WB_OFFSET, 0, 0, 0), segs, ws, n, torch.float64)
    # a NULL row keeps the running sum of the rows before it (pandas' cumsum puts NaN there instead)
    exp = pd.Series(np.nan_to_num(v)).groupby(part).cumsum().to_numpy()
    has = pd.Series(~np.isnan(v)).groupby(part).cumsum().to_numpy() > 0
    np.testing.assert_array_equal(ok, has)
    np.testing.assert_allclose(run[has], exp[has], rtol=1e-9, atol=1e-3 * np.abs(v[~np.isnan(v)]).max())


def test_rank_and_offset_kernels():
    import torch
    from dask_sql_b200 import _lib as L, device as D
    part = np.array([0, 0, 0, 0, 1, 1, 2], np.int64)
    order = np.array([1, 1, 2, 3, 5, 5, 0], np.int64)
    seg, segs, ws = _segments([part, order], 1)
    n = 7
    out = torch.empty(n, dtype=torch.int64, device="cuda")
    exp = {L.WIN_ROW_NUMBER: [1, 2, 3, 4, 1, 2, 1], L.WIN_RANK: [1, 1, 3, 4, 1, 1, 1],
           L.WIN_DENSE_RANK: [1, 1, 2, 3, 1, 1, 1]}
    for op, e in exp.items():
        L.window_rank(op, n, C.byref(segs), D.ptr(out), D.stream_ptr())
        assert out.cpu().tolist() == e
    (val,) = _cols([np.array([10, 11, 12, 13, 14, 15, 16], np.int64)])
    vs = val.as_struct()
    valid = torch.empty(1, dtype=torch.int32, device="cuda")
    L.window_offset(C.byref(vs), n, -1, 0, 0, C.byref(segs), D.ptr(out), D.ptr(valid), D.stream_ptr())
    bits = int(valid.cpu().numpy().view(np.uint32)[0])
    got = [v if (bits >> i) & 1 else None for i, v in enumerate(out.cpu().tolist())]
    assert got == [None, 10, 11, 12, None, 14, None]
    L.window_offset(C.byref(vs), n, 2, 1, -7, C.byref(segs), D.ptr(out), D.ptr(valid), D.stream_ptr())
    assert out.cpu().tolist() == [12, 13, -7, -7, -7, -7, -7]
