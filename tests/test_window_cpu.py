"""Window functions without a GPU: parsing, binding, the Window plan node and its method surface,
EXPLAIN text, filter placement, rejected forms, and the lazy WindowSource built by Context.sql()."""
import pandas as pd
import pytest

from dask_sql_b200.utils import ParsingException


def _catalog(schema, table):
    if table == "t":
        return "root", [("k", "BIGINT"), ("o", "BIGINT"), ("v", "DOUBLE"), ("rows", "BIGINT"), ("range", "BIGINT"),
                        ("row", "BIGINT")]
    return None


def _plan(sql):
    from dask_sql_b200.planner import plan_sql
    return plan_sql(sql, _catalog)


def _window_node(plan):
    from dask_sql_b200.planner import plan as P
    nodes = [n for n in P.walk(plan) if n.get_current_node_type() == "Window"]
    assert len(nodes) == 1
    return nodes[0]


@pytest.mark.parametrize("clause,lo,hi,unit", [
    ("ROWS BETWEEN UNBOUNDED PRECEDING AND CURRENT ROW", ("UNBOUNDED_PRECEDING", None), ("CURRENT", 0), "ROWS"),
    ("ROWS BETWEEN 3 PRECEDING AND 2 FOLLOWING", ("PRECEDING", 3), ("FOLLOWING", 2), "ROWS"),
    ("ROWS BETWEEN 2 FOLLOWING AND UNBOUNDED FOLLOWING", ("FOLLOWING", 2), ("UNBOUNDED_FOLLOWING", None), "ROWS"),
    ("ROWS BETWEEN 3 PRECEDING AND 1 PRECEDING", ("PRECEDING", 3), ("PRECEDING", 1), "ROWS"),
    ("ROWS 5 PRECEDING", ("PRECEDING", 5), ("CURRENT", 0), "ROWS"),
    ("ROWS BETWEEN 2147483647 PRECEDING AND CURRENT ROW", ("PRECEDING", 2147483647), ("CURRENT", 0), "ROWS"),
    ("RANGE BETWEEN CURRENT ROW AND UNBOUNDED FOLLOWING", ("CURRENT", 0), ("UNBOUNDED_FOLLOWING", None), "RANGE"),
    ("RANGE UNBOUNDED PRECEDING", ("UNBOUNDED_PRECEDING", None), ("CURRENT", 0), "RANGE"),
])
def test_frames_parse_and_bind(clause, lo, hi, unit):
    w = _window_node(_plan(f"SELECT SUM(v) OVER (PARTITION BY k ORDER BY o {clause}) AS s FROM t"))
    (call,) = w.getGroups()
    fr = w.getWindowFrame(call)
    assert fr.getFrameUnits() == unit
    for b, (kind, off) in ((fr.getLowerBound(), lo), (fr.getUpperBound(), hi)):
        assert b.isUnbounded() == kind.startswith("UNBOUNDED")
        assert b.isPreceding() == kind.endswith("PRECEDING") and b.isFollowing() == kind.endswith("FOLLOWING")
        assert b.isCurrentRow() == (kind == "CURRENT")
        assert b.getOffset() == (off if kind in ("PRECEDING", "FOLLOWING") else None)


def test_columns_named_like_frame_words_still_parse():
    p = _plan("SELECT rows, range, row, k over FROM t WHERE rows > 1 ORDER BY range")
    assert p.getRowType().getFieldNames() == ["t.rows", "t.range", "t.row", "over"]
    p = _plan("SELECT SUM(rows) over FROM t")        # OVER without "(" after a call is an alias
    assert p.getRowType().getFieldNames() == ["over"]


def test_window_node_surface_and_explain():
    p = _plan("""SELECT k, ROW_NUMBER() OVER (PARTITION BY k ORDER BY o DESC NULLS FIRST) AS rn,
                        LAG(v, 2, 0.5) OVER (ORDER BY o) AS lg, COUNT(*) OVER () AS n FROM t""")
    assert p.get_current_node_type() == "Projection"
    w = _window_node(p)
    assert w.get_inputs()[0].get_current_node_type() == "TableScan"
    rn, lg, n = w.window().getGroups()
    assert [w.getWindowFuncName(x) for x in (rn, lg, n)] == ["ROW_NUMBER", "LAG", "COUNT"]
    assert [e.display() for e in w.getPartitionExprs(rn)] == ["t.k"] and w.getPartitionExprs(n) == []
    (s,) = w.getSortExprs(rn)
    assert (s.getSortExpr().display(), s.isSortAscending(), s.isSortNullsFirst()) == ("t.o", False, True)
    (s,) = w.getSortExprs(lg)
    assert (s.isSortAscending(), s.isSortNullsFirst()) == (True, False)          # NULLS LAST for ASC
    assert w.getWindowFrame(rn) is None and [a.display() for a in w.getArgs(lg)] == ["t.v", "Int64(2)",
                                                                                      "Float64(0.5)"]
    names = w.getRowType().getFieldNames()
    assert names[:3] == ["t.k", "t.o", "t.v"] and len(names) == 6
    assert [f.sql_type for f in w.schema[3:]] == ["BIGINT", "DOUBLE", "BIGINT"]
    text = p.explain()
    assert text.splitlines()[1].strip().startswith(
        "Window: windowExpr=[[ROW_NUMBER() PARTITION BY [t.k] ORDER BY [t.o DESC NULLS FIRST]")
    assert "COUNT(*)]]" in text


def test_grouped_query_runs_the_window_after_aggregate_and_having():
    p = _plan("""SELECT k, SUM(v) AS s, RANK() OVER (ORDER BY SUM(v) DESC) AS r, SUM(SUM(v)) OVER () AS tot
                 FROM t GROUP BY k HAVING COUNT(*) > 1 ORDER BY r""")
    lines = [ln.strip() for ln in p.explain().splitlines()]
    kinds = [ln.split(":")[0] for ln in lines]
    assert kinds == ["Sort", "Projection", "Window", "Filter", "Aggregate", "TableScan"]
    assert "SUM(SUM(t.v))" in lines[2] and "ORDER BY [SUM(t.v) DESC NULLS FIRST]" in lines[2]
    # SUM(x) OVER () alone is not a GROUP BY
    p = _plan("SELECT k, SUM(v) OVER () AS s FROM t")
    assert "Aggregate" not in p.explain()


def test_filters_on_window_columns_stay_above_the_node():
    p = _plan("""SELECT * FROM (SELECT k, o, ROW_NUMBER() OVER (PARTITION BY k ORDER BY o) AS rn FROM t) s
                 WHERE rn <= 3 AND k > 1 AND o > 0""")
    lines = [ln.strip() for ln in p.explain().splitlines()]
    wi = next(i for i, ln in enumerate(lines) if ln.startswith("Window:"))
    assert lines[wi - 1].startswith("Filter:") and "ROW_NUMBER()" in lines[wi - 1] and "t.o > Int64(0)" in lines[wi - 1]
    assert lines[-1] == "TableScan: t projection=[k, o], full_filters=[t.k > Int64(1)]"


@pytest.mark.parametrize("sql,exc", [
    ("SELECT k FROM t WHERE ROW_NUMBER() OVER () > 1", ParsingException),
    ("SELECT k FROM t GROUP BY ROW_NUMBER() OVER ()", ParsingException),
    ("SELECT k FROM t GROUP BY k HAVING SUM(v) OVER () > 1", ParsingException),
    ("SELECT SUM(ROW_NUMBER() OVER ()) OVER () FROM t", ParsingException),
    ("SELECT LAG(v, o) OVER (ORDER BY o) FROM t", ParsingException),
    ("SELECT SUM(v) OVER (ORDER BY o ROWS BETWEEN 2147483648 PRECEDING AND CURRENT ROW) FROM t", ParsingException),
    ("SELECT SUM(v) OVER (ORDER BY o ROWS BETWEEN CURRENT ROW AND 1 PRECEDING) FROM t", ParsingException),
    ("SELECT SUM(v) OVER (ORDER BY o ROWS BETWEEN UNBOUNDED FOLLOWING AND CURRENT ROW) FROM t", ParsingException),
    ("SELECT SUM(v) OVER (PARTITION k) FROM t", ParsingException),
    ("SELECT SUM(v) OVER (ORDER BY o RANGE BETWEEN 1 PRECEDING AND CURRENT ROW) FROM t", NotImplementedError),
    ("SELECT COUNT(DISTINCT v) OVER () FROM t", NotImplementedError),
    ("SELECT SUM(v) FILTER (WHERE v > 0) OVER () FROM t", NotImplementedError),
    ("SELECT NTILE(4) OVER (ORDER BY o) FROM t", NotImplementedError),
])
def test_rejected_forms(sql, exc):
    with pytest.raises(exc):
        _plan(sql)


def test_context_builds_a_window_source_without_a_gpu():
    from dask_sql_b200 import Context
    from dask_sql_b200.frame import LazyFrame, WindowSource
    c = Context()
    c.create_table("t", pd.DataFrame({"k": [1, 1, 2], "o": [3, 1, 2], "v": [0.5, 1.5, 2.5], "b": [True, False, True]}))
    lf = c.sql("""SELECT k, ROW_NUMBER() OVER (PARTITION BY k ORDER BY o) AS rn,
                         SUM(v) OVER (PARTITION BY k ORDER BY o ROWS BETWEEN 1 PRECEDING AND CURRENT ROW) AS s,
                         AVG(o) OVER (PARTITION BY k ORDER BY o) AS a, LEAD(b) OVER (ORDER BY o) AS ld,
                         COUNT(*) OVER () AS n
                  FROM t""")
    assert isinstance(lf, LazyFrame) and lf.columns == ["k", "rn", "s", "a", "ld", "n"]
    src = lf.source
    assert isinstance(src, WindowSource)
    funcs = [w.func for w in src.calls]
    assert funcs == ["row_number", "sum", "avg", "lead", "count"]
    rn, s, a, ld, n = src.calls
    assert rn.partition == ("k",) and rn.order == (("o", True, False),)
    assert s.frame == ("ROWS", ("PRECEDING", 1), ("CURRENT", 0))
    assert a.frame == ("RANGE", ("UNBOUNDED_PRECEDING", None), ("CURRENT", 0))      # SQL's default frame
    assert ld.params == (1, None) and n.partition == () and n.order == ()
    assert [str(lf.dtype_of(x)) for x in lf.columns] == ["int64", "int64", "float64", "float64", "bool", "int64"]
