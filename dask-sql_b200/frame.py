"""Lazy, device-resident frame objects: the B200 layer's stand-in for dask.dataframe.

The reference's plugins return DataContainer(df, cc) where df is a lazy dask DataFrame that
supports df[cols], df[mask], .assign, .merge, .groupby().agg, .columns, .dtypes, .compute()
(SURVEY 8b; datacontainer.py:190-231, context.py:908-910).  LazyFrame offers that surface, but
instead of a task graph of pandas calls it records

    source  (device table | join | aggregate)
    exprs   {output column -> expression over the source's columns}
    pred    [conjuncts over the source's columns]

so chains of Filter / Projection / TableScan nodes collapse into ONE fused kernel pass at
.compute() (executor.py) rather than one pandas pass per operator.
"""
import itertools
from collections import OrderedDict
from typing import Dict, List, NamedTuple, Sequence

import numpy as np

from . import expr as E
from .expr import Expr, ColRef, Lit, I64, F64, U8

_NP_DTYPE = {I64: np.dtype("int64"), F64: np.dtype("float64"), U8: np.dtype("bool")}
_uid = itertools.count()


# ---------------------------------------------------------------------------------------------
# sources
# ---------------------------------------------------------------------------------------------
class Source:
    """schema: OrderedDict name -> (dtype, logical)"""
    schema: "OrderedDict[str, tuple]"

    def colref(self, name) -> ColRef:
        dt, lg = self.schema[name]
        return ColRef(name, dt, lg)


class TableSource(Source):
    def __init__(self, table):
        self.table = table
        self.schema = OrderedDict((n, (dt, lg)) for n, dt, lg in table.schema())


class JoinSource(Source):
    def __init__(self, left: "LazyFrame", right: "LazyFrame", left_on, right_on, how, broadcast=None):
        dup = set(left.columns) & set(right.columns)
        if dup:
            raise ValueError(f"join inputs share column names {sorted(dup)}; rename first")
        self.left, self.right = left, right
        self.left_on, self.right_on, self.how = list(left_on), list(right_on), how
        self.broadcast = broadcast
        self.schema = OrderedDict()
        for n in left.columns:
            self.schema[n] = left.col_type(n)
        if how not in ("leftsemi", "leftanti"):
            for n in right.columns:
                self.schema[n] = right.col_type(n)


MOMENT_FUNCS = ("var_samp", "var_pop", "stddev_samp", "stddev_pop")


class AggSource(Source):
    """group_cols: child columns; aggs: [(input child column or None, output name, fn)] with
    fn in sum | count | mean | min | max | size | var_samp | var_pop | stddev_samp | stddev_pop."""

    def __init__(self, child: "LazyFrame", group_cols, aggs, options=None):
        self.child, self.group_cols, self.aggs = child, list(group_cols), list(aggs)
        self.options = dict(options or {})
        self.schema = OrderedDict()
        for g in self.group_cols:
            self.schema[g] = child.col_type(g)
        for in_col, out, fn in self.aggs:
            if fn in ("count", "size"):
                self.schema[out] = (I64, "int64")
            elif fn == "mean" or fn in MOMENT_FUNCS:
                self.schema[out] = (F64, "float64")
            else:
                dt, lg = child.col_type(in_col)
                if dt == U8:
                    dt, lg = I64, "int64"
                self.schema[out] = (dt, lg)


class SortSource(Source):
    """ORDER BY: keys = [(child column, ascending, nulls_first)], most significant first."""

    def __init__(self, child: "LazyFrame", keys):
        self.child, self.keys = child, list(keys)
        self.schema = OrderedDict((n, child.col_type(n)) for n in child.columns)


class WindowCall(NamedTuple):
    """One window function of a WindowSource.  func: row_number | rank | dense_rank | lag | lead | sum |
    count | avg | min | max | first_value | last_value; args: child columns (none for COUNT(*) and the
    ranking functions); partition: child columns; order: [(child column, ascending, nulls_first)];
    frame: (ROWS | RANGE, lower, upper) with bounds (UNBOUNDED_PRECEDING | PRECEDING | CURRENT | FOLLOWING |
    UNBOUNDED_FOLLOWING, offset); out: output column; params: (k, default) of lag / lead."""
    func: str
    args: tuple
    partition: tuple
    order: tuple
    frame: tuple
    out: str
    params: tuple = ()


class WindowSource(Source):
    """Window functions over the child's rows: the child's columns followed by one column per call.
    Calls with the same (partition, order) share one sort (executor.run_window)."""

    def __init__(self, child: "LazyFrame", calls: Sequence[WindowCall]):
        self.child, self.calls = child, list(calls)
        self.schema = OrderedDict((n, child.col_type(n)) for n in child.columns)
        for w in self.calls:
            if w.func in ("row_number", "rank", "dense_rank", "count"):
                self.schema[w.out] = (I64, "int64")
            elif w.func == "avg":
                self.schema[w.out] = (F64, "float64")
            elif w.func == "sum":
                dt = child.col_type(w.args[0])[0]
                self.schema[w.out] = (F64, "float64") if dt == F64 else (I64, "int64")
            else:
                self.schema[w.out] = child.col_type(w.args[0])


class LimitSource(Source):
    """LIMIT / OFFSET over the child's row order."""

    def __init__(self, child: "LazyFrame", offset, fetch):
        self.child, self.offset, self.fetch = child, int(offset or 0), fetch
        self.schema = OrderedDict((n, child.col_type(n)) for n in child.columns)


# ---------------------------------------------------------------------------------------------
# series
# ---------------------------------------------------------------------------------------------
class LazySeries:
    """One lazily-evaluated column of a LazyFrame (an expression over the frame's source)."""

    def __init__(self, source: Source, pred: tuple, expr: Expr, name=None):
        self.source, self.pred, self.expr, self.name = source, pred, expr, name

    # -- pandas-ish metadata
    @property
    def dtype(self):
        if isinstance(self.expr, ColRef):
            lg = self.expr.logical
            try:
                return np.dtype(lg)
            except TypeError:
                import pandas as pd
                return pd.api.types.pandas_dtype(lg)
        return _NP_DTYPE[self.expr.dtype]

    def _wrap(self, e: Expr):
        return LazySeries(self.source, self.pred, e, self.name)

    def _other(self, o):
        if isinstance(o, LazySeries):
            if o.source is not self.source:
                raise ValueError("cannot combine columns of different frames without a join")
            return o.expr
        if isinstance(o, np.generic):
            o = o.item()
        return E.as_expr(o)

    def _bin(self, op, o, rev=False):
        a, b = self.expr, self._other(o)
        if rev:
            a, b = b, a
        return self._wrap(E.binop(op, a, b))

    def __add__(self, o): return self._bin("add", o)
    def __radd__(self, o): return self._bin("add", o, True)
    def __sub__(self, o): return self._bin("sub", o)
    def __rsub__(self, o): return self._bin("sub", o, True)
    def __mul__(self, o): return self._bin("mul", o)
    def __rmul__(self, o): return self._bin("mul", o, True)
    def __truediv__(self, o): return self._bin("truediv", o)
    def __rtruediv__(self, o): return self._bin("truediv", o, True)
    def __mod__(self, o): return self._bin("mod", o)
    def __gt__(self, o): return self._bin("gt", o)
    def __ge__(self, o): return self._bin("ge", o)
    def __lt__(self, o): return self._bin("lt", o)
    def __le__(self, o): return self._bin("le", o)
    def __eq__(self, o): return self._bin("eq", o)  # noqa: E711
    def __ne__(self, o): return self._bin("ne", o)
    def __and__(self, o): return self._bin("and", o)
    def __rand__(self, o): return self._bin("and", o, True)
    def __or__(self, o): return self._bin("or", o)
    def __ror__(self, o): return self._bin("or", o, True)
    def __invert__(self): return self._wrap(E.unop("not", self.expr))
    def __neg__(self): return self._wrap(E.unop("neg", self.expr))
    __hash__ = None

    def abs(self): return self._wrap(E.unop("abs", self.expr))
    def sqrt(self): return self._wrap(E.unop("sqrt", self.expr))
    def isna(self): return self._wrap(E.unop("isnull", self.expr))
    isnull = isna
    def notna(self): return ~self.isna()
    def fillna(self, v): return self._wrap(E.fillna(self.expr, self._other(v)))

    def sql_div(self, o, rev=False):
        """SQL division: truncating for integers (SQLDivisionOperator, call.py:165-189)."""
        return self._bin("divt", o, rev)

    def between(self, low, high, inclusive="both"):
        assert inclusive == "both"
        return (self >= low) & (self <= high)

    def isin(self, values):
        vals = list(values)
        if not vals:
            return self._wrap(Lit(False))
        out = None
        for v in vals:
            t = self == v
            out = t if out is None else (out | t)
        # pandas isin never yields NULL
        return out.fillna(False)

    def where(self, cond, other=None):
        return self._wrap(E.case(self._other(cond), self.expr, self._other(other)))

    def astype(self, dtype):
        s = str(dtype).lower()
        if s in ("boolean", "bool"):
            return self._wrap(E.cast(self.expr, U8))
        if s.startswith(("int", "uint")):
            return self._wrap(E.cast(self.expr, I64))
        if s.startswith("float"):
            return self._wrap(E.cast(self.expr, F64))
        raise NotImplementedError(f"astype({dtype}) is outside the int64/float64/bool hot path")

    def trunc(self):
        if self.expr.dtype != F64:
            return self
        return self._wrap(E.cast(E.cast(self.expr, I64), F64))

    def to_frame(self, name=None):
        name = name or self.name or "0"
        return LazyFrame(self.source, OrderedDict([(name, self.expr)]), list(self.pred))

    def compute(self):
        return self.to_frame().compute()[self.name or "0"]


# ---------------------------------------------------------------------------------------------
# frame
# ---------------------------------------------------------------------------------------------
class LazyFrame:
    def __init__(self, source: Source, exprs: "OrderedDict[str, Expr]" = None, pred: Sequence[Expr] = ()):
        self.source = source
        if exprs is None:
            exprs = OrderedDict((n, source.colref(n)) for n in source.schema)
        self.exprs: "OrderedDict[str, Expr]" = exprs
        self.pred: List[Expr] = list(pred)

    # -- metadata -------------------------------------------------------------------------
    @property
    def columns(self):
        return list(self.exprs.keys())

    @columns.setter
    def columns(self, names):
        names = [str(n) for n in names]
        assert len(names) == len(self.exprs)
        self.exprs = OrderedDict(zip(names, self.exprs.values()))

    def col_type(self, name):
        e = self.exprs[name]
        if isinstance(e, ColRef):
            return e.dtype, e.logical
        return e.dtype, {I64: "int64", F64: "float64", U8: "bool"}[e.dtype]

    def dtype_of(self, name):
        """numpy / pandas dtype of one column (cheap: no Series is built)."""
        return LazySeries(self.source, (), self.exprs[name]).dtype

    @property
    def dtypes(self):
        import pandas as pd
        return pd.Series({n: self.dtype_of(n) for n in self.exprs})

    @property
    def npartitions(self):
        from .executor import source_npartitions
        return source_npartitions(self.source)

    def _series(self, name):
        return LazySeries(self.source, tuple(self.pred), self.exprs[name], name)

    def copy(self):
        return LazyFrame(self.source, OrderedDict(self.exprs), list(self.pred))

    # -- indexing -------------------------------------------------------------------------
    def __getitem__(self, key):
        if isinstance(key, LazySeries):
            if key.source is not self.source:
                raise ValueError("filter condition belongs to a different frame")
            return LazyFrame(self.source, OrderedDict(self.exprs), self.pred + E.conjuncts(key.expr))
        if isinstance(key, (list, tuple)):
            return LazyFrame(self.source, OrderedDict((str(k), self.exprs[str(k)]) for k in key), self.pred)
        return self._series(str(key))

    @property
    def iloc(self):
        frame = self

        class _ILoc:
            def __getitem__(self, idx):
                rows, col = idx
                assert rows == slice(None)
                return frame._series(frame.columns[col])

        return _ILoc()

    def assign(self, **cols):
        exprs = OrderedDict(self.exprs)
        for n, v in cols.items():
            if isinstance(v, LazySeries):
                if v.source is not self.source:
                    raise ValueError("assigned column belongs to a different frame")
                exprs[n] = v.expr
            else:
                if isinstance(v, np.generic):
                    v = v.item()
                exprs[n] = E.as_expr(v)
        return LazyFrame(self.source, exprs, self.pred)

    def rename(self, columns):
        return LazyFrame(self.source, OrderedDict((columns.get(n, n), e) for n, e in self.exprs.items()), self.pred)

    def drop(self, columns, errors="raise"):
        columns = [columns] if isinstance(columns, str) else list(columns)
        return LazyFrame(self.source, OrderedDict((n, e) for n, e in self.exprs.items() if n not in columns),
                         self.pred)

    def head(self, n=5, compute=True, npartitions=-1):
        if n != 0:
            out = self.limit(n)
            return out.compute() if compute else out
        out = LazyFrame(self.source, OrderedDict(self.exprs), self.pred + [Lit(False)])
        return out.compute() if compute else out

    # -- relational ops -------------------------------------------------------------------
    def merge(self, right: "LazyFrame", on=None, left_on=None, right_on=None, how="inner", broadcast=None,
              indicator=False):
        if on is not None:
            left_on = right_on = [on] if isinstance(on, str) else list(on)
        left_on = [left_on] if isinstance(left_on, str) else list(left_on)
        right_on = [right_on] if isinstance(right_on, str) else list(right_on)
        if indicator:
            raise NotImplementedError("merge(indicator=True); use how='leftanti'")
        return LazyFrame(JoinSource(self, right, left_on, right_on, how, broadcast))

    def groupby(self, by, dropna=False):
        by = [by] if isinstance(by, str) else list(by)
        if dropna:
            raise NotImplementedError("groupby(dropna=True): SQL keeps the NULL group (aggregate.py:575-577)")
        return LazyGroupBy(self, by)

    def drop_duplicates(self, subset=None, **options):
        cols = list(subset) if subset is not None else self.columns
        return LazyFrame(AggSource(self[cols] if subset is None else self, cols, [], options))[cols]

    def reset_index(self, drop=False):
        return self

    def sort_values(self, by, ascending=True, na_position="last", nulls_first=None):
        by = [by] if isinstance(by, str) else list(by)
        asc = [ascending] * len(by) if isinstance(ascending, bool) else list(ascending)
        if nulls_first is None:
            nulls_first = [na_position == "first"] * len(by)
        elif isinstance(nulls_first, bool):
            nulls_first = [nulls_first] * len(by)
        return LazyFrame(SortSource(self, list(zip(by, asc, nulls_first))))

    def limit(self, fetch=None, offset=0):
        return LazyFrame(LimitSource(self, offset, fetch))

    # -- execution ------------------------------------------------------------------------
    def compute(self, **kwargs):
        from .executor import compute_frame
        return compute_frame(self)

    def persist(self):
        from .executor import persist_frame
        return persist_frame(self)

    def __len__(self):
        from .executor import count_rows
        return count_rows(self)

    def __repr__(self):
        return f"LazyFrame(columns={self.columns}, npred={len(self.pred)}, source={type(self.source).__name__})"


class LazyGroupBy:
    def __init__(self, frame: LazyFrame, by: List[str]):
        self.frame, self.by = frame, by

    def agg(self, spec: Dict[str, Dict[str, str]], **options):
        """spec: {input column: {output column: function}} (the shape DaskAggregatePlugin passes,
        aggregate.py:543-581).  Returns group columns followed by the outputs."""
        aggs = []
        for in_col, outs in spec.items():
            for out, fn in outs.items():
                aggs.append((in_col, out, fn))
        return LazyFrame(AggSource(self.frame, self.by, aggs, options))


def is_lazy(x):
    return isinstance(x, (LazyFrame, LazySeries))
