"""Logical plan and expression objects with the duck-typed method surface of the reference's
pyo3 classes (PyLogicalPlan src/sql/logical.rs:65-437, PyExpr src/expression.rs:47-900,
RelDataType(Field) src/sql/types/*.rs) — exactly the methods the hot-path plugins call
(SURVEY 8b).  The Rust planner crate cannot be built in this image; when real dask_sql is
importable its plans can be fed to the same plugins because they only rely on these methods.
"""
from typing import List, Optional, Sequence, Tuple

from ..mappings import SqlTypeName


# ---------------------------------------------------------------------------------------------
# row types
# ---------------------------------------------------------------------------------------------
class DataTypeMap:
    def __init__(self, sql_type: str):
        self.sql_type = sql_type

    def getSqlType(self):
        return SqlTypeName.fromString(self.sql_type)

    def getDataType(self):
        return self

    def getPrecisionScale(self):
        return (38, 10)


class RelDataTypeField:
    def __init__(self, qualifier: Optional[str], name: str, sql_type: str, index: int = 0):
        self.qualifier, self._name, self.sql_type, self.index = qualifier, name, sql_type, index

    def getName(self):
        return self._name

    def getQualifiedName(self):
        return f"{self.qualifier}.{self._name}" if self.qualifier else self._name

    def getType(self):
        return DataTypeMap(self.sql_type)

    def getIndex(self):
        return self.index

    def __repr__(self):
        return f"{self.getQualifiedName()}:{self.sql_type}"


class RelDataType:
    def __init__(self, fields: Sequence[RelDataTypeField]):
        self.fields = list(fields)

    def getFieldList(self):
        return list(self.fields)

    def getFieldNames(self):
        return [f.getQualifiedName() for f in self.fields]

    def getFieldCount(self):
        return len(self.fields)

    def getField(self, name, case_sensitive=True):
        for f in self.fields:
            if f.getName() == name or (not case_sensitive and f.getName().lower() == name.lower()):
                return f
        raise RuntimeError(f"Unable to find RelDataTypeField with name {name!r}")


class RexType:
    """Stand-in for the Rust enum; str() matches the keys of _REX_TYPE_TO_PLUGIN (rex/convert.py:16-22)."""

    def __init__(self, name):
        self.name = name

    def __str__(self):
        return f"RexType.{self.name}"

    def __eq__(self, other):
        return isinstance(other, RexType) and other.name == self.name

    def __hash__(self):
        return hash(self.name)


for _n in ("Reference", "Call", "Literal", "Alias", "ScalarSubquery"):
    setattr(RexType, _n, RexType(_n))


# ---------------------------------------------------------------------------------------------
# expressions
# ---------------------------------------------------------------------------------------------
_ARROW = {"BIGINT": "Int64", "DOUBLE": "Float64", "BOOLEAN": "Boolean", "VARCHAR": "Utf8", "NULL": "Null",
          "INTEGER": "Int32", "FLOAT": "Float32"}
AGG_FUNCS = {"SUM", "AVG", "COUNT", "MIN", "MAX", "MEAN", "STDDEV", "STDDEV_SAMP", "STDDEV_POP", "VAR_SAMP",
             "VAR_POP", "VARIANCE"}


WINDOW_FUNCS = {"ROW_NUMBER", "RANK", "DENSE_RANK", "LAG", "LEAD", "SUM", "COUNT", "AVG", "MEAN", "MIN", "MAX",
                "FIRST_VALUE", "LAST_VALUE", "SINGLE_VALUE"}
_BOUND_TEXT = {"UNBOUNDED_PRECEDING": "UNBOUNDED PRECEDING", "CURRENT": "CURRENT ROW",
               "UNBOUNDED_FOLLOWING": "UNBOUNDED FOLLOWING"}


class WindowSpec:
    """The OVER (...) of a window call: partition expressions, sort keys [(expr, asc, nulls_first)] and
    the frame (unit, lower, upper) with bounds (kind, offset) -- None when the query gives none."""

    def __init__(self, partition, order, frame):
        self.partition, self.order, self.frame = list(partition), list(order), frame

    def exprs(self):
        return self.partition + [e for e, _, _ in self.order]

    def map(self, fn) -> "WindowSpec":
        return WindowSpec([fn(e) for e in self.partition], [(fn(e), a, nf) for e, a, nf in self.order], self.frame)

    def display(self) -> str:
        parts = []
        if self.partition:
            parts.append(f"PARTITION BY [{', '.join(e.display() for e in self.partition)}]")
        if self.order:
            keys = ", ".join(f"{e.display()} {'ASC' if a else 'DESC'} NULLS {'FIRST' if nf else 'LAST'}"
                             for e, a, nf in self.order)
            parts.append(f"ORDER BY [{keys}]")
        if self.frame is not None:
            unit, lo, hi = self.frame
            show = lambda b: _BOUND_TEXT.get(b[0]) or f"{b[1]} {b[0]}"  # noqa: E731
            parts.append(f"{unit} BETWEEN {show(lo)} AND {show(hi)}")
        return " ".join(parts)


class WindowFrame:
    """getWindowFrame() of the Window node (the reference reads it at window.py:283-314)."""

    def __init__(self, unit, lo, hi):
        self.unit, self.lo, self.hi = unit, lo, hi

    def getFrameUnits(self):
        return self.unit

    def getLowerBound(self):
        return WindowFrameBound(*self.lo)

    def getUpperBound(self):
        return WindowFrameBound(*self.hi)


class WindowFrameBound:
    def __init__(self, kind, offset):
        self.kind, self.offset = kind, offset

    def isUnbounded(self):
        return self.kind.startswith("UNBOUNDED")

    def isPreceding(self):
        return self.kind.endswith("PRECEDING")

    def isFollowing(self):
        return self.kind.endswith("FOLLOWING")

    def isCurrentRow(self):
        return self.kind == "CURRENT"

    def getOffset(self):
        return self.offset if self.kind in ("PRECEDING", "FOLLOWING") else None


class PyExpr:
    """kind: column | literal | binary | not | isnull | isnotnull | negative | between | inlist |
    cast | case | agg | alias | scalarfn | istrue | window (name = function, args, window = WindowSpec)"""

    def __init__(self, kind, sql_type, **kw):
        self.kind = kind
        self.sql_type = sql_type            # BIGINT / DOUBLE / BOOLEAN / VARCHAR / NULL
        self.qualifier = kw.get("qualifier")
        self.name = kw.get("name")
        self.value = kw.get("value")
        self.op = kw.get("op")
        self.args: List["PyExpr"] = list(kw.get("args", ()))
        self.negated = kw.get("negated", False)
        self.distinct = kw.get("distinct", False)
        self.filter: Optional["PyExpr"] = kw.get("filter")
        self.window: Optional[WindowSpec] = kw.get("window")
        self.inputs: List["LogicalPlan"] = []   # plans whose concatenated schema getIndex() indexes

    # -- construction helpers
    def with_inputs(self, inputs):
        self.inputs = list(inputs)
        for a in self.args:
            a.with_inputs(inputs)
        if self.filter is not None:
            self.filter.with_inputs(inputs)
        for e in self.window_exprs():
            e.with_inputs(inputs)
        return self

    def window_exprs(self):
        return self.window.exprs() if self.window is not None else []

    def children(self):
        return self.args + ([self.filter] if self.filter is not None else []) + self.window_exprs()

    def columns(self, out=None):
        out = [] if out is None else out
        if self.kind == "column":
            out.append(self)
        for c in self.children():
            c.columns(out)
        return out

    def contains_agg(self):
        """A group aggregate somewhere in the expression.  A window call is not one, but its arguments,
        partition and sort keys may hold some: SUM(SUM(v)) OVER () runs after the GROUP BY."""
        return self.kind == "agg" or any(c.contains_agg() for c in self.args + self.window_exprs())

    def contains_window(self):
        return self.kind == "window" or any(c.contains_window() for c in self.children())

    def clone(self):
        e = PyExpr(self.kind, self.sql_type, qualifier=self.qualifier, name=self.name, value=self.value,
                   op=self.op, args=[a.clone() for a in self.args], negated=self.negated,
                   distinct=self.distinct, filter=self.filter.clone() if self.filter is not None else None,
                   window=self.window.map(lambda x: x.clone()) if self.window is not None else None)
        e.inputs = self.inputs
        return e

    # -- display (DataFusion-style names: they become output column names)
    def display(self) -> str:
        k = self.kind
        if k == "column":
            return f"{self.qualifier}.{self.name}" if self.qualifier else self.name
        if k == "literal":
            if self.value is None:
                return "NULL"
            if isinstance(self.value, bool):
                return f"Boolean({str(self.value).lower()})"
            if isinstance(self.value, int):
                return f"Int64({self.value})"
            if isinstance(self.value, float):
                return f"Float64({self.value!r})"
            return f'Utf8("{self.value}")'
        if k == "binary":
            return f"{self.args[0].display()} {self.op} {self.args[1].display()}"
        if k == "not":
            return f"NOT {self.args[0].display()}"
        if k == "isnull":
            return f"{self.args[0].display()} IS NULL"
        if k == "isnotnull":
            return f"{self.args[0].display()} IS NOT NULL"
        if k == "istrue":
            return f"{self.args[0].display()} IS {'NOT ' if self.negated else ''}{'TRUE' if self.value else 'FALSE'}"
        if k == "negative":
            return f"(- {self.args[0].display()})"
        if k == "between":
            return (f"{self.args[0].display()} {'NOT ' if self.negated else ''}BETWEEN "
                    f"{self.args[1].display()} AND {self.args[2].display()}")
        if k == "inlist":
            items = ", ".join(a.display() for a in self.args[1:])
            return f"{self.args[0].display()} {'NOT ' if self.negated else ''}IN ([{items}])"
        if k == "cast":
            return f"CAST({self.args[0].display()} AS {_ARROW.get(self.sql_type, self.sql_type)})"
        if k == "case":
            parts = ["CASE"]
            n = len(self.args) // 2
            for i in range(n):
                parts.append(f"WHEN {self.args[2 * i].display()} THEN {self.args[2 * i + 1].display()}")
            if len(self.args) % 2:
                parts.append(f"ELSE {self.args[-1].display()}")
            return " ".join(parts + ["END"])
        if k == "agg":
            inner = "*" if not self.args else ", ".join(a.display() for a in self.args)
            s = f"{self.name}({'DISTINCT ' if self.distinct else ''}{inner})"
            if self.filter is not None:
                s += f" FILTER (WHERE {self.filter.display()})"
            return s
        if k == "alias":
            return self.name
        if k == "sort":
            return self.args[0].display()
        if k == "scalarfn":
            return f"{self.name.lower()}({', '.join(a.display() for a in self.args)})"
        if k == "window":
            inner = "*" if self.value == "*" else ", ".join(a.display() for a in self.args)
            spec = self.window.display()
            return f"{self.name}({inner})" + (f" {spec}" if spec else "")
        return k

    __repr__ = display

    def output_field(self) -> Tuple[Optional[str], str]:
        if self.kind == "column":
            return self.qualifier, self.name
        return None, self.display()

    # -- reference surface (src/expression.rs)
    def toString(self):
        return self.display()

    def getRexType(self):
        if self.kind == "column":
            return RexType.Reference
        if self.kind == "literal":
            return RexType.Literal
        if self.kind == "alias":
            return RexType.Alias
        return RexType.Call

    def getExprType(self):
        return {"column": "Column", "literal": "Literal", "alias": "Alias", "agg": "AggregateFunction",
                "binary": "BinaryExpr", "not": "Not", "isnull": "IsNull", "isnotnull": "IsNotNull",
                "negative": "Negative", "between": "Between", "inlist": "InList", "cast": "Cast",
                "case": "Case", "scalarfn": "ScalarFunction", "istrue": "IsTrue",
                "window": "WindowFunction"}[self.kind]

    def column_name(self, rel=None) -> str:
        return self.display()

    def getIndex(self) -> int:
        """Position of this column in the concatenated schema of the node's inputs
        (expression.rs:193-263)."""
        assert self.kind == "column", f"getIndex() on {self.kind}"
        fields = [f for p in self.inputs for f in p.schema]
        # exact (qualifier, name) first, then unqualified unique match
        for i, f in enumerate(fields):
            if f.getName() == self.name and f.qualifier == self.qualifier:
                return i
        hits = [i for i, f in enumerate(fields) if f.getName() == self.name and
                (self.qualifier is None or f.qualifier is None)]
        if len(hits) == 1:
            return hits[0]
        # a computed column is referenced by its display name
        for i, f in enumerate(fields):
            if f.getQualifiedName() == self.display() or f.getName() == self.display():
                return i
        raise RuntimeError(f"Column {self.display()} not found in {fields}")

    def getOperands(self):
        return list(self.args)

    def getOperatorName(self) -> str:
        k = self.kind
        if k == "binary":
            return self.op
        return {"not": "not", "isnull": "is null", "isnotnull": "is not null", "negative": "negative",
                "between": "between", "inlist": "in list", "cast": "cast", "case": "case",
                "istrue": ("is not " if self.negated else "is ") + ("true" if self.value else "false")
                }.get(k, (self.name or k).lower())

    def getType(self) -> str:
        if self.kind == "literal":
            if self.value is None:
                return "Null"
            return _ARROW.get(self.sql_type, self.sql_type)
        return self.sql_type

    def isNegated(self):
        return bool(self.negated)

    # sort expressions (kind == "sort")
    def isSortAscending(self):
        return bool(getattr(self, "ascending", True))

    def isSortNullsFirst(self):
        return bool(getattr(self, "nulls_first", False))

    def getSortExpr(self):
        return self.args[0]

    def isDistinctAgg(self):
        return bool(self.distinct)

    def getFilterExpr(self):
        return self.filter

    def getPrecisionScale(self):
        return (38, 10)

    # literal getters
    def getBoolValue(self):
        if self.value is None:
            raise TypeError("NULL literal")
        return bool(self.value)

    def getInt64Value(self):
        return int(self.value)

    getInt32Value = getInt16Value = getInt8Value = getUInt64Value = getUInt32Value = getInt64Value
    getUInt16Value = getUInt8Value = getInt64Value

    def getFloat64Value(self):
        return float(self.value)

    getFloat32Value = getFloat64Value

    def getStringValue(self):
        return str(self.value)


def col(qualifier, name, sql_type):
    return PyExpr("column", sql_type, qualifier=qualifier, name=name)


def lit(value):
    if value is None:
        return PyExpr("literal", "NULL", value=None)
    if isinstance(value, bool):
        return PyExpr("literal", "BOOLEAN", value=value)
    if isinstance(value, int):
        return PyExpr("literal", "BIGINT", value=value)
    if isinstance(value, float):
        return PyExpr("literal", "DOUBLE", value=value)
    return PyExpr("literal", "VARCHAR", value=value)


def conjuncts(e: Optional[PyExpr]) -> List[PyExpr]:
    if e is None:
        return []
    if e.kind == "binary" and e.op == "AND":
        return conjuncts(e.args[0]) + conjuncts(e.args[1])
    return [e]


def conjunction(parts: Sequence[PyExpr]) -> Optional[PyExpr]:
    out = None
    for p in parts:
        out = p if out is None else PyExpr("binary", "BOOLEAN", op="AND", args=[out, p])
    return out


# ---------------------------------------------------------------------------------------------
# plan nodes
# ---------------------------------------------------------------------------------------------
class DaskTable:
    def __init__(self, schema_name, table_name, fields):
        self.schema_name, self.table_name, self.fields = schema_name, table_name, fields

    def getSchema(self):
        return self.schema_name

    def getTableName(self):
        return self.table_name

    def getRowType(self):
        return RelDataType(self.fields)


class DNFFilters:
    def __init__(self):
        self.filtered_exprs = []
        self.io_unfilterable_exprs = []


class LogicalPlan:
    node_type = "?"

    def __init__(self, inputs: Sequence["LogicalPlan"] = ()):
        self.inputs: List[LogicalPlan] = list(inputs)
        self.schema: List[RelDataTypeField] = []

    # -- reference surface (src/sql/logical.rs)
    def get_current_node_type(self):
        return self.node_type

    def get_inputs(self):
        return list(self.inputs)

    def getRowType(self):
        fields = [RelDataTypeField(f.qualifier, f.getName(), f.sql_type, i) for i, f in enumerate(self.schema)]
        return RelDataType(fields)

    def explain_original(self):
        return self.explain()

    def table_scan(self):
        return self

    filter = projection = join = aggregate = sort = limit = subquery_alias = distinct = explain_node = table_scan

    # -- display
    def describe(self) -> str:
        return self.node_type

    def explain(self, indent=0) -> str:
        lines = ["  " * indent + self.describe()]
        for i in self.inputs:
            lines.append(i.explain(indent + 1))
        return "\n".join(lines)

    __repr__ = describe

    def bind(self):
        """(Re)attach input plans to every expression so getIndex() resolves."""
        for e in self.expressions():
            e.with_inputs(self.inputs)
        return self

    def expressions(self) -> List[PyExpr]:
        return []


class TableScan(LogicalPlan):
    node_type = "TableScan"

    def __init__(self, schema_name, table_name, qualifier, all_fields):
        super().__init__([])
        self.schema_name, self.table_name, self.qualifier = schema_name, table_name, qualifier
        self.all_fields = [RelDataTypeField(qualifier, f.getName(), f.sql_type, i) for i, f in enumerate(all_fields)]
        self.projection_names: Optional[List[str]] = None
        self.filters: List[PyExpr] = []
        self.schema = list(self.all_fields)

    def set_projection(self, names: Optional[List[str]]):
        self.projection_names = names
        self.schema = list(self.all_fields) if names is None else \
            [f for f in self.all_fields if f.getName() in names]

    def getTable(self):
        return DaskTable(self.schema_name, self.table_name, self.all_fields)

    def getFilters(self):
        return list(self.filters)

    def getDNFFilters(self):
        return DNFFilters()     # IO-level (parquet) filter pushdown is out of scope (SURVEY 2 row 9)

    def containsProjections(self):
        return self.projection_names is not None

    def getTableScanProjects(self):
        return [f.getName() for f in self.schema]

    def bind(self):
        # scan filters index the table's full column list
        holder = LogicalPlan()
        holder.schema = self.all_fields
        for e in self.filters:
            e.with_inputs([holder])
        return self

    def expressions(self):
        return list(self.filters)

    def describe(self):
        s = f"TableScan: {self.qualifier}"
        if self.projection_names is not None:
            s += f" projection=[{', '.join(f.getName() for f in self.schema)}]"
        if self.filters:
            s += f", full_filters=[{', '.join(e.display() for e in self.filters)}]"
        return s


class SubqueryAlias(LogicalPlan):
    node_type = "SubqueryAlias"

    def __init__(self, child, alias):
        super().__init__([child])
        self.alias = alias
        self.schema = [RelDataTypeField(alias, f.getName(), f.sql_type, i) for i, f in enumerate(child.schema)]

    def describe(self):
        return f"SubqueryAlias: {self.alias}"


class Filter(LogicalPlan):
    node_type = "Filter"

    def __init__(self, child, predicate: PyExpr):
        super().__init__([child])
        self.predicate = predicate
        self.schema = list(child.schema)

    def getCondition(self):
        return self.predicate

    def expressions(self):
        return [self.predicate]

    def describe(self):
        return f"Filter: {self.predicate.display()}"


class Projection(LogicalPlan):
    node_type = "Projection"

    def __init__(self, child, exprs: Sequence[PyExpr]):
        super().__init__([child])
        self.exprs = list(exprs)
        self.schema = []
        for i, e in enumerate(self.exprs):
            inner = e.args[0] if e.kind == "alias" else e
            q, n = (None, e.name) if e.kind == "alias" else e.output_field()
            self.schema.append(RelDataTypeField(q, n, inner.sql_type, i))

    def getNamedProjects(self):
        out = []
        for e, f in zip(self.exprs, self.schema):
            out.append((f.getQualifiedName(), e.args[0] if e.kind == "alias" else e))
        return out

    def expressions(self):
        return list(self.exprs)

    def describe(self):
        def show(e):
            return f"{e.args[0].display()} AS {e.name}" if e.kind == "alias" else e.display()
        return "Projection: " + ", ".join(show(e) for e in self.exprs)


class Join(LogicalPlan):
    node_type = "Join"

    def __init__(self, left, right, how: str, on: Sequence[Tuple[PyExpr, PyExpr]], residual: Optional[PyExpr]):
        super().__init__([left, right])
        self.how, self.on, self.residual = how, list(on), residual
        self.schema = list(left.schema) + ([] if how in ("LEFTSEMI", "LEFTANTI") else list(right.schema))

    def getJoinType(self):
        return self.how

    def getCondition(self):
        """Equi pairs AND-ed with the residual filter (src/sql/logical/join.rs:26-71)."""
        parts = [PyExpr("binary", "BOOLEAN", op="=", args=[l, r]).with_inputs(self.inputs) for l, r in self.on]
        if self.residual is not None:
            parts += conjuncts(self.residual)
        c = conjunction(parts)
        return c.with_inputs(self.inputs) if c is not None else None

    def expressions(self):
        out = [e for pair in self.on for e in pair]
        if self.residual is not None:
            out.append(self.residual)
        return out

    def describe(self):
        names = {"INNER": "Inner", "LEFT": "Left", "RIGHT": "Right", "FULL": "Full", "LEFTSEMI": "LeftSemi",
                 "LEFTANTI": "LeftAnti"}
        on = ", ".join(f"{l.display()} = {r.display()}" for l, r in self.on)
        s = f"{names.get(self.how, self.how)} Join: {on}"
        if self.residual is not None:
            s += f" Filter: {self.residual.display()}"
        return s


class CrossJoin(LogicalPlan):
    node_type = "CrossJoin"

    def __init__(self, left, right):
        super().__init__([left, right])
        self.schema = list(left.schema) + list(right.schema)

    def describe(self):
        return "CrossJoin:"


class Aggregate(LogicalPlan):
    node_type = "Aggregate"

    def __init__(self, child, group_exprs: Sequence[PyExpr], agg_exprs: Sequence[PyExpr]):
        super().__init__([child])
        self.group_exprs, self.agg_exprs = list(group_exprs), list(agg_exprs)
        self.schema = []
        for i, e in enumerate(self.group_exprs + self.agg_exprs):
            q, n = e.output_field()
            self.schema.append(RelDataTypeField(q, n, e.sql_type, i))

    def getGroupSets(self):
        return list(self.group_exprs)

    def getNamedAggCalls(self):
        return list(self.agg_exprs)

    def getAggregationFuncName(self, e: PyExpr):
        e = e.args[0] if e.kind == "alias" else e
        return e.name

    def getArgs(self, e: PyExpr):
        e = e.args[0] if e.kind == "alias" else e
        return list(e.args)

    def isDistinctNode(self):
        return False

    def getDistinctColumns(self):
        return []

    def expressions(self):
        return self.group_exprs + self.agg_exprs

    def describe(self):
        return (f"Aggregate: groupBy=[[{', '.join(e.display() for e in self.group_exprs)}]], "
                f"aggr=[[{', '.join(e.display() for e in self.agg_exprs)}]]")


class Distinct(LogicalPlan):
    node_type = "Distinct"

    def __init__(self, child):
        super().__init__([child])
        self.schema = list(child.schema)

    # the Aggregate plugin also serves "Distinct" (aggregate.py:115)
    def getGroupSets(self):
        return []

    def getNamedAggCalls(self):
        return []

    def isDistinctNode(self):
        return True

    def getDistinctColumns(self):
        return [f.getQualifiedName() for f in self.schema]

    def describe(self):
        return "Distinct:"


class Sort(LogicalPlan):
    node_type = "Sort"

    def __init__(self, child, keys):   # keys: [(PyExpr, asc, nulls_first)]
        super().__init__([child])
        self.keys = list(keys)
        self.schema = list(child.schema)

    def getCollation(self):
        """Sort expressions with isSortAscending() / isSortNullsFirst() / column_name(rel), the
        surface rel/logical/sort.py uses."""
        out = []
        for e, asc, nulls_first in self.keys:
            s = PyExpr("sort", e.sql_type, args=[e]).with_inputs(self.inputs)
            s.ascending, s.nulls_first = asc, nulls_first
            out.append(s)
        return out

    def getNumRows(self):
        return None

    def expressions(self):
        return [k[0] for k in self.keys]

    def describe(self):
        return "Sort: " + ", ".join(f"{e.display()} {'ASC' if a else 'DESC'}" for e, a, _ in self.keys)


class Window(LogicalPlan):
    """Window functions over the input rows: the input's fields followed by one field per window call
    (named by its display).  The method surface is the one DaskWindowPlugin calls
    (dask_sql/physical/rel/logical/window.py:233-426): getGroups() lists the window calls, and the
    other accessors take one of them."""
    node_type = "Window"

    def __init__(self, child, window_exprs: Sequence[PyExpr]):
        super().__init__([child])
        self.window_exprs = list(window_exprs)
        self.schema = self._fields(child.schema)

    def _fields(self, child_schema):
        n = len(child_schema)
        return list(child_schema) + [RelDataTypeField(None, e.display(), e.sql_type, n + i)
                                     for i, e in enumerate(self.window_exprs)]

    def window(self):
        return self

    def getGroups(self):
        return list(self.window_exprs)

    def getPartitionExprs(self, w: PyExpr):
        return list(w.window.partition)

    def getSortExprs(self, w: PyExpr):
        out = []
        for e, asc, nulls_first in w.window.order:
            s = PyExpr("sort", e.sql_type, args=[e]).with_inputs(self.inputs)
            s.ascending, s.nulls_first = asc, nulls_first
            out.append(s)
        return out

    def getWindowFrame(self, w: PyExpr):
        return WindowFrame(*w.window.frame) if w.window.frame is not None else None

    def getWindowFuncName(self, w: PyExpr):
        return w.name

    def getArgs(self, w: PyExpr):
        return list(w.args)

    def expressions(self):
        return list(self.window_exprs)

    def describe(self):
        return f"Window: windowExpr=[[{', '.join(e.display() for e in self.window_exprs)}]]"


class Limit(LogicalPlan):
    node_type = "Limit"

    def __init__(self, child, skip, fetch):
        super().__init__([child])
        self.skip, self.fetch = skip, fetch
        self.schema = list(child.schema)

    def getSkip(self):
        return self.skip or 0

    def getFetch(self):
        return self.fetch

    def describe(self):
        return f"Limit: skip={self.skip or 0}, fetch={self.fetch}"


class Explain(LogicalPlan):
    node_type = "Explain"

    def __init__(self, child):
        super().__init__([child])
        self.schema = [RelDataTypeField(None, "plan", "VARCHAR", 0)]

    def getExplainString(self):
        return self.inputs[0].explain().split("\n")

    def describe(self):
        return "Explain"


class CreateMemoryTable(LogicalPlan):
    """CREATE TABLE|VIEW name AS query (src/sql/logical/create_memory_table.rs; consumed by
    physical/rel/custom/create_memory_table.py:36-76)."""
    node_type = "CreateMemoryTable"

    def __init__(self, child, name, or_replace, if_not_exists, is_table):
        super().__init__([child])
        self.name, self.or_replace, self.if_not_exists, self.is_table_ = name, or_replace, if_not_exists, is_table
        if not is_table:
            self.node_type = "CreateView"

    def create_memory_table(self):
        return self

    def getQualifiedName(self):
        return self.name

    def getOrReplace(self):
        return self.or_replace

    def getIfNotExists(self):
        return self.if_not_exists

    def getInput(self):
        return self.inputs[0]

    def isTable(self):
        return self.is_table_

    def describe(self):
        return f"{self.node_type}: {self.name}"


class CreateTable(LogicalPlan):
    """CREATE TABLE name WITH (...) (src/sql/logical/create_table.rs; custom/create_table.py:40-88)."""
    node_type = "CreateTable"

    def __init__(self, name, kwargs, or_replace, if_not_exists):
        super().__init__([])
        *schema, self.table_name = name.split(".")
        self.schema_name = schema[0] if schema else None
        self.kwargs, self.or_replace, self.if_not_exists = dict(kwargs), or_replace, if_not_exists

    def create_table(self):
        return self

    def getSchemaName(self):
        return self.schema_name

    def getTableName(self):
        return self.table_name

    def getOrReplace(self):
        return self.or_replace

    def getIfNotExists(self):
        return self.if_not_exists

    def getSQLWithOptions(self):
        return dict(self.kwargs)

    def describe(self):
        return f"CreateTable: {self.table_name}"


class DropTable(LogicalPlan):
    """DROP TABLE [IF EXISTS] name (src/sql/logical/drop_table.rs; custom/drop_table.py)."""
    node_type = "DropTable"

    def __init__(self, name, if_exists):
        super().__init__([])
        self.name, self.if_exists = name, if_exists

    def drop_table(self):
        return self

    def getQualifiedName(self):
        return self.name

    def getIfExists(self):
        return self.if_exists

    def describe(self):
        return f"DropTable: {self.name}"


def walk(plan: LogicalPlan):
    yield plan
    for i in plan.inputs:
        yield from walk(i)


def bind_all(plan: LogicalPlan) -> LogicalPlan:
    for p in walk(plan):
        p.bind()
    return plan
