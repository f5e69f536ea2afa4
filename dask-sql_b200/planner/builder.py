"""Syntax tree -> logical plan (the job of DataFusion's SqlToRel in the reference,
src/sql.rs:586-596), for the hot-path grammar.  Produces the same plan SHAPES the reference's
plugins expect: Projection / Aggregate / Filter / Join / SubqueryAlias / TableScan."""
from typing import Callable, Dict, List, Optional, Tuple

from ..utils import ParsingException
from . import plan as P
from .plan import PyExpr, RelDataTypeField
from .sqlparse import Node

_NUMERIC = ("BIGINT", "DOUBLE", "INTEGER", "FLOAT", "SMALLINT", "TINYINT", "REAL", "DECIMAL")
_CAST_TYPES = {"BIGINT": "BIGINT", "INT": "BIGINT", "INTEGER": "BIGINT", "SMALLINT": "BIGINT", "TINYINT": "BIGINT",
               "DOUBLE": "DOUBLE", "FLOAT": "DOUBLE", "REAL": "DOUBLE", "DECIMAL": "DOUBLE", "NUMERIC": "DOUBLE",
               "BOOLEAN": "BOOLEAN", "BOOL": "BOOLEAN", "VARCHAR": "VARCHAR", "STRING": "VARCHAR", "TEXT": "VARCHAR"}


def _norm_type(t: str) -> str:
    """Physical family of a SQL type: ints -> BIGINT, floats -> DOUBLE."""
    if t in ("INTEGER", "SMALLINT", "TINYINT", "BIGINT"):
        return "BIGINT"
    if t in ("FLOAT", "REAL", "DECIMAL", "DOUBLE"):
        return "DOUBLE"
    return t


def _arith_type(a: str, b: str) -> str:
    a, b = _norm_type(a), _norm_type(b)
    if "DOUBLE" in (a, b):
        return "DOUBLE"
    if a == "NULL":
        return b
    if b == "NULL":
        return a
    return "BIGINT"


class Binder:
    def __init__(self, sql: str, catalog: Callable[[Optional[str], str], Optional[Tuple[str, List[Tuple[str, str]]]]],
                 case_sensitive: bool = True):
        """catalog(schema_or_None, table) -> (schema_name, [(column, sql_type), ...]) or None."""
        self.sql, self.catalog, self.case_sensitive = sql, catalog, case_sensitive

    def err(self, msg):
        raise ParsingException(self.sql, msg)

    # -- queries ------------------------------------------------------------------------------
    def bind_statement(self, node: Node) -> P.LogicalPlan:
        if node.kind == "explain":
            return P.Explain(self.bind_query(node.query, {}))
        if node.kind == "create_memory_table":
            return P.CreateMemoryTable(self.bind_query(node.query, {}), node.name, node.or_replace,
                                       node.if_not_exists, node.is_table)
        if node.kind == "create_table":
            return P.CreateTable(node.name, node.kwargs, node.or_replace, node.if_not_exists)
        if node.kind == "drop_table":
            return P.DropTable(node.name, node.if_exists)
        return self.bind_query(node, {})

    def bind_query(self, q: Node, ctes: Dict[str, P.LogicalPlan]) -> P.LogicalPlan:
        ctes = dict(ctes)
        for name, sub in q.ctes or []:
            ctes[name] = self.bind_query(sub, ctes)
        plan = self.bind_from(q.source, ctes) if q.source is not None else self._empty_relation()
        if q.where is not None:
            pred = self.bind_expr(q.where, plan.schema)
            if pred.contains_agg():
                self.err("Aggregate functions are not allowed in WHERE")
            if pred.contains_window():
                self.err("Window functions are not allowed in WHERE")
            plan = P.Filter(plan, pred)

        # select list
        items: List[Tuple[PyExpr, Optional[str]]] = []
        for e, alias in q["items"]:
            if e.kind == "star":
                fields = [f for f in plan.schema if e.qualifier is None or f.qualifier == e.qualifier]
                if not fields:
                    self.err(f"Invalid qualifier {e.qualifier}")
                for f in fields:
                    items.append((P.col(f.qualifier, f.getName(), f.sql_type), None))
            else:
                items.append((self.bind_expr(e, plan.schema), alias))
        aliases = {a: e for e, a in items if a}
        having = self.bind_expr(q.having, plan.schema, aliases) if q.having is not None else None
        if having is not None and having.contains_window():
            self.err("Window functions are not allowed in HAVING")
        is_agg = bool(q.group_by) or any(e.contains_agg() for e, _ in items) or \
            (having is not None and having.contains_agg())

        if is_agg:
            group_exprs = []
            for g in q.group_by:
                if g.kind == "lit" and isinstance(g.value, int) and not isinstance(g.value, bool):
                    if not 1 <= g.value <= len(items):
                        self.err(f"GROUP BY position {g.value} is not in select list")
                    group_exprs.append(items[g.value - 1][0])
                elif g.kind == "col" and len(g.parts) == 1 and g.parts[0] in aliases and \
                        not self._resolves(g.parts[0], plan.schema):
                    group_exprs.append(aliases[g.parts[0]])
                else:
                    group_exprs.append(self.bind_expr(g, plan.schema))
                if group_exprs[-1].contains_window():
                    self.err("Window functions are not allowed in GROUP BY")
            agg_calls: List[PyExpr] = []

            def collect(e: PyExpr):
                if e.kind == "agg":
                    if not any(a.display() == e.display() for a in agg_calls):
                        agg_calls.append(e)
                    return
                for c in e.args + e.window_exprs():
                    collect(c)

            for e, _ in items:
                collect(e)
            if having is not None:
                collect(having)
            agg_plan = P.Aggregate(plan, group_exprs, agg_calls)

            def rewrite(e: PyExpr) -> PyExpr:
                for g in group_exprs:
                    if g.display() == e.display():
                        q_, n_ = g.output_field()
                        return P.col(q_, n_, g.sql_type)
                if e.kind == "agg":
                    return P.col(None, e.display(), e.sql_type)
                if e.kind == "column":
                    self.err(f"Column {e.display()} must appear in the GROUP BY clause or be used in an "
                             "aggregate function")
                out = e.clone()
                out.args = [rewrite(a) for a in e.args]
                if e.window is not None:            # a window over the groups: its keys name group outputs
                    out.window = e.window.map(rewrite)
                return out

            plan = agg_plan
            if having is not None:
                plan = P.Filter(plan, rewrite(having))
            plan, exprs = self._windows(plan, [rewrite(e) for e, _ in items])
            proj = []
            for r, (e, alias) in zip(exprs, items):
                name = alias if alias else None
                if name is None and e.kind != "column":
                    name = None  # display name of the aggregate output column
                proj.append(PyExpr("alias", r.sql_type, name=name, args=[r]) if name else r)
            plan = P.Projection(plan, proj)
        else:
            plan, exprs = self._windows(plan, [e for e, _ in items])
            proj = [PyExpr("alias", e.sql_type, name=a, args=[e]) if a else e for e, (_, a) in zip(exprs, items)]
            plan = P.Projection(plan, proj)

        if q.distinct:
            plan = P.Distinct(plan)
        if q.order_by:
            keys = []
            for e, asc, nulls_first in q.order_by:
                if e.kind == "lit" and isinstance(e.value, int) and not isinstance(e.value, bool):
                    f = plan.schema[e.value - 1]
                    b = P.col(f.qualifier, f.getName(), f.sql_type)
                else:
                    b = self.bind_expr(e, plan.schema, order_by_fallback=items)
                    if b.contains_window():
                        self.err("ORDER BY refers to a window function by its alias only")
                keys.append((b, asc, (not asc) if nulls_first is None else nulls_first))
            plan = P.Sort(plan, keys)
        if q.limit is not None or q.offset is not None:
            fetch = q.limit.value if q.limit is not None else None
            skip = q.offset.value if q.offset is not None else 0
            plan = P.Limit(plan, skip, fetch)
        return plan

    def _windows(self, plan, exprs):
        """Window calls of the select list become fields of one Window node on top of `plan` (the
        input, or the aggregate and its HAVING filter); the select list then reads those fields."""
        calls: List[PyExpr] = []

        def lift(e: PyExpr) -> PyExpr:
            if e.kind == "window":
                d = e.display()
                if not any(c.display() == d for c in calls):
                    calls.append(e)
                return P.col(None, d, e.sql_type)
            if not e.contains_window():
                return e
            out = e.clone()
            out.args = [lift(a) for a in e.args]
            return out

        exprs = [lift(e) for e in exprs]
        return (P.Window(plan, calls) if calls else plan), exprs

    def _empty_relation(self):
        p = P.LogicalPlan()
        p.node_type = "EmptyRelation"
        return p

    def _resolves(self, name, scope) -> bool:
        return any(f.getName() == name for f in scope)

    # -- FROM ---------------------------------------------------------------------------------
    def bind_from(self, src: Node, ctes) -> P.LogicalPlan:
        if src.kind == "table":
            parts = src.name
            if len(parts) == 1 and parts[0] in ctes:
                return P.SubqueryAlias(ctes[parts[0]], src.alias or parts[0])
            schema_name, table_name = (parts[-2], parts[-1]) if len(parts) >= 2 else (None, parts[0])
            found = self.catalog(schema_name, table_name)
            if found is None:
                self.err(f"Error during planning: table '{'.'.join(parts)}' not found")
            schema_name, cols = found
            fields = [RelDataTypeField(None, c, t, i) for i, (c, t) in enumerate(cols)]
            scan = P.TableScan(schema_name, table_name.lower(), table_name if not src.alias else table_name, fields)
            return P.SubqueryAlias(scan, src.alias) if src.alias else scan
        if src.kind == "subquery":
            return P.SubqueryAlias(self.bind_query(src.query, ctes), src.alias)
        if src.kind == "join":
            left, right = self.bind_from(src.left, ctes), self.bind_from(src.right, ctes)
            if src.how == "CROSS" or src.on is None:
                return P.CrossJoin(left, right)
            scope = left.schema + right.schema
            nleft = len(left.schema)
            if src.on.kind == "using":
                pairs = []
                for c in src.on.cols:
                    lf = [f for f in left.schema if f.getName() == c]
                    rf = [f for f in right.schema if f.getName() == c]
                    if len(lf) != 1 or len(rf) != 1:
                        self.err(f"USING column {c} must exist exactly once on both sides")
                    pairs.append((P.col(lf[0].qualifier, c, lf[0].sql_type), P.col(rf[0].qualifier, c, rf[0].sql_type)))
                return P.Join(left, right, src.how, pairs, None)
            cond = self.bind_expr(src.on, scope)
            pairs, residual = [], []
            holder = P.LogicalPlan()
            holder.schema = scope
            for c in P.conjuncts(cond):
                if c.kind == "binary" and c.op == "=" and c.args[0].kind == "column" and c.args[1].kind == "column":
                    a, b = c.args
                    ia, ib = a.with_inputs([holder]).getIndex(), b.with_inputs([holder]).getIndex()
                    if ia < nleft <= ib:
                        pairs.append((a, b))
                        continue
                    if ib < nleft <= ia:
                        pairs.append((b, a))
                        continue
                residual.append(c)
            return P.Join(left, right, src.how, pairs, P.conjunction(residual))
        self.err(f"Unsupported FROM item {src.kind}")

    # -- expressions --------------------------------------------------------------------------
    def bind_expr(self, e: Node, scope, aliases=None, order_by_fallback=None) -> PyExpr:
        k = e.kind
        if k == "lit":
            return P.lit(e.value)
        if k == "col":
            parts = e.parts
            if len(parts) == 1:
                name = parts[0]
                hits = [f for f in scope if f.getName() == name]
                if not hits and not self.case_sensitive:
                    hits = [f for f in scope if f.getName().lower() == name.lower()]
                if len(hits) == 1:
                    return P.col(hits[0].qualifier, hits[0].getName(), hits[0].sql_type)
                if len(hits) > 1:
                    if len({(h.qualifier, h.getName()) for h in hits}) == 1:
                        return P.col(hits[0].qualifier, hits[0].getName(), hits[0].sql_type)
                    self.err(f"Schema error: Ambiguous reference to unqualified field {name}")
                if aliases and name in aliases:
                    return aliases[name]
                if order_by_fallback:
                    for ex, al in order_by_fallback:
                        if al == name:
                            return P.col(None, name, ex.sql_type)
                self.err(f"Schema error: No field named {name}. Valid fields are "
                         f"{', '.join(f.getQualifiedName() for f in scope)}.")
            qual, name = parts[-2], parts[-1]
            hits = [f for f in scope if f.getName() == name and f.qualifier == qual]
            if len(hits) >= 1:
                return P.col(qual, name, hits[0].sql_type)
            self.err(f"Schema error: No field named {qual}.{name}. Valid fields are "
                     f"{', '.join(f.getQualifiedName() for f in scope)}.")
        rec = lambda x: self.bind_expr(x, scope, aliases, order_by_fallback)  # noqa: E731
        if k == "bin":
            l, r = rec(e.l), rec(e.r)
            op = e.op
            if op in ("AND", "OR"):
                return PyExpr("binary", "BOOLEAN", op=op, args=[l, r])
            if op in ("=", "!=", "<", "<=", ">", ">="):
                return PyExpr("binary", "BOOLEAN", op=op, args=[l, r])
            if op in ("+", "-", "*", "/", "%"):
                return PyExpr("binary", _arith_type(l.sql_type, r.sql_type), op=op, args=[l, r])
            self.err(f"Unsupported operator {op}")
        if k == "not":
            return PyExpr("not", "BOOLEAN", args=[rec(e.e)])
        if k == "neg":
            inner = rec(e.e)
            return PyExpr("negative", _norm_type(inner.sql_type), args=[inner])
        if k == "isnull":
            return PyExpr("isnotnull" if e.negated else "isnull", "BOOLEAN", args=[rec(e.e)])
        if k == "istrue":
            return PyExpr("istrue", "BOOLEAN", args=[rec(e.e)], negated=e.negated, value=e.value)
        if k == "between":
            return PyExpr("between", "BOOLEAN", args=[rec(e.e), rec(e.lo), rec(e.hi)], negated=e.negated)
        if k == "inlist":
            return PyExpr("inlist", "BOOLEAN", args=[rec(e.e)] + [rec(i) for i in e["items"]], negated=e.negated)
        if k == "cast":
            ty = _CAST_TYPES.get(e.type)
            if ty is None:
                self.err(f"Unsupported CAST target type {e.type}")
            return PyExpr("cast", ty, args=[rec(e.e)])
        if k == "case":
            args = []
            for w, t in e.whens:
                args += [rec(w), rec(t)]
            if e.other is not None:
                args.append(rec(e.other))
            thens = [args[i] for i in range(1, len(args) - (len(args) % 2), 2)] + \
                    ([args[-1]] if len(args) % 2 else [])
            ty = "NULL"
            for t in thens:
                ty = _arith_type(ty, t.sql_type) if t.sql_type in _NUMERIC + ("NULL",) and ty in _NUMERIC + ("NULL",) \
                    else t.sql_type
            return PyExpr("case", ty, args=args)
        if k == "func":
            name = e.name
            if e.over is not None:
                return self.bind_window(e, rec)
            if name in P.AGG_FUNCS:
                name = "AVG" if name == "MEAN" else name
                args = [] if e.star else [rec(a) for a in e.args]
                if name != "COUNT" and len(args) != 1:
                    self.err(f"{name} takes exactly one argument")
                if any(a.contains_agg() for a in args):
                    self.err("Aggregate function calls cannot be nested")
                if any(a.contains_window() for a in args):
                    self.err("Window function calls cannot be nested in an aggregate")
                if name == "COUNT":
                    ty = "BIGINT"
                elif name == "AVG" or name.startswith(("STDDEV", "VAR")):
                    ty = "DOUBLE"
                elif name == "SUM":
                    ty = _norm_type(args[0].sql_type) if args[0].sql_type != "BOOLEAN" else "BIGINT"
                else:
                    ty = args[0].sql_type
                filt = rec(e.filter) if e.filter is not None else None
                return PyExpr("agg", ty, name=name, args=args, distinct=e.distinct, filter=filt)
            args = [rec(a) for a in e.args]
            if name == "ABS" and len(args) == 1:
                return PyExpr("scalarfn", _norm_type(args[0].sql_type), name="abs", args=args)
            self.err(f"Function {name} is outside the int64/float64 hot path of the B200 layer")
        self.err(f"Unsupported expression {k}")

    _FRAME_ORDER = {"UNBOUNDED_PRECEDING": 0, "PRECEDING": 1, "CURRENT": 2, "FOLLOWING": 3, "UNBOUNDED_FOLLOWING": 4}

    def bind_window(self, e: Node, rec) -> PyExpr:
        """f(args) OVER (...) -> PyExpr("window").  Output types: ROW_NUMBER / RANK / DENSE_RANK / COUNT
        BIGINT, SUM int64 for integer and boolean input, AVG DOUBLE, the rest the argument's type."""
        name = "AVG" if e.name == "MEAN" else e.name
        if name not in P.WINDOW_FUNCS:
            raise NotImplementedError(f"window function {name} is not supported")
        if e.distinct:
            raise NotImplementedError(f"{name}(DISTINCT ...) OVER (...) is not supported")
        if e.filter is not None:
            raise NotImplementedError(f"FILTER (WHERE ...) on the window function {name} is not supported")
        if e.star and name != "COUNT":
            self.err(f"{name}(*) is not a window function")
        args = [] if e.star else [rec(a) for a in e.args]
        spec = e.over
        partition = [rec(p) for p in spec.partition]
        order = [(rec(x), asc, (not asc) if nf is None else nf) for x, asc, nf in spec.order]
        if any(x.contains_window() for x in args + partition + [o[0] for o in order]):
            self.err("Window function calls cannot be nested")
        nargs = {"ROW_NUMBER": (0, 0), "RANK": (0, 0), "DENSE_RANK": (0, 0), "LAG": (1, 3), "LEAD": (1, 3),
                 "COUNT": (0, 1)}.get(name, (1, 1))
        if not nargs[0] <= len(args) <= nargs[1]:
            self.err(f"{name} takes {nargs[0]}..{nargs[1]} argument(s) in a window, got {len(args)}")
        if name == "COUNT" and not args and not e.star:
            self.err("COUNT() needs an argument or *")
        if name in ("LAG", "LEAD"):
            if len(args) > 1:
                k = args[1]
                if k.kind != "literal" or not isinstance(k.value, int) or isinstance(k.value, bool) or k.value < 0:
                    self.err(f"the offset of {name} must be a non-negative integer literal")
            if len(args) > 2 and args[2].kind != "literal":
                self.err(f"the default of {name} must be a literal")
        if name in ("ROW_NUMBER", "RANK", "DENSE_RANK", "COUNT"):
            ty = "BIGINT"
        elif name == "AVG":
            ty = "DOUBLE"
        elif name == "SUM":
            ty = "BIGINT" if args[0].sql_type == "BOOLEAN" else _norm_type(args[0].sql_type)
        else:
            ty = args[0].sql_type
        frame = spec.frame
        if frame is not None:
            unit, lo, hi = frame
            for kind, off in (lo, hi):
                if off is not None and (not isinstance(off, int) or off > (1 << 31) - 1):
                    self.err(f"window frame offsets must be integers from 0 to 2^31-1, got {off}")
            if unit == "RANGE" and any(b[0] in ("PRECEDING", "FOLLOWING") for b in (lo, hi)):
                raise NotImplementedError("RANGE frames with a numeric offset are not supported "
                                          "(use ROWS, or UNBOUNDED / CURRENT ROW bounds)")
            if lo[0] == "UNBOUNDED_FOLLOWING" or hi[0] == "UNBOUNDED_PRECEDING" or \
                    self._FRAME_ORDER[lo[0]] > self._FRAME_ORDER[hi[0]]:
                self.err(f"invalid window frame: {unit} BETWEEN {lo[0]} AND {hi[0]}")
        return PyExpr("window", ty, name=name, args=args, value="*" if e.star else None,
                      window=P.WindowSpec(partition, order, frame))
