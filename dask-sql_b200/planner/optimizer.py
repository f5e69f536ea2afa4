"""The slice of the reference's optimizer (src/sql/optimizer.rs:53-98) that decides the SHAPE of
hot-path plans: predicate pushdown down to TableScan.filters (the Rust TableSource answers
`Exact` to every pushdown, src/sql/table.rs:70-91), IS NOT NULL on inner-join keys
(FilterNullJoinKeys, optimizer.rs:76) and projection pruning into the scans."""
from typing import List, Optional, Set

from . import plan as P
from .plan import PyExpr


def _rewrite_cols(e: PyExpr, mapping) -> Optional[PyExpr]:
    """Return a copy of e with columns replaced via mapping(col)->PyExpr|None; None if any fails."""
    if e.kind == "column":
        return mapping(e)
    out = e.clone()
    new_args = []
    for a in e.args:
        r = _rewrite_cols(a, mapping)
        if r is None:
            return None
        new_args.append(r)
    out.args = new_args
    if e.filter is not None:
        f = _rewrite_cols(e.filter, mapping)
        if f is None:
            return None
        out.filter = f
    return out


def _side(e: PyExpr, left: P.LogicalPlan, right: P.LogicalPlan) -> str:
    """'left' / 'right' / 'both' / 'none' by where the referenced columns resolve."""
    sides = set()
    for c in e.columns():
        in_l = any(f.getName() == c.name and (c.qualifier is None or f.qualifier == c.qualifier) for f in left.schema)
        in_r = any(f.getName() == c.name and (c.qualifier is None or f.qualifier == c.qualifier) for f in right.schema)
        if in_l and not in_r:
            sides.add("left")
        elif in_r and not in_l:
            sides.add("right")
        else:
            sides.add("both")
    if not sides:
        return "none"
    if sides == {"left"}:
        return "left"
    if sides == {"right"}:
        return "right"
    return "both"


def push_filters(plan: P.LogicalPlan, preds: List[PyExpr]) -> P.LogicalPlan:
    """Push the conjuncts `preds` (expressed over plan's output) as far down as they go."""
    if isinstance(plan, P.Filter):
        return push_filters(plan.inputs[0], preds + P.conjuncts(plan.predicate))

    if isinstance(plan, P.TableScan):
        plan.filters.extend(preds)
        return plan

    if isinstance(plan, P.SubqueryAlias):
        child = plan.inputs[0]

        def to_child(c: PyExpr):
            for f_out, f_in in zip(plan.schema, child.schema):
                if f_out.getName() == c.name and (c.qualifier in (None, plan.alias)):
                    return P.col(f_in.qualifier, f_in.getName(), f_in.sql_type)
            return None

        down, keep = [], []
        for p in preds:
            r = _rewrite_cols(p, to_child)
            (down if r is not None else keep).append(r if r is not None else p)
        new = P.SubqueryAlias(push_filters(child, down), plan.alias)
        return _wrap(new, keep)

    if isinstance(plan, P.Projection):
        child = plan.inputs[0]

        def to_child(c: PyExpr):
            for f_out, e in zip(plan.schema, plan.exprs):
                if f_out.getName() == c.name and (c.qualifier is None or c.qualifier == f_out.qualifier):
                    inner = e.args[0] if e.kind == "alias" else e
                    if inner.contains_agg():
                        return None
                    return inner.clone()
            return None

        down, keep = [], []
        for p in preds:
            r = _rewrite_cols(p, to_child)
            (down if r is not None else keep).append(r if r is not None else p)
        new = P.Projection(push_filters(child, down), plan.exprs)
        return _wrap(new, keep)

    if isinstance(plan, P.Join):
        left, right = plan.inputs
        lp, rp, keep = [], [], []
        for p in preds:
            s = _side(p, left, right)
            if s == "left" and plan.how in ("INNER", "LEFT", "LEFTSEMI", "LEFTANTI"):
                lp.append(p)
            elif s == "right" and plan.how in ("INNER", "RIGHT"):
                rp.append(p)
            else:
                keep.append(p)
        residual = P.conjuncts(plan.residual)
        res_keep = []
        if plan.how == "INNER":
            # single-sided parts of the ON clause are ordinary filters for an inner join
            for p in residual:
                s = _side(p, left, right)
                if s == "left":
                    lp.append(p)
                elif s == "right":
                    rp.append(p)
                else:
                    res_keep.append(p)
            # FilterNullJoinKeys: NULL keys never match, drop them before the join
            for a, b in plan.on:
                lp.append(PyExpr("isnotnull", "BOOLEAN", args=[a.clone()]))
                rp.append(PyExpr("isnotnull", "BOOLEAN", args=[b.clone()]))
        else:
            # outer joins: an ON-clause term over the NULL-SUPPLYING side alone only decides which of
            # that side's rows can be partners, so it filters that input (DataFusion's push_down_filter
            # does the same with join on-filters); terms over the preserved side must stay in the ON clause
            into_right = plan.how in ("LEFT", "LEFTSEMI", "LEFTANTI")
            into_left = plan.how == "RIGHT"
            for p in residual:
                s = _side(p, left, right)
                if s == "right" and into_right:
                    rp.append(p)
                elif s == "left" and into_left:
                    lp.append(p)
                else:
                    res_keep.append(p)
        lp, rp = _dedup(lp), _dedup(rp)
        new = P.Join(push_filters(left, lp), push_filters(right, rp), plan.how, plan.on, P.conjunction(res_keep))
        return _wrap(new, keep)

    if isinstance(plan, P.Aggregate):
        child = plan.inputs[0]
        group_names = {g.display() for g in plan.group_exprs if g.kind == "column"}
        down, keep = [], []
        for p in preds:
            cols = p.columns()
            if cols and all(c.display() in group_names for c in cols):
                down.append(p)
            else:
                keep.append(p)
        new = P.Aggregate(push_filters(child, down), plan.group_exprs, plan.agg_exprs)
        return _wrap(new, keep)

    if isinstance(plan, P.Window):
        # a filter decides which rows the windows see: only one over columns that every window
        # partitions by removes whole partitions and may go below; filters on window outputs stay above
        child = plan.inputs[0]
        shared = None
        for w in plan.window_exprs:
            keys = {e.display() for e in w.window.partition if e.kind == "column"}
            shared = keys if shared is None else shared & keys
        down, keep = [], []
        for p in preds:
            cols = p.columns()
            (down if cols and shared and all(c.display() in shared for c in cols) else keep).append(p)
        new = P.Window(push_filters(child, down), plan.window_exprs)
        return _wrap(new, keep)

    # Distinct / Sort / Limit / CrossJoin / Explain: optimise below, keep predicates above
    plan.inputs = [push_filters(i, []) for i in plan.inputs]
    return _wrap(plan, preds)


def _dedup(preds: List[PyExpr]) -> List[PyExpr]:
    seen, out = set(), []
    for p in preds:
        d = p.display()
        if d not in seen:
            seen.add(d)
            out.append(p)
    return out


def _wrap(plan: P.LogicalPlan, preds: List[PyExpr]) -> P.LogicalPlan:
    c = P.conjunction(preds)
    return P.Filter(plan, c) if c is not None else plan


def prune_columns(plan: P.LogicalPlan) -> P.LogicalPlan:
    """Projection pushdown: every TableScan keeps only columns whose name is referenced somewhere
    above it (name-based and therefore conservative), filters included."""
    names: Set[str] = set()
    star_scans = []
    for node in P.walk(plan):
        for e in node.expressions():
            for c in e.columns():
                names.add(c.name)
        if isinstance(node, P.Distinct):
            for f in node.schema:
                names.add(f.getName())
    for node in P.walk(plan):
        if isinstance(node, P.TableScan):
            keep = [f.getName() for f in node.all_fields if f.getName() in names]
            if not keep and node.all_fields:
                keep = [node.all_fields[0].getName()]
            node.set_projection(keep)
    _refresh_schemas(plan)
    return plan


def _refresh_schemas(plan: P.LogicalPlan):
    """Recompute pass-through schemas bottom-up after scans changed their projection."""
    for i in plan.inputs:
        _refresh_schemas(i)
    if isinstance(plan, P.SubqueryAlias):
        child = plan.inputs[0]
        plan.schema = [P.RelDataTypeField(plan.alias, f.getName(), f.sql_type, i) for i, f in enumerate(child.schema)]
    elif isinstance(plan, (P.Filter, P.Distinct, P.Sort, P.Limit)):
        plan.schema = list(plan.inputs[0].schema)
    elif isinstance(plan, P.Join):
        l, r = plan.inputs
        plan.schema = list(l.schema) + ([] if plan.how in ("LEFTSEMI", "LEFTANTI") else list(r.schema))
    elif isinstance(plan, P.CrossJoin):
        plan.schema = list(plan.inputs[0].schema) + list(plan.inputs[1].schema)
    elif isinstance(plan, P.Window):
        plan.schema = plan._fields(plan.inputs[0].schema)


def optimize(plan: P.LogicalPlan) -> P.LogicalPlan:
    if isinstance(plan, (P.Explain, P.CreateMemoryTable)):
        plan.inputs = [optimize(plan.inputs[0])]
        return plan
    if isinstance(plan, (P.CreateTable, P.DropTable)):
        return plan
    plan = push_filters(plan, [])
    plan = prune_columns(plan)
    return P.bind_all(plan)
