"""Physical execution of LazyFrame trees on one GPU per process.

This is where the reference's per-partition pandas calls are replaced by fused CUDA passes:

  Filter/Projection/TableScan chains -> predicate terms evaluated inside the consuming kernel
  Aggregate over a scan               -> b2_scan_agg / b2_groupby_{dense,hash1,hashk}
  Join                                -> b2_join_build(_dense) + b2_join_count/write + b2_gather
  Aggregate over an inner join with a unique build key, grouped by build columns
                                      -> star pipeline: one pass over the probe side
                                         (b2_star_build_* + b2_star_agg), nothing materialised

There is no CPU fallback anywhere in this module: every row-level operation is a call into
libb200sql.so; host code only plans, allocates and moves metadata.
"""
import ctypes as C
import os
from typing import Dict, List, Optional, Sequence, Set

import numpy as np
import torch

from . import _lib as L
from . import device as D
from . import expr as E
from . import parallel as P
from .device import DeviceColumn, TermSpec, I64, F64, U8
from .expr import Expr, ColRef, Lit, Call
from .frame import LazyFrame, Source, TableSource, JoinSource, AggSource, SortSource, LimitSource, WindowSource
from .table import DeviceTable, HostColumn

DENSE_MAX_SLOTS = 1 << 27          # direct-address group tables up to 128M slots
_TORCH_DT = {I64: torch.int64, F64: torch.float64, U8: torch.uint8}
_LOGICAL = {I64: "int64", F64: "float64", U8: "bool"}

# counters the bench / tests read to prove which kernels ran
stats = {"launches": 0, "star_fused": 0, "dense_groupby": 0, "hash_groupby": 0, "dense_join": 0,
         "chain_join": 0, "keyed_join": 0, "partitioned_groupby": 0, "h2d_bytes": 0, "d2h_bytes": 0}


# Optional per-launch timing of the dominant kernels (bench.py sets this to a list): each entry
# is [kernel name, rows, start event, end event], recorded on the launching stream.
kernel_events = None


_timing_events = []      # pre-created timing events: cudaEventCreate costs tens of microseconds of host time


def prefill_timing_events(n: int):
    """bench.py calls this before its timed region so that the per-launch events it asks for are free."""
    while len(_timing_events) < n:
        _timing_events.append(torch.cuda.Event(enable_timing=True))


def _timing_event():
    return _timing_events.pop() if _timing_events else torch.cuda.Event(enable_timing=True)


def _kernel_event_begin(name, rows):
    if kernel_events is None:
        return None
    e0, e1 = _timing_event(), _timing_event()
    e0.record(D.cur_stream())
    rec = [name, rows, e0, e1]
    kernel_events.append(rec)
    return rec


def _kernel_event_end(rec):
    if rec is not None:
        rec[3].record(D.cur_stream())


# Optional per-phase timing of a query's exchange steps (bench.py sets this to a list): entries are
# [phase name, start event, end event] on the launching stream -- "where does an N>1 step go".
phase_events = None


class _Phase:
    __slots__ = ("rec", "stream")

    def __init__(self, name, stream=None):
        self.rec = None
        if phase_events is not None:
            self.rec = [name, _timing_event(), _timing_event()]
            self.stream = stream if stream is not None else D.cur_stream()

    def __enter__(self):
        if self.rec is not None:
            self.rec[1].record(self.stream)
        return self

    def __exit__(self, *exc):
        if self.rec is not None:
            self.rec[2].record(self.stream)
            phase_events.append(self.rec)
        return False


def _dev():
    return D.cur_device()


class Part(dict):
    """One materialised partition: column name -> DeviceColumn, all of length n."""

    # "replicated": every rank holds these rows (or there is one rank); "keyrange": the rows of a
    # multi-GPU aggregate, of which every rank holds the groups of its own slice of the key range
    dist = "replicated"

    def __init__(self, cols=(), n=0):
        super().__init__(cols)
        self.n = int(n)

    def resolve(self):
        return self


class PendingPart(Part):
    """A partition whose row count is still on the device.

    The kernels that produce it are already enqueued (outputs allocated at their upper bound), the
    count travels to a pinned host word behind them; the first access to `.n` or to a column waits
    for it and finishes the partition.  A query whose result nobody looks at yet -- the next
    Context.sql() of a loop, the next operator's launch code -- therefore never stalls the host
    behind the GPU: the reference's lazy dask graph, restated as "kernels first, sync on use"."""

    def __init__(self, thunk):
        dict.__init__(self)
        self._thunk = thunk
        self._n = 0

    @property
    def resolved(self):
        return self._thunk is None

    def resolve(self):
        if self._thunk is not None:
            thunk, self._thunk = self._thunk, None
            D.reset_stream()
            real = thunk().resolve()
            dict.update(self, real)
            self._n = real.n
            self.dist = real.dist     # a fallback path may have produced a differently distributed result
        return self

    @property
    def n(self):
        return self.resolve()._n

    @n.setter
    def n(self, v):
        self._n = int(v)

    def __getitem__(self, k):
        return dict.__getitem__(self.resolve(), k)

    def __iter__(self):
        return dict.__iter__(self.resolve())

    def __len__(self):
        return dict.__len__(self.resolve())

    def __contains__(self, k):
        return dict.__contains__(self.resolve(), k)

    def keys(self):
        return dict.keys(self.resolve())

    def values(self):
        return dict.values(self.resolve())

    def items(self):
        return dict.items(self.resolve())

    def get(self, k, default=None):
        return dict.get(self.resolve(), k, default)


class _PinnedRing:
    """A fixed pool of pinned 64-byte slots for the counts that travel to the host behind the kernels.
    (A fresh pin_memory tensor per query means a cudaHostAlloc whenever the host runs ahead of the GPU
    -- the allocator cannot recycle a block whose copy has not finished -- and that call costs far more
    than the query's launches.)  A slot is reused only after the copy that last used it completed."""

    SLOTS = 1024

    def __init__(self):
        self.buf = torch.empty(self.SLOTS * 8, dtype=torch.int64, pin_memory=True)
        self.events = [None] * self.SLOTS
        self.i = 0

    def take(self):
        i = self.i
        self.i = (i + 1) % self.SLOTS
        ev = self.events[i]
        if ev is not None:
            ev.synchronize()           # 1024 counts in flight: wait for the oldest
        return i, self.buf[i * 8:(i + 1) * 8]


_pinned_ring = None


class DeviceCount:
    """Small integer tensors produced on the device (a row count, duplicate-key flags), copied to pinned
    host memory behind the kernels that wrote them; .get() waits for those copies only and returns the
    values of all tensors in order."""

    def __init__(self, *tensors):
        global _pinned_ring
        if _pinned_ring is None:
            _pinned_ring = _PinnedRing()
        self.views, slots = [], []
        for t in tensors:
            t = t.reshape(-1)
            assert t.numel() * t.element_size() <= 64, "DeviceCount carries a handful of integers"
            i, slot = _pinned_ring.take()
            dst = slot.view(t.dtype)[: t.numel()]
            dst.copy_(t, non_blocking=True)
            self.views.append(dst)
            slots.append(i)
        self.event = torch.cuda.Event()
        self.event.record(D.cur_stream())
        for i in slots:
            _pinned_ring.events[i] = self.event

    def get(self):
        self.event.synchronize()
        out = []
        for v in self.views:
            stats["d2h_bytes"] += v.numel() * v.element_size()
            out.extend(v.tolist())
        return out


# ---------------------------------------------------------------------------------------------
# small helpers
# ---------------------------------------------------------------------------------------------
def simplify_pred(pred: Sequence[Expr]):
    """-> (conjuncts, always_false)"""
    out = []
    for p in pred:
        for c in E.conjuncts(p):
            if isinstance(c, Lit):
                if c.value is None or not c.value:
                    return [], True
                continue
            out.append(c)
    return out, False


def eval_expr(part: Part, e: Expr) -> DeviceColumn:
    """Materialise expression `e` over the columns of `part` (one b2_expr_eval pass)."""
    if isinstance(e, ColRef):
        return part[e.name]
    names = sorted(e.refs())
    cols = [part[n] for n in names]
    prog = E.compile_expr(e, names)
    nullable = E.may_be_null(e, lambda n: part[n].valid is not None)
    stats["launches"] += 1
    return D.expr_eval(prog, cols, part.n, nullable)


def const_column(value, dtype, n, dev) -> DeviceColumn:
    if value is None:
        data = torch.zeros(n, dtype=_TORCH_DT[dtype], device=dev)
        if dtype == F64:
            data.fill_(float("nan"))
        return DeviceColumn(data, torch.zeros(D.bitmap_words(n), dtype=torch.int32, device=dev), dtype)
    return DeviceColumn(torch.full((n,), value, dtype=_TORCH_DT[dtype], device=dev), None, dtype)


def null_column(dtype, logical, n, dev) -> DeviceColumn:
    c = const_column(None, dtype, n, dev)
    c.logical = logical
    return c


def concat_columns(cols: List[DeviceColumn]) -> DeviceColumn:
    """Row-wise concatenation (plumbing: torch.cat on buffers; validity re-packed on device)."""
    if len(cols) == 1:
        return cols[0]
    dev = cols[0].device
    data = torch.cat([c.data for c in cols])
    if all(c.valid is None for c in cols):
        return DeviceColumn(data, None, cols[0].dtype, cols[0].logical)
    # expand each piece's validity to one byte per row, concatenate, re-pack with b2_expr_eval
    masks = []
    for c in cols:
        if c.valid is None:
            masks.append(torch.ones(c.n, dtype=torch.uint8, device=dev))
        else:
            p = Part({"x": c}, c.n)
            m = eval_expr(p, E.unop("not", Call("isnull", [ColRef("x", I64 if c.dtype != U8 else U8)], U8)))
            masks.append(m.data)
    mask = DeviceColumn(torch.cat(masks), None, U8)
    whole = DeviceColumn(data, None, cols[0].dtype, cols[0].logical)
    p = Part({"m": mask, "v": whole}, whole.n)
    out = eval_expr(p, E.case(ColRef("m", U8), ColRef("v", whole.dtype), Lit(None, whole.dtype)))
    if out.valid is None:
        out = DeviceColumn(out.data, None, out.dtype)
    out.logical = cols[0].logical
    return out


def concat_parts(parts: List[Part], names: Sequence[str]) -> Part:
    parts = [p for p in parts if p.n > 0] or parts[:1]
    if len(parts) == 1:
        return Part({n: parts[0][n] for n in names}, parts[0].n)
    return Part({n: concat_columns([p[n] for p in parts]) for n in names}, sum(p.n for p in parts))


class ScanCtx:
    """Binds a partition and a predicate to a b2_scan_t: chooses the column slots, turns
    conjuncts into kernel terms, evaluates what is not a simple term into a mask column."""

    def __init__(self, part: Part, pred: Sequence[Expr]):
        self.part = part
        self.cols: List[DeviceColumn] = []
        self.index: Dict[str, int] = {}
        self.terms: List[TermSpec] = []
        complex_ = []
        for c in pred:
            t = E.as_term(c)
            if t is not None and len(self.terms) < L.MAX_TERMS - 1:
                name, op, lit = t
                col = part[name]
                if op == L.IS_NOT_NULL and col.valid is None and col.dtype != F64:
                    continue  # statically true (e.g. the planner's IS NOT NULL on join keys): no load, no term
                self.terms.append(TermSpec(self._slot_for_name(name), op, lit))
            else:
                complex_.append(c)
        if complex_:
            e = complex_[0]
            for c in complex_[1:]:
                e = E.binop("and", e, c)
            mask = eval_expr(part, E.cast(e, U8))
            self.terms.append(TermSpec(self._add("mask:" + repr(e), mask), L.IS_TRUE, 0))

    def _add(self, key, col: DeviceColumn) -> int:
        if key in self.index:
            return self.index[key]
        if len(self.cols) >= L.MAX_COLS:
            raise NotImplementedError(f"a fused pass reads at most {L.MAX_COLS} columns")
        self.index[key] = len(self.cols)
        self.cols.append(col)
        return self.index[key]

    def _slot_for_name(self, name) -> int:
        return self._add("col:" + name, self.part[name])

    def slot(self, e: Expr) -> int:
        """Column slot holding expression `e` (source column, or materialised temp)."""
        if isinstance(e, ColRef):
            return self._slot_for_name(e.name)
        key = "tmp:" + repr(e)
        if key in self.index:
            return self.index[key]
        if isinstance(e, Lit):
            col = const_column(e.value, e.dtype, self.part.n, _dev())
        else:
            col = eval_expr(self.part, e)
        return self._add(key, col)

    def scan(self) -> L.Scan:
        return D.make_scan(self.cols, self.terms, self.part.n)


def select_part(part: Part, pred: Sequence[Expr], names: Sequence[str]) -> Part:
    """Rows of `part` passing `pred`, restricted to source columns `names` (order-preserving)."""
    ctx = ScanCtx(part, pred)
    slots = [ctx.slot(ColRef(n, part[n].dtype)) for n in names]
    scan = ctx.scan()
    first, rest = slots[: L.MAX_GATHER], slots[L.MAX_GATHER:]
    stats["launches"] += 3
    idx, outs, total = D.select(scan, _dev(), first, want_idx=bool(rest) or not first, cols=ctx.cols)
    res = Part({}, total)
    for n, o in zip(names, outs):
        res[n] = o
    for n, s in zip(names[L.MAX_GATHER:], rest):
        stats["launches"] += 1
        res[n] = D.gather(ctx.cols[s], idx, False)
    return res


# ---------------------------------------------------------------------------------------------
# sources
# ---------------------------------------------------------------------------------------------
def _split_out(src: Source) -> int:
    return max(1, int((getattr(src, "options", None) or {}).get("split_out") or 1))


def source_npartitions(src: Source) -> int:
    if isinstance(src, TableSource):
        return src.table.npartitions
    if isinstance(src, JoinSource):
        return max(source_npartitions(src.left.source), source_npartitions(src.right.source))
    if isinstance(src, AggSource):
        return _split_out(src)           # sql.aggregate.split_out (aggregate.py:321,581): output partitions
    return 1


def split_part(part: Part, k: int) -> List[Part]:
    """The rows of `part` as k contiguous partitions (boundaries on multiples of 32 rows, so validity
    bitmaps split on word boundaries; column slices are views).  A compacted dense group table is in
    key order, so these are key ranges: every group lives in exactly one output partition, which is
    what dask's split_out guarantees (there by hashing the keys)."""
    part = part.resolve()
    n = part.n
    step = max(32, (-(-n // k) + 31) // 32 * 32)
    out = []
    for i in range(k):
        lo, hi = min(n, i * step), min(n, (i + 1) * step)
        if hi > lo:
            piece = Part({name: c.slice(lo, hi) for name, c in part.items()}, hi - lo)
        else:
            piece = Part({name: DeviceColumn(c.data[:0], None, c.dtype, c.logical) for name, c in part.items()}, 0)
        piece.dist = part.dist
        out.append(piece)
    return out


def frame_distribution(frame: LazyFrame) -> str:
    src = frame.source
    if isinstance(src, TableSource):
        return src.table.distribution
    if isinstance(src, JoinSource):
        return join_sides(src)[1]
    if isinstance(src, (SortSource, LimitSource, WindowSource)):
        return "replicated" if P.world()[1] > 1 else "local"
    return "replicated" if P.world()[1] > 1 else "local"


def _global_rows(frame: LazyFrame) -> int:
    """Row estimate every rank agrees on (local estimates differ: a 'root' table is empty off rank 0
    and shards are uneven).  Table counts are gathered once and cached on the immutable table."""
    src = frame.source
    world = P.world()[1]
    if isinstance(src, TableSource):
        t = src.table
        if world == 1 or t.distribution not in ("sharded", "root"):
            return t.nrows
        if "_global_nrows" not in t.__dict__:
            t.__dict__["_global_nrows"] = sum(r[0] for r in P.all_gather_ints([t.nrows], _dev()))
        return t.__dict__["_global_nrows"]
    if isinstance(src, JoinSource):
        return max(_global_rows(src.left), _global_rows(src.right))
    return _global_rows(src.child)


def join_sides(js: JoinSource):
    """(swap, distribution of the result).  swap=True: the LEFT input is hashed (build side) and the
    right one streams.  Decided only from facts every rank shares -- the join type, the inputs'
    distributions and globally agreed row counts -- never from rank-local sizes: ranks that disagree
    on the build side would enter different collectives and hang."""
    how = js.how
    ld, rd = frame_distribution(js.left), frame_distribution(js.right)
    if how == "right":
        swap = True
    elif how != "inner":
        swap = False
    elif P.world()[1] > 1 and (ld == "sharded") != (rd == "sharded"):
        swap = rd == "sharded"          # the sharded side streams, the other one is broadcast
    else:
        swap = _global_rows(js.left) < _global_rows(js.right)
    probe_d, build_d = (rd, ld) if swap else (ld, rd)
    # the build side is made whole on every rank (run_join), so the output rows live where the
    # probe rows live
    return swap, probe_d


def estimated_rows(frame: LazyFrame) -> int:
    src = frame.source
    if isinstance(src, TableSource):
        return src.table.nrows
    if isinstance(src, JoinSource):
        return max(estimated_rows(src.left), estimated_rows(src.right))
    return estimated_rows(src.child)


def gather_keyrange(part: Part) -> Part:
    """Key-range-sharded aggregate -> the same rows on every rank (all-gather in rank order)."""
    if P.world()[1] == 1:
        return part                    # single GPU: nothing to gather, and a pending result stays pending
    part = part.resolve()
    if part.dist != "keyrange":
        return part
    from .merge import allgather_part
    with _Phase("gather_result"):
        out = allgather_part(Part(dict(part), part.n), _dev())
    return out


def _pushdown_terms(pred) -> list:
    """the `column <cmp> literal` conjuncts of a pushed-down predicate as (column, B2 op, literal)"""
    out = []
    for c in pred or ():
        t = E.as_term(c)
        if t is not None:
            out.append(t)
    return out


def materialize(src: Source, needed: Set[str], top: bool = False, pred=None) -> List[Part]:
    """top: the caller is the outermost frame of a query -- a multi-GPU aggregate may then stay
    sharded by key range (one slice of the groups per rank, the dask result with split_out = world
    size); any operator stacked on top of an aggregate needs all groups and gets them gathered."""
    if isinstance(src, TableSource):
        dev = _dev()
        parts = []
        table = src.table
        if hasattr(table, "scan_pruned"):
            # lazy Parquet table: only the referenced columns of the row groups whose statistics admit
            # a row passing the pushed-down conjuncts (conservative: the kernels still filter every row)
            before = table.stats["row_groups_skipped"]
            table_parts = table.scan_pruned(needed, _pushdown_terms(pred))
            stats["rowgroups_skipped"] = stats.get("rowgroups_skipped", 0) + table.stats["row_groups_skipped"] - before
        else:
            table_parts = table.partitions
        for p in table_parts:
            n = next(iter(p.values())).n if p else 0
            cols = {}
            for name in needed:
                c = p[name]
                if isinstance(c, HostColumn):
                    stats["h2d_bytes"] += c.nbytes()
                    hc, c = c, c.to_device(dev)
                    if hc.stats is None:
                        # statistics ride on the first upload and stay with the (immutable) host column
                        hc.stats = c.ensure_stats()
                cols[name] = c
            parts.append(Part(cols, n))
        return parts
    if isinstance(src, JoinSource):
        return run_join(src, needed)
    if isinstance(src, AggSource):
        part = run_aggregate(src)
        part = part if top else gather_keyrange(part)
        k = _split_out(src)
        return split_part(part, k) if k > 1 else [part]
    if isinstance(src, SortSource):
        return [run_sort(src, needed)]
    if isinstance(src, LimitSource):
        return [run_limit(src, needed)]
    if isinstance(src, WindowSource):
        return [run_window(src, needed)]
    raise TypeError(f"unknown source {type(src).__name__}")


def run_sort(src: SortSource, needed: Set[str]) -> Part:
    """ORDER BY: one stable radix sort of row ids per key (last key first), then one gather per
    output column (b2_sort_by + b2_gather)."""
    dev = _dev()
    names = [n for n in src.child.columns if n in needed or any(n == k for k, _, _ in src.keys)]
    whole = concat_parts(execute(src.child, names), names)
    n = whole.n
    if n <= 1:
        return Part({k: whole[k] for k in names if k in needed}, n)
    idx = torch.empty(n, dtype=torch.int32, device=dev)
    L.iota(D.ptr(idx), n, D.stream_ptr())
    ws = torch.empty(L.sort_ws_bytes(n), dtype=torch.uint8, device=dev)
    for name, asc, nulls_first in reversed(src.keys):
        cs = whole[name].as_struct()
        stats["launches"] += 29
        L.sort_by(C.byref(cs), n, 0 if asc else 1, 1 if nulls_first else 0, D.ptr(idx), D.ptr(ws), D.stream_ptr())
    out = Part({}, n)
    for k in names:
        if k in needed:
            stats["launches"] += 1
            out[k] = D.gather(whole[k], idx, False)
    return out


_WIN_OP = {"row_number": L.WIN_ROW_NUMBER, "rank": L.WIN_RANK, "dense_rank": L.WIN_DENSE_RANK, "sum": L.WIN_SUM,
           "count": L.WIN_COUNT, "avg": L.WIN_AVG, "min": L.WIN_MIN, "max": L.WIN_MAX, "first_value": L.WIN_FIRST,
           "last_value": L.WIN_LAST}


def run_window(src: WindowSource, needed: Set[str]) -> Part:
    """Window functions (window.py:227-348 of the reference: one groupby().apply() per call).  The child
    is made whole (and, at world > 1, gathered from its shards: every rank computes the same rows);
    calls with identical (PARTITION BY, ORDER BY) share one sort -- b2_sort_by per key, order keys then
    partition keys, last key first -- and one gather of the columns still needed, then
    b2_window_segments and one kernel per call.  The result is in the last sort's row order."""
    dev = _dev()
    refs = set()
    for w in src.calls:
        refs.update(w.args)
        refs.update(w.partition)
        refs.update(k for k, _, _ in w.order)
    names = [n for n in src.child.columns if n in needed or n in refs]
    whole = concat_parts(execute(src.child, names), names)
    if P.world()[1] > 1 and frame_distribution(src.child) in ("sharded", "root"):
        from .merge import allgather_part
        with _Phase("window_gather"):
            whole = allgather_part(Part(dict(whole), whole.n), dev)
    n = whole.n
    if n >= 1 << 31:
        raise NotImplementedError(f"window functions over {n} rows: the input must hold fewer than 2^31 rows "
                                  "(the sort's int32 row ids)")
    calls = [w for w in src.calls if w.out in needed]
    specs: Dict[tuple, list] = {}
    for w in calls:
        specs.setdefault((tuple(w.partition), tuple(w.order)), []).append(w)
    cur = {k: whole[k] for k in names}
    if n == 0:
        for w in calls:
            dt, lg = src.schema[w.out]
            cur[w.out] = DeviceColumn(torch.empty(0, dtype=_TORCH_DT[dt], device=dev), None, dt, lg)
        return Part({k: cur[k] for k in src.schema if k in needed}, 0)
    ws = torch.empty(max(L.sort_ws_bytes(n), L.window_ws_bytes(n)), dtype=torch.uint8, device=dev)
    seg = torch.empty((5, n), dtype=torch.int32, device=dev)
    segs = L.WSegs(*[seg[i].data_ptr() for i in range(5)])
    for (part_keys, order_keys), group in specs.items():
        keys = [(k, True, False) for k in part_keys] + list(order_keys)
        if len(keys) > L.WIN_MAX_KEYS:
            raise NotImplementedError(f"a window partitions and orders by at most {L.WIN_MAX_KEYS} columns")
        if keys:
            idx = torch.empty(n, dtype=torch.int32, device=dev)
            rec = _kernel_event_begin("window_sort", n)
            stats["launches"] += 1
            L.iota(D.ptr(idx), n, D.stream_ptr())
            for name, asc, nulls_first in reversed(keys):
                cs = cur[name].as_struct()
                stats["launches"] += 29
                L.sort_by(C.byref(cs), n, 0 if asc else 1, 1 if nulls_first else 0, D.ptr(idx), D.ptr(ws),
                          D.stream_ptr())
            _kernel_event_end(rec)
            rec = _kernel_event_begin("window_gather", n)
            for k in list(cur):
                stats["launches"] += 1
                cur[k] = D.gather(cur[k], idx, False)
            _kernel_event_end(rec)
        kc = (L.Col * max(1, len(keys)))(*[cur[k].as_struct() for k, _, _ in keys])
        rec = _kernel_event_begin("window_segments", n)
        stats["launches"] += 3
        L.window_segments(kc, len(part_keys), len(keys), n, C.byref(segs), D.ptr(ws), D.stream_ptr())
        _kernel_event_end(rec)
        for w in group:
            rec = _kernel_event_begin("window_" + w.func, n)
            cur[w.out] = _window_call(w, cur, n, segs, ws, src.schema[w.out][1])
            _kernel_event_end(rec)
        stats["window_specs"] = stats.get("window_specs", 0) + 1
    return Part({k: cur[k] for k in src.schema if k in needed}, n)


def _frame_struct(frame) -> "L.WFrame":
    unit, lo, hi = frame

    def bound(b):
        kind, off = b
        if kind.startswith("UNBOUNDED"):
            return L.WB_UNBOUNDED, 0
        if kind == "CURRENT":
            return L.WB_OFFSET, 0
        return L.WB_OFFSET, (-off if kind == "PRECEDING" else off)

    (lk, lo_off), (hk, hi_off) = bound(lo), bound(hi)
    return L.WFrame(1 if unit == "RANGE" else 0, lk, hk, 0, lo_off, hi_off)


def _window_call(w, cur, n, segs, ws, logical) -> DeviceColumn:
    dev = _dev()
    if w.func in ("row_number", "rank", "dense_rank"):
        out = torch.empty(n, dtype=torch.int64, device=dev)
        stats["launches"] += 1
        L.window_rank(_WIN_OP[w.func], n, C.byref(segs), D.ptr(out), D.stream_ptr())
        return DeviceColumn(out, None, I64)
    val = cur[w.args[0]] if w.args else None
    back_to_bool = False
    if val is not None and val.dtype == U8:
        # booleans run as int64 0/1 (SUM counts TRUEs); MIN / MAX / FIRST / LAST / LAG / LEAD cast back
        stats["launches"] += 1
        val = eval_expr(Part({"v": val}, n), E.cast(ColRef("v", U8), I64))
        back_to_bool = w.func not in ("sum", "count", "avg")
    vs = val.as_struct() if val is not None else L.Col()
    valid = torch.empty(D.bitmap_words(n), dtype=torch.int32, device=dev)
    if w.func in ("lag", "lead"):
        k, default = w.params
        out = torch.empty(n, dtype=_TORCH_DT[val.dtype], device=dev)
        raw = 0
        if default is not None:
            raw = int(np.array([default], dtype=np.float64 if val.dtype == F64 else np.int64).view(np.int64)[0])
        stats["launches"] += 1
        L.window_offset(C.byref(vs), n, -k if w.func == "lag" else k, default is not None, raw, C.byref(segs),
                        D.ptr(out), D.ptr(valid), D.stream_ptr())
        dt = val.dtype
    else:
        dt = I64 if w.func == "count" else F64 if w.func == "avg" else val.dtype
        out = torch.empty(n, dtype=_TORCH_DT[dt], device=dev)
        if w.func == "count":
            valid = None
        fr = _frame_struct(w.frame)
        stats["launches"] += 4
        L.window_agg(C.byref(vs), _WIN_OP[w.func], C.byref(fr), n, C.byref(segs), D.ptr(out), D.ptr(valid),
                     D.ptr(ws), D.stream_ptr())
    res = DeviceColumn(out, valid, dt, logical if dt != U8 else None)
    if back_to_bool:
        stats["launches"] += 1
        res = eval_expr(Part({"v": res}, n), E.cast(ColRef("v", I64), U8))
        res.logical = logical
    return res


def run_limit(src: LimitSource, needed: Set[str]) -> Part:
    dev = _dev()
    names = [n for n in src.child.columns if n in needed]
    whole = concat_parts(execute(src.child, names), names)
    lo = min(src.offset, whole.n)
    hi = whole.n if src.fetch is None else min(whole.n, lo + int(src.fetch))
    if lo == 0 and hi == whole.n:
        return whole
    idx = torch.arange(lo, hi, dtype=torch.int32, device=dev)
    out = Part({}, hi - lo)
    for k in names:
        c = whole[k]
        if c.valid is None:
            out[k] = DeviceColumn(c.data[lo:hi], None, c.dtype, c.logical)   # a view: no copy
        else:
            stats["launches"] += 1
            out[k] = D.gather(c, idx, False)
    return out


def empty_part(exprs: Dict[str, Expr]) -> Part:
    dev = _dev()
    out = Part({}, 0)
    for n, e in exprs.items():
        lg = e.logical if isinstance(e, ColRef) else _LOGICAL[e.dtype]
        out[n] = DeviceColumn(torch.empty(0, dtype=_TORCH_DT[e.dtype], device=dev), None, e.dtype, lg)
    return out


def execute(frame: LazyFrame, needed: Optional[Sequence[str]] = None, top: bool = False) -> List[Part]:
    """Materialise `needed` output columns of `frame`, partition by partition.  top=True lets the
    groups of a multi-GPU aggregate stay with the rank that owns their key range (Part.dist ==
    "keyrange"); compute_frame gathers them on the way to the host."""
    D.reset_stream()
    names = list(needed) if needed is not None else frame.columns
    exprs = {n: frame.exprs[n] for n in names}
    pred, never = simplify_pred(frame.pred)
    if never:
        return [empty_part(exprs)]
    src_needed: Set[str] = set()
    for e in exprs.values():
        e.refs(src_needed)
    for p in pred:
        p.refs(src_needed)
    parts = materialize(frame.source, src_needed, top, pred)

    def project(part: Part) -> Part:
        dist = part.dist
        if pred:
            colrefs = sorted({r for e in exprs.values() for r in e.refs()})
            part = select_part(part, pred, colrefs)
        res = Part({}, part.n)
        res.dist = dist
        for n, e in exprs.items():
            if isinstance(e, Lit):
                res[n] = const_column(e.value, e.dtype, part.n, _dev())
            else:
                res[n] = eval_expr(part, e)
        return res

    out = []
    for part in parts:
        if isinstance(part, PendingPart) and not part.resolved:
            lazy = PendingPart(lambda part=part: project(part.resolve()))   # stays lazy
            lazy.dist = part.dist
            out.append(lazy)
        else:
            out.append(project(part))
    return out


# ---------------------------------------------------------------------------------------------
# aggregation
# ---------------------------------------------------------------------------------------------
MOMENT_FUNCS = ("var_samp", "var_pop", "stddev_samp", "stddev_pop")


class KAgg:
    __slots__ = ("expr", "op", "need_cnt", "dtype", "nullable")

    def __init__(self, expr, op, dtype, nullable=True):
        self.expr, self.op, self.need_cnt, self.dtype, self.nullable = expr, op, False, dtype, nullable


class AggPlan:
    """Maps SQL aggregates onto kernel accumulators, sharing accumulators and counts.

    Semantics follow aggregate.py:486-495: SUM is sum(min_count=1) (all-NULL group -> NULL),
    AVG = mean (NULLs skipped), COUNT(col) skips NULLs, COUNT(*) counts rows."""

    def __init__(self, aggs, nullable, shifts=None):
        self.kaggs: List[KAgg] = []
        self.need_rows = False
        self.outs = []  # (out_name, fn, acc_idx, cnt_ref, in_dtype, logical)  cnt_ref: int | 'rows' | None
        self.second = {}   # moment functions: out_name -> accumulator of the sum of squared deviations
        for e, out, fn in aggs:
            fn = fn.lower()
            if fn in MOMENT_FUNCS:
                # VAR / STDDEV from (n, sum(x-K), sum((x-K)^2)): the three sums are additive over
                # partitions and GPUs, and with K near the data (the midpoint of the column's range,
                # agreed by all ranks) the subtraction S2 - S1^2/n no longer cancels catastrophically
                # for large-mean data the way sum-of-squares around zero does.  (pandas' groupby var is
                # Welford's update, aggregate.py:129-231 builds on it.)
                x = E.cast(e, F64)
                k_shift = float((shifts or {}).get(repr(e), 0.0))
                d = E.binop("sub", x, k_shift) if k_shift else x
                a1 = self._slot(d, L.AGG_SUM, True)
                self.second[out] = self._slot(E.binop("mul", d, d), L.AGG_SUM, True)
                self.outs.append((out, fn, a1, self._cnt(d), F64, "float64"))
                continue
            lg = (e.logical if isinstance(e, ColRef) else _LOGICAL[e.dtype]) if e is not None else "int64"
            if fn == "size" or e is None:
                self.need_rows = True
                self.outs.append((out, "size", None, "rows", I64, "int64"))
                continue
            nul = nullable(e)
            if fn == "count":
                if nul:
                    self.outs.append((out, "count", None, self._cnt(e), e.dtype, lg))
                else:
                    self.need_rows = True
                    self.outs.append((out, "count", None, "rows", e.dtype, lg))
            elif fn == "sum":
                a = self._slot(e, L.AGG_SUM, nul)
                self.outs.append((out, "sum", a, self._cnt(e) if nul else None, e.dtype, lg))
            elif fn in ("mean", "avg"):
                a = self._slot(e, L.AGG_SUM if e.dtype == F64 else L.AGG_SUMF, nul)
                if nul:
                    c = self._cnt(e)
                else:
                    self.need_rows = True
                    c = "rows"
                self.outs.append((out, "mean", a, c, e.dtype, lg))
            elif fn in ("min", "max"):
                a = self._slot(e, L.AGG_MIN if fn == "min" else L.AGG_MAX, nul)
                self.outs.append((out, fn, a, self._cnt(e) if nul else None, e.dtype, lg))
            else:
                raise NotImplementedError(f"aggregate function {fn} is a 'next' row of the hot-path scope")
        if len(self.kaggs) > L.MAX_AGGS:
            raise NotImplementedError(f"more than {L.MAX_AGGS} distinct accumulators in one GROUP BY")
        # a float SUM over a never-NULL input receives an add from every row of its group: started
        # at -0.0 it doubles as the group's existence flag (device.GroupTable.indicator)
        self.indicator = None
        if not self.need_rows and os.environ.get("B200SQL_NO_INDICATOR") != "1":
            for i, k in enumerate(self.kaggs):
                if not k.nullable and (k.op == L.AGG_SUMF or (k.op == L.AGG_SUM and k.dtype == F64)):
                    self.indicator = i
                    break

    def _slot(self, e, op, nullable=True):
        for i, k in enumerate(self.kaggs):
            if k.op == op and repr(k.expr) == repr(e):
                return i
        self.kaggs.append(KAgg(e, op, e.dtype, nullable))
        return len(self.kaggs) - 1

    def _cnt(self, e):
        for i, k in enumerate(self.kaggs):
            if repr(k.expr) == repr(e):
                k.need_cnt = True
                return i
        self.kaggs.append(KAgg(e, L.AGG_COUNT, e.dtype, True))
        self.kaggs[-1].need_cnt = True
        return len(self.kaggs) - 1


def _nullable_fn(child: LazyFrame, sharded: bool = False):
    """Can an aggregate input be NULL?  bitmap present, float column (NaN), or computed.
    sharded: the answer decides which accumulator arrays a group table carries (count next to the sum,
    -0.0 indicator or presence bitmap), and the ranks' partial tables are merged array by array -- so for
    a sharded input the ranks agree on it (MAX over the ranks: NULL anywhere = nullable everywhere).
    Every rank asks the same questions in the same order (same plan), one tiny all-reduce each."""
    src = child.source

    def nullable(e: Expr):
        if isinstance(e, Lit):
            return e.value is None
        if isinstance(e, ColRef) and isinstance(src, TableSource):
            t = src.table
            has_bitmap = t.column_nullable(e.name)
            if e.dtype != F64:
                return has_bitmap
            if hasattr(t, "scan_pruned"):
                return True          # lazy Parquet: NaNs are not in the file's null counts; keep the count
            # NaN is NULL for float inputs: whether a count must be kept next to the sum depends on
            # the data.  One statistics pass per resident column (cached) saves an atomic per row
            # on every later query; host-resident columns are not uploaded twice for this.
            for p in t.partitions:
                c = p[e.name]
                if c.stats is None and isinstance(c, DeviceColumn):
                    c.ensure_stats()
            sts = [p[e.name].stats for p in t.partitions]
            if all(s is not None for s in sts):
                return has_bitmap or any(s.nulls > 0 for s in sts)
            return True
        if e.dtype == F64:
            return True
        return E.may_be_null(e, lambda n: True)

    if not sharded or P.world()[1] == 1:
        return nullable

    def agreed(e: Expr):
        t = torch.tensor([1 if nullable(e) else 0], dtype=torch.int64, device=_dev())
        return bool(int(P.allreduce_(t, "max").item()))

    return agreed


def _one_row(value, dtype, logical, dev) -> DeviceColumn:
    if value is None:
        c = null_column(dtype, logical, 1, dev)
        return c
    c = const_column(value, dtype, 1, dev)
    c.logical = logical
    return c


def _moment_shifts(aggs, parts, child, sharded):
    """{repr(input expr): K} for the VAR / STDDEV aggregates: K = midpoint of the input's value range
    (cached table statistics for plain columns), the same on every rank."""
    shifts = {}
    for e, _, fn in aggs:
        if e is None or fn.lower() not in MOMENT_FUNCS or repr(e) in shifts:
            continue
        st = _key_stats(parts, e, child)
        lo, hi = (float(st.vmin), float(st.vmax)) if st.vmin is not None else (float("inf"), float("-inf"))
        if sharded:
            t = torch.tensor([lo, -hi], dtype=torch.float64, device=_dev())
            P.allreduce_(t, "min")
            lo, hi = float(t[0].item()), -float(t[1].item())
        mid = (lo + hi) / 2 if lo <= hi else 0.0
        shifts[repr(e)] = mid if np.isfinite(mid) else 0.0
    return shifts


def run_aggregate(src: AggSource, allow_fast=True) -> Part:
    if allow_fast:
        # a fused star query that was prepared before: straight to its cached launch descriptors
        last = src.__dict__.get("_prepared_last")
        if last is not None and last[0] == (P.world()[1], _dev().index) and last[1] in PreparedStar._live \
                and os.environ.get("B200SQL_NO_PREPARED") != "1":
            return last[1].run(src)
    child = src.child
    pred, never = simplify_pred(child.pred)
    gexprs = [child.exprs[g] for g in src.group_cols]
    aggs = [(child.exprs[i] if i is not None else None, out, fn) for i, out, fn in src.aggs]
    sharded = P.world()[1] > 1 and frame_distribution(child) in ("sharded", "root")
    if gexprs and isinstance(child.source, JoinSource) and not never:
        res = try_star(src, child, gexprs, aggs, pred, sharded, allow_fast)
        if res is not None:
            return res
    if not gexprs and isinstance(child.source, JoinSource) and not never and allow_fast:
        res = try_join_agg(src, child, aggs, pred, sharded)
        if res is not None:
            return res
    needed: Set[str] = set()
    for e in gexprs:
        e.refs(needed)
    for e, _, _ in aggs:
        if e is not None:
            e.refs(needed)
    for p in pred:
        p.refs(needed)
    parts = [] if never else materialize(child.source, needed, pred=pred)
    plan = AggPlan(aggs, _nullable_fn(child, sharded), _moment_shifts(aggs, parts, child, sharded))
    if not gexprs:
        return global_aggregate(parts, pred, plan, sharded)
    return grouped_aggregate(parts, pred, gexprs, src.group_cols, plan, child, sharded, src.options)


def global_aggregate(parts: List[Part], pred, plan: AggPlan, sharded: bool) -> Part:
    dev = _dev()
    # kernel aggregates: every KAgg, plus COUNT(*) (last) to know whether any row passed
    k = len(plan.kaggs)
    if k + 1 > L.MAX_AGGS:
        raise NotImplementedError("too many aggregates for one global pass")
    ga = None
    for part in parts:
        if part.n == 0:
            continue
        ctx = ScanCtx(part, pred)
        specs = [(ctx.slot(ka.expr), ka.op) for ka in plan.kaggs] + [(-1, L.AGG_COUNT)]
        if ga is None:
            ga = D.GlobalAgg(dev, specs)
        else:
            ga.specs = specs
            ga.aggs = D.make_aggs(specs)
        stats["launches"] += 2
        ev = _kernel_event_begin("b2_scan_agg_kernel", part.n)
        ga.update(ctx.scan())
        _kernel_event_end(ev)
    if ga is None:
        acc = np.array([{L.AGG_MIN: (1 << 63) - 1, L.AGG_MAX: -(1 << 63)}.get(ka.op, 0) for ka in plan.kaggs] + [0],
                       dtype=np.int64)
        cnt = np.zeros(k + 1, dtype=np.int64)
    else:
        acc, cnt = ga.result()
        stats["d2h_bytes"] += 16 * (k + 1)
    if sharded:
        acc, cnt = _allreduce_global(acc, cnt, plan, dev)
    return _finish_global(plan, acc, cnt, dev)


def _finish_global(plan: AggPlan, acc, cnt, dev, float_acc=None) -> Part:
    """One-row result of a global aggregate from the raw accumulators (host numpy int64 bit patterns;
    entry len(plan.kaggs) of `cnt` is the number of rows that took part).  float_acc[i]: accumulator
    i holds a float64 although its input expression is typed int (never the case for plain scans)."""
    k = len(plan.kaggs)
    rows = int(cnt[k])
    out = Part({}, 1 if rows > 0 else 0)
    for name, fn, a, c, in_dt, lg in plan.outs:
        n_valid = rows if c == "rows" else (int(cnt[c]) if c is not None else rows)
        is_f = in_dt == F64 or bool(float_acc and a is not None and float_acc[a])
        if fn in ("size", "count"):
            val, dt, lgo = n_valid, I64, "int64"
        elif fn in MOMENT_FUNCS:
            dt, lgo = F64, "float64"
            ddof = 0 if fn.endswith("pop") else 1
            if n_valid <= ddof:
                val = None
            else:
                s1 = acc[a:a + 1].view(np.float64)[0].item()
                a2 = plan.second[name]
                s2 = acc[a2:a2 + 1].view(np.float64)[0].item()
                val = max((s2 - s1 * s1 / n_valid) / (n_valid - ddof), 0.0)
                if fn.startswith("stddev"):
                    val = val ** 0.5
        elif fn == "sum":
            dt, lgo = (F64, lg if in_dt == F64 else "float64") if is_f else (I64, lg if lg != "bool" else "int64")
            val = None if n_valid == 0 else (acc[a:a + 1].view(np.float64)[0].item() if is_f else int(acc[a]))
        elif fn == "mean":
            dt, lgo = F64, "float64"
            val = None if n_valid == 0 else acc[a:a + 1].view(np.float64)[0].item() / n_valid
        else:  # min / max
            dt, lgo = (F64, lg if in_dt == F64 else "float64") if is_f else (I64, lg)
            if n_valid == 0:
                val = None
            elif is_f:
                val = L.ordered_to_f64(int(acc[a]))
            else:
                val = int(acc[a])
        col = _one_row(val, dt, lgo, dev)
        if rows == 0:
            col = DeviceColumn(col.data[:0], None, dt, lgo)
        out[name] = col
    return out


def _allreduce_global(acc, cnt, plan: AggPlan, dev):
    """Combine per-rank scalars: all-gather the tiny vectors, fold on the host."""
    import torch.distributed as dist
    size = P.world()[1]
    t = torch.from_numpy(np.concatenate([acc, cnt])).to(dev)
    gathered = [torch.empty_like(t) for _ in range(size)]
    dist.all_gather(gathered, t)
    allv = torch.stack(gathered).cpu().numpy()
    k = len(acc)
    accs, cnts = allv[:, :k], allv[:, k:]
    out = accs[0].copy()
    for i, ka in enumerate(plan.kaggs):
        col = accs[:, i]
        if ka.op in (L.AGG_SUM, L.AGG_SUMF):
            if ka.op == L.AGG_SUMF or ka.dtype == F64:
                out[i:i + 1] = np.array([col.view(np.float64).sum()]).view(np.int64)
            else:
                out[i] = np.sum(col.astype(np.uint64), dtype=np.uint64).astype(np.int64)
        elif ka.op == L.AGG_MIN:
            out[i] = col.min()
        elif ka.op == L.AGG_MAX:
            out[i] = col.max()
    return out, cnts.sum(axis=0)


# -- grouped ----------------------------------------------------------------------------------
def _padded_slots(nslots: int, sharded: bool) -> int:
    """Slots to allocate: a table that will be reduce-scattered is padded to a multiple of
    32 x world size (equal, bitmap-word-aligned slices for every rank)."""
    size = P.world()[1]
    if not sharded or size == 1:
        return nslots
    q = 32 * size
    return (nslots + q - 1) // q * q


class GroupState:
    """Accumulators + key storage of one GROUP BY, independent of how slots are found."""

    def __init__(self, dev, nslots, plan: AggPlan, need_present, force_rows=False, alloc=None, new=None):
        need_rows = plan.need_rows or force_rows
        specs = [(0, ka.op) for ka in plan.kaggs]
        self.table = D.GroupTable(dev, nslots, specs, [ka.dtype for ka in plan.kaggs],
                                  [ka.need_cnt for ka in plan.kaggs], need_rows,
                                  need_present and not need_rows,
                                  indicator=None if need_rows else plan.indicator, alloc=alloc, new=new)
        self.plan = plan
        self.nslots = nslots

    def bind(self, ctx: ScanCtx):
        specs = [(ctx.slot(ka.expr), ka.op) for ka in self.plan.kaggs]
        self.table.specs = specs
        self.table.aggs = D.make_aggs(specs)


def _key_stats(parts: List[Part], e: Expr, child: LazyFrame):
    """min/max/nulls of a group/join key over all partitions (cached on table columns)."""
    if isinstance(e, ColRef) and isinstance(child.source, TableSource):
        return child.source.table.column_stats(e.name)
    mn = mx = None
    nulls = 0
    repeat = 0.0
    for p in parts:
        if p.n == 0:
            continue
        st = eval_expr(p, e).ensure_stats()
        nulls += st.nulls
        repeat = max(repeat, st.repeat)
        if st.vmin is not None:
            mn = st.vmin if mn is None else min(mn, st.vmin)
            mx = st.vmax if mx is None else max(mx, st.vmax)
    return D.Stats(mn, mx, nulls, repeat)


def grouped_aggregate(parts, pred, gexprs, gnames, plan: AggPlan, child, sharded, options) -> Part:
    dev = _dev()
    total_rows = sum(p.n for p in parts)
    if sharded:
        t = torch.tensor([total_rows], dtype=torch.int64, device=dev)
        total_rows_all = int(P.allreduce_(t).item())
    else:
        total_rows_all = total_rows
    glog = [(e.logical if isinstance(e, ColRef) else _LOGICAL[e.dtype]) for e in gexprs]
    if total_rows_all == 0:
        out = Part({}, 0)
        for g, e, lg in zip(gnames, gexprs, glog):
            out[g] = DeviceColumn(torch.empty(0, dtype=_TORCH_DT[e.dtype], device=dev), None, e.dtype, lg)
        for name, fn, a, c, in_dt, lg in plan.outs:
            dt = I64 if fn in ("size", "count") else (F64 if fn == "mean" or in_dt == F64 else I64)
            out[name] = DeviceColumn(torch.empty(0, dtype=_TORCH_DT[dt], device=dev), None, dt)
        return out

    # ---- choose the table kind
    mode = "hashk"
    kmin = rng = None
    if len(gexprs) == 1 and gexprs[0].dtype in (I64, U8):
        st = _key_stats(parts, gexprs[0], child)
        lo, hi = st.vmin, st.vmax
        if sharded:  # agree on the global key range
            big = (1 << 62)
            t = torch.tensor([lo if lo is not None else big, -(hi if hi is not None else -big)],
                             dtype=torch.int64, device=dev)
            P.allreduce_(t, "min")
            lo, hi = int(t[0].item()), -int(t[1].item())
            if lo == big:
                lo = hi = None
        if lo is None:
            lo = hi = 0
        if hi - lo + 2 <= DENSE_MAX_SLOTS and (hi - lo) <= 8 * max(total_rows_all, 1) + 1024:
            mode, kmin, rng = "dense", lo, hi - lo + 1
            # keys that repeat inside a warp: pre-aggregate per warp / CTA (b2_groupby_dense_grouped).
            # A rank-local choice: both kernels fill the same table.
            repeats = st.repeat >= REPEAT_MIN and os.environ.get("B200SQL_NO_WARPAGG") != "1"
        elif gexprs[0].dtype == I64:
            mode = "hash1"
    elif len(gexprs) == 1 and gexprs[0].dtype == F64:
        mode = "hash1"
    if len(gexprs) > L.MAX_KEYS:
        raise NotImplementedError(f"GROUP BY over more than {L.MAX_KEYS} columns")

    if mode == "dense":
        stats["dense_groupby"] += 1
        nslots = rng + 1
        work = []
        for part in parts:
            if part.n == 0:
                continue
            ctx = ScanCtx(part, pred)
            kslot = ctx.slot(gexprs[0])
            work.append((part, ctx, kslot, [ctx.slot(ka.expr) for ka in plan.kaggs]))
        buckets = _partition_plan(nslots, plan, work, total_rows)
        if buckets is not None:
            # table far beyond L2: reorder (key, inputs) by key range first so the atomics of the
            # aggregation pass stay inside one L2-sized slice of the table at a time
            stats["partitioned_groupby"] += 1
            shift, nbuckets = buckets
            gs = GroupState(dev, nslots + 1, plan, need_present=True,      # +1: see b2_range_partition
                            alloc=_padded_slots(nslots + 1, sharded))
            # all input partitions are reordered into ONE bucket-ordered array: the aggregation pass
            # then meets every slice of the table exactly once (per-partition passes would reload it
            # once per partition)
            carried = sorted({v for _, _, _, vs in work for v in vs})
            n_all = sum(part.n for part, _, _, _ in work)
            ws = torch.zeros(L.range_partition_ws_bytes(nbuckets) // 8, dtype=torch.int64, device=dev)
            for part, ctx, kslot, vslots in work:
                stats["launches"] += 1
                ev = _kernel_event_begin("b2_part_hist_kernel", part.n)
                L.range_partition_hist(C.byref(ctx.scan()), kslot, kmin, nslots, shift, nbuckets, D.ptr(ws),
                                       D.stream_ptr())
                _kernel_event_end(ev)
            stats["launches"] += 1
            L.range_partition_scan(nbuckets, D.ptr(ws), D.stream_ptr())
            ctx0 = work[0][1]
            out_key = torch.full((n_all,), kmin + nslots + 1, dtype=torch.int64, device=dev)
            outs = [torch.empty(n_all, dtype=_TORCH_DT[ctx0.cols[c].dtype], device=dev) for c in carried]
            cc = (C.c_int32 * max(1, len(carried)))(*carried)
            oc = (C.c_void_p * max(1, len(carried)))(*[o.data_ptr() for o in outs])
            for part, ctx, kslot, vslots in work:
                stats["launches"] += 1
                ev = _kernel_event_begin("b2_part_scatter_kernel", part.n)
                L.range_partition_scatter(C.byref(ctx.scan()), kslot, kmin, nslots, shift, nbuckets, len(carried), cc,
                                          D.ptr(out_key), oc, D.ptr(ws), D.stream_ptr())
                _kernel_event_end(ev)
            cols2 = [DeviceColumn(out_key, None, I64)] + \
                    [DeviceColumn(o, None, ctx0.cols[c].dtype) for o, c in zip(outs, carried)]
            specs = [(1 + carried.index(v), ka.op) for v, ka in zip(work[0][3], plan.kaggs)]
            gs.table.specs, gs.table.aggs = specs, D.make_aggs(specs)
            stats["launches"] += 1
            ticket = torch.zeros(1, dtype=torch.int64, device=dev)
            scan2 = D.make_scan(cols2, [], n_all)
            ev = _kernel_event_begin("b2_groupby_dense_ordered", n_all)
            L.groupby_dense_ordered(C.byref(scan2), 0, int(kmin), gs.table.nslots, gs.table.aggs, len(gs.table.specs),
                                    C.byref(gs.table.state), D.ptr(ticket), D.stream_ptr())
            _kernel_event_end(ev)
        else:
            gs = GroupState(dev, nslots, plan, need_present=True, alloc=_padded_slots(nslots, sharded))
            # keys that repeat: "hot" = heavy hitters (sampled once per query from the first partition) go
            # to thread-private partials; "warp" = match-based warp aggregation + per-CTA table
            skew = os.environ.get("B200SQL_SKEW", "hot") if repeats else None
            hot = None
            for part, ctx, kslot, _ in work:
                gs.bind(ctx)
                if skew == "hot" and hot is None:
                    kcol = ctx.cols[kslot]
                    if kcol.dtype == I64 and nslots < (1 << 31):
                        stats["launches"] += 1
                        hot = D.hot_slots(kcol, kmin, nslots)
                    else:
                        skew = "warp"
                stats["launches"] += 1
                ev = _kernel_event_begin("b2_groupby_dense_kernel", part.n)
                D.groupby_dense(ctx.scan(), kslot, kmin, gs.table, skew=skew, hot=hot)
                _kernel_event_end(ev)
            stats["grouped_groupby"] = stats.get("grouped_groupby", 0) + (1 if repeats else 0)
        key_nullable = E.may_be_null(gexprs[0], lambda n: any(n in p and p[n].valid is not None for p in parts))
        if sharded:
            # a rank whose shard has no NULL key must still agree that the NULL slot may be occupied
            t = torch.tensor([1 if key_nullable else 0], dtype=torch.int64, device=dev)
            key_nullable = bool(int(P.allreduce_(t, "max").item()))
        view = _merge_dense(gs.table, plan, sharded, dev)
        # the NULL group sits in slot rng of the key range; the range-partitioned path allocates one slot
        # more than that (b2_range_partition encodes NULL as the key value kmin + rng), which stays empty
        view.nslots = nslots
        if view.lo == 0 and view.count > nslots and view.dist != "keyrange":
            view.count = nslots
        return _finalize_dense(view, kmin, gnames[0], gexprs[0], glog[0], plan, dev, key_nullable)

    # ---- hash tables: size from the row count, grow on overflow
    stats["hash_groupby"] += 1
    cap = D._pow2_at_least(max(1024, min(2 * total_rows, 1 << 22)))
    while True:
        flags = D.new_flags(dev)
        gs = GroupState(dev, cap + 2 if mode == "hash1" else cap, plan, need_present=(mode == "hashk"))
        if mode == "hash1":
            tkeys = torch.full((cap + 2,), L.EMPTY_KEY, dtype=torch.int64, device=dev)
        else:
            nk = len(gexprs)
            tkeys = torch.zeros(nk * cap, dtype=torch.int64, device=dev)
            tnulls = torch.zeros(cap, dtype=torch.uint8, device=dev)
            tstate = torch.zeros(cap, dtype=torch.int32, device=dev)
        for part in parts:
            if part.n == 0:
                continue
            ctx = ScanCtx(part, pred)
            kslots = [ctx.slot(e) for e in gexprs]
            gs.bind(ctx)
            stats["launches"] += 1
            if mode == "hash1":
                D.groupby_hash1(ctx.scan(), kslots[0], tkeys, cap, gs.table, flags)
            else:
                D.groupby_hashk(ctx.scan(), kslots, tkeys, tnulls, tstate, cap, gs.table, flags)
        fl = flags.cpu().tolist()
        if fl[0] == 0:
            break
        if cap >= (1 << 31):
            raise MemoryError("group table would exceed 2^31 slots")
        cap *= 4
    if mode == "hash1":
        raw = _extract_hash1(gs, tkeys, cap, fl, gnames[0], gexprs[0], glog[0], dev)
    else:
        raw = _extract_hashk(gs, tkeys, tnulls, cap, gnames, gexprs, glog, dev)
    if sharded:
        from .merge import tree_merge_raw
        raw = tree_merge_raw(raw, plan, options, dev)
    return finish(raw, plan)


REPEAT_MIN = 0.05      # Stats.repeat above which a dense GROUP BY pre-aggregates (uniform 1M keys: 0.0005; Zipf 1.1: > 0.3)
PARTITION_MIN_TABLE_BYTES = 256 << 20     # below this the table (mostly) lives in the 126 MB L2 anyway
PARTITION_BUCKET_BYTES = 24 << 20         # slice of the group table touched by one bucket


def _partition_plan(nslots, plan: AggPlan, work, total_rows):
    """(shift, nbuckets) for b2_range_partition, or None when the dense table is small enough for
    L2, the inputs are not plain 8-byte columns, or there are too few rows to pay for the extra pass."""
    if os.environ.get("B200SQL_NO_PARTITION") == "1" or not work:
        return None
    per_slot = 8 * (sum(1 for k in plan.kaggs if k.op != L.AGG_COUNT) + sum(1 for k in plan.kaggs if k.need_cnt)
                    + (1 if plan.need_rows else 0))
    min_bytes = int(os.environ.get("B200SQL_PARTITION_MIN_BYTES", PARTITION_MIN_TABLE_BYTES))
    if per_slot == 0 or nslots * per_slot < min_bytes or total_rows * 4 < nslots:
        return None
    if len({v for _, _, _, vs in work for v in vs}) > L.MAX_GATHER:
        return None
    for part, ctx, kslot, vslots in work:
        if ctx.cols[kslot].dtype != I64:
            return None
        for v in vslots:
            if ctx.cols[v].dtype == U8 or ctx.cols[v].valid is not None:
                return None
    bucket_bytes = int(os.environ.get("B200SQL_PARTITION_BUCKET_BYTES", PARTITION_BUCKET_BYTES))
    shift = max(0, (max(1, bucket_bytes // per_slot)).bit_length() - 1)
    while ((nslots - 1) >> shift) + 1 > 1024:
        shift += 1
    return shift, ((nslots - 1) >> shift) + 1


class SlotView:
    """A window [lo, lo + count) of a dense group table's slots: the accumulator arrays restricted to
    it and the rule that tells which of its slots hold a group.  Single GPU: the whole table.
    Multi-GPU: this rank's slice of the reduce-scattered table (executor._merge_dense)."""

    def __init__(self, nslots, lo, count, acc, cnt, rows, occ_kind, occ, dist="replicated"):
        self.nslots, self.lo, self.count = nslots, lo, count      # nslots: logical table size (NULL slot = nslots-1)
        self.acc, self.cnt, self.rows = acc, cnt, rows
        self.occ_kind, self.occ = occ_kind, occ                    # 'rows' | 'indicator' | 'bitmap' | 'bytes'
        self.dist = dist

    @classmethod
    def whole(cls, t: D.GroupTable, count=None):
        n = t.nslots if count is None else count
        cut = lambda x: None if x is None else x[:n]
        if t.rows is not None:
            kind, occ = "rows", cut(t.rows)
        elif t.indicator is not None:
            kind, occ = "indicator", cut(t.acc[t.indicator])
        else:
            kind, occ = "bitmap", t.present
        return cls(t.nslots, 0, n, [cut(a) for a in t.acc], [cut(c) for c in t.cnt], cut(t.rows), kind, occ)

    def occupancy(self, keys: torch.Tensor):
        """(column, predicate term) selecting the slots of the window that received at least one row."""
        if self.occ_kind == "rows":
            return DeviceColumn(self.occ, None, I64), TermSpec(0, L.GT, 0)
        if self.occ_kind == "indicator":
            # untouched float SUM accumulator = -0.0 = the INT64_MIN bit pattern (single GPU only:
            # a collective is free to lose the sign of a zero, see _merge_dense)
            return DeviceColumn(self.occ.view(torch.int64), None, I64), TermSpec(0, L.NE, L.EMPTY_KEY)
        if self.occ_kind == "bytes":
            return DeviceColumn(self.occ, None, U8), TermSpec(0, L.IS_TRUE, 0)
        return DeviceColumn(keys, self.occ, I64), TermSpec(0, L.IS_NOT_NULL, 0)


_PRESENCE_PROG = {}      # compiled once: the three ways a table records "this slot holds a group"


def _presence_bytes(t: D.GroupTable, dev, out=None) -> torch.Tensor:
    """uint8[alloc]: 1 where this rank's partial table holds a group.  Derived from whatever the
    kernels maintained (row counter, -0.0 indicator accumulator, presence bitmap) in one
    b2_expr_eval pass, so that existence crosses the ranks as DATA: NCCL may pick an algorithm
    (in-switch NVLS reduction, zero-initialised scratch) under which -0.0 + -0.0 comes back +0.0."""
    n = t.alloc
    if t.rows is not None:
        kind, col = "rows", DeviceColumn(t.rows, None, I64)
    elif t.indicator is not None:
        kind, col = "indicator", DeviceColumn(t.acc[t.indicator].view(torch.int64), None, I64)
    else:
        # only the validity bitmap is read; any 8-byte buffer of the right length serves as values
        vals = next((a for a in list(t.acc) + list(t.cnt) if a is not None), None)
        if vals is None:
            vals = torch.zeros(n, dtype=torch.int64, device=dev)
        kind, col = "bitmap", DeviceColumn(vals.view(torch.int64), t.present, I64)
    prog = _PRESENCE_PROG.get(kind)
    if prog is None:
        x = ColRef("x", I64)
        e = {"rows": lambda: E.binop("gt", x, 0), "indicator": lambda: E.binop("ne", x, L.EMPTY_KEY),
             "bitmap": lambda: E.unop("not", Call("isnull", [x], U8))}[kind]()
        prog = _PRESENCE_PROG[kind] = E.compile_expr(E.cast(e, U8), ["x"])
    return D.expr_eval(prog, [col], n, False, out=out).data


def _merge_dense(t: D.GroupTable, plan: AggPlan, sharded: bool, dev, keep=None) -> SlotView:
    """Combine the ranks' partial dense tables: reduce-scatter by slot range (sum of sums / counts,
    min of mins, max of maxes, OR of existence), so that every rank ends up owning the merged
    groups of one contiguous key range -- the reference's tree reduction (aggregate.py:575-581,
    groupby(...).agg(split_every)) restated for direct-address tables, with split_out = world size.
    Existence travels explicitly (a uint8 per slot, MAX-reduced); nothing depends on how the
    collective treats signed zeros."""
    rank, size = P.world()
    if not sharded or size == 1:
        return SlotView.whole(t)
    assert t.alloc % (32 * size) == 0, "sharded group tables are padded to 32 x world slots"
    chunk = t.alloc // size
    # keep: buffers of a prepared query, reused run after run.  Tensors handed to a collective are tied
    # to the communicator's stream by the allocator; fresh ones every run cannot be recycled while the
    # host is ahead of the GPU, and every run then pays cudaMalloc for its lookup and table buffers.
    with _Phase("presence"):
        pbuf = None
        if keep is not None:
            pbuf = keep.get("pres_in")
            if pbuf is None:
                pbuf = keep["pres_in"] = torch.empty(t.alloc, dtype=torch.uint8, device=dev)
        pres = _presence_bytes(t, dev, out=pbuf)
        stats["launches"] += 1

    def kept(key, like):
        if keep is None:
            return None
        buf = keep.get(key)
        if buf is None:
            buf = keep[key] = torch.empty(chunk, dtype=like.dtype, device=dev)
        return buf

    with _Phase("reduce_scatter"):
        accs, cnts = [], []
        for i, (ka, acc, cnt) in enumerate(zip(plan.kaggs, t.acc, t.cnt)):
            accs.append(None if acc is None else
                        P.reduce_scatter_(acc, {L.AGG_MIN: "min", L.AGG_MAX: "max"}.get(ka.op, "sum"),
                                          out=kept(("a", i), acc)))
            cnts.append(None if cnt is None else P.reduce_scatter_(cnt, "sum", out=kept(("c", i), cnt)))
        rows = None if t.rows is None else P.reduce_scatter_(t.rows, "sum", out=kept("r", t.rows))
        pres = P.reduce_scatter_(pres, "max", out=kept("p", pres))
    return SlotView(t.nslots, rank * chunk, chunk, accs, cnts, rows, "bytes", pres, dist="keyrange")


class RawGroups:
    """Compacted raw state of a GROUP BY: one row per group, accumulators not yet finished
    (so partial results of several GPUs can still be merged)."""

    def __init__(self, keys: Dict[str, DeviceColumn], acc, cnt, rows, n):
        self.keys, self.acc, self.cnt, self.rows, self.n = keys, acc, cnt, rows, n


def finish(raw: RawGroups, plan: AggPlan) -> Part:
    out = Part(dict(raw.keys), raw.n)
    _finish_outputs(plan, raw.acc, raw.cnt, raw.rows, raw.n, out)
    return out


def _finish_outputs(plan: AggPlan, acc_cols, cnt_cols, rows_col, n, out: Part):
    """Per-group output columns from gathered accumulators (device expressions)."""
    for name, fn, a, c, in_dt, lg in plan.outs:
        cnt = rows_col if c == "rows" else (cnt_cols[c] if c is not None else None)
        env = Part({}, n)
        if cnt is not None:
            env["c"] = cnt
        if fn in ("size", "count"):
            out[name] = DeviceColumn(cnt.data, None, I64, "int64")
            continue
        acc = acc_cols[a]
        env["a"] = acc
        if fn in MOMENT_FUNCS:
            env["b"] = acc_cols[plan.second[name]]
            ddof = 0 if fn.endswith("pop") else 1
            nf = E.cast(ColRef("c", I64), F64)
            s1, s2 = ColRef("a", F64), ColRef("b", F64)
            var = E.binop("truediv", E.binop("sub", s2, E.binop("truediv", E.binop("mul", s1, s1), nf)),
                          E.binop("sub", nf, float(ddof)))
            var = E.case(E.binop("lt", var, 0.0), Lit(0.0), var)      # a constant group may round to -1e-17
            val = E.unop("sqrt", var) if fn.startswith("stddev") else var
            col = eval_expr(env, E.case(E.binop("gt", ColRef("c", I64), ddof), val, Lit(None, F64)))
            col.logical = "float64"
            out[name] = col
            continue
        if fn == "mean":
            e = E.binop("truediv", ColRef("a", F64), ColRef("c", I64))
            e = E.case(E.binop("gt", ColRef("c", I64), 0), e, Lit(None, F64))
            col = eval_expr(env, e)
            col.logical = "float64"
        else:
            is_f = (in_dt == F64)
            val: Expr = ColRef("a", I64 if (fn in ("min", "max") or not is_f) else F64)
            if fn in ("min", "max") and is_f:
                val = Call("ord2f", [val], F64)
            if cnt is not None:
                val = E.case(E.binop("gt", ColRef("c", I64), 0), val, Lit(None, val.dtype))
            col = eval_expr(env, val) if not isinstance(val, ColRef) else acc
            col = DeviceColumn(col.data, col.valid, F64 if is_f else I64, lg if lg != "bool" else "int64")
        out[name] = col


def _gather_view(view: SlotView, idx, dev):
    """Accumulator / count / row-count arrays of `view` gathered at the (window-local) slots `idx`."""
    acc_cols, cnt_cols = [], []
    for acc, cnt in zip(view.acc, view.cnt):
        if acc is not None:
            dt = F64 if acc.dtype == torch.float64 else I64
            stats["launches"] += 1
            acc_cols.append(D.gather(DeviceColumn(acc, None, dt), idx, False))
        else:
            acc_cols.append(None)
        if cnt is not None:
            stats["launches"] += 1
            cnt_cols.append(D.gather(DeviceColumn(cnt, None, I64), idx, False))
        else:
            cnt_cols.append(None)
    rows_col = None
    if view.rows is not None:
        stats["launches"] += 1
        rows_col = D.gather(DeviceColumn(view.rows, None, I64), idx, False)
    return acc_cols, cnt_cols, rows_col


DEFER_MAX_SLOTS = 1 << 23    # deferred compaction allocates its outputs at one row per slot of the window


def _finalize_dense(view: SlotView, kmin, gname, gexpr, glog, plan, dev, key_nullable=True,
                    check=None, fallback=None) -> Part:
    """Window of a dense table -> result partition (group key = kmin + slot; the table's last slot
    is the NULL group).  `check`: optional int32 device flags whose first word must be 0 for the
    result to stand (star pipeline: duplicate build keys), else `fallback()` is the result.  With a
    NULL-free int64 key the compaction is enqueued without waiting for its count (PendingPart); the
    flags ride on the same host copy."""
    count = view.count
    ncols = 1 + sum(a is not None for a in view.acc) + sum(c is not None for c in view.cnt) + (view.rows is not None)
    if not key_nullable and gexpr.dtype == I64 and count <= DEFER_MAX_SLOTS and ncols <= L.MAX_GATHER \
            and os.environ.get("B200SQL_NO_DEFER") != "1":
        with _Phase("compact"):
            slot_keys = torch.arange(kmin + view.lo, kmin + view.lo + count, dtype=torch.int64, device=dev)
            occ, term = view.occupancy(slot_keys)
            cols, where = [occ, DeviceColumn(slot_keys, None, I64)], {}
            for i, (acc, cnt) in enumerate(zip(view.acc, view.cnt)):
                if acc is not None:
                    where[("a", i)] = len(cols)
                    cols.append(DeviceColumn(acc, None, F64 if acc.dtype == torch.float64 else I64))
                if cnt is not None:
                    where[("c", i)] = len(cols)
                    cols.append(DeviceColumn(cnt, None, I64))
            if view.rows is not None:
                where[("r", 0)] = len(cols)
                cols.append(DeviceColumn(view.rows, None, I64))
            gcols = list(range(1, len(cols)))
            stats["launches"] += 3
            outs, cnt_dev = D.select_launch(D.make_scan(cols, [term], count), dev, gcols, cols)
            pending = DeviceCount(cnt_dev, check) if check is not None else DeviceCount(cnt_dev)

        def thunk():
            vals = pending.get()
            total = int(vals[0])
            if check is not None and vals[1]:
                return fallback()
            got = {g: DeviceColumn(o[:total], None, cols[g].dtype) for g, o in zip(gcols, outs)}
            kcol = DeviceColumn(got[1].data, None, I64, glog)
            acc_cols = [got.get(where.get(("a", i))) for i in range(len(view.acc))]
            cnt_cols = [got.get(where.get(("c", i))) for i in range(len(view.cnt))]
            res = finish(RawGroups({gname: kcol}, acc_cols, cnt_cols, got.get(where.get(("r", 0))), total), plan)
            res.dist = view.dist
            return res

        out = PendingPart(thunk)
        out.dist = view.dist
        return out
    with _Phase("compact"):
        raw = _extract_dense(view, kmin, gname, gexpr, glog, dev, key_nullable)
    with _Phase("finish"):
        out = finish(raw, plan)
    out.dist = view.dist
    if check is not None and int(check[0].item()):
        return fallback()
    return out


def _extract_dense(view: SlotView, kmin, gname, gexpr, glog, dev, key_nullable=True) -> RawGroups:
    count = view.count
    slot_keys = torch.arange(kmin + view.lo, kmin + view.lo + count, dtype=torch.int64, device=dev)
    occ, term = view.occupancy(slot_keys)
    if not key_nullable and gexpr.dtype == I64:
        # the key column has no NULLs, so the NULL slot stays empty: no validity work.
        # compaction and gathers in one write pass: keys and every accumulator array ride along as
        # gather columns of b2_select_write (<= 8), instead of one b2_gather launch each
        cols = [occ, DeviceColumn(slot_keys, None, I64)]
        where = {}
        for i, (acc, cnt) in enumerate(zip(view.acc, view.cnt)):
            if acc is not None:
                where[("a", i)] = len(cols)
                cols.append(DeviceColumn(acc, None, F64 if acc.dtype == torch.float64 else I64))
            if cnt is not None:
                where[("c", i)] = len(cols)
                cols.append(DeviceColumn(cnt, None, I64))
        if view.rows is not None:
            where[("r", 0)] = len(cols)
            cols.append(DeviceColumn(view.rows, None, I64))
        if len(cols) - 1 <= L.MAX_GATHER:
            gcols = list(range(1, len(cols)))
            stats["launches"] += 3
            _, outs, total = D.select(D.make_scan(cols, [term], count), dev, gcols, want_idx=False, cols=cols)
            got = {g: DeviceColumn(o.data, None, o.dtype) for g, o in zip(gcols, outs)}
            kcol = DeviceColumn(got[1].data, None, I64, glog)
            acc_cols = [got.get(where.get(("a", i))) for i in range(len(view.acc))]
            cnt_cols = [got.get(where.get(("c", i))) for i in range(len(view.cnt))]
            return RawGroups({gname: kcol}, acc_cols, cnt_cols, got.get(where.get(("r", 0))), total)
        stats["launches"] += 4
        idx, _, total = D.select(D.make_scan([occ], [term], count), dev, (), want_idx=True, cols=[occ])
        kcol = D.gather(DeviceColumn(slot_keys, None, I64, glog), idx, False)
        kcol = DeviceColumn(kcol.data, None, I64, glog)
        acc_cols, cnt_cols, rows_col = _gather_view(view, idx, dev)
        return RawGroups({gname: kcol}, acc_cols, cnt_cols, rows_col, total)
    # occupied slots of the window
    stats["launches"] += 3
    idx, _, total = D.select(D.make_scan([occ], [term], count), dev, (), want_idx=True, cols=[occ])
    # key column: the table's last slot is the NULL group (it lies in exactly one rank's window)
    kvalid = torch.full((D.bitmap_words(count),), -1, dtype=torch.int32, device=dev)
    last = view.nslots - 1 - view.lo
    if 0 <= last < count:
        kvalid[last >> 5] = int(np.array([~(1 << (last & 31)) & 0xFFFFFFFF], dtype=np.uint32).view(np.int32)[0])
    stats["launches"] += 1
    kcol = D.gather(DeviceColumn(slot_keys, kvalid, I64), idx, True)
    if gexpr.dtype == U8:
        kc = eval_expr(Part({"k": kcol}, total), E.cast(ColRef("k", I64), U8))
        kcol = DeviceColumn(kc.data, kcol.valid, U8, glog)
    kcol.logical = glog
    kcol = _drop_full_valid(kcol)
    acc_cols, cnt_cols, rows_col = _gather_view(view, idx, dev)
    return RawGroups({gname: kcol}, acc_cols, cnt_cols, rows_col, total)


def _drop_full_valid(col: DeviceColumn) -> DeviceColumn:
    """Drop a validity bitmap that marks nothing NULL (keeps numpy dtypes on the way out)."""
    if col.valid is None or col.n == 0:
        return DeviceColumn(col.data, None, col.dtype, col.logical)
    p = Part({"x": DeviceColumn(col.data, col.valid, I64 if col.dtype != U8 else U8)}, col.n)
    isn = eval_expr(p, Call("isnull", [ColRef("x", I64 if col.dtype != U8 else U8)], U8))
    if int(isn.data.max().item()) == 0:
        return DeviceColumn(col.data, None, col.dtype, col.logical)
    return col


def _extract_hash1(gs, tkeys, cap, fl, gname, gexpr, glog, dev) -> RawGroups:
    occ = DeviceColumn(tkeys[:cap], None, I64)
    scan = D.make_scan([occ], [TermSpec(0, L.NE, L.EMPTY_KEY)], cap)
    stats["launches"] += 3
    idx, _, total = D.select(scan, dev, (), want_idx=True, cols=[occ])
    extra = []
    if fl[1]:
        extra.append(cap)
    if fl[2]:
        extra.append(cap + 1)
    null_pos = None
    if extra:
        if fl[1]:
            null_pos = total
        idx = torch.cat([idx, torch.tensor(extra, dtype=torch.int32, device=dev)])
        total += len(extra)
    stats["launches"] += 1
    kcol = D.gather(DeviceColumn(tkeys, None, gexpr.dtype), idx, False)
    if null_pos is not None:
        if gexpr.dtype == F64:
            kcol.data[null_pos] = float("nan")
        else:
            valid = torch.full((D.bitmap_words(total),), -1, dtype=torch.int32, device=dev)
            valid[null_pos >> 5] = int(np.array([~(1 << (null_pos & 31)) & 0xFFFFFFFF], dtype=np.uint32).view(np.int32)[0])
            kcol = DeviceColumn(kcol.data, valid, kcol.dtype)
    kcol.logical = glog
    acc_cols, cnt_cols, rows_col = _gather_view(SlotView.whole(gs.table, gs.table.alloc), idx, dev)
    return RawGroups({gname: kcol}, acc_cols, cnt_cols, rows_col, total)


def _extract_hashk(gs, tkeys, tnulls, cap, gnames, gexprs, glogs, dev) -> RawGroups:
    view = SlotView.whole(gs.table, cap)
    occ, term = view.occupancy(tkeys[:cap])
    scan = D.make_scan([occ], [term], cap)
    stats["launches"] += 3
    idx, _, total = D.select(scan, dev, (), want_idx=True, cols=[occ])
    stats["launches"] += 1
    nulls = D.gather(DeviceColumn(tnulls, None, U8), idx, False)
    any_null = total > 0 and int(nulls.data.max().item()) > 0
    out = {}
    for k, (g, e, lg) in enumerate(zip(gnames, gexprs, glogs)):
        stats["launches"] += 1
        kc = D.gather(DeviceColumn(tkeys[k * cap:(k + 1) * cap], None, I64), idx, False)
        if any_null:
            env = Part({"k": kc, "m": nulls}, total)
            bit = E.binop("mod", E.binop("divt", ColRef("m", U8), 1 << k), 2)
            val = E.case(E.binop("eq", bit, 0), ColRef("k", I64), Lit(None, I64))
            kc = _drop_full_valid(eval_expr(env, val))
        if e.dtype == F64:
            col = DeviceColumn(kc.data.view(torch.float64), None, F64, lg)
            if kc.valid is not None:  # NULL float key = NaN
                col = eval_expr(Part({"k": DeviceColumn(col.data, kc.valid, F64)}, total),
                                E.fillna(ColRef("k", F64), float("nan")))
                col = DeviceColumn(col.data, None, F64, lg)
        elif e.dtype == U8:
            c8 = eval_expr(Part({"k": DeviceColumn(kc.data, None, I64)}, total), E.cast(ColRef("k", I64), U8))
            col = DeviceColumn(c8.data, kc.valid, U8, lg)
        else:
            col = DeviceColumn(kc.data, kc.valid, I64, lg)
        out[g] = col
    acc_cols, cnt_cols, rows_col = _gather_view(view, idx, dev)
    return RawGroups(out, acc_cols, cnt_cols, rows_col, total)


# ---------------------------------------------------------------------------------------------
# fused star pipeline: Aggregate <- Inner Join(fk = unique pk), grouped by build-side columns
# ---------------------------------------------------------------------------------------------
def _side_of(e: Expr, left_names: Set[str], right_names: Set[str]):
    r = e.refs()
    if not r:
        return "none"
    if r <= left_names:
        return "left"
    if r <= right_names:
        return "right"
    return "both"


class PreparedStar:
    """Everything about one fused star query that does not change between executions, kept with the
    (immutable) plan: launch descriptors of every dim / fact partition (ctypes structs over resident
    columns), the aggregate plan, the lookup buffers and the group table (re-initialised, not
    re-allocated, per run).  A step of a repeated query then costs the host a few dozen calls instead
    of re-deriving all of it -- at 8 GPUs a step is ~1 ms of device work, so host time IS the step time.

    One stream, in order: lookup fill -> b2_star_build_scan (every rank that holds dim rows; a 'root' table
    is followed by one NCCL broadcast of the finished lookup) -> b2_star_agg per fact partition -> merge ->
    compaction.  The lookup buffer is refilled in stream order; with the NVLink peer merge two group
    tables alternate between consecutive executions (peers read a table while its owner has moved on).
    The host issues run k + 2 only after run k has FINISHED (event): at most two executions in flight.
    Results are always freshly allocated and never alias the reused buffers."""

    _live: "List[PreparedStar]" = []
    MAX_LIVE = 4          # prepared plans keep ~100 MB of HBM each: keep only the most recent ones

    @classmethod
    def get(cls, src, fact, dim, fk_e, pk_e, ge, gexpr0, aggs, fpred, dpred, meta, owner, bcast, sharded, dev):
        key = (sharded, P.world()[1], _dev().index)
        cache = src.__dict__.setdefault("_prepared_star", {})
        if key in cache:
            prep = cache[key]
            if prep is not None and prep not in cls._live:      # evicted meanwhile: its buffers are gone
                prep = None
                cache.pop(key)
            else:
                return prep
        try:
            prep = cls(src, fact, dim, fk_e, pk_e, ge, gexpr0, aggs, fpred, dpred, meta, owner, bcast, sharded, dev)
        except _NotPreparable:
            prep = None
        if P.world()[1] > 1:
            # every rank must take the same path (the prepared one issues its own collectives): agree once
            ok = torch.tensor([1 if prep is not None else 0], dtype=torch.int64, device=dev)
            if int(P.allreduce_(ok, "min").item()) == 0:
                prep = None
            else:
                if sharded and P.peer_memory_available():
                    # collective (symmetric allocation + handle exchange): entered by all ranks or by none.
                    # A rank on which it fails (no peer access, mapping refused) says so and ALL ranks stay
                    # on the NCCL merge.
                    state, why = None, None
                    try:
                        state = prep.build_peer_merge()
                    except Exception as e:  # noqa: BLE001 -- any failure means "no peer path", never a wrong result
                        why = f"{type(e).__name__}: {e}"
                    ok = torch.tensor([1 if state is not None else 0], dtype=torch.int64, device=dev)
                    if int(P.allreduce_(ok, "min").item()) == 1:
                        prep.install_peer_merge(state)
                    elif why is not None:
                        import warnings
                        warnings.warn(f"NVLink peer merge unavailable, using ncclReduceScatter: {why}")
        cache[key] = prep
        if prep is not None:
            src.__dict__["_prepared_last"] = ((P.world()[1], _dev().index), prep)
            cls._live.append(prep)
            while len(cls._live) > cls.MAX_LIVE:
                cls._live.pop(0)
        return prep

    def __init__(self, src, fact, dim, fk_e, pk_e, ge, gexpr0, aggs, fpred, dpred, meta, owner, bcast, sharded, dev):
        self.dev, self.owner, self.bcast, self.sharded = dev, owner, bcast, sharded
        self.pmin, self.prange, self.gmin, self.grng, self.gnull = meta
        self.nslots = self.grng + 1
        self.gname = src.group_cols[0]
        self.gexpr0 = gexpr0
        self.glog = dim.col_type(gexpr0.name)[1] if isinstance(gexpr0, ColRef) else "int64"
        self.plan = AggPlan([(E.substitute(e, fact.exprs) if e is not None else None, o, f) for e, o, f in aggs],
                            _nullable_fn(fact, sharded))
        if any(not isinstance(ka.expr, ColRef) for ka in self.plan.kaggs):
            raise _NotPreparable()
        # ---- launch descriptors (every referenced column must be resident and used as it is)
        self.keep = []
        self.dim_launch = []
        if owner:
            needed = {pk_e.name, ge.name}
            for p in dpred:
                p.refs(needed)
            for part in self._resident_parts(dim.source.table, needed):
                ctx = ScanCtx(part, dpred)
                pk_slot, g_slot = ctx.slot(pk_e), ctx.slot(ge)
                self._only_table_columns(ctx)
                self.dim_launch.append((ctx.scan(), pk_slot, g_slot))
                self.keep.append(ctx)
        needed = set(fk_e.refs())
        for ka in self.plan.kaggs:
            ka.expr.refs(needed)
        for p in fpred:
            p.refs(needed)
        self.fact_launch = []
        for part in self._resident_parts(fact.source.table, needed):
            ctx = ScanCtx(part, fpred)
            fk_slot = ctx.slot(fk_e)
            specs = [(ctx.slot(ka.expr), ka.op) for ka in self.plan.kaggs]
            self._only_table_columns(ctx)
            self.fact_launch.append((ctx.scan(), fk_slot, D.make_aggs(specs), len(specs), part.n))
            self.keep.append(ctx)
        # ---- reused device buffers
        # ONE lookup buffer: every run refills it in stream order, after the previous run's scan.  (Two
        # alternating buffers -- needed while the build ran on its own stream -- keep 2 x 40 MB of
        # evict_last lines in a 126 MB L2 next to the group tables, and a step with one fact partition
        # per GPU then meets a lookup that the other buffer's protected lines have half displaced:
        # b2_star_agg measured 0.70-0.72 ms per 125M rows at N = 2 / 4 / 8 against 0.577 ms at N = 1.)
        self.lookup = torch.empty(self.prange + 4, dtype=torch.int32, device=dev)
        self.lk = L.StarLookup()
        self.lk.dense, self.lk.lookup, self.lk.kmin, self.lk.range = 1, self.lookup.data_ptr(), self.pmin, self.prange
        # group tables: ONE (re-initialised per run) on the NCCL / single-GPU path; enable_peer_merge()
        # replaces it with two in symmetric memory that alternate run by run
        self.tabs = [GroupState(dev, self.nslots, self.plan, need_present=True,
                                alloc=_padded_slots(self.nslots, sharded))]
        self.refill = [self._refill_list(self.tabs[0].table)]
        self.dirty = [False]      # a fresh table is already initialised
        self.peer = None          # per-table b2_peer_merge descriptors once enabled
        self.epoch = 0
        self.free = [None, None]  # event recorded at the end of run k, waited for before run k + 2 is issued
        self.merge_bufs = {}      # presence / reduce-scatter outputs, reused run after run
        self.runs = 0

    @staticmethod
    def _refill_list(t: D.GroupTable):
        """(tensor, initial value) of every array of the table: what a run has to restore first."""
        out = []
        for acc in t.acc:
            if acc is not None:
                out.append((acc, float(acc[0].item()) if acc.dtype == torch.float64 else int(acc[0].item())))
        for cnt in t.cnt:
            if cnt is not None:
                out.append((cnt, 0))
        if t.rows is not None:
            out.append((t.rows, 0))
        if t.present is not None:
            out.append((t.present, 0))
        return out

    def install_peer_merge(self, state):
        self.tabs, self.refill, self.dirty, self.peer, self.arena, self.local_ready = state
        stats["peer_merge_plans"] = stats.get("peer_merge_plans", 0) + 1

    def build_peer_merge(self):
        """Group tables in symmetric memory and the description of their merge for b2_peer_merge: one
        kernel per step (barrier + reduction of this rank's slot range over every peer's table + merge
        of existence, csrc/peer.cuh) instead of a presence pass and two to five NCCL reduce-scatters.
        Two tables alternate, so that a table is refilled only after all peers have read it (see peer.cuh).
        Returns the state install_peer_merge() takes; nothing of `self` is touched before that."""
        rank, size = P.world()
        dev = self.dev
        alloc = _padded_slots(self.nslots, True)
        proto = self.tabs[0].table
        narr = sum(a is not None for a in proto.acc) + sum(c is not None for c in proto.cnt) + (proto.rows is not None)
        per_table = (narr * alloc * 8 + D.bitmap_words(alloc) * 4) + (narr + 2) * P.PeerArena.ALIGN
        arena = P.PeerArena(2 * per_table + 4 * P.PeerArena.ALIGN, dev)
        _, sig_off = arena.carve(L.MAX_PEERS, torch.int64, 0)
        chunk = alloc // size
        tabs, refill, dirty, peer = [], [], [], []
        local_ready = torch.zeros(1, dtype=torch.int64, device=dev)
        for _ in range(2):
            offs = {}

            def new(n, dtype, fill, offs=offs):
                t, off = arena.carve(n, dtype, fill)
                offs[t.data_ptr()] = off
                return t

            gs = GroupState(dev, self.nslots, self.plan, need_present=True, alloc=alloc, new=new)
            t = gs.table
            m = L.PeerMerge()
            m.world, m.rank, m.lo, m.count = size, rank, rank * chunk, chunk
            m.signal_off = sig_off
            m.local_ready = local_ready.data_ptr()
            for p_, b in enumerate(arena.base):
                m.peer_base[p_] = b
            arrays, accs, cnts, rows = [], [], [], None      # arrays: (tensor, op) in the kernel's order
            for ka, acc, cnt in zip(self.plan.kaggs, t.acc, t.cnt):
                if acc is not None:
                    op = {L.AGG_MIN: L.PEER_MIN_I64, L.AGG_MAX: L.PEER_MAX_I64}.get(
                        ka.op, L.PEER_SUM_F64 if acc.dtype == torch.float64 else L.PEER_SUM_I64)
                    arrays.append((acc, op))
                if cnt is not None:
                    arrays.append((cnt, L.PEER_SUM_I64))
            if t.rows is not None:
                arrays.append((t.rows, L.PEER_SUM_I64))
            outs = {}
            for a, (src, op) in enumerate(arrays):
                m.ops[a], m.array_off[a] = op, offs[src.data_ptr()]
                outs[src.data_ptr()] = torch.empty(chunk, dtype=src.dtype, device=dev)
                m.out[a] = outs[src.data_ptr()].data_ptr()
            m.narrays = len(arrays)
            index = {src.data_ptr(): a for a, (src, _) in enumerate(arrays)}
            if t.rows is not None:
                m.presence_kind, m.presence_array = L.PEER_PRESENT_ROWS, index[t.rows.data_ptr()]
            elif t.indicator is not None:
                m.presence_kind, m.presence_array = L.PEER_PRESENT_INDICATOR, index[t.acc[t.indicator].data_ptr()]
            else:
                m.presence_kind, m.presence_array = L.PEER_PRESENT_BITMAP, 0
                m.bitmap_off = offs[t.present.data_ptr()]
            pres = torch.empty(chunk, dtype=torch.uint8, device=dev)
            m.out_present = pres.data_ptr()
            pick = lambda x: None if x is None else outs[x.data_ptr()]
            view = SlotView(t.nslots, rank * chunk, chunk, [pick(a) for a in t.acc], [pick(c) for c in t.cnt],
                            pick(t.rows), "bytes", pres, dist="keyrange")
            tabs.append(gs)
            refill.append(self._refill_list(t))
            dirty.append(False)
            peer.append((m, view))
        return tabs, refill, dirty, peer, arena, local_ready

    @staticmethod
    def _resident_parts(table, needed):
        parts = []
        for p in table.partitions:
            n = next(iter(p.values())).n if p else 0
            if n == 0:
                continue
            cols = {}
            for name in needed:
                c = p[name]
                if not isinstance(c, DeviceColumn):
                    raise _NotPreparable()          # host-resident table: uploaded per query, classic path
                cols[name] = c
            parts.append(Part(cols, n))
        return parts

    @staticmethod
    def _only_table_columns(ctx: "ScanCtx"):
        if any(not k.startswith("col:") for k in ctx.index):
            raise _NotPreparable()                  # computed inputs / mask predicates are evaluated per query

    def run(self, src) -> Part:
        i = self.runs & 1
        self.runs += 1
        buf = self.lookup
        main = D.cur_stream()
        sp = D.stream_ptr()
        # The host waits here until the run before the previous one has FINISHED: at most two executions
        # of this query are in flight.  That hides the host's issue latency, and no more: letting the host
        # run many collectives ahead of the GPUs measurably stretches the steps (ranks drift apart and the
        # allocator cannot recycle buffers the communicator still holds).
        if self.free[i] is not None:
            self.free[i].synchronize()
        # ---- build side, in order on the caller's stream.  (Round 2 first ran it on a second stream and
        # communicator so that the next step's build + broadcast overlapped the current scan.  Measured at
        # N=2 there is nothing to gain: the scan kernels are persistent grids that fill every SM, so the
        # build kernels wait for a whole fact partition anyway -- 0.75 ms of "build" for 0.08 ms of work,
        # 0.70 ms of "broadcast" for 40 MB -- and the extra stream, communicator and events only add cost.)
        with _Phase("build"):
            # lookup := -1 everywhere (0xFF bytes), the 4 flag words behind it := 0
            L.memset(C.c_void_p(buf.data_ptr()), 0xFF, 4 * self.prange, sp)
            L.memset(C.c_void_p(buf.data_ptr() + 4 * self.prange), 0, 16, sp)
            for scan, pk_slot, g_slot in self.dim_launch:
                stats["launches"] += 1
                L.star_build_scan(C.byref(scan), pk_slot, g_slot, self.pmin, self.prange, self.gmin,
                                  self.nslots - 1, C.c_void_p(buf.data_ptr()),
                                  C.c_void_p(buf.data_ptr() + 4 * self.prange), sp)
        if self.bcast:
            with _Phase("bcast"):
                P.broadcast_(buf, 0)
        # ---- probe side
        ti = i if self.peer is not None else 0
        t = self.tabs[ti].table
        with _Phase("scan"):
            if self.dirty[ti]:
                for tensor, value in self.refill[ti]:
                    tensor.fill_(value)
            self.dirty[ti] = True
            for scan, fk_slot, aggs_arr, naggs, n in self.fact_launch:
                stats["launches"] += 1
                ev = _kernel_event_begin("b2_star_agg_kernel", n)
                L.star_agg(C.byref(scan), fk_slot, C.byref(self.lk), aggs_arr, naggs, C.byref(t.state), sp)
                _kernel_event_end(ev)
        if self.peer is not None:
            m, view = self.peer[ti]
            self.epoch += 1
            m.epoch = self.epoch
            with _Phase("peer_merge"):
                stats["launches"] += 1
                ev = _kernel_event_begin("b2_peer_merge_kernel", m.count)
                L.peer_merge(C.byref(m), sp)
                _kernel_event_end(ev)
        else:
            view = _merge_dense(t, self.plan, self.sharded, self.dev, keep=self.merge_bufs)
        stats["star_fused"] += 1

        def general():   # a duplicate build key showed up: the general path redoes the query
            stats["star_fused"] -= 1
            return run_aggregate(src, allow_fast=False)

        out = _finalize_dense(view, self.gmin, self.gname, self.gexpr0, self.glog, self.plan, self.dev,
                              key_nullable=self.gnull, check=buf[self.prange:], fallback=general)
        done = torch.cuda.Event()
        done.record(main)
        self.free[i] = done
        return out


class _NotPreparable(Exception):
    pass


def _star_dense_fast(src, fact, dim, fk_e, pk_e, gexprs, aggs, fact_pred, dim_pred, sharded, dev) -> Optional[Part]:
    """Star pipeline when the dimension side is a registered table whose join key and (single)
    group key are dense int64 columns: b2_star_build_scan per dim partition, b2_star_agg per fact
    partition, one compaction at the end.  Returns None when the shape does not apply or a
    duplicate build key shows up (the general path then takes over)."""
    if len(gexprs) != 1 or not isinstance(dim.source, TableSource) or not isinstance(pk_e, ColRef):
        return None
    ge = E.substitute(gexprs[0], dim.exprs)
    if not isinstance(ge, ColRef) or ge.dtype != I64 or pk_e.dtype != I64:
        return None
    rank, world = P.world()
    dist = frame_distribution(dim)
    if world > 1 and dist == "sharded":
        return None
    table = dim.source.table
    owner = world == 1 or dist != "root" or rank == 0
    meta = None
    if owner:
        pst, gst = table.column_stats(pk_e.name), table.column_stats(ge.name)
        gnull = table.column_nullable(ge.name)
        meta = (pst.vmin, pst.vmax, gst.vmin, gst.vmax, table.nrows, gnull)
    if world > 1 and dist == "root":
        # key ranges of the root-only table: one object broadcast per (table, columns), then cached on
        # the (immutable) table object of every rank -- a blocking host round trip per query otherwise
        cache = table.__dict__.setdefault("_root_meta", {})
        ck = (pk_e.name, ge.name)
        if ck not in cache:
            cache[ck] = P.broadcast_object(meta, 0)
        meta = cache[ck]
    pmin, pmax, gmin, gmax, dn, gnull = meta
    if pmin is None or gmin is None or dn == 0:
        return None
    prange, grng = pmax - pmin + 1, gmax - gmin + 1
    if not (prange <= max(4 * dn, 1 << 16) and prange < (1 << 31)):
        return None
    if not (grng + 1 <= DENSE_MAX_SLOTS and grng <= 8 * dn + 1024):
        return None
    dpred, never = simplify_pred(dim.pred + [E.substitute(p, dim.exprs) for p in dim_pred])
    fpred, fnever = simplify_pred(fact.pred + [E.substitute(p, fact.exprs) for p in fact_pred])
    if never or fnever:
        return None
    nslots = grng + 1
    if os.environ.get("B200SQL_NO_PREPARED") != "1":
        prep = PreparedStar.get(src, fact, dim, fk_e, pk_e, ge, gexprs[0], aggs, fpred, dpred,
                                (pmin, prange, gmin, grng, gnull), owner, world > 1 and dist == "root", sharded, dev)
        if prep is not None:
            return prep.run(src)
    # lookup and the 4 flag words share one buffer: one broadcast carries both
    buf = torch.full((prange + 4,), -1, dtype=torch.int32, device=dev)
    lookup, flags = buf[:prange], buf[prange:]
    flags.zero_()
    with _Phase("build"):
        if owner:
            needed: Set[str] = {pk_e.name, ge.name}
            for p in dpred:
                p.refs(needed)
            for part in materialize(dim.source, needed):
                if part.n == 0:
                    continue
                ctx = ScanCtx(part, dpred)
                pk_slot, g_slot = ctx.slot(pk_e), ctx.slot(ge)     # slots first: scan() snapshots the columns
                stats["launches"] += 1
                L.star_build_scan(C.byref(ctx.scan()), pk_slot, g_slot, pmin, prange, gmin, nslots - 1,
                                  D.ptr(lookup), D.ptr(flags), D.stream_ptr())
    if world > 1 and dist == "root":
        # the build side crosses NVLink as the finished 4-byte-per-key lookup, not as its columns
        with _Phase("bcast"):
            P.broadcast_(buf, 0)
    plan = AggPlan([(E.substitute(e, fact.exprs) if e is not None else None, o, f) for e, o, f in aggs],
                   _nullable_fn(fact, sharded))
    gs = GroupState(dev, nslots, plan, need_present=True, alloc=_padded_slots(nslots, sharded))
    lk = L.StarLookup()
    lk.dense, lk.lookup, lk.kmin, lk.range = 1, lookup.data_ptr(), pmin, prange
    needed = set(fk_e.refs())
    for ka in plan.kaggs:
        ka.expr.refs(needed)
    for p in fpred:
        p.refs(needed)
    with _Phase("scan"):
        for part in materialize(fact.source, needed, pred=fpred):
            if part.n == 0:
                continue
            ctx = ScanCtx(part, fpred)
            fk_slot = ctx.slot(fk_e)
            gs.bind(ctx)
            stats["launches"] += 1
            ev = _kernel_event_begin("b2_star_agg_kernel", part.n)
            L.star_agg(C.byref(ctx.scan()), fk_slot, C.byref(lk), gs.table.aggs, len(gs.table.specs),
                       C.byref(gs.table.state), D.stream_ptr())
            _kernel_event_end(ev)
    view = _merge_dense(gs.table, plan, sharded, dev)
    glog = dim.col_type(gexprs[0].name)[1] if isinstance(gexprs[0], ColRef) else "int64"
    stats["star_fused"] += 1

    def general():   # a duplicate build key showed up: the general path redoes the query
        stats["star_fused"] -= 1
        return run_aggregate(src, allow_fast=False)

    # the duplicate-key flags ride on the (deferred) host copy of the group count
    return _finalize_dense(view, gmin, src.group_cols[0], gexprs[0], glog, plan, dev, key_nullable=gnull,
                           check=flags, fallback=general)


def try_star(src: AggSource, child: LazyFrame, gexprs, aggs, pred, sharded, allow_fast=True) -> Optional[Part]:
    js: JoinSource = child.source
    if js.how != "inner" or len(js.left_on) != 1 or any(fn.lower() in MOMENT_FUNCS for _, _, fn in aggs):
        return None
    lnames, rnames = set(js.left.columns), set(js.right.columns)
    gsides = {_side_of(e, lnames, rnames) for e in gexprs}
    if len(gsides) != 1 or gsides & {"both", "none"}:
        return None
    dim_side = gsides.pop()
    fact_side = "left" if dim_side == "right" else "right"
    for e, _, _ in aggs:
        if e is not None and _side_of(e, lnames, rnames) not in (fact_side, "none"):
            return None
    fact_pred, dim_pred = [], []
    for p in pred:
        s = _side_of(p, lnames, rnames)
        if s == fact_side:
            fact_pred.append(p)
        elif s == dim_side:
            dim_pred.append(p)
        else:
            return None
    fact: LazyFrame = js.left if fact_side == "left" else js.right
    dim: LazyFrame = js.right if fact_side == "left" else js.left
    fk_name = js.left_on[0] if fact_side == "left" else js.right_on[0]
    pk_name = js.right_on[0] if fact_side == "left" else js.left_on[0]
    if not isinstance(fact.source, TableSource):
        return None
    fk_e, pk_e = fact.exprs[fk_name], dim.exprs[pk_name]
    if fk_e.dtype != I64 or pk_e.dtype != I64:
        return None
    dev = _dev()

    # ---- fast path: dense join key and dense group key straight from a registered table: the
    # whole build side is one kernel per dim partition (filter -> slot -> lookup), no host sync
    fast = _star_dense_fast(src, fact, dim, fk_e, pk_e, gexprs, aggs, fact_pred, dim_pred, sharded, dev) \
        if allow_fast else None
    if fast is not None:
        return fast

    # ---- build side: filtered dim rows, their group slots, and the pk -> slot lookup
    dim_f = LazyFrame(dim.source, dim.exprs, dim.pred + [E.substitute(p, dim.exprs) for p in dim_pred])
    gcols = [f"__g{i}" for i in range(len(gexprs))]
    dim_exprs = {"__pk": pk_e}
    for gc, ge in zip(gcols, gexprs):
        dim_exprs[gc] = E.substitute(ge, dim.exprs)
    dim_q = LazyFrame(dim.source, dim_exprs, dim_f.pred)
    dparts = execute(dim_q)
    dist = frame_distribution(dim)
    d = concat_parts(dparts, ["__pk"] + gcols)
    if P.world()[1] > 1 and dist in ("root", "sharded"):
        from .merge import broadcast_part, allgather_part
        d = broadcast_part(d, dev) if dist == "root" else allgather_part(d, dev)
    if d.n == 0:
        return None
    pk = d["__pk"]
    def _stats(expr, col):
        # a filtered subset lies within the table-level range, and table statistics are cached:
        # no kernel and no host sync per query
        if isinstance(expr, ColRef) and isinstance(dim.source, TableSource) and dist not in ("root", "sharded"):
            return dim.source.table.column_stats(expr.name)
        return col.ensure_stats()

    pst = _stats(pk_e, pk)
    if pst.vmin is None:
        return None
    plan = AggPlan([(E.substitute(e, fact.exprs) if e is not None else None, o, f) for e, o, f in aggs],
                   _nullable_fn(fact, sharded))
    glog = [(e.logical if isinstance(e, ColRef) else _LOGICAL[e.dtype]) for e in gexprs]
    glog = [dim.col_type(e.name)[1] if isinstance(e, ColRef) else l for e, l in zip(gexprs, glog)]

    # group slots of the dim rows
    gkey_cols = [d[g] for g in gcols]
    dense_groups = False
    if len(gcols) == 1 and gkey_cols[0].dtype in (I64,):
        gst = _stats(E.substitute(gexprs[0], dim.exprs), gkey_cols[0])
        if gst.vmin is not None and gst.vmax - gst.vmin + 2 <= DENSE_MAX_SLOTS and \
                (gst.vmax - gst.vmin) <= 8 * d.n + 1024:
            dense_groups = True
    flags = D.new_flags(dev)
    slot_of_row = torch.empty(d.n, dtype=torch.int32, device=dev)
    if dense_groups:
        gmin, grng = gst.vmin, gst.vmax - gst.vmin + 1
        nslots = grng + 1
        ks = gkey_cols[0].as_struct()
        stats["launches"] += 1
        L.dense_slots(C.byref(ks), d.n, gmin, nslots - 1, D.ptr(slot_of_row), D.stream_ptr())
    else:
        # factorize the dim's group columns with the composite-key table; slots = table slots
        cap = D._pow2_at_least(max(1024, 2 * d.n))
        nk = len(gcols)
        tkeys = torch.zeros(nk * cap, dtype=torch.int64, device=dev)
        tnulls = torch.zeros(cap, dtype=torch.uint8, device=dev)
        tstate = torch.zeros(cap, dtype=torch.int32, device=dev)
        ftab = D.GroupTable(dev, cap, [], [], [], False, False)
        ftab.state.out_slot = slot_of_row.data_ptr()
        scan = D.make_scan(gkey_cols, [], d.n)
        stats["launches"] += 1
        D.groupby_hashk(scan, list(range(nk)), tkeys, tnulls, tstate, cap, ftab, flags)
        if int(flags[0].item()):
            return None
        nslots = cap
    gs = GroupState(dev, nslots, plan, need_present=True,
                    alloc=_padded_slots(nslots, sharded) if dense_groups else None)

    # pk -> slot lookup
    lk = L.StarLookup()
    prange = pst.vmax - pst.vmin + 1
    pks = pk.as_struct()
    flags.zero_()
    if prange <= max(4 * d.n, 1 << 16) and prange < (1 << 31):
        lookup = torch.full((prange,), -1, dtype=torch.int32, device=dev)
        stats["launches"] += 1
        L.star_build_dense(C.byref(pks), None, d.n, D.ptr(slot_of_row), pst.vmin, prange, D.ptr(lookup),
                           D.ptr(flags), D.stream_ptr())
        lk.dense, lk.lookup, lk.kmin, lk.range = 1, lookup.data_ptr(), pst.vmin, prange
    else:
        lcap = D._pow2_at_least(max(1024, 2 * d.n))
        ltk = torch.full((lcap,), L.EMPTY_KEY, dtype=torch.int64, device=dev)
        lts = torch.full((lcap,), -1, dtype=torch.int32, device=dev)
        stats["launches"] += 1
        L.star_build_hash(C.byref(pks), None, d.n, D.ptr(slot_of_row), D.ptr(ltk), D.ptr(lts), lcap,
                          D.ptr(flags), D.stream_ptr())
        lk.dense, lk.table_keys, lk.table_slots, lk.cap = 0, ltk.data_ptr(), lts.data_ptr(), lcap
    fl = flags.cpu().tolist()
    if fl[0] or fl[1]:
        return None  # duplicate build keys (or overflow): the general join path handles it

    # ---- one pass over the fact partitions
    fpred, never = simplify_pred(fact.pred + [E.substitute(p, fact.exprs) for p in fact_pred])
    if never:
        fparts = []
    else:
        needed: Set[str] = set(fk_e.refs())
        for ka in plan.kaggs:
            ka.expr.refs(needed)
        for p in fpred:
            p.refs(needed)
        fparts = materialize(fact.source, needed, pred=fpred)
    for part in fparts:
        if part.n == 0:
            continue
        ctx = ScanCtx(part, fpred)
        fk_slot = ctx.slot(fk_e)
        gs.bind(ctx)
        stats["launches"] += 1
        ev = _kernel_event_begin("b2_star_agg_kernel", part.n)
        L.star_agg(C.byref(ctx.scan()), fk_slot, C.byref(lk), gs.table.aggs, len(gs.table.specs),
                   C.byref(gs.table.state), D.stream_ptr())
        _kernel_event_end(ev)
    stats["star_fused"] += 1
    if dense_groups:
        # dense slots = key - gmin on every rank (gmin comes from the broadcast dim rows): mergeable by slot
        view = _merge_dense(gs.table, plan, sharded, dev)
        return _finalize_dense(view, gmin, src.group_cols[0], gexprs[0], glog[0], plan, dev,
                               key_nullable=gkey_cols[0].valid is not None)
    # hashed slots are assigned by CAS races, i.e. differently on every rank: partial tables are
    # merged BY KEY along the reduction tree (like any hash GROUP BY), never element-wise by slot
    raw = _extract_hashk(gs, tkeys, tnulls, nslots, src.group_cols, gexprs, glog, dev)
    if sharded:
        from .merge import tree_merge_raw
        raw = tree_merge_raw(raw, plan, src.options, dev)
    return finish(raw, plan)


# ---------------------------------------------------------------------------------------------
# fused join + global aggregate: Aggregate(no GROUP BY) <- Inner Join(fk = unique dense pk)
# ---------------------------------------------------------------------------------------------
def _strip_f64_cast(e: Expr) -> Expr:
    """cast(int expr -> float64) -> the int expr: b2_join_agg converts inside the kernel, and an
    int64 payload can then be stored as 4-byte offsets (half the L2 footprint of the build side)."""
    if isinstance(e, Call) and e.op == "cast" and e.dtype == F64 and e.args[0].dtype == I64:
        return e.args[0]
    return e


def _split_two_sided(e: Expr, pnames: Set[str], bnames: Set[str]):
    """-> (probe-side expr | None, build-side expr | None, B2_JA_* combine), or None when `e` is not
    of the shape  P,  B,  P*B,  P+B,  P-B,  B-P."""
    side = _side_of(e, pnames, bnames)
    if side == "left":
        return e, None, L.JA_P
    if side == "right":
        return None, e, L.JA_B
    if side != "both" or not isinstance(e, Call) or e.op not in ("mul", "add", "sub"):
        return None
    x, y = e.args
    sx, sy = _side_of(x, pnames, bnames), _side_of(y, pnames, bnames)
    comb = {"mul": L.JA_MUL, "add": L.JA_ADD, "sub": L.JA_SUB}[e.op]
    if sx == "left" and sy == "right":
        return _strip_f64_cast(x), _strip_f64_cast(y), comb
    if sx == "right" and sy == "left":
        return _strip_f64_cast(y), _strip_f64_cast(x), (L.JA_RSUB if e.op == "sub" else comb)
    return None


def try_join_agg(src: AggSource, child: LazyFrame, aggs, pred, sharded) -> Optional[Part]:
    """Global aggregates straight off the probe scan of an inner join on a unique dense key
    (b2_join_agg): nothing of the join is materialised.  None = shape does not apply."""
    js: JoinSource = child.source
    if js.how != "inner" or len(js.left_on) != 1 or any(fn.lower() in MOMENT_FUNCS for _, _, fn in aggs):
        return None
    swap, _ = join_sides(js)
    probe, build = (js.right, js.left) if swap else (js.left, js.right)
    pkey, bkey = (js.right_on[0], js.left_on[0]) if swap else (js.left_on[0], js.right_on[0])
    if not isinstance(probe.source, TableSource):
        return None
    pk_e, bk_e = probe.exprs[pkey], build.exprs[bkey]
    if pk_e.dtype != I64 or bk_e.dtype != I64:
        return None
    pnames, bnames = set(probe.columns), set(build.columns)
    probe_pred, build_pred = [], []
    for p in pred:
        s_ = _side_of(p, pnames, bnames)
        if s_ == "left":
            probe_pred.append(p)
        elif s_ == "right":
            build_pred.append(p)
        else:
            return None
    # aggregate inputs in terms of the join's inputs, split into a probe part and a build part
    plan = AggPlan(aggs, lambda e: True)      # NULLs are tracked per aggregate by the kernel anyway
    if len(plan.kaggs) + 1 > L.MAX_AGGS:
        return None
    split, bexprs = [], []
    for ka in plan.kaggs:
        sp = _split_two_sided(ka.expr, pnames, bnames)
        if sp is None:
            return None
        pe, be, comb = sp
        if pe is not None and pe.dtype == U8 or be is not None and be.dtype == U8:
            return None
        bi = -1
        if be is not None:
            be = E.substitute(be, build.exprs)
            for i, x in enumerate(bexprs):
                if repr(x) == repr(be):
                    bi = i
            if bi < 0:
                bexprs.append(be)
                bi = len(bexprs) - 1
        split.append((E.substitute(pe, probe.exprs) if pe is not None else None, bi, comb))
    if len(bexprs) > L.JA_MAX_BUILD:
        return None
    dev = _dev()

    # ---- build side: key + payload expressions of the (filtered) build rows, whole on every rank
    b_exprs = {"__bk": bk_e}
    for i, be in enumerate(bexprs):
        b_exprs[f"__b{i}"] = be
    bpred = build.pred + [E.substitute(p, build.exprs) for p in build_pred]
    with _Phase("build"):
        bpart = concat_parts(execute(LazyFrame(build.source, b_exprs, bpred)), list(b_exprs))
    if P.world()[1] > 1:
        bd = frame_distribution(build)
        if bd in ("root", "sharded") and not (bd == "root" and frame_distribution(probe) == "root"):
            from .merge import broadcast_part, allgather_part
            with _Phase("bcast"):
                bpart = broadcast_part(bpart, dev) if bd == "root" else allgather_part(bpart, dev)
    if bpart.n == 0:
        return None
    jt = D.JoinTable([bpart["__bk"]])
    stats["launches"] += 1
    if not jt.dense:
        return None                      # duplicate or sparse build keys: the general join handles it
    stats["launches"] += max(1, len(bexprs))
    jt.key_layout([bpart[f"__b{i}"] for i in range(len(bexprs))])

    # ---- one pass over the probe partitions
    ppred, never = simplify_pred(probe.pred + [E.substitute(p, probe.exprs) for p in probe_pred])
    k = len(plan.kaggs)
    acc_d = torch.zeros(k + 1, dtype=torch.int64, device=dev)
    cnt_d = torch.zeros(k + 1, dtype=torch.int64, device=dev)
    ws = D._workspace(dev, L.scan_agg_ws_bytes())
    nb = len(bexprs)
    bc = (L.Col * max(1, nb))(*[c.as_struct() for c in jt.keyed_cols])
    bb = (C.c_int64 * max(1, nb))(*jt.keyed_base)
    needed: Set[str] = set(pk_e.refs())
    for pe, _, _ in split:
        if pe is not None:
            pe.refs(needed)
    for p in ppred:
        p.refs(needed)
    first = True
    float_acc = [False] * k
    for part in ([] if never else materialize(probe.source, needed, pred=ppred)):
        if part.n == 0:
            continue
        ctx = ScanCtx(part, ppred)
        kslot = ctx.slot(pk_e)
        arr = (L.JoinAgg * (k + 1))()
        for i, (ka, (pe, bi, comb)) in enumerate(zip(plan.kaggs, split)):
            arr[i].pcol = ctx.slot(pe) if pe is not None else -1
            arr[i].bcol, arr[i].combine, arr[i].op = bi, comb, ka.op
            pf = pe is not None and pe.dtype == F64
            bf = bi >= 0 and jt.keyed_cols[bi].dtype == F64
            float_acc[i] = pf or bf or ka.op == L.AGG_SUMF
        arr[k].pcol, arr[k].bcol, arr[k].combine, arr[k].op = -1, -1, L.JA_ROWS, L.AGG_COUNT
        stats["launches"] += 2
        ev = _kernel_event_begin("b2_join_agg_kernel", part.n)
        L.join_agg(C.byref(ctx.scan()), kslot, C.byref(jt.struct), nb, bc, bb, arr, k + 1, D.ptr(acc_d), D.ptr(cnt_d),
                   0 if first else 1, D.ptr(ws), D.stream_ptr())
        _kernel_event_end(ev)
        first = False
    if first:
        acc = np.array([{L.AGG_MIN: (1 << 63) - 1, L.AGG_MAX: -(1 << 63)}.get(ka.op, 0) for ka in plan.kaggs] + [0],
                       dtype=np.int64)
        cnt = np.zeros(k + 1, dtype=np.int64)
    else:
        acc, cnt = acc_d.cpu().numpy(), cnt_d.cpu().numpy()
        stats["d2h_bytes"] += 16 * (k + 1)
    stats["join_agg"] = stats.get("join_agg", 0) + 1
    if sharded:
        # the all-reduce folds by the accumulator's arithmetic type: mark float accumulators as such
        for ka, f in zip(plan.kaggs, float_acc):
            if f:
                ka.dtype = F64
        acc, cnt = _allreduce_global(acc, cnt, plan, dev)
    return _finish_global(plan, acc, cnt, dev, float_acc)


# ---------------------------------------------------------------------------------------------
# join
# ---------------------------------------------------------------------------------------------
def run_join(js: JoinSource, needed: Set[str]) -> List[Part]:
    dev = _dev()
    how = js.how
    left, right = js.left, js.right
    lkeys, rkeys = js.left_on, js.right_on
    # which side is hashed (build) and which streams (probe): agreed by all ranks
    swap, _ = join_sides(js)
    probe, build = (right, left) if swap else (left, right)
    pkeys, bkeys = (rkeys, lkeys) if swap else (lkeys, rkeys)
    mode = {"inner": L.JOIN_INNER, "left": L.JOIN_LEFT, "right": L.JOIN_LEFT, "outer": L.JOIN_LEFT,
            "leftsemi": L.JOIN_SEMI, "leftanti": L.JOIN_ANTI}[how]

    # key expressions; mixed int/float keys compare as float64 (pandas upcasts the same way)
    pk_exprs = [probe.exprs[k] for k in pkeys]
    bk_exprs = [build.exprs[k] for k in bkeys]
    for i, (a, b) in enumerate(zip(pk_exprs, bk_exprs)):
        if a.dtype == U8:
            a = pk_exprs[i] = E.cast(a, I64)
        if b.dtype == U8:
            b = bk_exprs[i] = E.cast(b, I64)
        if a.dtype != b.dtype:
            pk_exprs[i], bk_exprs[i] = E.cast(a, F64), E.cast(b, F64)

    build_out = [n for n in build.columns if n in needed] if how not in ("leftsemi", "leftanti") else []
    probe_out = [n for n in probe.columns if n in needed]

    # ---- build side: materialise (filtered) needed columns + keys into one partition
    b_exprs = {n: build.exprs[n] for n in build_out}
    for i, e in enumerate(bk_exprs):
        b_exprs[f"__bk{i}"] = e
    bparts = execute(LazyFrame(build.source, b_exprs, build.pred))
    bpart = concat_parts(bparts, list(b_exprs))
    probe_dist = frame_distribution(probe)
    if P.world()[1] > 1:
        bd = frame_distribution(build)
        # the build side must be whole wherever probe rows live: broadcast it from its owner, or
        # all-gather its shards (also for LEFT / SEMI / ANTI / OUTER joins: a probe row is
        # "unmatched" only if NO rank holds a partner).  Both sides on rank 0 only: nothing to move.
        if bd in ("root", "sharded") and not (bd == "root" and probe_dist == "root"):
            from .merge import broadcast_part, allgather_part
            with _Phase("bcast"):
                bpart = broadcast_part(bpart, dev) if bd == "root" else allgather_part(bpart, dev)
    bkey_cols = [bpart[f"__bk{i}"] for i in range(len(bk_exprs))]
    jt = D.JoinTable(bkey_cols)
    stats["launches"] += 1
    stats["dense_join" if jt.dense else "chain_join"] += 1
    build_matched = torch.zeros(max(bpart.n, 1), dtype=torch.uint8, device=dev) if how == "outer" else None
    prefs = sorted({r for n in probe_out for r in probe.exprs[n].refs()})
    fused_gather = len(prefs) <= L.MAX_GATHER and len(build_out) <= L.MAX_GATHER
    if jt.dense and fused_gather and how != "outer" and estimated_rows(probe) >= bpart.n \
            and os.environ.get("B200SQL_NO_KEY_LAYOUT") != "1":
        # unique dense keys probed by at least as many rows as were built: one pass over the build
        # columns puts them in key order, every probe row then saves a random access
        stats["launches"] += max(1, len(build_out))
        stats["keyed_join"] += 1
        jt.key_layout([bpart[n] for n in build_out])

    # ---- probe side, partition by partition
    ppred, never = simplify_pred(probe.pred)
    src_needed: Set[str] = set()
    for n in probe_out:
        probe.exprs[n].refs(src_needed)
    for e in pk_exprs:
        e.refs(src_needed)
    for p in ppred:
        p.refs(src_needed)
    pparts = [] if never else materialize(probe.source, src_needed, pred=ppred)
    outs: List[Part] = []
    for part in pparts:
        if part.n == 0:
            continue
        ctx = ScanCtx(part, ppred)
        kslots = [ctx.slot(e) for e in pk_exprs]
        refs = prefs
        if fused_gather and jt.dense and build_matched is None and os.environ.get("B200SQL_NO_ONEPASS") != "1":
            # direct-address table: single-pass probe (look-back offsets), row count left on the device
            rslots = [ctx.slot(ColRef(r, part[r].dtype)) for r in refs]
            stats["launches"] += 3
            ev = _kernel_event_begin("b2_join_onepass", part.n)
            trim, count = D.join_probe_onepass(ctx.scan(), kslots, jt, mode, dev, ctx.cols, rslots,
                                               [bpart[n] for n in build_out], mode == L.JOIN_LEFT)
            _kernel_event_end(ev)
            pending = DeviceCount(count)

            def finish_part(trim=trim, pending=pending, keep=(ctx, jt, bpart)):
                total = int(pending.get()[0])
                pres, bres = trim(total)
                g = Part(dict(zip(refs, pres)), total)
                res = Part({}, total)
                for n, col in zip(build_out, bres):
                    res[n] = col
                for n in probe_out:
                    e = probe.exprs[n]
                    res[n] = const_column(e.value, e.dtype, total, dev) if isinstance(e, Lit) else eval_expr(g, e)
                return res

            outs.append(PendingPart(finish_part))
            continue
        if fused_gather:
            # probe + gather of both sides' columns in one pass (b2_join_write_gather)
            rslots = [ctx.slot(ColRef(r, part[r].dtype)) for r in refs]
            stats["launches"] += 3
            pres, bres, total = D.join_probe_gather(ctx.scan(), kslots, jt, mode, dev, ctx.cols, rslots,
                                                    [bpart[n] for n in build_out], mode == L.JOIN_LEFT,
                                                    build_matched)
            g = Part(dict(zip(refs, pres)), total)
            res = Part({}, total)
            for n, col in zip(build_out, bres):
                res[n] = col
        else:
            stats["launches"] += 3
            pidx, bidx, total = D.join_probe(ctx.scan(), kslots, jt, mode, dev, build_matched)
            res = Part({}, total)
            g = Part({r: D.gather(part[r], pidx, False) for r in refs}, total)
            stats["launches"] += len(refs)
            for n in build_out:
                stats["launches"] += 1
                res[n] = D.gather(bpart[n], bidx, mode == L.JOIN_LEFT)
        # probe-side output expressions are evaluated on the gathered source columns
        for n in probe_out:
            e = probe.exprs[n]
            res[n] = const_column(e.value, e.dtype, total, dev) if isinstance(e, Lit) else eval_expr(g, e)
        outs.append(res)
    emit_unmatched = how == "outer" and bpart.n > 0
    if emit_unmatched and P.world()[1] > 1 and probe_dist in ("sharded", "root"):
        # a build row is unmatched only if no rank's probe rows matched it: OR the flags over the
        # ranks, and let exactly one rank emit the leftovers
        P.allreduce_(build_matched, "max")
        emit_unmatched = P.world()[0] == 0
    if emit_unmatched:
        # build rows nobody matched, with NULL probe columns
        um = DeviceColumn(build_matched[: bpart.n], None, U8)
        scan = D.make_scan([um], [TermSpec(0, L.EQ, 0)], bpart.n)
        stats["launches"] += 3
        idx, _, total = D.select(scan, dev, (), want_idx=True, cols=[um])
        if total > 0:
            res = Part({}, total)
            for n in probe_out:
                dt, lg = probe.col_type(n)
                res[n] = null_column(dt, lg, total, dev)
            for n in build_out:
                stats["launches"] += 1
                res[n] = D.gather(bpart[n], idx, False)
            outs.append(res)
    if not outs:
        cols = {}
        for n in probe_out:
            dt, lg = probe.col_type(n)
            cols[n] = DeviceColumn(torch.empty(0, dtype=_TORCH_DT[dt], device=dev), None, dt, lg)
        for n in build_out:
            dt, lg = build.col_type(n)
            cols[n] = DeviceColumn(torch.empty(0, dtype=_TORCH_DT[dt], device=dev), None, dt, lg)
        outs = [Part(cols, 0)]
    return outs


# ---------------------------------------------------------------------------------------------
# entry points used by LazyFrame
# ---------------------------------------------------------------------------------------------
def compute_frame(frame: LazyFrame):
    """Execute and bring the result to the host as a pandas DataFrame (Context.sql(...).compute())."""
    import pandas as pd

    parts = [gather_keyrange(p) for p in execute(frame, top=True)]
    torch.cuda.current_stream().synchronize()
    frames = []
    for p in parts:
        data = {}
        for n in frame.columns:
            stats["d2h_bytes"] += p[n].nbytes()
            data[n] = D.column_to_host(p[n])
        frames.append(pd.DataFrame(data, columns=frame.columns) if data else pd.DataFrame(index=range(p.n)))
    if len(frames) == 1:
        return frames[0]
    nonempty = [f for f in frames if len(f)]
    if not nonempty:
        return frames[0]
    return pd.concat(nonempty, ignore_index=True)


def persist_frame(frame: LazyFrame) -> LazyFrame:
    parts = execute(frame)
    table = DeviceTable([dict(p.resolve()) for p in parts], frame_distribution(frame))
    return LazyFrame(TableSource(table))


def count_rows(frame: LazyFrame) -> int:
    pred, never = simplify_pred(frame.pred)
    if never:
        return 0
    if not pred and isinstance(frame.source, TableSource):
        return frame.source.table.nrows
    cnt = LazyFrame(AggSource(frame, [], [(None, "n", "size")])).compute()
    return int(cnt["n"].iloc[0]) if len(cnt) else 0
