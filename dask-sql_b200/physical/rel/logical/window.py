"""Window: f(...) OVER (PARTITION BY ... ORDER BY ... ROWS|RANGE ...) (the reference's plugin is
dask_sql/physical/rel/logical/window.py:201-428, DaskWindowPlugin).

The reference runs every window call as groupby(partition keys).apply(sort -> expanding() / rolling()),
one pandas call per partition and per call.  Here the node becomes one lazy WindowSource: each call is
described by child column names (computed arguments and keys become lazy columns of the child, fused
into whatever produces it), and the executor sorts once per distinct (PARTITION BY, ORDER BY) and runs
the segmented CUDA kernels of csrc/window.cuh.

Without a frame clause the frame is SQL's default, RANGE BETWEEN UNBOUNDED PRECEDING AND CURRENT ROW:
the whole partition when there is no ORDER BY, and the rows up to the current row's last peer when there
is one (the reference uses expanding(), which splits ties; DESIGN.md section 6)."""
from ....datacontainer import DataContainer
from ....frame import LazyFrame, LazySeries, WindowCall, WindowSource
from ....utils import new_temporary_column
from ...rex import RexConverter
from ..base import BaseRelPlugin

# SQL name -> executor function (the reference's OPERATION_MAPPING, window.py:214-225, plus RANK,
# DENSE_RANK, LAG and LEAD; SINGLE_VALUE is FIRST_VALUE there too)
_FUNCS = {"row_number": "row_number", "rank": "rank", "dense_rank": "dense_rank", "lag": "lag", "lead": "lead",
          "sum": "sum", "$sum0": "sum", "count": "count", "avg": "avg", "mean": "avg", "min": "min", "max": "max",
          "first_value": "first_value", "single_value": "first_value", "last_value": "last_value"}
_DEFAULT_FRAME = ("RANGE", ("UNBOUNDED_PRECEDING", None), ("CURRENT", 0))


class DaskWindowPlugin(BaseRelPlugin):
    class_name = "Window"

    def convert(self, rel, context) -> DataContainer:
        (dc,) = self.assert_inputs(rel, 1, context)
        frame, names = dc.df, dc.column_container
        node = rel.window()
        input_rel = rel.get_inputs()[0]
        field_names = [str(f) for f in rel.getRowType().getFieldNames()]
        nin = len(names.columns)
        calls, outputs = [], []

        def column_of(rex):
            """(frame, child column) holding the value of `rex`: an input column as it is, anything else
            as a new lazy column."""
            nonlocal frame
            name = rex.column_name(input_rel)
            if names.knows(name):
                return names.get_backend_by_frontend_name(name)
            value = RexConverter.convert(input_rel, rex, DataContainer(frame, names), context=context)
            tmp = new_temporary_column(frame)
            if isinstance(value, LazySeries):
                frame = frame.assign(**{tmp: value})
            else:
                frame = frame.assign(**{tmp: value if value is not None else float("nan")})
            return tmp

        for i, w in enumerate(node.getGroups()):
            sql_name = node.getWindowFuncName(w).lower()
            func = _FUNCS.get(sql_name)
            if func is None:
                raise NotImplementedError(f"window function {sql_name} is not implemented")
            args = node.getArgs(w)
            params = ()
            if func in ("lag", "lead"):
                k = args[1].getInt64Value() if len(args) > 1 else 1
                default = None
                if len(args) > 2 and str(args[2].getType()) != "Null":
                    default = args[2].value
                    default = float(default) if args[0].sql_type == "DOUBLE" else int(default)
                params, args = (int(k), default), args[:1]
            arg_cols = tuple(column_of(a) for a in args)
            partition = tuple(column_of(p) for p in node.getPartitionExprs(w))
            order = tuple((column_of(s.getSortExpr()), s.isSortAscending(), s.isSortNullsFirst())
                          for s in node.getSortExprs(w))
            fr = node.getWindowFrame(w)
            if fr is None:
                frame_t = _DEFAULT_FRAME
            else:
                def bound(b):
                    if b.isCurrentRow():
                        return ("CURRENT", 0)
                    side = "PRECEDING" if b.isPreceding() else "FOLLOWING"
                    return ("UNBOUNDED_" + side, None) if b.isUnbounded() else (side, int(b.getOffset()))
                frame_t = (fr.getFrameUnits(), bound(fr.getLowerBound()), bound(fr.getUpperBound()))
            out = new_temporary_column(frame)
            calls.append(WindowCall(func, arg_cols, partition, order, frame_t, out, params))
            outputs.append((field_names[nin + i], out))

        result = LazyFrame(WindowSource(frame, calls))
        for field, backend in outputs:
            names = names.add(field, backend)
        names = self.fix_column_to_row_type(names, rel.getRowType())
        return self.fix_dtype_to_row_type(DataContainer(result, names), rel.getRowType())
