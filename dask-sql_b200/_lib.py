"""ctypes binding of libb200sql.so (C-ABI declared in include/b200sql.h).

There is deliberately no fallback: if the library is missing the import fails loudly, and
every call checks the int32 status and raises with b2_last_error().
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200SQL_LIB") or os.path.join(HERE, "libb200sql.so")   # override: A/B builds

# ---- constants (mirror include/b200sql.h) ----
I64, F64, U8 = 0, 1, 2
U32 = 3          # storage-only: narrowed key-ordered join payload
COL_SENTINEL = 1
MAX_COLS, MAX_TERMS, MAX_AGGS, MAX_KEYS, MAX_GATHER, MAX_PROG = 16, 8, 8, 4, 8, 64
TILE = 4096
EQ, NE, LT, LE, GT, GE, IS_NULL, IS_NOT_NULL, IS_TRUE = range(9)
AGG_SUM, AGG_SUMF, AGG_MIN, AGG_MAX, AGG_COUNT = range(5)
JOIN_INNER, JOIN_LEFT, JOIN_SEMI, JOIN_ANTI = range(4)
EMPTY_KEY = -(1 << 63)

OP_LOAD, OP_CONST_I, OP_CONST_F, OP_CONST_NULL, OP_I2F, OP_F2I = 0, 1, 2, 3, 4, 5
OP_ADD_I, OP_SUB_I, OP_MUL_I, OP_DIV_I, OP_NEG_I, OP_ABS_I, OP_MOD_I = 10, 11, 12, 13, 14, 15, 16
OP_ADD_F, OP_SUB_F, OP_MUL_F, OP_DIV_F, OP_NEG_F, OP_ABS_F, OP_SQRT_F = 20, 21, 22, 23, 24, 25, 26
OP_EQ_I, OP_EQ_F = 30, 40
OP_AND, OP_OR, OP_NOT, OP_ISNULL_I, OP_ISNULL_F, OP_CASE, OP_FILLNA, OP_ORD2F = 50, 51, 52, 53, 54, 55, 56, 57


class Col(C.Structure):
    _fields_ = [("data", C.c_void_p), ("valid", C.c_void_p), ("dtype", C.c_int32), ("flags", C.c_int32)]


class Term(C.Structure):
    _fields_ = [("col", C.c_int32), ("op", C.c_int32), ("as_f64", C.c_int32), ("pad_", C.c_int32),
                ("lit_i", C.c_int64), ("lit_f", C.c_double)]


class Scan(C.Structure):
    _fields_ = [("cols", Col * MAX_COLS), ("terms", Term * MAX_TERMS), ("ncols", C.c_int32),
                ("nterms", C.c_int32), ("n", C.c_int64)]


class Agg(C.Structure):
    _fields_ = [("col", C.c_int32), ("op", C.c_int32)]


class AggState(C.Structure):
    _fields_ = [("acc", C.c_void_p * MAX_AGGS), ("cnt", C.c_void_p * MAX_AGGS), ("rows", C.c_void_p),
                ("present", C.c_void_p), ("out_slot", C.c_void_p)]


class Instr(C.Structure):
    _fields_ = [("op", C.c_int32), ("a", C.c_int32), ("imm_i", C.c_int64), ("imm_f", C.c_double)]


class Prog(C.Structure):
    _fields_ = [("code", Instr * MAX_PROG), ("n", C.c_int32), ("out_dtype", C.c_int32)]


class JoinTable(C.Structure):
    _fields_ = [("keys", Col * MAX_KEYS), ("nkeys", C.c_int32), ("dense", C.c_int32), ("head", C.c_void_p),
                ("next", C.c_void_p), ("cap", C.c_int64), ("lookup", C.c_void_p), ("kmin", C.c_int64),
                ("range", C.c_int64)]


JA_P, JA_B, JA_MUL, JA_ADD, JA_SUB, JA_RSUB, JA_ROWS = range(7)
JA_MAX_BUILD = 4


class JoinAgg(C.Structure):
    _fields_ = [("pcol", C.c_int32), ("bcol", C.c_int32), ("combine", C.c_int32), ("op", C.c_int32)]


class StarLookup(C.Structure):
    _fields_ = [("dense", C.c_int32), ("pad_", C.c_int32), ("lookup", C.c_void_p), ("kmin", C.c_int64),
                ("range", C.c_int64), ("table_keys", C.c_void_p), ("table_slots", C.c_void_p),
                ("cap", C.c_int64)]


MAX_PEERS, PEER_MAX_ARRAYS = 16, 2 * MAX_AGGS + 1
PEER_SUM_F64, PEER_SUM_I64, PEER_MIN_I64, PEER_MAX_I64 = range(4)
PEER_PRESENT_ROWS, PEER_PRESENT_INDICATOR, PEER_PRESENT_BITMAP = 1, 2, 3


class PeerMerge(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("narrays", C.c_int32), ("presence_kind", C.c_int32),
                ("presence_array", C.c_int32), ("ops", C.c_int32 * PEER_MAX_ARRAYS),
                ("array_off", C.c_int64 * PEER_MAX_ARRAYS), ("bitmap_off", C.c_int64), ("signal_off", C.c_int64),
                ("peer_base", C.c_void_p * MAX_PEERS), ("out", C.c_void_p * PEER_MAX_ARRAYS),
                ("out_present", C.c_void_p), ("lo", C.c_int64), ("count", C.c_int64), ("local_ready", C.c_void_p),
                ("epoch", C.c_uint64)]


WIN_MAX_KEYS = 8
WB_UNBOUNDED, WB_OFFSET = 0, 1
(WIN_ROW_NUMBER, WIN_RANK, WIN_DENSE_RANK, WIN_SUM, WIN_COUNT, WIN_AVG, WIN_MIN, WIN_MAX, WIN_FIRST,
 WIN_LAST) = range(10)


class WSegs(C.Structure):
    _fields_ = [("part_start", C.c_void_p), ("part_end", C.c_void_p), ("peer_start", C.c_void_p),
                ("peer_end", C.c_void_p), ("dense", C.c_void_p)]


class WFrame(C.Structure):
    _fields_ = [("range", C.c_int32), ("lo_kind", C.c_int32), ("hi_kind", C.c_int32), ("pad_", C.c_int32),
                ("lo", C.c_int64), ("hi", C.c_int64)]


assert C.sizeof(WSegs) == 40 and C.sizeof(WFrame) == 32
assert C.sizeof(Col) == 24 and C.sizeof(Term) == 32 and C.sizeof(Scan) == 656
assert C.sizeof(AggState) == 152 and C.sizeof(Instr) == 24 and C.sizeof(Prog) == 1544
assert C.sizeof(JoinTable) == 152 and C.sizeof(StarLookup) == 56 and C.sizeof(PeerMerge) == 544


class B200SqlError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the B200 execution layer has no CPU fallback. Build it with "
            "`python __graft_entry__.py build` (nvcc -gencode arch=compute_100a,code=sm_100a).")
    return C.CDLL(LIB_PATH)


_lib = _load()
_lib.b2_last_error.restype = C.c_char_p
_lib.b2_num_tiles.restype = C.c_int64
_lib.b2_num_tiles.argtypes = [C.c_int64]
_lib.b2_stats_ws_bytes.restype = C.c_int64
_lib.b2_scan_agg_ws_bytes.restype = C.c_int64
_lib.b2_join_onepass_ws_bytes.restype = C.c_int64
_lib.b2_join_onepass_ws_bytes.argtypes = [C.c_int64]
_lib.b2_range_partition_ws_bytes.restype = C.c_int64
_lib.b2_range_partition_ws_bytes.argtypes = [C.c_int32]
_lib.b2_f64_to_ordered.restype = C.c_int64
_lib.b2_f64_to_ordered.argtypes = [C.c_double]
_lib.b2_ordered_to_f64.restype = C.c_double
_lib.b2_ordered_to_f64.argtypes = [C.c_int64]

_P = C.c_void_p
_SIGS = {
    "b2_version": [],
    "b2_device_info": [C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                       C.POINTER(C.c_int32), C.POINTER(C.c_int64)],
    "b2_d2h": [_P, _P, C.c_int64, _P],
    "b2_sync": [_P],
    "b2_memset": [_P, C.c_int32, C.c_int64, _P],
    "b2_col_stats": [C.POINTER(Col), C.c_int64, _P, _P, _P],
    "b2_expr_eval": [C.POINTER(Prog), C.POINTER(Col), C.c_int32, C.c_int64, _P, _P, _P],
    "b2_scan_agg": [C.POINTER(Scan), C.POINTER(Agg), C.c_int32, _P, _P, C.c_int32, _P, _P],
    "b2_select_count": [C.POINTER(Scan), _P, _P],
    "b2_select_write": [C.POINTER(Scan), _P, _P, C.c_int32, C.POINTER(C.c_int32), C.POINTER(_P),
                        C.POINTER(_P), _P],
    "b2_gather": [C.POINTER(Col), _P, C.c_int64, _P, _P, _P],
    "b2_groupby_dense": [C.POINTER(Scan), C.c_int32, C.c_int64, C.c_int64, C.POINTER(Agg), C.c_int32,
                         C.POINTER(AggState), _P],
    "b2_groupby_dense_grouped": [C.POINTER(Scan), C.c_int32, C.c_int64, C.c_int64, C.POINTER(Agg), C.c_int32,
                                 C.POINTER(AggState), _P],
    "b2_hot_slots": [C.POINTER(Col), C.c_int64, C.c_int64, C.c_int64, _P, _P],
    "b2_groupby_dense_hot": [C.POINTER(Scan), C.c_int32, C.c_int64, C.c_int64, C.POINTER(Agg), C.c_int32,
                             C.POINTER(AggState), _P, _P],
    "b2_groupby_dense_ordered": [C.POINTER(Scan), C.c_int32, C.c_int64, C.c_int64, C.POINTER(Agg), C.c_int32,
                                 C.POINTER(AggState), _P, _P],
    "b2_groupby_hash1": [C.POINTER(Scan), C.c_int32, _P, C.c_int64, C.POINTER(Agg), C.c_int32,
                         C.POINTER(AggState), _P, _P],
    "b2_groupby_hashk": [C.POINTER(Scan), C.POINTER(C.c_int32), C.c_int32, _P, _P, _P, C.c_int64,
                         C.POINTER(Agg), C.c_int32, C.POINTER(AggState), _P, _P],
    "b2_join_build": [C.POINTER(Col), C.c_int32, C.c_int64, _P, _P, C.c_int64, _P],
    "b2_join_build_dense": [C.POINTER(Col), C.c_int64, C.c_int64, C.c_int64, _P, _P, _P],
    "b2_join_count": [C.POINTER(Scan), C.POINTER(C.c_int32), C.POINTER(JoinTable), C.c_int32, _P, _P],
    "b2_join_write": [C.POINTER(Scan), C.POINTER(C.c_int32), C.POINTER(JoinTable), C.c_int32, _P, _P, _P,
                      _P, _P],
    "b2_join_write_gather": [C.POINTER(Scan), C.POINTER(C.c_int32), C.POINTER(JoinTable), C.c_int32, _P, _P, _P,
                             _P, C.c_int32, C.POINTER(C.c_int32), C.POINTER(_P), C.POINTER(_P), C.c_int32,
                             C.POINTER(Col), C.POINTER(_P), C.POINTER(_P), _P],
    "b2_join_key_layout": [C.POINTER(Col), C.c_int64, C.c_int64, C.c_int64, C.POINTER(Col), C.c_int32, C.c_int64,
                           _P, _P, _P, _P],
    "b2_join_write_gather_keyed": [C.POINTER(Scan), C.POINTER(C.c_int32), C.POINTER(JoinTable), C.c_int32, _P, _P,
                                   _P, _P, C.c_int32, C.POINTER(C.c_int32), C.POINTER(_P), C.POINTER(_P),
                                   C.c_int32, C.POINTER(Col), C.POINTER(C.c_int64), C.POINTER(_P), C.POINTER(_P),
                                   _P],
    "b2_join_onepass": [C.POINTER(Scan), C.POINTER(C.c_int32), C.POINTER(JoinTable), C.c_int32, C.c_int32, _P, C.c_int32,
                        C.POINTER(C.c_int32), C.POINTER(_P), C.POINTER(_P), C.c_int32, C.POINTER(Col),
                        C.POINTER(C.c_int64), C.POINTER(_P), C.POINTER(_P), _P],
    "b2_join_agg": [C.POINTER(Scan), C.c_int32, C.POINTER(JoinTable), C.c_int32, C.POINTER(Col), C.POINTER(C.c_int64),
                    C.POINTER(JoinAgg), C.c_int32, _P, _P, C.c_int32, _P, _P],
    "b2_range_partition_hist": [C.POINTER(Scan), C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_int32, _P, _P],
    "b2_range_partition_scan": [C.c_int32, _P, _P],
    "b2_range_partition_scatter": [C.POINTER(Scan), C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                   C.POINTER(C.c_int32), _P, C.POINTER(_P), _P, _P],
    "b2_range_partition": [C.POINTER(Scan), C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                           C.POINTER(C.c_int32), _P, C.POINTER(_P), _P, _P],
    "b2_iota": [_P, C.c_int64, _P],
    "b2_bitmap_or": [_P, _P, C.c_int64, _P],
    "b2_peer_merge": [C.POINTER(PeerMerge), _P],
    "b2_sort_by": [C.POINTER(Col), C.c_int64, C.c_int32, C.c_int32, _P, _P, _P],
    "b2_dense_slots": [C.POINTER(Col), C.c_int64, C.c_int64, C.c_int32, _P, _P],
    "b2_star_build_dense": [C.POINTER(Col), _P, C.c_int64, _P, C.c_int64, C.c_int64, _P, _P, _P],
    "b2_star_build_scan": [C.POINTER(Scan), C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _P,
                           _P, _P],
    "b2_star_build_hash": [C.POINTER(Col), _P, C.c_int64, _P, _P, _P, C.c_int64, _P, _P],
    "b2_star_agg": [C.POINTER(Scan), C.c_int32, C.POINTER(StarLookup), C.POINTER(Agg), C.c_int32,
                    C.POINTER(AggState), _P],
    "b2_window_segments": [C.POINTER(Col), C.c_int32, C.c_int32, C.c_int64, C.POINTER(WSegs), _P, _P],
    "b2_window_rank": [C.c_int32, C.c_int64, C.POINTER(WSegs), _P, _P],
    "b2_window_offset": [C.POINTER(Col), C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.POINTER(WSegs), _P, _P, _P],
    "b2_window_agg": [C.POINTER(Col), C.c_int32, C.POINTER(WFrame), C.c_int64, C.POINTER(WSegs), _P, _P, _P, _P],
}

EXPORTS = sorted(list(_SIGS) + ["b2_last_error", "b2_num_tiles", "b2_stats_ws_bytes", "b2_scan_agg_ws_bytes",
                                "b2_sort_ws_bytes", "b2_window_ws_bytes", "b2_join_onepass_ws_bytes",
                                "b2_range_partition_ws_bytes",
                                "b2_f64_to_ordered", "b2_ordered_to_f64"])


call_times = {} if os.environ.get("B200SQL_CALL_TIMES") == "1" else None    # name -> [calls, host seconds]


def _wrap(name):
    fn = getattr(_lib, name)
    fn.restype = C.c_int32
    fn.argtypes = _SIGS[name]

    if call_times is not None:
        import time

        def call(*args):
            t0 = time.perf_counter()
            rc = fn(*args)
            rec = call_times.setdefault(name, [0, 0.0])
            rec[0] += 1
            rec[1] += time.perf_counter() - t0
            if rc != 0:
                raise B200SqlError(f"{name} failed ({rc}): {_lib.b2_last_error().decode()}")
            return rc

        call.__name__ = name
        return call

    def call(*args):
        rc = fn(*args)
        if rc != 0:
            raise B200SqlError(f"{name} failed ({rc}): {_lib.b2_last_error().decode()}")
        return rc

    call.__name__ = name
    return call


version = getattr(_lib, "b2_version")
version.restype = C.c_int32
device_info = _wrap("b2_device_info")
d2h = _wrap("b2_d2h")
sync = _wrap("b2_sync")
memset = _wrap("b2_memset")
col_stats = _wrap("b2_col_stats")
expr_eval = _wrap("b2_expr_eval")
scan_agg = _wrap("b2_scan_agg")
select_count = _wrap("b2_select_count")
select_write = _wrap("b2_select_write")
gather = _wrap("b2_gather")
groupby_dense = _wrap("b2_groupby_dense")
groupby_dense_ordered = _wrap("b2_groupby_dense_ordered")
groupby_dense_grouped = _wrap("b2_groupby_dense_grouped")
groupby_dense_hot = _wrap("b2_groupby_dense_hot")
hot_slots = _wrap("b2_hot_slots")
groupby_hash1 = _wrap("b2_groupby_hash1")
groupby_hashk = _wrap("b2_groupby_hashk")
join_build = _wrap("b2_join_build")
join_build_dense = _wrap("b2_join_build_dense")
join_count = _wrap("b2_join_count")
join_write = _wrap("b2_join_write")
join_write_gather = _wrap("b2_join_write_gather")
join_write_gather_keyed = _wrap("b2_join_write_gather_keyed")
join_key_layout = _wrap("b2_join_key_layout")
join_onepass = _wrap("b2_join_onepass")
join_onepass_ws_bytes = _lib.b2_join_onepass_ws_bytes
join_agg = _wrap("b2_join_agg")
range_partition = _wrap("b2_range_partition")
range_partition_hist = _wrap("b2_range_partition_hist")
range_partition_scan = _wrap("b2_range_partition_scan")
range_partition_scatter = _wrap("b2_range_partition_scatter")
range_partition_ws_bytes = _lib.b2_range_partition_ws_bytes
iota = _wrap("b2_iota")
bitmap_or = _wrap("b2_bitmap_or")
peer_merge = _wrap("b2_peer_merge")
sort_by = _wrap("b2_sort_by")
_lib.b2_sort_ws_bytes.restype = C.c_int64
_lib.b2_sort_ws_bytes.argtypes = [C.c_int64]
sort_ws_bytes = _lib.b2_sort_ws_bytes
dense_slots = _wrap("b2_dense_slots")
star_build_dense = _wrap("b2_star_build_dense")
star_build_scan = _wrap("b2_star_build_scan")
star_build_hash = _wrap("b2_star_build_hash")
star_agg = _wrap("b2_star_agg")
window_segments = _wrap("b2_window_segments")
window_rank = _wrap("b2_window_rank")
window_offset = _wrap("b2_window_offset")
window_agg = _wrap("b2_window_agg")
_lib.b2_window_ws_bytes.restype = C.c_int64
_lib.b2_window_ws_bytes.argtypes = [C.c_int64]
window_ws_bytes = _lib.b2_window_ws_bytes
num_tiles = _lib.b2_num_tiles
stats_ws_bytes = _lib.b2_stats_ws_bytes
scan_agg_ws_bytes = _lib.b2_scan_agg_ws_bytes
f64_to_ordered = _lib.b2_f64_to_ordered
ordered_to_f64 = _lib.b2_ordered_to_f64


def has_symbol(name):
    try:
        getattr(_lib, name)
        return True
    except AttributeError:
        return False
