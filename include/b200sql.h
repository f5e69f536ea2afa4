/*
 * b200sql.h — C-ABI of libb200sql.so: the B200-native (sm_100a) execution kernels
 * behind dask-sql's filter -> hash-join -> hash-groupby-aggregate hot path.
 *
 * The reference (dask-contrib/dask-sql @ f186de3) has no FFI of its own for this
 * path: its plugins call pandas / dask.dataframe methods.  Each entry point below
 * therefore names the reference call site(s) whose per-partition arithmetic it
 * replaces (paths relative to /root/reference).  The Python plugins in
 * dask-sql_b200/physical/ reach these functions through ctypes (dask-sql_b200/_lib.py);
 * INTEGRATION.md shows the binding a dask-sql maintainer would add.
 *
 * Conventions
 *  - every function returns int32 status: 0 = OK, <0 = error; text via b2_last_error().
 *  - no C++ exceptions, no torch types; plain pointers and sizes only.
 *  - all data pointers are DEVICE pointers owned by the caller, 16-byte aligned
 *    (value buffers) unless stated otherwise.  The library never allocates device memory.
 *  - validity bitmaps are Arrow layout (LSB bit order, 1 = valid); NULL pointer = all valid.
 *    For B2_F64 columns NaN additionally counts as NULL wherever pandas treats it so
 *    (isna, join keys, group keys, aggregate inputs) but NOT in comparisons (IEEE).
 *  - `stream` is a cudaStream_t passed as void*; every call is asynchronous with respect to
 *    the host and writes results to device memory.  b2_d2h()/b2_sync() are the sync points.
 *  - row indices are int32 (a partition holds < 2^31 rows); -1 means "no row" (NULL fill).
 *  - thread-safe across distinct streams.
 */
#ifndef B200SQL_H
#define B200SQL_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define B2_OK            0
#define B2_ERR_CUDA     -1
#define B2_ERR_ARG      -2

/* physical column types */
#define B2_I64 0   /* int64  (BIGINT and narrower ints, widened at ingest) */
#define B2_F64 1   /* float64 (DOUBLE) */
#define B2_U8  2   /* boolean, one byte per row (0/1) */
#define B2_U32 3   /* storage only: uint32 offsets from a base, for key-ordered join payloads
                    * (b2_join_key_layout / b2_join_write_gather_keyed); never a column type */

#define B2_MAX_COLS   16
#define B2_MAX_TERMS   8
#define B2_MAX_AGGS    8
#define B2_MAX_KEYS    4
#define B2_MAX_GATHER  8
#define B2_MAX_PROG   64
#define B2_TILE     4096   /* rows per selection tile (b2_select_*, b2_join_*) */

/* predicate term operators (b2_term_t.op) */
#define B2_EQ 0
#define B2_NE 1
#define B2_LT 2
#define B2_LE 3
#define B2_GT 4
#define B2_GE 5
#define B2_IS_NULL     6
#define B2_IS_NOT_NULL 7
#define B2_IS_TRUE     8   /* column is a B2_U8 mask: pass iff valid and != 0 */

/* aggregate operators (b2_agg_t.op) */
#define B2_AGG_SUM    0   /* native type: int64 wraps (two's complement) / float64 */
#define B2_AGG_SUMF   1   /* value converted to float64 before adding (AVG over ints) */
#define B2_AGG_MIN    2
#define B2_AGG_MAX    3
#define B2_AGG_COUNT  4   /* only the non-null count is kept (acc may be NULL) */

/* join flags */
#define B2_JOIN_INNER        0
#define B2_JOIN_LEFT         1   /* also emit unmatched probe rows with build index -1 */
#define B2_JOIN_SEMI         2   /* emit each probe row once if it has >= 1 match (build index = -1) */
#define B2_JOIN_ANTI         3   /* emit each probe row once if it has no match */

/* empty-slot sentinel of int64 hash tables (b2_groupby_hash1, b2_star_build_hash) */
#define B2_EMPTY_KEY ((int64_t)0x8000000000000000LL)

typedef struct b2_col {
  const void*    data;    /* int64_t* / double* / uint8_t* */
  const uint8_t* valid;   /* Arrow validity bitmap or NULL */
  int32_t        dtype;   /* B2_I64 / B2_F64 / B2_U8 */
  int32_t        flags;   /* B2_COL_* (0 for ordinary columns) */
} b2_col_t;
/* a B2_U32 key-ordered join payload in which every offset WITHOUT a build row holds 0xFFFFFFFF: the
 * probe learns "no partner" from the payload itself and skips the presence bitmap -- one random L2
 * request per probe row instead of two (the probe kernels are bound by the L2's request rate). */
#define B2_COL_SENTINEL 1

/* one conjunct of a pushed-down predicate:  cols[col] <op> literal */
typedef struct b2_term {
  int32_t col;
  int32_t op;
  int32_t as_f64;   /* compare as float64 (int column value is converted) */
  int32_t pad_;
  int64_t lit_i;
  double  lit_f;
} b2_term_t;

/* a filtered scan of one partition: rows [0,n) of `cols` that satisfy ALL terms.
 * Replaces DaskTableScanPlugin._apply_filters (physical/rel/logical/table_scan.py:80-119)
 * and filter_or_scalar (physical/rel/logical/filter.py:20-45): a NULL predicate is False. */
typedef struct b2_scan {
  b2_col_t  cols[B2_MAX_COLS];
  b2_term_t terms[B2_MAX_TERMS];
  int32_t   ncols;
  int32_t   nterms;
  int64_t   n;
} b2_scan_t;

typedef struct b2_agg {
  int32_t col;   /* input column in scan.cols; -1 = COUNT(*) */
  int32_t op;
} b2_agg_t;

/* per-slot accumulators of a group table (caller-allocated, caller-initialised:
 * SUM/COUNT arrays 0, MIN arrays INT64_MAX, MAX arrays INT64_MIN).
 * float64 MIN/MAX accumulators hold the order-preserving int64 image of the double
 * (see b2_f64_to_ordered in DESIGN.md); b2_ordered_to_f64() converts back. */
typedef struct b2_aggstate {
  void*     acc[B2_MAX_AGGS];   /* int64_t* or double*, [nslots]; NULL = not kept */
  int64_t*  cnt[B2_MAX_AGGS];   /* non-null input count per slot; NULL = not kept */
  int64_t*  rows;               /* rows per slot (COUNT(*)); NULL = not kept */
  uint32_t* present;            /* presence bitmap over slots; NULL = not kept */
  int32_t*  out_slot;           /* int32[n]: slot each input row landed in (-1 = filtered); NULL = not kept.
                                   Turns the group-by kernels into a factorize (pandas groupby's first half). */
} b2_aggstate_t;

/* expression program (postfix) evaluated per row by b2_expr_eval.
 * Replaces the per-operator pandas passes of RexCallPlugin.convert
 * (physical/rex/core/call.py:1158-1216, OPERATION_MAPPING :1047-1062). */
typedef struct b2_instr {
  int32_t op;
  int32_t a;       /* column index for LOAD */
  int64_t imm_i;
  double  imm_f;
} b2_instr_t;

typedef struct b2_prog {
  b2_instr_t code[B2_MAX_PROG];
  int32_t    n;
  int32_t    out_dtype;   /* B2_I64 / B2_F64 / B2_U8 */
} b2_prog_t;

/* b2_instr_t.op */
#define B2_OP_LOAD      0   /* push cols[a] (U8 pushed as int 0/1) */
#define B2_OP_CONST_I   1
#define B2_OP_CONST_F   2
#define B2_OP_CONST_NULL 3
#define B2_OP_I2F       4
#define B2_OP_F2I       5   /* truncate toward zero */
#define B2_OP_ADD_I    10
#define B2_OP_SUB_I    11
#define B2_OP_MUL_I    12
#define B2_OP_DIV_I    13   /* SQL truncated division (call.py:165-189); x/0 -> NULL */
#define B2_OP_NEG_I    14
#define B2_OP_ABS_I    15
#define B2_OP_MOD_I    16
#define B2_OP_ADD_F    20
#define B2_OP_SUB_F    21
#define B2_OP_MUL_F    22
#define B2_OP_DIV_F    23
#define B2_OP_NEG_F    24
#define B2_OP_ABS_F    25
#define B2_OP_SQRT_F   26   /* IEEE sqrt (STDDEV = sqrt(VAR), aggregate.py:200-231) */
#define B2_OP_EQ_I     30   /* 30..35 = EQ NE LT LE GT GE on ints   */
#define B2_OP_EQ_F     40   /* 40..45 = EQ NE LT LE GT GE on doubles (IEEE: NaN != x is true) */
#define B2_OP_AND      50   /* Kleene */
#define B2_OP_OR       51   /* Kleene */
#define B2_OP_NOT      52
#define B2_OP_ISNULL_I 53   /* -> never-null bool */
#define B2_OP_ISNULL_F 54   /* NaN counts as NULL */
#define B2_OP_CASE     55   /* pops else, then, cond: cond true -> then, else (or NULL cond) -> else */
#define B2_OP_FILLNA   56   /* pops fill, x: x if valid else fill */
#define B2_OP_ORD2F    57   /* order-preserving int64 image -> float64 (float MIN/MAX accumulators) */

/* ---- runtime --------------------------------------------------------------------- */
const char* b2_last_error(void);
int32_t b2_version(void);
/* sm count, L2 bytes, compute capability, total HBM bytes of `device` */
int32_t b2_device_info(int32_t device, int32_t* sm_count, int64_t* l2_bytes,
                       int32_t* cc_major, int32_t* cc_minor, int64_t* hbm_bytes);
int32_t b2_d2h(void* host_dst, const void* dev_src, int64_t bytes, void* stream); /* copies then syncs stream */
int32_t b2_sync(void* stream);
/* cudaMemsetAsync on `stream` (re-initialising lookup / table buffers that a prepared query reuses) */
int32_t b2_memset(void* dev_ptr, int32_t byte, int64_t nbytes, void* stream);
/* number of B2_TILE tiles covering n rows */
int64_t b2_num_tiles(int64_t n);

/* ---- ingest ---------------------------------------------------------------------- */
/* Column statistics computed once at Context.create_table (context.py:168-293 keeps only
 * Statistics(row_count)); d_out = int64[6]: {min, max, null_count, n_nan, repeats, sampled};
 * min/max are the raw 64-bit pattern of the column type and cover non-null (non-NaN) values only.
 * repeats / sampled: of `sampled` rows taken as groups of 32 consecutive rows spread over the
 * column, `repeats` share their value with another row of their group -- the skew estimate that
 * selects b2_groupby_dense_grouped.  ws: device scratch of >= b2_stats_ws_bytes() bytes. */
int64_t b2_stats_ws_bytes(void);
int32_t b2_col_stats(const b2_col_t* col, int64_t n, int64_t* d_out, void* ws, void* stream);

/* ---- expressions ----------------------------------------------------------------- */
/* Evaluate `prog` for rows [0,n) of cols; writes out_data (type prog->out_dtype) and, when
 * out_valid != NULL, the Arrow validity bitmap of the result ((n+31)/32 uint32 words). */
int32_t b2_expr_eval(const b2_prog_t* prog, const b2_col_t* cols, int32_t ncols, int64_t n,
                     void* out_data, uint32_t* out_valid, void* stream);

/* ---- filter ---------------------------------------------------------------------- */
/* Global (no GROUP BY) aggregates over a filtered scan, no survivor materialisation.
 * Replaces df[cond] + groupby(<const col>).agg(...) of DaskAggregatePlugin._do_aggregations
 * (physical/rel/logical/aggregate.py:288-375, constant-key trick :305-306,:576).
 * d_out_acc: int64[naggs] raw 64-bit accumulators (int64, or double bits, or ordered-int64
 * for float MIN/MAX); d_out_cnt: int64[naggs] non-null counts.  If `accumulate` != 0 the
 * call combines into the existing outputs (next partition of the same table), otherwise it
 * initialises them.  ws >= b2_scan_agg_ws_bytes(). */
int64_t b2_scan_agg_ws_bytes(void);
int32_t b2_scan_agg(const b2_scan_t* scan, const b2_agg_t* aggs, int32_t naggs,
                    int64_t* d_out_acc, int64_t* d_out_cnt, int32_t accumulate,
                    void* ws, void* stream);

/* Order-preserving selection (df[cond], filter.py:39-40), two passes.
 * b2_select_count: d_tile_off = int64[b2_num_tiles(n)+1]; on return d_tile_off[t] is the
 * number of passing rows before tile t and d_tile_off[ntiles] the total.
 * b2_select_write: writes the passing row ids to out_idx (may be NULL) and, for each of the
 * ngather columns scan.cols[gather_cols[g]], the surviving values to out_data[g] and validity
 * words to out_valid[g] (NULL = not needed; must be zero-initialised by the caller because
 * bits are OR-ed in). */
int32_t b2_select_count(const b2_scan_t* scan, int64_t* d_tile_off, void* stream);
int32_t b2_select_write(const b2_scan_t* scan, const int64_t* d_tile_off, int32_t* out_idx,
                        int32_t ngather, const int32_t* gather_cols, void* const* out_data,
                        uint32_t* const* out_valid, void* stream);

/* out[i] = col[idx[i]] (idx[i] == -1 -> NULL).  The take() at the end of pandas
 * boolean indexing / merge (join.py:241-246).  out_valid: (n_idx+31)/32 words or NULL. */
int32_t b2_gather(const b2_col_t* col, const int32_t* idx, int64_t n_idx,
                  void* out_data, uint32_t* out_valid, void* stream);

/* ---- group-by -------------------------------------------------------------------- */
/* Dense (direct-address) group table: slot = key - kmin for kmin <= key <= kmax, NULL key
 * -> slot nslots-1 (nslots = kmax-kmin+2).  Fused with the scan's predicate.
 * Replaces groupby(by, dropna=False).agg(...) per partition (aggregate.py:575-581). */
int32_t b2_groupby_dense(const b2_scan_t* scan, int32_t key_col, int64_t kmin, int64_t nslots,
                         const b2_agg_t* aggs, int32_t naggs, const b2_aggstate_t* st,
                         void* stream);

/* b2_groupby_dense for keys that REPEAT within a warp (skewed distributions, e.g. Zipf): same
 * arguments and results (float sums up to summation order), but a batch whose rows share slots
 * combines them per warp (match + shuffles, one atomic per distinct slot and 32-row step) and
 * collects slots seen twice in a step in a per-CTA shared-memory table that is flushed with one atomic
 * per accumulator at the end.  The L2 serialises atomics per ADDRESS: without this a key that takes
 * 12 % of the rows costs several times the whole uniform-key query.  nslots < 2^31. */
int32_t b2_groupby_dense_grouped(const b2_scan_t* scan, int32_t key_col, int64_t kmin, int64_t nslots,
                                 const b2_agg_t* aggs, int32_t naggs, const b2_aggstate_t* st,
                                 void* stream);

/* Heavy hitters of a dense group key, by sampling: d_hot = int32[32] receives the slots (key - kmin) that
 * occur most often among ~32k sampled rows of `key` (at least 6 times, i.e. a share above ~0.02 %), most
 * frequent first, padded with -1.  A performance hint for b2_groupby_dense_hot; results never depend on it. */
int32_t b2_hot_slots(const b2_col_t* key, int64_t n, int64_t kmin, int64_t nslots, int32_t* d_hot, void* stream);
/* b2_groupby_dense in which the rows of the listed heavy hitters accumulate in thread-private shared
 * memory partials (SUM / COUNT / COUNT(*) accumulators; no atomics, no cross-lane traffic) that every
 * CTA flushes with one atomic per hitter and accumulator at its end; all other rows take the per-row
 * atomic.  For Zipf-like keys: the few addresses that would otherwise serialise in the L2. */
int32_t b2_groupby_dense_hot(const b2_scan_t* scan, int32_t key_col, int64_t kmin, int64_t nslots,
                             const b2_agg_t* aggs, int32_t naggs, const b2_aggstate_t* st, const int32_t* d_hot,
                             void* stream);

/* Hash group table on ONE 64-bit key (int64, or float64 bits normalised -0.0 -> 0.0).
 * table_keys = int64[cap+2] pre-filled with B2_EMPTY_KEY, cap a power of two; slot cap holds
 * the NULL(/NaN) key group and slot cap+1 the group whose key equals B2_EMPTY_KEY.
 * Accumulator arrays have cap+2 slots.  d_flags = int32[4]: [0] set to 1 if the table
 * overflowed (caller retries with larger cap), [1] NULL-key group present, [2] sentinel-key
 * group present. */
int32_t b2_groupby_hash1(const b2_scan_t* scan, int32_t key_col, int64_t* table_keys,
                         int64_t cap, const b2_agg_t* aggs, int32_t naggs,
                         const b2_aggstate_t* st, int32_t* d_flags, void* stream);

/* Hash group table on 1..B2_MAX_KEYS key columns of any type (NULL keys group together).
 * table_keys = int64[nkeys*cap] key bit patterns, key k of slot h at [k*cap+h], table_nulls = uint8[cap] per-slot key-null
 * mask, table_state = int32[cap] zero-initialised (0 empty, 1 being written, 2 ready). */
int32_t b2_groupby_hashk(const b2_scan_t* scan, const int32_t* key_cols, int32_t nkeys,
                         int64_t* table_keys, uint8_t* table_nulls, int32_t* table_state,
                         int64_t cap, const b2_agg_t* aggs, int32_t naggs,
                         const b2_aggstate_t* st, int32_t* d_flags, void* stream);

/* dst |= src over nwords 32-bit words: merges the presence bitmaps of per-GPU dense group tables
 * after an all-gather (NCCL has no bitwise reduction). */
int32_t b2_bitmap_or(uint32_t* dst, const uint32_t* src, int64_t nwords, void* stream);

/* ---- multi-GPU merge of dense partial tables over NVLink peer memory ----------------------
 * Replaces dask's tree reduction of per-partition partial aggregates (aggregate.py:575-581,
 * `groupby(...).agg(..., split_every)`; tests/integration/test_groupby.py:526-598) for
 * direct-address tables, with split_out = world size: ONE kernel per GPU does the cross-GPU
 * barrier, the reduction of this rank's slot range over all peers' tables (read through peer
 * mappings of a symmetric allocation), and the merge of group existence.
 *
 * Every rank holds the same layout inside a buffer that all ranks have mapped: peer_base[p] is
 * rank p's buffer as seen from THIS process.  array_off[a] = byte offset of 8-byte-per-slot array
 * a, bitmap_off = offset of the presence bitmap (LSB order), signal_off = offset of
 * uint64[B2_MAX_PEERS] zero-initialised signal words used by the in-kernel barrier.  epoch must
 * increase by one per call on all ranks (same sequence everywhere); local_ready is a zero-
 * initialised uint64 in this GPU's memory.  out[a] receives count merged elements (slots
 * [lo, lo+count) of the table), out_present one byte per slot (1 = some rank saw the group).
 * Arrays are combined in rank order 0..world-1 (bit-reproducible float sums).
 * The caller double-buffers the tables: the table of call k may be rewritten once call k+1 has
 * been enqueued on this rank's stream. */
#define B2_MAX_PEERS        16
#define B2_PEER_MAX_ARRAYS  (2 * B2_MAX_AGGS + 1)
#define B2_PEER_SUM_F64 0
#define B2_PEER_SUM_I64 1   /* wraps (two's complement), like the single-GPU accumulators */
#define B2_PEER_MIN_I64 2   /* MIN / MAX accumulators hold int64 values or ordered images of doubles */
#define B2_PEER_MAX_I64 3
#define B2_PEER_PRESENT_ROWS      1   /* group exists iff merged array[presence_array] > 0 */
#define B2_PEER_PRESENT_INDICATOR 2   /* ... iff some rank's array[presence_array] bits != B2_EMPTY_KEY (-0.0) */
#define B2_PEER_PRESENT_BITMAP    3   /* ... iff some rank's bitmap bit is set */
typedef struct b2_peer_merge {
  int32_t   world, rank;
  int32_t   narrays;
  int32_t   presence_kind, presence_array;
  int32_t   ops[B2_PEER_MAX_ARRAYS];
  int64_t   array_off[B2_PEER_MAX_ARRAYS];
  int64_t   bitmap_off;
  int64_t   signal_off;
  void*     peer_base[B2_MAX_PEERS];
  void*     out[B2_PEER_MAX_ARRAYS];
  uint8_t*  out_present;
  int64_t   lo, count;                /* multiples of 32 */
  uint64_t* local_ready;
  uint64_t  epoch;
} b2_peer_merge_t;
int32_t b2_peer_merge(const b2_peer_merge_t* m, void* stream);

/* bit-exact order-preserving double<->int64 images used by float MIN/MAX accumulators */
int64_t b2_f64_to_ordered(double x);
double  b2_ordered_to_f64(int64_t k);

/* ---- hash join ------------------------------------------------------------------- */
/* Chained hash table over the build side's key columns: head = int32[cap] pre-filled with
 * -1 (cap a power of two), next = int32[n].  Rows with a NULL/NaN key are skipped
 * (join.py:202-213).  Replaces the factorize half of pandas.merge (join.py:241-246). */
int32_t b2_join_build(const b2_col_t* keys, int32_t nkeys, int64_t n,
                      int32_t* head, int32_t* next, int64_t cap, void* stream);

/* Direct-address table for a single int64 key: lookup = int32[range] pre-filled with -1,
 * lookup[key-kmin] = row.  d_flags[0] is set to 1 if two rows share a key (caller falls
 * back to b2_join_build). */
int32_t b2_join_build_dense(const b2_col_t* key, int64_t n, int64_t kmin, int64_t range,
                            int32_t* lookup, int32_t* d_flags, void* stream);

typedef struct b2_jointable {
  b2_col_t  keys[B2_MAX_KEYS];  /* build-side key columns */
  int32_t   nkeys;
  int32_t   dense;              /* 0 = chained (head/next/cap), 1 = direct (lookup/kmin/range),
                                 * 2 = key-ordered: lookup is the presence BITMAP (uint32 words,
                                 *     range bits) and the build row of a match is key-kmin */
  const int32_t* head;
  const int32_t* next;
  int64_t   cap;
  const int32_t* lookup;
  int64_t   kmin;
  int64_t   range;
} b2_jointable_t;

/* Probe with the rows of `scan` that pass its terms; probe_keys index scan.cols.
 * Same two-pass protocol as b2_select_*: count fills d_tile_off (int64[ntiles+1], exclusive
 * scan, total last), write emits (probe row, build row) pairs in probe-row order.
 * mode = B2_JOIN_*.  build_matched (uint8[n_build], may be NULL) is set to 1 for every build
 * row that found a partner (RIGHT / FULL joins, join.py:41-48). */
int32_t b2_join_count(const b2_scan_t* scan, const int32_t* probe_keys, const b2_jointable_t* jt,
                      int32_t mode, int64_t* d_tile_off, void* stream);
int32_t b2_join_write(const b2_scan_t* scan, const int32_t* probe_keys, const b2_jointable_t* jt,
                      int32_t mode, const int64_t* d_tile_off, int32_t* out_probe_idx,
                      int32_t* out_build_idx, uint8_t* build_matched, void* stream);

/* b2_join_write that also gathers output columns in the same pass (the take() on every column of
 * both sides that ends pandas.merge, join.py:241-246): for each emitted pair, probe columns
 * scan.cols[probe_cols[k]] are copied to probe_out[k] and build-side columns build_cols[k] (indexed
 * by the build row, NULL for an unmatched LEFT row) to build_out[k].  *_valid[k]: validity words of
 * the output (zero-initialised by the caller, bits are OR-ed in) or NULL.  out_probe_idx /
 * out_build_idx may be NULL when the caller only wants the gathered columns. */
int32_t b2_join_write_gather(const b2_scan_t* scan, const int32_t* probe_keys, const b2_jointable_t* jt,
                             int32_t mode, const int64_t* d_tile_off, int32_t* out_probe_idx,
                             int32_t* out_build_idx, uint8_t* build_matched, int32_t nprobe,
                             const int32_t* probe_cols, void* const* probe_out, uint32_t* const* probe_valid,
                             int32_t nbuild, const b2_col_t* build_cols, void* const* build_out,
                             uint32_t* const* build_valid, void* stream);

/* Key-ordered layout for a unique dense-key build side (the broadcast dimension of C3): the probe's
 * "take" on a build column (join.py:241-246) then costs ONE random access at the key offset instead
 * of lookup[key] -> row -> col[row], and int64 payloads whose value range fits 32 bits are stored as
 * uint32 offsets so the whole payload array stays L2-resident.
 *   out_data[key[i]-kmin] = col[i]           out_dtype == col->dtype  (8 or 1 bytes per key)
 *   out_data[key[i]-kmin] = col[i] - base    out_dtype == B2_U32      (col int64, 4 bytes per key)
 * out_valid (may be NULL): validity words in key order, zero-initialised by the caller.
 * present (may be NULL): bit key-kmin is set for every build row; it is the `lookup` of a
 * b2_jointable_t with dense == 2.  col may be NULL to produce only `present`.  Rows with a NULL key
 * or a key outside [kmin, kmin+range) are skipped.  Unique keys are the caller's responsibility
 * (b2_join_build_dense reports duplicates). */
int32_t b2_join_key_layout(const b2_col_t* key, int64_t n, int64_t kmin, int64_t range, const b2_col_t* col,
                           int32_t out_dtype, int64_t base, void* out_data, uint32_t* out_valid,
                           uint32_t* present, void* stream);
/* b2_join_write_gather for build columns in key order: build_cols[k].dtype may be B2_U32 with
 * build_base[k] the base of the offsets (build_base may be NULL when no column is narrowed). */
int32_t b2_join_write_gather_keyed(const b2_scan_t* scan, const int32_t* probe_keys, const b2_jointable_t* jt,
                                   int32_t mode, const int64_t* d_tile_off, int32_t* out_probe_idx,
                                   int32_t* out_build_idx, uint8_t* build_matched, int32_t nprobe,
                                   const int32_t* probe_cols, void* const* probe_out,
                                   uint32_t* const* probe_valid, int32_t nbuild, const b2_col_t* build_cols,
                                   const int64_t* build_base, void* const* build_out,
                                   uint32_t* const* build_valid, void* stream);

/* Probe of a direct-address table (jt->dense 1 or 2; every probe row emits at most one output row in
 * all four modes) WITHOUT a host round trip: outputs are caller-allocated at their upper bound
 * (scan.n rows) and filled in probe-row order, the row count stays on the device.
 *   lookback == 0: count (key + presence only) -> scan -> write, three launches on `stream`;
 *   lookback != 0: one launch; each 2048-row tile learns its offset by a decoupled look-back over
 *                  the tiles before it (reads every input byte exactly once).
 * The write kernel front-loads its loads (key + first probe column, then presence word + the first
 * key-ordered payload speculatively), i.e. two dependent memory round trips per tile.
 * d_ws: b2_join_onepass_ws_bytes(n) bytes, ZEROED by the caller; its first int64 receives the number
 * of rows emitted.  Gather arguments as for b2_join_write_gather_keyed. */
int64_t b2_join_onepass_ws_bytes(int64_t n);
int32_t b2_join_onepass(const b2_scan_t* scan, const int32_t* probe_keys, const b2_jointable_t* jt, int32_t mode,
                        int32_t lookback, void* d_ws, int32_t nprobe, const int32_t* probe_cols,
                        void* const* probe_out, uint32_t* const* probe_valid, int32_t nbuild,
                        const b2_col_t* build_cols, const int64_t* build_base, void* const* build_out,
                        uint32_t* const* build_valid, void* stream);

/* ---- inner join fused with GLOBAL aggregates over both sides (C3, non-materialising) ---------- */
/* One pass over the probe partition: predicate -> presence + payload lookup at the key offset ->
 * combine -> aggregate; no join row is materialised.  Replaces, fused, join.py:189-248 (merge:
 * factorize + indexers + take of every column) followed by the constant-key global aggregate of
 * aggregate.py:305-306,576 for plans  Aggregate(no GROUP BY) <- Inner Join(fk = unique dense pk)
 * whose aggregate inputs are  P,  B,  P*B,  P+B,  P-B  or  B-P  with P a probe-side and B a
 * build-side column (single-sided sub-expressions are evaluated into columns first).
 * jt must be the key-ordered layout (dense == 2, b2_join_key_layout); build_cols[b] are its payload
 * columns in key order (B2_I64 / B2_F64, or B2_U32 with build_base[b]).  Arithmetic is float64 as soon
 * as one side is float64 (the int side is converted, like pandas' upcast), else wrapping int64.
 * A row contributes to an aggregate iff it finds a build row and neither input is NULL/NaN.
 * Outputs as for b2_scan_agg (raw 64-bit accumulators + non-null counts, `accumulate` to combine
 * partitions); an aggregate with combine == B2_JA_ROWS only counts the join's rows.
 * ws >= b2_scan_agg_ws_bytes(). */
#define B2_JA_MAX_BUILD 4
#define B2_JA_P     0   /* value = P                */
#define B2_JA_B     1   /* value = B                */
#define B2_JA_MUL   2   /* value = P * B            */
#define B2_JA_ADD   3   /* value = P + B            */
#define B2_JA_SUB   4   /* value = P - B            */
#define B2_JA_RSUB  5   /* value = B - P            */
#define B2_JA_ROWS  6   /* COUNT(*) of the join     */
typedef struct b2_joinagg {
  int32_t pcol;      /* probe input: index into scan.cols, or -1 */
  int32_t bcol;      /* build input: index into build_cols, or -1 */
  int32_t combine;   /* B2_JA_* */
  int32_t op;        /* B2_AGG_* applied to the combined value */
} b2_joinagg_t;
int32_t b2_join_agg(const b2_scan_t* scan, int32_t probe_key, const b2_jointable_t* jt, int32_t nbuild,
                    const b2_col_t* build_cols, const int64_t* build_base, const b2_joinagg_t* aggs, int32_t naggs,
                    int64_t* d_out_acc, int64_t* d_out_cnt, int32_t accumulate, void* ws, void* stream);

/* ---- group tables far beyond L2 (C5: 100M keys) ----------------------------------------------- */
/* Reorder the rows of `scan` that pass its terms by key RANGE, so that b2_groupby_dense over the
 * reordered arrays touches one L2-sized slice of the group table after the other (instead of a random
 * DRAM read-modify-write per row).  bucket = slot >> shift with slot = key - kmin (NULL key ->
 * nslots-1, the NULL slot of b2_groupby_dense), nbuckets <= 1024 and > (nslots-1) >> shift.
 *   out_key[i]      = kmin + slot   (int64, no bitmap: run the consumer with nslots+1 slots)
 *   out_cols[c][i]  = scan.cols[carry_cols[c]] of the same row (8-byte columns without bitmap)
 * All outputs are caller-allocated with scan.n rows; rows past the number of passing rows are left
 * untouched (pre-fill out_key with an out-of-range key, e.g. kmin + nslots + 1, so the consumer
 * ignores them).  d_ws: b2_range_partition_ws_bytes(nbuckets) bytes, ZEROED; afterwards
 * ws[0..nbuckets] are the bucket starts (ws[nbuckets] = rows written).  No host round trip.
 * Replaces nothing in the reference (pandas' groupby hashes in place); it is what makes
 * aggregate.py:522-589 on 100M groups stream instead of thrash. */
/* b2_groupby_dense for input that b2_range_partition has ordered by key range: 2048-row tiles are
 * handed to the CTAs in order through *d_ticket (device uint64, ZEROED by the caller), so the rows in
 * flight always form one contiguous window and touch one slice of the table at a time. */
int32_t b2_groupby_dense_ordered(const b2_scan_t* scan, int32_t key_col, int64_t kmin, int64_t nslots,
                                 const b2_agg_t* aggs, int32_t naggs, const b2_aggstate_t* st, uint64_t* d_ticket,
                                 void* stream);
int64_t b2_range_partition_ws_bytes(int32_t nbuckets);
/* The three phases separately, so that SEVERAL input partitions can be reordered into ONE output (the
 * dask-style partitions of a table would otherwise each revisit every slice of the group table):
 * _hist per input (accumulates into ws), _scan once, _scatter per input into the shared outputs (sized
 * for the sum of the inputs' rows).  b2_range_partition = the three on one input. */
int32_t b2_range_partition_hist(const b2_scan_t* scan, int32_t key_col, int64_t kmin, int64_t nslots, int32_t shift,
                                int32_t nbuckets, void* d_ws, void* stream);
int32_t b2_range_partition_scan(int32_t nbuckets, void* d_ws, void* stream);
int32_t b2_range_partition_scatter(const b2_scan_t* scan, int32_t key_col, int64_t kmin, int64_t nslots, int32_t shift,
                                   int32_t nbuckets, int32_t ncarry, const int32_t* carry_cols, int64_t* out_key,
                                   void* const* out_cols, void* d_ws, void* stream);
int32_t b2_range_partition(const b2_scan_t* scan, int32_t key_col, int64_t kmin, int64_t nslots, int32_t shift,
                           int32_t nbuckets, int32_t ncarry, const int32_t* carry_cols, int64_t* out_key,
                           void* const* out_cols, void* d_ws, void* stream);

/* ---- ORDER BY ("next" row of the scope: the tail of TPC-H Q3) ------------------------------- */
/* Stable LSD radix sort of row ids by one key column.  idx = int32[n] permutation (b2_iota for the
 * identity) reordered in place so that col[idx[i]] is sorted (descending != 0: DESC; nulls_first
 * != 0: NULL/NaN rows first).  Multi-key ORDER BY: call once per key from the LAST key to the FIRST.
 * Replaces sort_values / nsmallest of physical/utils/sort.py:9-140.  ws >= b2_sort_ws_bytes(n). */
int64_t b2_sort_ws_bytes(int64_t n);
int32_t b2_iota(int32_t* out, int64_t n, void* stream);
int32_t b2_sort_by(const b2_col_t* col, int64_t n, int32_t descending, int32_t nulls_first, int32_t* idx,
                   void* ws, void* stream);

/* ---- fused filter -> join -> group-by (star pipeline) ----------------------------- */
/* out_slot[i] = key[i]-kmin (NULL key -> null_slot) as int32: turns a dense group-key column of
 * the build side into group-table slot numbers. */
int32_t b2_dense_slots(const b2_col_t* key, int64_t n, int64_t kmin, int32_t null_slot,
                       int32_t* out_slot, void* stream);

/* Build the join->group lookup of the fused pipeline from the (already filtered) build side:
 * for build row r = sel ? sel[i] : i, lookup[pk[r]-kmin] = slot_of_row[i].  Dense variant;
 * d_flags[0] = 1 on duplicate pk. */
int32_t b2_star_build_dense(const b2_col_t* pk, const int32_t* sel, int64_t n_sel,
                            const int32_t* slot_of_row, int64_t kmin, int64_t range,
                            int32_t* lookup, int32_t* d_flags, void* stream);
/* The same lookup straight from the UNFILTERED build partition when join key and group key are both
 * dense int64: rows of `scan` passing its terms write lookup[pk-pk_min] = grp-grp_min (NULL grp ->
 * null_slot, NULL pk skipped).  Fuses table_scan.py:80-119 (dim filter) into the build; nothing is
 * materialised.  Call once per build partition; d_flags[0] = 1 on duplicate pk. */
int32_t b2_star_build_scan(const b2_scan_t* scan, int32_t pk_col, int32_t grp_col, int64_t pk_min,
                           int64_t pk_range, int64_t grp_min, int32_t null_slot, int32_t* lookup,
                           int32_t* d_flags, void* stream);
/* Hash variant: table_keys = int64[cap] pre-filled with B2_EMPTY_KEY, table_slots = int32[cap].
 * d_flags[0] = 1 on duplicate pk, d_flags[1] = 1 on overflow. */
int32_t b2_star_build_hash(const b2_col_t* pk, const int32_t* sel, int64_t n_sel,
                           const int32_t* slot_of_row, int64_t* table_keys, int32_t* table_slots,
                           int64_t cap, int32_t* d_flags, void* stream);

typedef struct b2_starlookup {
  int32_t dense;
  int32_t pad_;
  const int32_t* lookup;   /* dense: int32[range], -1 = no partner */
  int64_t kmin;
  int64_t range;
  const int64_t* table_keys;  /* hash */
  const int32_t* table_slots;
  int64_t cap;
} b2_starlookup_t;

/* One pass over the probe (fact) partition: predicate -> key lookup -> aggregate into the
 * group slot of the matching build row.  Replaces, fused, table_scan.py:80-119 +
 * join.py:189-248 + aggregate.py:522-589 for plans of the shape
 *   Aggregate(group by build cols; aggs over probe cols) <- Inner Join(fk = unique pk). */
int32_t b2_star_agg(const b2_scan_t* scan, int32_t fk_col, const b2_starlookup_t* lk,
                    const b2_agg_t* aggs, int32_t naggs, const b2_aggstate_t* st, void* stream);

/* ---- window functions: f(...) OVER (PARTITION BY ... ORDER BY ... ROWS|RANGE ...) ---------------
 * Replaces the reference's per-partition pandas pass of DaskWindowPlugin
 * (dask_sql/physical/rel/logical/window.py:145-198, map_on_each_group: sort, then expanding() /
 * rolling(Indexer) per group; and :330-332, groupby(partition keys).apply(...)).  All entry points
 * work on columns already sorted by (partition keys, order keys) -- b2_iota + b2_sort_by per key,
 * then b2_gather -- so a partition and a peer group (rows with equal ORDER BY values) are each a
 * contiguous row range.  Row ranges are int32: the input holds < 2^31 rows. */
#define B2_WIN_MAX_KEYS 8

/* per-row segment arrays (int32[n] each, caller-allocated): [part_start, part_end) is the row's
 * partition, [peer_start, peer_end) its peer group, dense[i] the number of peer-group starts in
 * rows 0..i (DENSE_RANK helper). */
typedef struct b2_wsegs {
  int32_t* part_start;
  int32_t* part_end;
  int32_t* peer_start;
  int32_t* peer_end;
  int32_t* dense;
} b2_wsegs_t;

/* window frame.  kind B2_WB_UNBOUNDED: UNBOUNDED PRECEDING (lower bound) / UNBOUNDED FOLLOWING
 * (upper bound).  kind B2_WB_OFFSET: a row offset from the current row, -a = a PRECEDING,
 * 0 = CURRENT ROW, +b = b FOLLOWING.  range != 0: RANGE frame, whose B2_WB_OFFSET bounds must be 0
 * and mean the first / last peer of the current row. */
#define B2_WB_UNBOUNDED 0
#define B2_WB_OFFSET    1
typedef struct b2_wframe {
  int32_t range;
  int32_t lo_kind;
  int32_t hi_kind;
  int32_t pad_;
  int64_t lo;
  int64_t hi;
} b2_wframe_t;

/* window functions (b2_window_rank / b2_window_agg op) */
#define B2_WIN_ROW_NUMBER  0
#define B2_WIN_RANK        1
#define B2_WIN_DENSE_RANK  2
#define B2_WIN_SUM         3   /* int64 (wrapping) for B2_I64 input, float64 for B2_F64 */
#define B2_WIN_COUNT       4   /* non-NULL values; val->data == NULL: COUNT(*) */
#define B2_WIN_AVG         5   /* float64 */
#define B2_WIN_MIN         6
#define B2_WIN_MAX         7
#define B2_WIN_FIRST       8   /* value at the frame's first row (NULL if that value is NULL) */
#define B2_WIN_LAST        9

/* device scratch of b2_window_segments / b2_window_agg for n rows */
int64_t b2_window_ws_bytes(int64_t n);

/* keys[0..npart) = partition keys, keys[npart..nkeys) = order keys, all gathered into sorted order.
 * NULL equals NULL, NaN is NULL, -0.0 equals 0.0 (the conventions of b2_sort_by's key image).
 * Starts: one pass with a decoupled look-back of the tile carries; ends: scattered at each
 * segment's last row and gathered.  Every array of `segs` is written. */
int32_t b2_window_segments(const b2_col_t* keys, int32_t npart, int32_t nkeys, int64_t n, const b2_wsegs_t* segs,
                           void* ws, void* stream);

/* ROW_NUMBER / RANK / DENSE_RANK -> int64[n] (window.py:187-190 computes ROW_NUMBER as range(1, len+1)) */
int32_t b2_window_rank(int32_t op, int64_t n, const b2_wsegs_t* segs, int64_t* out, void* stream);

/* LAG (offset = -k) / LEAD (offset = +k): out[i] = val[i + offset] when that row is in i's partition,
 * else the default (has_default: default_raw, the value's 64-bit pattern; else NULL).  val: B2_I64 or
 * B2_F64; out has val's type; out_valid: (n+31)/32 words. */
int32_t b2_window_offset(const b2_col_t* val, int64_t n, int64_t offset, int32_t has_default, int64_t default_raw,
                         const b2_wsegs_t* segs, void* out, uint32_t* out_valid, void* stream);

/* Framed aggregate (window.py:161-192: expanding() / rolling() per group).  val: B2_I64 or B2_F64.
 * Lower bound UNBOUNDED: segmented inclusive scan read at the frame end; upper bound UNBOUNDED: reverse
 * scan read at the frame start; both bounded: evaluated over the frame (int64 SUM / COUNT over frames
 * wider than 32 rows: difference of the exact wrapping prefix sums).  Float scans combine tile carries
 * in a fixed order, so results are bit-identical from run to run.  Empty frame or no non-NULL value:
 * NULL (COUNT: 0).  out: int64 (COUNT, int SUM/MIN/MAX/FIRST/LAST) or float64 (AVG, float input);
 * out_valid: (n+31)/32 words or NULL for COUNT.  ws >= b2_window_ws_bytes(n). */
int32_t b2_window_agg(const b2_col_t* val, int32_t op, const b2_wframe_t* frame, int64_t n, const b2_wsegs_t* segs,
                      void* out, uint32_t* out_valid, void* ws, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200SQL_H */
