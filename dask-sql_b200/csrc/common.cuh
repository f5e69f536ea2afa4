// common.cuh — shared device helpers for libb200sql (sm_100a).
// Everything here is hand-written CUDA; no CUB/Thrust/cuDF.
//
// Design rule learnt from the first ncu capture (profiles/r01_first_capture.md): these kernels
// are HBM-bound only if the per-row instruction count stays small.  All run-time dispatch
// (operator, column type, nullable or not) therefore happens ONCE PER BATCH of R rows per lane
// (`switch` outside), and the unrolled per-row loops inside are template instances with
// compile-time operator/type and immediate-offset addressing.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "b200sql.h"

#define B2_BLOCK 256
#define B2_WARPS (B2_BLOCK / 32)
#define FULL_MASK 0xffffffffu

// ---------------------------------------------------------------------------------------
// host-side error plumbing
// ---------------------------------------------------------------------------------------
extern thread_local char g_b2_err[512];
static inline int32_t b2_fail(int32_t code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_b2_err, sizeof(g_b2_err), fmt, ap);
  va_end(ap);
  return code;
}
#define B2_CUDA_TRY(expr)                                                              \
  do {                                                                                 \
    cudaError_t e__ = (expr);                                                          \
    if (e__ != cudaSuccess)                                                            \
      return b2_fail(B2_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                     __FILE__, __LINE__);                                              \
  } while (0)
#define B2_CHECK_LAUNCH(name)                                                          \
  do {                                                                                 \
    cudaError_t e__ = cudaGetLastError();                                              \
    if (e__ != cudaSuccess)                                                            \
      return b2_fail(B2_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e__)); \
  } while (0)
#define B2_REQUIRE(cond, msg)                                                          \
  do {                                                                                 \
    if (!(cond)) return b2_fail(B2_ERR_ARG, "%s: %s", __func__, msg);                  \
  } while (0)

// persistent grid: one resident wave of CTAs (sm_count x occupancy), rows are grid-strided.
int b2_sm_count();
template <class K>
static inline int b2_wave_grid(K kernel, int block, int64_t work_items_blocks) {
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, block, 0);
  if (occ < 1) occ = 1;
  int64_t g = (int64_t)b2_sm_count() * occ;
  if (g > work_items_blocks) g = work_items_blocks;
  if (g < 1) g = 1;
  return (int)g;
}

// ---------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t b2_mix64(uint64_t k) {  // murmur3 fmix64
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdULL;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ULL;
  k ^= k >> 33;
  return k;
}

// ---- decoupled look-back (single-pass order-preserving compaction) -------------------------------
// status[tile]: bits 63..62 = 0 not ready / 1 tile aggregate / 2 inclusive prefix, low 62 bits = value.
// Called by the 32 lanes of one warp once the tile's own count `agg` is known; publishes it, sums the
// predecessors' aggregates back to the nearest inclusive prefix and returns the tile's exclusive
// prefix.  Only the 64-bit status word is exchanged, so relaxed volatile accesses suffice.  Progress:
// the grid is resident (b2_wave_grid) and every block takes its tiles in increasing order, so the
// lowest unfinished tile never waits.
#define B2_LB_AGG (1ULL << 62)
#define B2_LB_PREFIX (2ULL << 62)
#define B2_LB_MASK ((1ULL << 62) - 1)
__device__ __forceinline__ uint64_t b2_ld_volatile_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void b2_st_volatile_u64(uint64_t* p, uint64_t v) {
  asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// The combining operator is a template parameter: commutative and associative over non-negative
// values below 2^62, with identity 0 (sum of counts; max of row positions, window.cuh).
struct b2_lb_sum {
  static __device__ __forceinline__ int64_t op(int64_t a, int64_t b) { return a + b; }
};
struct b2_lb_max {
  static __device__ __forceinline__ int64_t op(int64_t a, int64_t b) { return a > b ? a : b; }
};
template <class OP>
__device__ __forceinline__ int64_t b2_lookback_op(uint64_t* __restrict__ status, int64_t tile, int64_t agg, int lane) {
  if (tile == 0) {
    if (lane == 0) b2_st_volatile_u64(status, B2_LB_PREFIX | (uint64_t)agg);
    return 0;
  }
  if (lane == 0) b2_st_volatile_u64(status + tile, B2_LB_AGG | (uint64_t)agg);
  int64_t excl = 0;
  for (int64_t t = tile - 1;; t -= 32) {
    const int64_t idx = t - lane;                       // lane 0 = nearest predecessor
    uint64_t v = B2_LB_PREFIX;                          // before tile 0: prefix 0
    if (idx >= 0) {
      do { v = b2_ld_volatile_u64(status + idx); } while ((v >> 62) == 0);
    }
    const uint32_t pmask = __ballot_sync(FULL_MASK, (v >> 62) == 2);
    const int first = pmask ? __ffs(pmask) - 1 : 31;    // nearest lane holding an inclusive prefix
    int64_t val = lane <= first ? (int64_t)(v & B2_LB_MASK) : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) val = OP::op(val, __shfl_xor_sync(FULL_MASK, val, o));
    excl = OP::op(excl, val);
    if (pmask) break;
  }
  if (lane == 0) b2_st_volatile_u64(status + tile, B2_LB_PREFIX | (uint64_t)OP::op(excl, agg));
  return excl;
}
__device__ __forceinline__ int64_t b2_lookback(uint64_t* __restrict__ status, int64_t tile, int64_t agg, int lane) {
  return b2_lookback_op<b2_lb_sum>(status, tile, agg, lane);
}

__device__ __forceinline__ bool b2_bit(const uint8_t* __restrict__ bm, int64_t i) {
  return (bm[i >> 3] >> (i & 7)) & 1;
}

// L2 eviction policies (createpolicy; plain ld only takes .L2::evict_* on 256-bit vectors).
// Non-volatile asm without inputs: the compiler hoists/CSEs it, one instruction per kernel.
__device__ __forceinline__ uint64_t b2_policy_stream() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t b2_policy_keep() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// streaming 8-byte load: read-only path, first-out of L2 so that the L2-resident lookup / group
// tables survive the scan.  (L1 allocation is left on: a column that is both a predicate and an
// aggregate input is re-read a few instructions later and should hit L1.)
__device__ __forceinline__ int64_t b2_ld_stream(const int64_t* p) {
  int64_t v;
  asm("ld.global.nc.L2::cache_hint.b64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(b2_policy_stream()));
  return v;
}
// table load that should stay in L2
__device__ __forceinline__ int32_t b2_ld_keep_i32(const int32_t* p) {
  int32_t v;
  asm("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(b2_policy_keep()));
  return v;
}
// streaming stores: result columns are written once and not read again by the kernel, so they must
// not push the randomly accessed tables (evict_last) out of L2
__device__ __forceinline__ void b2_st_stream(int64_t* p, int64_t v) {
  asm volatile("st.global.L2::cache_hint.b64 [%0], %1, %2;" ::"l"(p), "l"(v), "l"(b2_policy_stream()) : "memory");
}
__device__ __forceinline__ int64_t b2_ld_keep_i64(const int64_t* p) {
  int64_t v;
  asm("ld.global.nc.L2::cache_hint.b64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(b2_policy_keep()));
  return v;
}
__device__ __forceinline__ int64_t b2_ld_cg_i64(const int64_t* p) {
  return __ldcg(reinterpret_cast<const long long*>(p));
}

__host__ __device__ __forceinline__ int64_t b2_ordered_from_bits(int64_t b) {
  return b ^ ((b >> 63) & 0x7fffffffffffffffLL);
}

// run-time comparators: used only by the per-row interpreter (expr.cuh), never in scan loops
__device__ __forceinline__ bool b2_cmp_i(int op, int64_t a, int64_t b) {
  switch (op) {
    case B2_EQ: return a == b;
    case B2_NE: return a != b;
    case B2_LT: return a < b;
    case B2_LE: return a <= b;
    case B2_GT: return a > b;
    default: return a >= b;
  }
}
__device__ __forceinline__ bool b2_cmp_f(int op, double a, double b) {
  switch (op) {
    case B2_EQ: return a == b;
    case B2_NE: return a != b;   // IEEE: true when either is NaN (numpy semantics)
    case B2_LT: return a < b;
    case B2_LE: return a <= b;
    case B2_GT: return a > b;
    default: return a >= b;
  }
}
// compile-time comparators for the scan loops
template <int OP, class T>
__device__ __forceinline__ bool b2_cmp_t(T a, T b) {
  if (OP == B2_EQ) return a == b;
  if (OP == B2_NE) return a != b;
  if (OP == B2_LT) return a < b;
  if (OP == B2_LE) return a <= b;
  if (OP == B2_GT) return a > b;
  return a >= b;
}

// raw 64-bit load of any column type (U8 widened to 0/1); per-row helper for non-hot paths
__device__ __forceinline__ int64_t b2_load_raw(const b2_col_t& c, int64_t row) {
  if (c.dtype == B2_U8) return (int64_t) reinterpret_cast<const uint8_t*>(c.data)[row];
  return b2_ld_stream(reinterpret_cast<const int64_t*>(c.data) + row);
}
// NULL test in the pandas sense: bitmap bit clear, or NaN in a float column
__device__ __forceinline__ bool b2_is_null(const b2_col_t& c, int64_t row, int64_t raw) {
  if (c.valid && !b2_bit(c.valid, row)) return true;
  if (c.dtype == B2_F64) { double d = __longlong_as_double(raw); return d != d; }
  return false;
}

// ---------------------------------------------------------------------------------------
// batch helpers.  A "batch" is R rows of one lane: rows row0 + 32*j, j < R.  `bits` has bit j
// set for the rows that are (still) live.  When the whole warp batch is in bounds (`full`),
// loads are unconditional with immediate offsets.
// ---------------------------------------------------------------------------------------
template <int R>
__device__ __forceinline__ uint32_t b2_bounds_bits(int64_t row0, int64_t n, bool& full) {
  full = row0 + (int64_t)(R - 1) * 32 < n;   // lane-local; callers use it only for load predication
  if (full) return (R == 32) ? 0xffffffffu : ((1u << R) - 1u);
  uint32_t bits = 0;
#pragma unroll
  for (int j = 0; j < R; ++j)
    if (row0 + (int64_t)j * 32 < n) bits |= 1u << j;
  return bits;
}

// load R raw 64-bit values of a 64-bit column
template <int R>
__device__ __forceinline__ void b2_load_batch64(const void* data, int64_t row0, uint32_t bits, bool full,
                                                int64_t (&raw)[R]) {
  const int64_t* p = reinterpret_cast<const int64_t*>(data) + row0;
  if (full) {
#pragma unroll
    for (int j = 0; j < R; ++j) raw[j] = b2_ld_stream(p + j * 32);
  } else {
#pragma unroll
    for (int j = 0; j < R; ++j) raw[j] = (bits >> j) & 1 ? b2_ld_stream(p + j * 32) : 0;
  }
}
template <int R>
__device__ __forceinline__ void b2_load_batch8(const void* data, int64_t row0, uint32_t bits, bool full,
                                               int64_t (&raw)[R]) {
  const uint8_t* p = reinterpret_cast<const uint8_t*>(data) + row0;
#pragma unroll
  for (int j = 0; j < R; ++j) raw[j] = (full || ((bits >> j) & 1)) ? (int64_t)p[j * 32] : 0;
}
template <int R>
__device__ __forceinline__ void b2_load_batch(const b2_col_t& c, int64_t row0, uint32_t bits, bool full,
                                              int64_t (&raw)[R]) {
  if (c.dtype == B2_U8) b2_load_batch8<R>(c.data, row0, bits, full, raw);
  else b2_load_batch64<R>(c.data, row0, bits, full, raw);
}

// validity bits of the batch (bit j = row j valid).  Bitmap bytes: row0+32j -> byte (row0>>3)+4j
template <int R>
__device__ __forceinline__ uint32_t b2_valid_bits(const uint8_t* __restrict__ valid, int64_t row0, uint32_t bits) {
  const uint8_t* p = valid + (row0 >> 3);
  const int sh = (int)(row0 & 7);
  uint32_t v = 0;
#pragma unroll
  for (int j = 0; j < R; ++j)
    if ((bits >> j) & 1) v |= (uint32_t)((p[j * 4] >> sh) & 1) << j;
  return v;
}
// NULL bits of a batch in the pandas sense (bitmap, plus NaN for float columns)
template <int R>
__device__ __forceinline__ uint32_t b2_null_bits(const b2_col_t& c, int64_t row0, uint32_t bits,
                                                 const int64_t (&raw)[R]) {
  uint32_t nul = 0;
  if (c.valid) nul = bits & ~b2_valid_bits<R>(c.valid, row0, bits);
  if (c.dtype == B2_F64) {
#pragma unroll
    for (int j = 0; j < R; ++j) {
      const double d = __longlong_as_double(raw[j]);
      nul |= (uint32_t)(d != d) << j;
    }
    nul &= bits;
  }
  return nul;
}

// Branch-free comparison against a literal: every SQL comparison is a choice among the three
// outcomes (less, equal, greater) plus "unordered" for NaN, so the operator becomes four masks
// computed once per batch and the per-row work is two compares and two selects, with no jump
// table and one code path for all six operators.
struct b2_cmpmask {
  uint32_t lt, eq, gt, un;  // 0 or 0xffffffff
};
__device__ __forceinline__ b2_cmpmask b2_make_cmpmask(int op) {
  b2_cmpmask m;
  m.lt = (op == B2_LT || op == B2_LE || op == B2_NE) ? 0xffffffffu : 0u;
  m.eq = (op == B2_EQ || op == B2_LE || op == B2_GE) ? 0xffffffffu : 0u;
  m.gt = (op == B2_GT || op == B2_GE || op == B2_NE) ? 0xffffffffu : 0u;
  m.un = (op == B2_NE) ? 0xffffffffu : 0u;  // IEEE: NaN != x is true, everything else false
  return m;
}
template <int R>
__device__ __forceinline__ uint32_t b2_cmp_batch_i(const int64_t (&raw)[R], int64_t lit, const b2_cmpmask m) {
  uint32_t ok = 0;
#pragma unroll
  for (int j = 0; j < R; ++j) {
    const uint32_t r = raw[j] < lit ? m.lt : (raw[j] == lit ? m.eq : m.gt);
    ok |= r & (1u << j);
  }
  return ok;
}
template <int R, bool CVT>  // CVT: the column holds int64 and is compared as float64
__device__ __forceinline__ uint32_t b2_cmp_batch_f(const int64_t (&raw)[R], double lit, const b2_cmpmask m) {
  uint32_t ok = 0;
#pragma unroll
  for (int j = 0; j < R; ++j) {
    const double a = CVT ? (double)raw[j] : __longlong_as_double(raw[j]);
    const uint32_t r = a < lit ? m.lt : (a == lit ? m.eq : (a > lit ? m.gt : m.un));
    ok |= r & (1u << j);
  }
  return ok;
}

// ---------------------------------------------------------------------------------------
// column loaders: where a batch's values come from
// ---------------------------------------------------------------------------------------
struct b2_gld {  // straight from global memory
  const b2_scan_t* s;
  int64_t row0;
  template <int R>
  __device__ __forceinline__ void load(int col, uint32_t bits, bool full, int64_t (&raw)[R]) const {
    b2_load_batch<R>(s->cols[col], row0, bits, full, raw);
  }
};
struct b2_sld {  // from the shared-memory tile staged by the TMA producer warp (pipeline.cuh)
  const b2_scan_t* s;
  int64_t row0;            // global row of this lane's first row (bitmaps, out_slot)
  const uint8_t* stage;    // base of the current stage in shared memory
  const int32_t* col_off;  // byte offset of each column's tile within a stage
  int tile_off;            // this lane's first row within the tile
  template <int R>
  __device__ __forceinline__ void load(int col, uint32_t bits, bool full, int64_t (&raw)[R]) const {
    if (s->cols[col].dtype == B2_U8) {
      const uint8_t* p = stage + col_off[col] + tile_off;
#pragma unroll
      for (int j = 0; j < R; ++j) raw[j] = (int64_t)p[j * 32];
    } else {
      const int64_t* p = reinterpret_cast<const int64_t*>(stage + col_off[col]) + tile_off;
#pragma unroll
      for (int j = 0; j < R; ++j) raw[j] = p[j * 32];
    }
  }
};

// Evaluate all predicate terms for the batch.  Returns the surviving row bits and whether the
// batch is fully in bounds.
template <int R, class LD>
__device__ __forceinline__ uint32_t b2_eval_terms(const b2_scan_t& s, const LD& ld, bool& full, int& last_col,
                                                  int64_t (&raw)[R]) {
  // On return `raw` still holds the values of column `last_col` (the last term's column, -1 if
  // none) for the surviving rows: consumers that need the same column again (SUM(x) ... WHERE x > 0,
  // a join key that is also filtered) reuse the registers instead of re-loading.
  const int64_t row0 = ld.row0;
  uint32_t bits = b2_bounds_bits<R>(row0, s.n, full);
  last_col = -1;
  for (int t = 0; t < s.nterms; ++t) {
    const b2_term_t& tm = s.terms[t];
    const b2_col_t& c = s.cols[tm.col];
    const int op = tm.op;
    ld.template load<R>(tm.col, bits, full, raw);
    last_col = tm.col;
    uint32_t ok;
    if (op == B2_IS_NULL || op == B2_IS_NOT_NULL) {
      const uint32_t nul = b2_null_bits<R>(c, row0, bits, raw);
      ok = op == B2_IS_NULL ? nul : ~nul;
    } else {
      if (op == B2_IS_TRUE) {
        ok = 0;
#pragma unroll
        for (int j = 0; j < R; ++j) ok |= (uint32_t)(raw[j] != 0) << j;
      } else {
        const b2_cmpmask m = b2_make_cmpmask(op);
        if (c.dtype == B2_F64) ok = b2_cmp_batch_f<R, false>(raw, tm.lit_f, m);
        else if (tm.as_f64) ok = b2_cmp_batch_f<R, true>(raw, tm.lit_f, m);
        else ok = b2_cmp_batch_i<R>(raw, tm.lit_i, m);
      }
      if (c.valid) ok &= b2_valid_bits<R>(c.valid, row0, bits);
    }
    bits &= ok;
  }
  return bits;
}
template <int R, class LD>
__device__ __forceinline__ uint32_t b2_eval_terms(const b2_scan_t& s, const LD& ld, bool& full) {
  int last_col;
  int64_t raw[R];
  return b2_eval_terms<R>(s, ld, full, last_col, raw);
}
template <int R>
__device__ __forceinline__ uint32_t b2_eval_terms(const b2_scan_t& s, int64_t row0, bool& full) {
  const b2_gld ld{&s, row0};
  return b2_eval_terms<R>(s, ld, full);
}
template <int R>
__device__ __forceinline__ uint32_t b2_eval_terms(const b2_scan_t& s, int64_t row0) {
  bool full;
  return b2_eval_terms<R>(s, row0, full);
}

// ---------------------------------------------------------------------------------------
// aggregate updates into group tables (global-memory atomics)
// ---------------------------------------------------------------------------------------
// accumulator kinds: op x input type, resolved once per batch
#define B2_K_SUM_I   0
#define B2_K_SUM_F   1   // SUM of float64, and SUMF of float64
#define B2_K_SUMF_I  2   // int converted to float64, then added
#define B2_K_MIN_I   3
#define B2_K_MAX_I   4
#define B2_K_MIN_F   5   // ordered-int64 image
#define B2_K_MAX_F   6
#define B2_K_NONE    7   // COUNT only

__device__ __forceinline__ int b2_agg_kind(int op, int dtype) {
  const bool f = dtype == B2_F64;
  switch (op) {
    case B2_AGG_SUM: return f ? B2_K_SUM_F : B2_K_SUM_I;
    case B2_AGG_SUMF: return f ? B2_K_SUM_F : B2_K_SUMF_I;
    case B2_AGG_MIN: return f ? B2_K_MIN_F : B2_K_MIN_I;
    case B2_AGG_MAX: return f ? B2_K_MAX_F : B2_K_MAX_I;
    default: return B2_K_NONE;
  }
}

template <int KIND>
__device__ __forceinline__ void b2_atomic_k(void* acc, int64_t slot, int64_t raw) {
  if (KIND == B2_K_SUM_I) atomicAdd(reinterpret_cast<unsigned long long*>(acc) + slot, (unsigned long long)raw);
  // x + 0.0 turns -0.0 into +0.0 (pandas' running sum starts at +0.0, so the results agree) and
  // lets a float SUM accumulator that starts at -0.0 double as the "group was seen" flag: only an
  // untouched slot still holds the -0.0 bit pattern (see GroupTable.indicator on the host side)
  else if (KIND == B2_K_SUM_F) atomicAdd(reinterpret_cast<double*>(acc) + slot, __dadd_rn(__longlong_as_double(raw), 0.0));
  else if (KIND == B2_K_SUMF_I) atomicAdd(reinterpret_cast<double*>(acc) + slot, (double)raw);
  else if (KIND == B2_K_MIN_I) atomicMin(reinterpret_cast<long long*>(acc) + slot, (long long)raw);
  else if (KIND == B2_K_MAX_I) atomicMax(reinterpret_cast<long long*>(acc) + slot, (long long)raw);
  else if (KIND == B2_K_MIN_F) atomicMin(reinterpret_cast<long long*>(acc) + slot, (long long)b2_ordered_from_bits(raw));
  else if (KIND == B2_K_MAX_F) atomicMax(reinterpret_cast<long long*>(acc) + slot, (long long)b2_ordered_from_bits(raw));
}

template <int R, int KIND, bool CNT>
__device__ __forceinline__ void b2_atomic_batch2(void* acc, int64_t* cnt, const int64_t (&slot)[R],
                                                 const int64_t (&raw)[R], uint32_t live) {
#pragma unroll
  for (int j = 0; j < R; ++j) {
    if ((live >> j) & 1) {
      if (KIND != B2_K_NONE) b2_atomic_k<KIND>(acc, slot[j], raw[j]);
      if (CNT) atomicAdd(reinterpret_cast<unsigned long long*>(cnt) + slot[j], 1ULL);
    }
  }
}
template <int R, int KIND>
__device__ __forceinline__ void b2_atomic_batch(void* acc, int64_t* cnt, const int64_t (&slot)[R],
                                                const int64_t (&raw)[R], uint32_t live) {
  if (cnt) b2_atomic_batch2<R, KIND, true>(acc, cnt, slot, raw, live);
  else b2_atomic_batch2<R, KIND, false>(acc, cnt, slot, raw, live);
}

struct b2_aggs_arg {  // aggs passed by value in kernel params
  b2_agg_t a[B2_MAX_AGGS];
  int32_t n;
};

// For the batch at row0 with resolved slots (slot < 0 = row does not contribute): per aggregate,
// load its input column for the contributing rows, drop NULLs, apply the atomics.
// `pre` (optional): values of aggregate 0's input column already loaded by the caller for the rows
// in `pre_bits` (a superset of the contributing rows), so that this load overlapped the slot lookup.
template <int R, class LD>
__device__ __forceinline__ void b2_apply_aggs(const b2_scan_t& s, const LD& ld, const b2_agg_t* __restrict__ aggs,
                                              int naggs, const b2_aggstate_t& st,
                                              const int64_t (&slot)[R], const int64_t* pre = nullptr) {
  const int64_t row0 = ld.row0;
  uint32_t live = 0;
#pragma unroll
  for (int j = 0; j < R; ++j) live |= (uint32_t)(slot[j] >= 0) << j;
  if (st.out_slot) {
#pragma unroll
    for (int j = 0; j < R; ++j)
      if (row0 + (int64_t)j * 32 < s.n) st.out_slot[row0 + (int64_t)j * 32] = (int32_t)slot[j];
  }
  if (st.rows) {
#pragma unroll
    for (int j = 0; j < R; ++j)
      if ((live >> j) & 1) atomicAdd(reinterpret_cast<unsigned long long*>(st.rows) + slot[j], 1ULL);
  }
  if (st.present) {
    // read first (L1-cached: a stale miss only costs a redundant atomicOr): after warm-up almost
    // every group is already marked, so the atomic is rare
    uint32_t word[R];
#pragma unroll
    for (int j = 0; j < R; ++j) word[j] = (live >> j) & 1 ? __ldca(st.present + (slot[j] >> 5)) : 0xffffffffu;
#pragma unroll
    for (int j = 0; j < R; ++j) {
      const uint32_t b = 1u << (slot[j] & 31);
      if (((live >> j) & 1) && !(word[j] & b)) atomicOr(st.present + (slot[j] >> 5), b);
    }
  }
  for (int a = 0; a < naggs; ++a) {
    const b2_agg_t ag = aggs[a];
    if (ag.col < 0) continue;  // COUNT(*) is st.rows
    const b2_col_t& c = s.cols[ag.col];
    int64_t raw[R];
    if (a == 0 && pre) {
#pragma unroll
      for (int j = 0; j < R; ++j) raw[j] = pre[j];
    } else {
      ld.template load<R>(ag.col, live, false, raw);
    }
    uint32_t ok = live;
    if (c.valid || c.dtype == B2_F64) ok &= ~b2_null_bits<R>(c, row0, live, raw);
    void* acc = st.acc[a];
    int64_t* cnt = st.cnt[a];
    const int kind = acc ? b2_agg_kind(ag.op, c.dtype) : B2_K_NONE;
    switch (kind) {
      case B2_K_SUM_I: b2_atomic_batch<R, B2_K_SUM_I>(acc, cnt, slot, raw, ok); break;
      case B2_K_SUM_F: b2_atomic_batch<R, B2_K_SUM_F>(acc, cnt, slot, raw, ok); break;
      case B2_K_SUMF_I: b2_atomic_batch<R, B2_K_SUMF_I>(acc, cnt, slot, raw, ok); break;
      case B2_K_MIN_I: b2_atomic_batch<R, B2_K_MIN_I>(acc, cnt, slot, raw, ok); break;
      case B2_K_MAX_I: b2_atomic_batch<R, B2_K_MAX_I>(acc, cnt, slot, raw, ok); break;
      case B2_K_MIN_F: b2_atomic_batch<R, B2_K_MIN_F>(acc, cnt, slot, raw, ok); break;
      case B2_K_MAX_F: b2_atomic_batch<R, B2_K_MAX_F>(acc, cnt, slot, raw, ok); break;
      default: b2_atomic_batch<R, B2_K_NONE>(acc, cnt, slot, raw, ok); break;
    }
  }
}
