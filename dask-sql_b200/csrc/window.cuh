// window.cuh — window functions over sorted columns: segment boundaries, ranking, LAG/LEAD and
// framed aggregates.  The reference evaluates OVER (...) with one pandas call per partition
// (dask_sql/physical/rel/logical/window.py:145-198 map_on_each_group, :330-332 groupby().apply());
// here the input is sorted once by (partition keys, order keys) (b2_sort_by + b2_gather) and every
// partition is a contiguous row range, so a window function is a segmented scan or a bounded
// gather over that range -- the cost does not depend on how many partitions there are.
//
// Tiles: 256 threads x 8 consecutive rows = 2048 rows.  Float scans are reduce-then-scan with a
// fixed tile size and a fixed combination order (tile totals -> one-block scan of the tiles ->
// downsweep): float64 results are bit-identical from run to run, like b2_scan_agg.
#pragma once
#include "common.cuh"

#define B2_WIN_BLOCK 256
#define B2_WIN_WARPS (B2_WIN_BLOCK / 32)
#define B2_WIN_ROWS 8
#define B2_WIN_TILE (B2_WIN_BLOCK * B2_WIN_ROWS)
#define B2_WIN_CARRY_BLOCK 512

struct b2_wkeys_arg {  // keys passed by value in kernel params
  b2_col_t k[B2_WIN_MAX_KEYS];
  int32_t npart, nkeys;
};

__device__ __forceinline__ int64_t b2_win_raw(const b2_col_t& c, int64_t r) {
  return c.dtype == B2_U8 ? (int64_t) reinterpret_cast<const uint8_t*>(c.data)[r]
                          : (int64_t)__ldg(reinterpret_cast<const long long*>(c.data) + r);
}
// rows a and b hold the same key: NULL == NULL (NaN is NULL), -0.0 == 0.0
__device__ __forceinline__ bool b2_win_same(const b2_col_t& c, int64_t a, int64_t b) {
  const int64_t ra = b2_win_raw(c, a), rb = b2_win_raw(c, b);
  const bool na = b2_is_null(c, a, ra), nb = b2_is_null(c, b, rb);
  if (na || nb) return na && nb;
  if (c.dtype == B2_F64) return __longlong_as_double(ra) == __longlong_as_double(rb);
  return ra == rb;
}

// ---------------------------------------------------------------------------------------
// segments: starts by one look-back pass, ends by scatter + gather
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(B2_WIN_BLOCK)
b2_win_starts_kernel(const __grid_constant__ b2_wkeys_arg keys, int64_t n, int64_t ntiles, uint64_t* __restrict__ status,
                     int32_t* __restrict__ part_start, int32_t* __restrict__ peer_start, int32_t* __restrict__ dense) {
  __shared__ int64_t wsum[3][B2_WIN_WARPS + 1];
  __shared__ int64_t carry[3];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t row0 = tile * B2_WIN_TILE + (int64_t)threadIdx.x * B2_WIN_ROWS;
    uint32_t pf = 0, qf = 0;
#pragma unroll
    for (int j = 0; j < B2_WIN_ROWS; ++j) {
      const int64_t i = row0 + j;
      if (i >= n) break;
      bool p = i == 0, q = p;
      if (!p) {
        for (int k = 0; k < keys.nkeys && !q; ++k) {
          if (!b2_win_same(keys.k[k], i, i - 1)) {
            q = true;
            p = k < keys.npart;
          }
        }
      }
      pf |= (uint32_t)p << j;
      qf |= (uint32_t)q << j;
    }
    // this thread's aggregates: last partition start, last peer start (max), peer starts (sum)
    int64_t v[3] = {pf ? row0 + 31 - __clz(pf) : 0, qf ? row0 + 31 - __clz(qf) : 0, __popc(qf)};
    // inclusive scan over the block in thread order
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t u0 = __shfl_up_sync(FULL_MASK, v[0], o), u1 = __shfl_up_sync(FULL_MASK, v[1], o),
                    u2 = __shfl_up_sync(FULL_MASK, v[2], o);
      if (lane >= o) {
        v[0] = max(v[0], u0);
        v[1] = max(v[1], u1);
        v[2] += u2;
      }
    }
    if (lane == 31) {
      wsum[0][warp] = v[0];
      wsum[1][warp] = v[1];
      wsum[2][warp] = v[2];
    }
    __syncthreads();
    if (threadIdx.x < 3) {  // exclusive scan of the warp totals, tile total in slot B2_WIN_WARPS
      const int s = threadIdx.x;
      int64_t run = 0;
      for (int w = 0; w < B2_WIN_WARPS; ++w) {
        const int64_t t = wsum[s][w];
        wsum[s][w] = run;
        run = s == 2 ? run + t : max(run, t);
      }
      wsum[s][B2_WIN_WARPS] = run;
    }
    __syncthreads();
    if (warp == 0) {
      const int64_t c0 = b2_lookback_op<b2_lb_max>(status, tile, wsum[0][B2_WIN_WARPS], lane);
      const int64_t c1 = b2_lookback_op<b2_lb_max>(status + ntiles, tile, wsum[1][B2_WIN_WARPS], lane);
      const int64_t c2 = b2_lookback_op<b2_lb_sum>(status + 2 * ntiles, tile, wsum[2][B2_WIN_WARPS], lane);
      if (lane == 0) {
        carry[0] = c0;
        carry[1] = c1;
        carry[2] = c2;
      }
    }
    __syncthreads();
    // exclusive prefix of this thread = carry (+) warp-exclusive (+) lanes before it
    const int64_t e0 = __shfl_up_sync(FULL_MASK, v[0], 1), e1 = __shfl_up_sync(FULL_MASK, v[1], 1),
                  e2 = __shfl_up_sync(FULL_MASK, v[2], 1);
    int64_t rp = max(carry[0], wsum[0][warp]), rq = max(carry[1], wsum[1][warp]), rc = carry[2] + wsum[2][warp];
    if (lane > 0) {
      rp = max(rp, e0);
      rq = max(rq, e1);
      rc += e2;
    }
#pragma unroll
    for (int j = 0; j < B2_WIN_ROWS; ++j) {
      const int64_t i = row0 + j;
      if (i >= n) break;
      if ((pf >> j) & 1) rp = i;
      if ((qf >> j) & 1) {
        rq = i;
        ++rc;
      }
      part_start[i] = (int32_t)rp;
      peer_start[i] = (int32_t)rq;
      dense[i] = (int32_t)rc;
    }
    __syncthreads();  // wsum / carry are reused by the next tile
  }
}

// each segment's last row writes the segment's end at the segment's first row
__global__ void __launch_bounds__(B2_BLOCK)
b2_win_ends_scatter_kernel(int64_t n, const int32_t* __restrict__ ps, const int32_t* __restrict__ qs,
                           int32_t* __restrict__ pe, int32_t* __restrict__ qe) {
  for (int64_t i = (int64_t)blockIdx.x * B2_BLOCK + threadIdx.x; i < n; i += (int64_t)gridDim.x * B2_BLOCK) {
    const bool last = i == n - 1;
    if (last || ps[i + 1] == i + 1) pe[ps[i]] = (int32_t)(i + 1);
    if (last || qs[i + 1] == i + 1) qe[qs[i]] = (int32_t)(i + 1);
  }
}
// every other row reads it there (rows that start a segment already hold their end)
__global__ void __launch_bounds__(B2_BLOCK)
b2_win_ends_gather_kernel(int64_t n, const int32_t* __restrict__ ps, const int32_t* __restrict__ qs, int32_t* pe,
                          int32_t* qe) {
  for (int64_t i = (int64_t)blockIdx.x * B2_BLOCK + threadIdx.x; i < n; i += (int64_t)gridDim.x * B2_BLOCK) {
    const int32_t p = ps[i], q = qs[i];
    if (p != i) pe[i] = pe[p];
    if (q != i) qe[i] = qe[q];
  }
}

// ---------------------------------------------------------------------------------------
// ranking and offsets (one row per thread, warps on 32-row aligned groups for the bitmap)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(B2_BLOCK)
b2_win_rank_kernel(int32_t op, int64_t n, const b2_wsegs_t s, int64_t* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * B2_BLOCK + threadIdx.x; i < n; i += (int64_t)gridDim.x * B2_BLOCK) {
    const int64_t ps = s.part_start[i];
    int64_t r;
    if (op == B2_WIN_ROW_NUMBER) r = i - ps + 1;
    else if (op == B2_WIN_RANK) r = (int64_t)s.peer_start[i] - ps + 1;
    else r = (int64_t)s.dense[i] - s.dense[ps] + 1;
    b2_st_stream(out + i, r);
  }
}

__global__ void __launch_bounds__(B2_BLOCK)
b2_win_offset_kernel(const __grid_constant__ b2_col_t val, int64_t n, int64_t off, int32_t has_default, int64_t def,
                     const b2_wsegs_t s, int64_t* __restrict__ out, uint32_t* __restrict__ out_valid) {
  const int lane = threadIdx.x & 31;
  for (int64_t base = (int64_t)blockIdx.x * B2_BLOCK + (threadIdx.x & ~31); base < n;
       base += (int64_t)gridDim.x * B2_BLOCK) {
    const int64_t i = base + lane;
    bool ok = false;
    if (i < n) {
      const int64_t j = i + off;
      int64_t raw = def;
      ok = has_default != 0;
      if (j >= s.part_start[i] && j < s.part_end[i]) {
        raw = b2_win_raw(val, j);
        ok = !b2_is_null(val, j, raw);
      }
      if (!ok && val.dtype == B2_F64) raw = 0x7ff8000000000000LL;  // NULL float: NaN
      b2_st_stream(out + i, raw);
    }
    const uint32_t bits = __ballot_sync(FULL_MASK, ok);
    if (lane == 0) out_valid[base >> 5] = bits;
  }
}

// ---------------------------------------------------------------------------------------
// framed aggregates
// ---------------------------------------------------------------------------------------
// accumulator kinds are common.cuh's B2_K_*; float kinds hold float64 bit patterns
__device__ __forceinline__ double b2_wd(int64_t b) { return __longlong_as_double(b); }
__device__ __forceinline__ int64_t b2_wb(double d) { return __double_as_longlong(d); }

template <int K>
__device__ __forceinline__ int64_t b2_wa_id() {
  if (K == B2_K_MIN_I) return INT64_MAX;
  if (K == B2_K_MAX_I) return INT64_MIN;
  if (K == B2_K_MIN_F) return 0x7ff0000000000000LL;           // +inf
  if (K == B2_K_MAX_F) return (int64_t)0xfff0000000000000ULL;  // -inf
  return 0;                                                    // 0 and +0.0
}
template <int K>
__device__ __forceinline__ int64_t b2_wa_lift(int64_t raw) {
  if (K == B2_K_SUMF_I) return b2_wb((double)raw);
  if (K == B2_K_SUM_F) return b2_wb(__dadd_rn(b2_wd(raw), 0.0));  // -0.0 -> +0.0, as pandas' sum
  return raw;
}
template <int K>
__device__ __forceinline__ int64_t b2_wa_op(int64_t a, int64_t b) {
  if (K == B2_K_SUM_I) return (int64_t)((uint64_t)a + (uint64_t)b);  // wraps like numpy
  if (K == B2_K_SUM_F || K == B2_K_SUMF_I) return b2_wb(__dadd_rn(b2_wd(a), b2_wd(b)));
  if (K == B2_K_MIN_I) return b < a ? b : a;
  if (K == B2_K_MAX_I) return b > a ? b : a;
  if (K == B2_K_MIN_F) return b2_wd(b) < b2_wd(a) ? b : a;
  if (K == B2_K_MAX_F) return b2_wd(b) > b2_wd(a) ? b : a;
  return 0;
}

// segmented-scan state: f = a segment starts inside, a = accumulator, c = non-NULL count
struct b2_wst {
  int32_t f;
  int64_t a, c;
};
template <int K>
__device__ __forceinline__ b2_wst b2_wcomb(const b2_wst& l, const b2_wst& r) {
  if (r.f) return r;
  return b2_wst{l.f, b2_wa_op<K>(l.a, r.a), l.c + r.c};
}
template <int K>
__device__ __forceinline__ b2_wst b2_wst_id() {
  return b2_wst{0, b2_wa_id<K>(), 0};
}

// physical row of logical row j (REV: the scan runs from the last row to the first)
template <bool REV>
__device__ __forceinline__ int64_t b2_wrow(int64_t j, int64_t n) { return REV ? n - 1 - j : j; }
template <bool REV>
__device__ __forceinline__ bool b2_wseg_start(const b2_wsegs_t& s, int64_t i) {
  return REV ? s.part_end[i] - 1 == i : s.part_start[i] == i;
}

// the state of one thread's B2_WIN_ROWS logical rows
template <int K, bool REV, bool STAR>
__device__ __forceinline__ b2_wst b2_wthread(const b2_col_t& val, const b2_wsegs_t& s, int64_t j0, int64_t n) {
  b2_wst st = b2_wst_id<K>();
#pragma unroll
  for (int r = 0; r < B2_WIN_ROWS; ++r) {
    const int64_t j = j0 + r;
    if (j >= n) break;
    const int64_t i = b2_wrow<REV>(j, n);
    if (b2_wseg_start<REV>(s, i)) st = b2_wst{1, b2_wa_id<K>(), 0};
    if (STAR) {
      ++st.c;
    } else {
      const int64_t raw = b2_win_raw(val, i);
      if (!b2_is_null(val, i, raw)) {
        st.a = b2_wa_op<K>(st.a, b2_wa_lift<K>(raw));
        ++st.c;
      }
    }
  }
  return st;
}

// block-wide exclusive scan in thread order (fixed order: deterministic); `total` = block aggregate
template <int K>
__device__ __forceinline__ b2_wst b2_wscan_block(b2_wst v, b2_wst& total, b2_wst* sh) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  b2_wst inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    b2_wst u;
    u.f = __shfl_up_sync(FULL_MASK, inc.f, o);
    u.a = __shfl_up_sync(FULL_MASK, inc.a, o);
    u.c = __shfl_up_sync(FULL_MASK, inc.c, o);
    if (lane >= o) inc = b2_wcomb<K>(u, inc);
  }
  if (lane == 31) sh[warp] = inc;
  __syncthreads();
  if (threadIdx.x == 0) {
    b2_wst run = b2_wst_id<K>();
    for (int w = 0; w < B2_WIN_WARPS; ++w) {
      const b2_wst t = sh[w];
      sh[w] = run;
      run = b2_wcomb<K>(run, t);
    }
    sh[B2_WIN_WARPS] = run;
  }
  __syncthreads();
  b2_wst prev;
  prev.f = __shfl_up_sync(FULL_MASK, inc.f, 1);
  prev.a = __shfl_up_sync(FULL_MASK, inc.a, 1);
  prev.c = __shfl_up_sync(FULL_MASK, inc.c, 1);
  const b2_wst ex = lane == 0 ? sh[warp] : b2_wcomb<K>(sh[warp], prev);
  total = sh[B2_WIN_WARPS];
  __syncthreads();
  return ex;
}

// pass 1: per-tile aggregates
template <int K, bool REV, bool STAR>
__global__ void __launch_bounds__(B2_WIN_BLOCK)
b2_win_reduce_kernel(const __grid_constant__ b2_col_t val, int64_t n, int64_t ntiles, const b2_wsegs_t s,
                     int32_t* __restrict__ tf, int64_t* __restrict__ ta, int64_t* __restrict__ tc) {
  __shared__ b2_wst sh[B2_WIN_WARPS + 1];
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const b2_wst v = b2_wthread<K, REV, STAR>(val, s, tile * B2_WIN_TILE + (int64_t)threadIdx.x * B2_WIN_ROWS, n);
    b2_wst total;
    b2_wscan_block<K>(v, total, sh);
    if (threadIdx.x == 0) {
      tf[tile] = total.f;
      ta[tile] = total.a;
      tc[tile] = total.c;
    }
  }
}

// pass 2 (one block): exclusive carry of every tile, each thread owning a contiguous run of tiles
template <int K>
__global__ void __launch_bounds__(B2_WIN_CARRY_BLOCK)
b2_win_carry_kernel(int64_t ntiles, const int32_t* __restrict__ tf, const int64_t* __restrict__ ta,
                    const int64_t* __restrict__ tc, int64_t* __restrict__ ca, int64_t* __restrict__ cc) {
  __shared__ int32_t shf[B2_WIN_CARRY_BLOCK];
  __shared__ int64_t sha[B2_WIN_CARRY_BLOCK], shc[B2_WIN_CARRY_BLOCK];
  const int64_t per = (ntiles + B2_WIN_CARRY_BLOCK - 1) / B2_WIN_CARRY_BLOCK;
  const int64_t lo = (int64_t)threadIdx.x * per, hi = min(ntiles, lo + per);
  b2_wst run = b2_wst_id<K>();
#pragma unroll 1
  for (int64_t t = lo; t < hi; ++t) run = b2_wcomb<K>(run, b2_wst{tf[t], ta[t], tc[t]});
  shf[threadIdx.x] = run.f;
  sha[threadIdx.x] = run.a;
  shc[threadIdx.x] = run.c;
  __syncthreads();
  if (threadIdx.x == 0) {
    b2_wst acc = b2_wst_id<K>();
#pragma unroll 1
    for (int w = 0; w < B2_WIN_CARRY_BLOCK; ++w) {
      const b2_wst t{shf[w], sha[w], shc[w]};
      shf[w] = acc.f;
      sha[w] = acc.a;
      shc[w] = acc.c;
      acc = b2_wcomb<K>(acc, t);
    }
  }
  __syncthreads();
  run = b2_wst{shf[threadIdx.x], sha[threadIdx.x], shc[threadIdx.x]};
#pragma unroll 1
  for (int64_t t = lo; t < hi; ++t) {
    ca[t] = run.a;
    cc[t] = run.c;
    run = b2_wcomb<K>(run, b2_wst{tf[t], ta[t], tc[t]});
  }
}

// pass 3: inclusive segmented scan written per row (P_a, P_c at the physical row)
template <int K, bool REV, bool STAR>
__global__ void __launch_bounds__(B2_WIN_BLOCK)
b2_win_down_kernel(const __grid_constant__ b2_col_t val, int64_t n, int64_t ntiles, const b2_wsegs_t s,
                   const int64_t* __restrict__ ca, const int64_t* __restrict__ cc, int64_t* __restrict__ pa,
                   int32_t* __restrict__ pc) {
  __shared__ b2_wst sh[B2_WIN_WARPS + 1];
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t j0 = tile * B2_WIN_TILE + (int64_t)threadIdx.x * B2_WIN_ROWS;
    const b2_wst v = b2_wthread<K, REV, STAR>(val, s, j0, n);
    b2_wst total;
    const b2_wst ex = b2_wscan_block<K>(v, total, sh);
    b2_wst st = b2_wcomb<K>(b2_wst{0, ca[tile], cc[tile]}, ex);
#pragma unroll
    for (int r = 0; r < B2_WIN_ROWS; ++r) {
      const int64_t j = j0 + r;
      if (j >= n) break;
      const int64_t i = b2_wrow<REV>(j, n);
      if (b2_wseg_start<REV>(s, i)) st = b2_wst{1, b2_wa_id<K>(), 0};
      if (STAR) {
        ++st.c;
      } else {
        const int64_t raw = b2_win_raw(val, i);
        if (!b2_is_null(val, i, raw)) {
          st.a = b2_wa_op<K>(st.a, b2_wa_lift<K>(raw));
          ++st.c;
        }
      }
      pa[i] = st.a;
      pc[i] = (int32_t)st.c;
    }
  }
}

// frame of row i as an inclusive row range [fs, fe] (empty when fs > fe)
__device__ __forceinline__ void b2_win_frame(const b2_wframe_t& fr, int64_t i, const b2_wsegs_t& s, int64_t& fs,
                                             int64_t& fe) {
  const int64_t ps = s.part_start[i], pe = s.part_end[i];
  if (fr.lo_kind == B2_WB_UNBOUNDED) fs = ps;
  else if (fr.range) fs = s.peer_start[i];
  else fs = max(i + fr.lo, ps);
  if (fr.hi_kind == B2_WB_UNBOUNDED) fe = pe - 1;
  else if (fr.range) fe = (int64_t)s.peer_end[i] - 1;
  else fe = min(i + fr.hi, pe - 1);
}

#define B2_WM_SCAN 0   // read the forward scan at the frame end
#define B2_WM_RSCAN 1  // read the reverse scan at the frame start
#define B2_WM_DIFF 2   // difference of forward prefixes (exact: int64 SUM, COUNT)
#define B2_WM_DIRECT 3 // combine the frame's rows
#define B2_WM_FIRST 4
#define B2_WM_LAST 5
#define B2_WOUT_VALUE 0
#define B2_WOUT_COUNT 1
#define B2_WOUT_AVG 2

template <int K, int MODE, bool STAR>
__global__ void __launch_bounds__(B2_BLOCK)
b2_win_agg_kernel(const __grid_constant__ b2_col_t val, int32_t out_kind, int32_t out_f64, const b2_wframe_t fr,
                  int64_t n, const b2_wsegs_t s, const int64_t* __restrict__ pa, const int32_t* __restrict__ pc,
                  int64_t* __restrict__ out, uint32_t* __restrict__ out_valid) {
  const int lane = threadIdx.x & 31;
  for (int64_t base = (int64_t)blockIdx.x * B2_BLOCK + (threadIdx.x & ~31); base < n;
       base += (int64_t)gridDim.x * B2_BLOCK) {
    const int64_t i = base + lane;
    bool ok = false;
    if (i < n) {
      int64_t fs, fe, res = 0;
      b2_win_frame(fr, i, s, fs, fe);
      if (fs <= fe) {
        if (MODE == B2_WM_FIRST || MODE == B2_WM_LAST) {
          const int64_t j = MODE == B2_WM_FIRST ? fs : fe;
          res = b2_win_raw(val, j);
          ok = !b2_is_null(val, j, res);
        } else {
          int64_t a, c;
          if (MODE == B2_WM_SCAN) {
            a = pa[fe];
            c = pc[fe];
          } else if (MODE == B2_WM_RSCAN) {
            a = pa[fs];
            c = pc[fs];
          } else if (MODE == B2_WM_DIFF) {
            a = pa[fe];
            c = pc[fe];
            if (fs > s.part_start[i]) {
              a = (int64_t)((uint64_t)a - (uint64_t)pa[fs - 1]);
              c -= pc[fs - 1];
            }
          } else {
            a = b2_wa_id<K>();
            c = 0;
            for (int64_t j = fs; j <= fe; ++j) {
              if (STAR) {
                ++c;
              } else {
                const int64_t raw = b2_win_raw(val, j);
                if (!b2_is_null(val, j, raw)) {
                  a = b2_wa_op<K>(a, b2_wa_lift<K>(raw));
                  ++c;
                }
              }
            }
          }
          if (out_kind == B2_WOUT_COUNT) {
            res = c;
            ok = true;
          } else {
            ok = c > 0;
            res = out_kind == B2_WOUT_AVG ? b2_wb(b2_wd(a) / (double)c) : a;
          }
        }
      } else if (out_kind == B2_WOUT_COUNT) {
        ok = true;  // empty frame: COUNT is 0
      }
      if (!ok && out_f64) res = 0x7ff8000000000000LL;
      b2_st_stream(out + i, res);
    }
    if (out_valid) {
      const uint32_t bits = __ballot_sync(FULL_MASK, ok);
      if (lane == 0) out_valid[base >> 5] = bits;
    }
  }
}

// host side: workspace layout shared by segments and aggregates
struct b2_wws {
  int64_t ntiles;
  uint64_t* status;  // 3 * ntiles (segments)
  int64_t* pa;       // n
  int32_t* pc;       // n
  int32_t* tf;       // ntiles
  int64_t *ta, *tc, *ca, *cc;
};
static inline b2_wws b2_wws_layout(void* ws, int64_t n) {
  b2_wws w;
  w.ntiles = (n + B2_WIN_TILE - 1) / B2_WIN_TILE;
  uint8_t* p = reinterpret_cast<uint8_t*>(ws);
  auto take = [&](int64_t bytes) { uint8_t* r = p; p += (bytes + 255) & ~(int64_t)255; return r; };
  w.pa = reinterpret_cast<int64_t*>(take(n * 8));
  w.pc = reinterpret_cast<int32_t*>(take(n * 4));
  w.tf = reinterpret_cast<int32_t*>(take(w.ntiles * 4));
  w.ta = reinterpret_cast<int64_t*>(take(w.ntiles * 8));
  w.tc = reinterpret_cast<int64_t*>(take(w.ntiles * 8));
  w.ca = reinterpret_cast<int64_t*>(take(w.ntiles * 8));
  w.cc = reinterpret_cast<int64_t*>(take(w.ntiles * 8));
  w.status = reinterpret_cast<uint64_t*>(w.pa);  // the segment pass runs before any scan: reuse
  return w;
}

template <int K, bool REV, bool STAR>
static int32_t b2_win_scan(const b2_col_t& val, int64_t n, const b2_wsegs_t& s, const b2_wws& w, cudaStream_t st) {
  const int64_t nt = w.ntiles;
  int grid = b2_wave_grid(b2_win_reduce_kernel<K, REV, STAR>, B2_WIN_BLOCK, nt);
  b2_win_reduce_kernel<K, REV, STAR><<<grid, B2_WIN_BLOCK, 0, st>>>(val, n, nt, s, w.tf, w.ta, w.tc);
  b2_win_carry_kernel<K><<<1, B2_WIN_CARRY_BLOCK, 0, st>>>(nt, w.tf, w.ta, w.tc, w.ca, w.cc);
  grid = b2_wave_grid(b2_win_down_kernel<K, REV, STAR>, B2_WIN_BLOCK, nt);
  b2_win_down_kernel<K, REV, STAR><<<grid, B2_WIN_BLOCK, 0, st>>>(val, n, nt, s, w.ca, w.cc, w.pa, w.pc);
  B2_CHECK_LAUNCH("b2_win_scan kernels");
  return B2_OK;
}

template <int K, int MODE, bool STAR>
static int32_t b2_win_finish(const b2_col_t& val, int32_t out_kind, int32_t out_f64, const b2_wframe_t& fr, int64_t n,
                             const b2_wsegs_t& s, const b2_wws& w, void* out, uint32_t* out_valid, cudaStream_t st) {
  const int grid = b2_wave_grid(b2_win_agg_kernel<K, MODE, STAR>, B2_BLOCK, (n + B2_BLOCK - 1) / B2_BLOCK);
  b2_win_agg_kernel<K, MODE, STAR><<<grid, B2_BLOCK, 0, st>>>(val, out_kind, out_f64, fr, n, s, w.pa, w.pc,
                                                               reinterpret_cast<int64_t*>(out), out_valid);
  B2_CHECK_LAUNCH("b2_win_agg_kernel");
  return B2_OK;
}

template <int K, bool STAR>
static int32_t b2_win_agg_k(const b2_col_t& val, int32_t out_kind, int32_t out_f64, const b2_wframe_t& fr, int64_t n,
                            const b2_wsegs_t& s, const b2_wws& w, void* out, uint32_t* out_valid, cudaStream_t st) {
  int32_t rc;
  if (fr.lo_kind == B2_WB_UNBOUNDED) {
    if ((rc = b2_win_scan<K, false, STAR>(val, n, s, w, st)) != B2_OK) return rc;
    return b2_win_finish<K, B2_WM_SCAN, STAR>(val, out_kind, out_f64, fr, n, s, w, out, out_valid, st);
  }
  if (fr.hi_kind == B2_WB_UNBOUNDED) {
    if ((rc = b2_win_scan<K, true, STAR>(val, n, s, w, st)) != B2_OK) return rc;
    return b2_win_finish<K, B2_WM_RSCAN, STAR>(val, out_kind, out_f64, fr, n, s, w, out, out_valid, st);
  }
  const bool wide = fr.range || fr.hi - fr.lo >= 32;
  if ((K == B2_K_SUM_I || K == B2_K_NONE) && wide) {
    if ((rc = b2_win_scan<K, false, STAR>(val, n, s, w, st)) != B2_OK) return rc;
    return b2_win_finish<K, B2_WM_DIFF, STAR>(val, out_kind, out_f64, fr, n, s, w, out, out_valid, st);
  }
  return b2_win_finish<K, B2_WM_DIRECT, STAR>(val, out_kind, out_f64, fr, n, s, w, out, out_valid, st);
}

extern "C" {

int64_t b2_window_ws_bytes(int64_t n) {
  const int64_t nt = (n + B2_WIN_TILE - 1) / B2_WIN_TILE;
  const int64_t scan = n * 12 + nt * 36 + 8 * 256;
  const int64_t seg = nt * 24 + 256;
  return (scan > seg ? scan : seg) + 256;
}

// replaces window.py:330-332 (groupby(partition keys, dropna=False).apply) and the per-group sort of
// window.py:156-159: partitions and peer groups of the sorted rows
int32_t b2_window_segments(const b2_col_t* keys, int32_t npart, int32_t nkeys, int64_t n, const b2_wsegs_t* segs,
                           void* ws, void* stream) {
  B2_REQUIRE(segs && (keys || nkeys == 0) && (ws || n == 0), "null argument");
  B2_REQUIRE(nkeys >= 0 && nkeys <= B2_WIN_MAX_KEYS && npart >= 0 && npart <= nkeys, "bad key count");
  B2_REQUIRE(n < ((int64_t)1 << 31), "window input must hold < 2^31 rows");
  if (n <= 0) return B2_OK;
  cudaStream_t st = (cudaStream_t)stream;
  b2_wkeys_arg k;
  memset(&k, 0, sizeof(k));
  for (int i = 0; i < nkeys; ++i) k.k[i] = keys[i];
  k.npart = npart;
  k.nkeys = nkeys;
  const b2_wws w = b2_wws_layout(ws, n);
  B2_CUDA_TRY(cudaMemsetAsync(w.status, 0, (size_t)w.ntiles * 3 * 8, st));
  int grid = b2_wave_grid(b2_win_starts_kernel, B2_WIN_BLOCK, w.ntiles);
  b2_win_starts_kernel<<<grid, B2_WIN_BLOCK, 0, st>>>(k, n, w.ntiles, w.status, segs->part_start, segs->peer_start,
                                                      segs->dense);
  grid = b2_wave_grid(b2_win_ends_scatter_kernel, B2_BLOCK, (n + B2_BLOCK - 1) / B2_BLOCK);
  b2_win_ends_scatter_kernel<<<grid, B2_BLOCK, 0, st>>>(n, segs->part_start, segs->peer_start, segs->part_end,
                                                        segs->peer_end);
  grid = b2_wave_grid(b2_win_ends_gather_kernel, B2_BLOCK, (n + B2_BLOCK - 1) / B2_BLOCK);
  b2_win_ends_gather_kernel<<<grid, B2_BLOCK, 0, st>>>(n, segs->part_start, segs->peer_start, segs->part_end,
                                                       segs->peer_end);
  B2_CHECK_LAUNCH("b2_window_segments kernels");
  return B2_OK;
}

// replaces window.py:187-190 (ROW_NUMBER as range(1, len(group) + 1)); RANK / DENSE_RANK from peers
int32_t b2_window_rank(int32_t op, int64_t n, const b2_wsegs_t* segs, int64_t* out, void* stream) {
  B2_REQUIRE(segs && (out || n == 0), "null argument");
  B2_REQUIRE(op == B2_WIN_ROW_NUMBER || op == B2_WIN_RANK || op == B2_WIN_DENSE_RANK, "not a ranking function");
  if (n <= 0) return B2_OK;
  const int grid = b2_wave_grid(b2_win_rank_kernel, B2_BLOCK, (n + B2_BLOCK - 1) / B2_BLOCK);
  b2_win_rank_kernel<<<grid, B2_BLOCK, 0, (cudaStream_t)stream>>>(op, n, *segs, out);
  B2_CHECK_LAUNCH("b2_win_rank_kernel");
  return B2_OK;
}

// LAG / LEAD: one gather inside the partition (no reference counterpart; window.py:214-225 lists its functions)
int32_t b2_window_offset(const b2_col_t* val, int64_t n, int64_t offset, int32_t has_default, int64_t default_raw,
                         const b2_wsegs_t* segs, void* out, uint32_t* out_valid, void* stream) {
  B2_REQUIRE(val && segs && ((out && out_valid) || n == 0), "null argument");
  B2_REQUIRE(val->dtype == B2_I64 || val->dtype == B2_F64, "LAG / LEAD take int64 or float64 values");
  if (n <= 0) return B2_OK;
  const int grid = b2_wave_grid(b2_win_offset_kernel, B2_BLOCK, (n + B2_BLOCK - 1) / B2_BLOCK);
  b2_win_offset_kernel<<<grid, B2_BLOCK, 0, (cudaStream_t)stream>>>(*val, n, offset, has_default, default_raw, *segs,
                                                                    reinterpret_cast<int64_t*>(out), out_valid);
  B2_CHECK_LAUNCH("b2_win_offset_kernel");
  return B2_OK;
}

// replaces window.py:161-192: expanding() / rolling(window) / rolling(Indexer) + the OverOperation
// classes (window.py:24-62) of every group
int32_t b2_window_agg(const b2_col_t* val, int32_t op, const b2_wframe_t* frame, int64_t n, const b2_wsegs_t* segs,
                      void* out, uint32_t* out_valid, void* ws, void* stream) {
  B2_REQUIRE(val && frame && segs && ((out && ws) || n == 0), "null argument");
  B2_REQUIRE(op >= B2_WIN_SUM && op <= B2_WIN_LAST, "not a framed aggregate");
  const bool star = val->data == nullptr;
  B2_REQUIRE(!star || op == B2_WIN_COUNT, "only COUNT takes no value column");
  B2_REQUIRE(star || val->dtype == B2_I64 || val->dtype == B2_F64, "window aggregates take int64 or float64 values");
  B2_REQUIRE(op == B2_WIN_COUNT || out_valid || n == 0, "out_valid is required");
  const b2_wframe_t& fr = *frame;
  B2_REQUIRE(fr.lo_kind == B2_WB_UNBOUNDED || fr.lo_kind == B2_WB_OFFSET, "bad lower bound");
  B2_REQUIRE(fr.hi_kind == B2_WB_UNBOUNDED || fr.hi_kind == B2_WB_OFFSET, "bad upper bound");
  B2_REQUIRE(!fr.range || ((fr.lo_kind == B2_WB_UNBOUNDED || fr.lo == 0) && (fr.hi_kind == B2_WB_UNBOUNDED || fr.hi == 0)),
             "RANGE frames take only UNBOUNDED and CURRENT ROW bounds");
  B2_REQUIRE(n < ((int64_t)1 << 31), "window input must hold < 2^31 rows");
  if (n <= 0) return B2_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const b2_wws w = b2_wws_layout(ws, n);
  const bool f = !star && val->dtype == B2_F64;
  const b2_col_t v = *val;
  if (op == B2_WIN_FIRST || op == B2_WIN_LAST) {
    if (op == B2_WIN_FIRST) return b2_win_finish<B2_K_NONE, B2_WM_FIRST, false>(v, B2_WOUT_VALUE, f, fr, n, *segs, w, out, out_valid, st);
    return b2_win_finish<B2_K_NONE, B2_WM_LAST, false>(v, B2_WOUT_VALUE, f, fr, n, *segs, w, out, out_valid, st);
  }
  uint32_t* ov = op == B2_WIN_COUNT ? nullptr : out_valid;
  switch (op) {
    case B2_WIN_COUNT:
      if (star) return b2_win_agg_k<B2_K_NONE, true>(v, B2_WOUT_COUNT, 0, fr, n, *segs, w, out, ov, st);
      return b2_win_agg_k<B2_K_NONE, false>(v, B2_WOUT_COUNT, 0, fr, n, *segs, w, out, ov, st);
    case B2_WIN_SUM:
      if (f) return b2_win_agg_k<B2_K_SUM_F, false>(v, B2_WOUT_VALUE, 1, fr, n, *segs, w, out, ov, st);
      return b2_win_agg_k<B2_K_SUM_I, false>(v, B2_WOUT_VALUE, 0, fr, n, *segs, w, out, ov, st);
    case B2_WIN_AVG:
      if (f) return b2_win_agg_k<B2_K_SUM_F, false>(v, B2_WOUT_AVG, 1, fr, n, *segs, w, out, ov, st);
      return b2_win_agg_k<B2_K_SUMF_I, false>(v, B2_WOUT_AVG, 1, fr, n, *segs, w, out, ov, st);
    case B2_WIN_MIN:
      if (f) return b2_win_agg_k<B2_K_MIN_F, false>(v, B2_WOUT_VALUE, 1, fr, n, *segs, w, out, ov, st);
      return b2_win_agg_k<B2_K_MIN_I, false>(v, B2_WOUT_VALUE, 0, fr, n, *segs, w, out, ov, st);
    default:
      if (f) return b2_win_agg_k<B2_K_MAX_F, false>(v, B2_WOUT_VALUE, 1, fr, n, *segs, w, out, ov, st);
      return b2_win_agg_k<B2_K_MAX_I, false>(v, B2_WOUT_VALUE, 0, fr, n, *segs, w, out, ov, st);
  }
}

}  // extern "C"
