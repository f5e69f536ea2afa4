// b200sql.cu — libb200sql.so: C-ABI + kernels (see include/b200sql.h).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
#include "common.cuh"
#include <limits.h>
#include <string.h>

#include <cstdlib>
thread_local char g_b2_err[512] = {0};

static int g_sm_count_cache[64] = {0};
int b2_sm_count() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev < 0 || dev >= 64) return 148;
  if (g_sm_count_cache[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    g_sm_count_cache[dev] = n;
    // First use of this device: optionally set aside part of L2 for evict_last ("persisting") lines --
    // the lookup / payload / group tables the kernels mark with b2_policy_keep().  B200SQL_L2_PERSIST_MB
    // (default 0 = leave the driver default) is clamped to the device maximum.
    const char* e = getenv("B200SQL_L2_PERSIST_MB");
    if (e && atoi(e) > 0) {
      int maxb = 0;
      cudaDeviceGetAttribute(&maxb, cudaDevAttrMaxPersistingL2CacheSize, dev);
      size_t want = (size_t)atoi(e) << 20;
      if (maxb > 0 && want > (size_t)maxb) want = (size_t)maxb;
      if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) != cudaSuccess) cudaGetLastError();
    }
  }
  return g_sm_count_cache[dev];
}

#include "expr.cuh"
#include "filter.cuh"
#include "groupby.cuh"
#include "join.cuh"
#include "joinagg.cuh"
#include "sort.cuh"
#include "partition.cuh"
#include "peer.cuh"
#include "window.cuh"

extern "C" {

const char* b2_last_error(void) { return g_b2_err; }
int32_t b2_version(void) { return 100; }

int32_t b2_device_info(int32_t device, int32_t* sm_count, int64_t* l2_bytes, int32_t* cc_major,
                       int32_t* cc_minor, int64_t* hbm_bytes) {
  cudaDeviceProp p;
  B2_CUDA_TRY(cudaGetDeviceProperties(&p, device));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (l2_bytes) *l2_bytes = p.l2CacheSize;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  if (hbm_bytes) *hbm_bytes = (int64_t)p.totalGlobalMem;
  return B2_OK;
}

int32_t b2_d2h(void* host_dst, const void* dev_src, int64_t bytes, void* stream) {
  B2_CUDA_TRY(cudaMemcpyAsync(host_dst, dev_src, (size_t)bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  B2_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return B2_OK;
}

int32_t b2_memset(void* dev_ptr, int32_t byte, int64_t nbytes, void* stream) {
  B2_REQUIRE(dev_ptr || nbytes == 0, "null argument");
  if (nbytes > 0) B2_CUDA_TRY(cudaMemsetAsync(dev_ptr, byte, (size_t)nbytes, (cudaStream_t)stream));
  return B2_OK;
}

int32_t b2_sync(void* stream) {
  B2_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return B2_OK;
}

int64_t b2_num_tiles(int64_t n) { return (n + B2_TILE - 1) / B2_TILE; }

int64_t b2_f64_to_ordered(double x) {
  int64_t b;
  memcpy(&b, &x, 8);
  return b2_ordered_from_bits(b);
}
double b2_ordered_to_f64(int64_t k) {
  int64_t b = b2_ordered_from_bits(k);
  double x;
  memcpy(&x, &b, 8);
  return x;
}

}  // extern "C"
