// Shared plumbing for the dmosopt_b200 CUDA library (sm_100a).
// Context, stream-ordered scratch buffers, host/device pointer staging,
// launch accounting, order-preserving float transforms and Philox4x32-10.
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include <string>
#include <vector>

#include "../../include/dmosopt_b200.h"

struct dmo_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaMemPool_t pool = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int sm_count = 148;
  int64_t launches = 0;
  std::string err;
  void* flush_buf = nullptr;
  size_t flush_bytes = 0;
  int* dev_flag = nullptr;  // device-side error / watchdog flag (int[4])
  uint64_t h2d_bytes = 0, d2h_bytes = 0;  // bytes staged for host buffers (In<> / Out<>)
  // optional per-kernel CUDA-event timers (dmo_profile_enable); bench.py reads them for the roofline
  bool profiling = false;
  struct Timer {
    std::string name;
    cudaEvent_t a, b;
  };
  std::vector<Timer> timers;
};

// RAII: records a start/stop event pair around a kernel (or a group of launches) when profiling is on
struct ProfileScope {
  dmo_ctx* ctx;
  int idx = -1;
  ProfileScope(dmo_ctx* c, const char* name) : ctx(c) {
    if (!c->profiling) return;
    dmo_ctx::Timer t;
    t.name = name;
    if (cudaEventCreate(&t.a) != cudaSuccess || cudaEventCreate(&t.b) != cudaSuccess) return;
    cudaEventRecord(t.a, c->stream);
    c->timers.push_back(t);
    idx = (int)c->timers.size() - 1;
  }
  ~ProfileScope() {
    if (idx >= 0) cudaEventRecord(ctx->timers[idx].b, ctx->stream);
  }
};

int dmo_fail(dmo_ctx* ctx, int code, const char* fmt, ...);

#define DMO_CUDA(call)                                                                        \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return dmo_fail(ctx, DMO_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                      __FILE__, __LINE__);                                                    \
  } while (0)

#define DMO_TRY(expr)              \
  do {                             \
    int s__ = (expr);              \
    if (s__ != DMO_OK) return s__; \
  } while (0)

#define DMO_REQUIRE(cond, ...)                                 \
  do {                                                         \
    if (!(cond)) return dmo_fail(ctx, DMO_ERR_ARG, __VA_ARGS__); \
  } while (0)

// every kernel launch of the library goes through this macro so that
// dmo_launch_count() is the library's own count of launched kernels
#define DMO_LAUNCH(kernel, grid, block, smem, ...)                       \
  do {                                                                   \
    kernel<<<(grid), (block), (smem), ctx->stream>>>(__VA_ARGS__);       \
    ctx->launches++;                                                     \
  } while (0)

#define DMO_CHECK_LAUNCH() DMO_CUDA(cudaGetLastError())

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------
// Stream-ordered scratch buffer (cudaMallocAsync on the context's pool).
template <typename T>
struct DevBuf {
  dmo_ctx* ctx = nullptr;
  T* p = nullptr;
  size_t n = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  int alloc(dmo_ctx* c, size_t count) {
    release();
    ctx = c;
    n = count;
    if (count == 0) count = 1;
    cudaError_t e = cudaMallocAsync((void**)&p, count * sizeof(T), c->stream);
    if (e != cudaSuccess) {
      p = nullptr;
      return dmo_fail(c, DMO_ERR_CUDA, "cudaMallocAsync(%zu bytes) failed: %s", count * sizeof(T),
                      cudaGetErrorString(e));
    }
    return DMO_OK;
  }
  void release() {
    if (p) cudaFreeAsync(p, ctx->stream);
    p = nullptr;
  }
};

bool dmo_is_device_ptr(const void* p);

// Input array that may live on the host: gives a device pointer valid on ctx->stream.
template <typename T>
struct In {
  DevBuf<T> buf;
  const T* d = nullptr;
  int init(dmo_ctx* ctx, const T* src, size_t count) {
    if (src == nullptr || count == 0) {
      d = nullptr;
      return DMO_OK;
    }
    if (dmo_is_device_ptr(src)) {
      d = src;
      return DMO_OK;
    }
    DMO_TRY(buf.alloc(ctx, count));
    DMO_CUDA(cudaMemcpyAsync(buf.p, src, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    ctx->h2d_bytes += count * sizeof(T);
    d = buf.p;
    return DMO_OK;
  }
};

// Output array that may live on the host: kernels write to .d, finish() copies back.
template <typename T>
struct Out {
  DevBuf<T> buf;
  T* d = nullptr;
  T* host = nullptr;
  size_t count = 0;
  int init(dmo_ctx* ctx, T* dst, size_t cnt) {
    count = cnt;
    if (dst == nullptr) {
      d = nullptr;
      return DMO_OK;
    }
    if (dmo_is_device_ptr(dst)) {
      d = dst;
      return DMO_OK;
    }
    host = dst;
    DMO_TRY(buf.alloc(ctx, cnt));
    d = buf.p;
    return DMO_OK;
  }
  int finish(dmo_ctx* ctx, size_t cnt = (size_t)-1) {
    if (host && d) {
      size_t c = (cnt == (size_t)-1) ? count : cnt;
      if (c) DMO_CUDA(cudaMemcpyAsync(host, d, c * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
      ctx->d2h_bytes += c * sizeof(T);
    }
    return DMO_OK;
  }
};

// ---------------------------------------------------------------------------
// device helpers
#ifdef __CUDACC__

// IEEE-754 order-preserving maps (radix-sortable keys).  -0.0 is canonicalised to +0.0
// first so that it compares equal to +0.0 like numpy does.
__device__ __forceinline__ uint64_t f64_to_ordered(double x) {
  x = x + 0.0;
  uint64_t b = (uint64_t)__double_as_longlong(x);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double ordered_to_f64(uint64_t k) {
  uint64_t b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}
__device__ __forceinline__ uint32_t f32_to_ordered(float x) {
  x = x + 0.0f;
  uint32_t b = __float_as_uint(x);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// Philox4x32-10 (Salmon, Moraes, Dror, Shaw 2011): counter-based, no state in memory.
struct Philox {
  uint32_t k0, k1;
  __device__ __forceinline__ Philox(uint64_t seed) : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)) {}
  __device__ __forceinline__ uint4 operator()(uint64_t ctr_lo, uint64_t ctr_hi) const {
    uint32_t c0 = (uint32_t)ctr_lo, c1 = (uint32_t)(ctr_lo >> 32);
    uint32_t c2 = (uint32_t)ctr_hi, c3 = (uint32_t)(ctr_hi >> 32);
    uint32_t a = k0, b = k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
      uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
      uint32_t n0 = h1 ^ c1 ^ a, n1 = l1, n2 = h0 ^ c3 ^ b, n3 = l0;
      c0 = n0;
      c1 = n1;
      c2 = n2;
      c3 = n3;
      a += 0x9E3779B9u;
      b += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
};
// 53-bit uniform in [0, 1) from two 32-bit words (same construction as numpy's Generator.random)
__device__ __forceinline__ double u01_53(uint32_t hi, uint32_t lo) {
  return (double)((((uint64_t)(hi >> 5)) << 26) | (uint64_t)(lo >> 6)) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

#endif  // __CUDACC__

// ---------------------------------------------------------------------------
// primitives implemented in prims.cu (CUB is only included there)
int prim_sort_pairs_u64(dmo_ctx* ctx, const uint64_t* kin, uint64_t* kout, const uint32_t* vin,
                        uint32_t* vout, int64_t n, int begin_bit, int end_bit);
int prim_sort_pairs_u32(dmo_ctx* ctx, const uint32_t* kin, uint32_t* kout, const uint32_t* vin,
                        uint32_t* vout, int64_t n, int begin_bit, int end_bit);
int prim_inclusive_sum_u32(dmo_ctx* ctx, const uint32_t* in, uint32_t* out, int64_t n);
int prim_exclusive_sum_i32(dmo_ctx* ctx, const int32_t* in, int32_t* out, int64_t n);
int prim_iota_u32(dmo_ctx* ctx, uint32_t* out, int64_t n);

// internal device-pointer entry points shared between translation units
// (all pointers are device pointers; outputs in caller-provided device buffers)
int rank_nd_device(dmo_ctx* ctx, const double* dY, int64_t n, int M, int32_t* d_rank);
int rank_nd_device_keep(dmo_ctx* ctx, const double* dY, int64_t n, int M, int64_t keep, int32_t* d_rank);
// 0 for non-dominated rows, non-zero otherwise (no ranks: no dependency chain)
int nondominated_flags_device(dmo_ctx* ctx, const double* dY, int64_t n, int M, int32_t* d_flag01);
int crowding_device(dmo_ctx* ctx, const double* dY, int64_t n, int M, double* dD);
int euclidean_device(dmo_ctx* ctx, const double* dY, int64_t n, int M, double* dD);
// perm (uint32, n) sorted by (rank asc, then each desc key descending, stable on index)
int lexsort_device(dmo_ctx* ctx, const int32_t* d_rank, const double* const* d_desc_keys, int nkeys,
                   int64_t n, uint32_t* d_perm);
int hypervolume_device(dmo_ctx* ctx, const double* dF, int64_t n, int M, const double* h_ref, double* h_out);
// the same when the rows carry their non-dominated ranks within a superset (rank > 0 rows are skipped, no filter pass)
int hypervolume_device_ranked(dmo_ctx* ctx, const double* dF, int64_t n, int M, const double* h_ref, const int32_t* d_rank,
                              double* h_out);
