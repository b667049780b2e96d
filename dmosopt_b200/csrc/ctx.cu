// Context management, error reporting, memory helpers of the C ABI
// (include/dmosopt_b200.h, section "context").
#include <stdarg.h>

#include "common.cuh"

int dmo_fail(dmo_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

bool dmo_is_device_ptr(const void* p) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    cudaGetLastError();  // clear
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

extern "C" {

int dmo_version(void) { return 100; }

int dmo_create(int device, dmo_ctx** out) {
  if (!out) return DMO_ERR_ARG;
  *out = nullptr;
  dmo_ctx* ctx = new dmo_ctx();
  ctx->device = device;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) {
    fprintf(stderr, "dmosopt_b200: cudaSetDevice(%d) failed: %s\n", device, cudaGetErrorString(e));
    delete ctx;
    return DMO_ERR_CUDA;
  }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    delete ctx;
    return DMO_ERR_CUDA;
  }
  ctx->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess) {
    delete ctx;
    return DMO_ERR_CUDA;
  }
  // keep freed scratch memory cached in the default pool (stream-ordered allocator)
  if (cudaDeviceGetDefaultMemPool(&ctx->pool, device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  if (cudaMalloc((void**)&ctx->dev_flag, 4 * sizeof(int)) != cudaSuccess) {
    delete ctx;
    return DMO_ERR_CUDA;
  }
  cudaMemset(ctx->dev_flag, 0, 4 * sizeof(int));
  *out = ctx;
  return DMO_OK;
}

int dmo_destroy(dmo_ctx* ctx) {
  if (!ctx) return DMO_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->flush_buf) cudaFree(ctx->flush_buf);
  if (ctx->dev_flag) cudaFree(ctx->dev_flag);
  cudaEventDestroy(ctx->ev0);
  cudaEventDestroy(ctx->ev1);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
  return DMO_OK;
}

const char* dmo_last_error(dmo_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int dmo_synchronize(dmo_ctx* ctx) {
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  return DMO_OK;
}

void* dmo_stream(dmo_ctx* ctx) { return (void*)ctx->stream; }
int64_t dmo_launch_count(dmo_ctx* ctx) { return ctx->launches; }
int dmo_sm_count(dmo_ctx* ctx) { return ctx->sm_count; }

int dmo_timer_begin(dmo_ctx* ctx) {
  DMO_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  return DMO_OK;
}

int dmo_timer_end(dmo_ctx* ctx, float* ms) {
  DMO_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  DMO_CUDA(cudaEventSynchronize(ctx->ev1));
  DMO_CUDA(cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
  return DMO_OK;
}

int dmo_host_alloc(void** out, uint64_t bytes) {
  return cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault) == cudaSuccess ? DMO_OK : DMO_ERR_CUDA;
}
int dmo_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? DMO_OK : DMO_ERR_CUDA; }

int dmo_device_alloc(dmo_ctx* ctx, void** out, uint64_t bytes) {
  // stream-ordered, from the context's pool (release threshold = unlimited): a per-generation buffer costs
  // microseconds, not a cudaMalloc / cudaFree pair
  if (!ctx || !out) return DMO_ERR_ARG;
  DMO_CUDA(cudaSetDevice(ctx->device));
  DMO_CUDA(cudaMallocAsync(out, bytes ? bytes : 1, ctx->stream));
  return DMO_OK;
}
int dmo_device_free(dmo_ctx* ctx, void* p) {
  if (!ctx) return DMO_ERR_ARG;
  if (!p) return DMO_OK;
  DMO_CUDA(cudaFreeAsync(p, ctx->stream));
  return DMO_OK;
}

int dmo_memcpy(dmo_ctx* ctx, void* dst, const void* src, uint64_t bytes) {
  if (!ctx) return DMO_ERR_ARG;
  if (bytes == 0) return DMO_OK;
  DMO_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, ctx->stream));
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  const bool sd = dmo_is_device_ptr(src), dd = dmo_is_device_ptr(dst);
  if (!sd && dd) ctx->h2d_bytes += bytes;
  if (sd && !dd) ctx->d2h_bytes += bytes;
  return DMO_OK;
}

int dmo_transfer_bytes(dmo_ctx* ctx, uint64_t* h2d, uint64_t* d2h) {
  if (h2d) *h2d = ctx->h2d_bytes;
  if (d2h) *d2h = ctx->d2h_bytes;
  return DMO_OK;
}

int dmo_profile_enable(dmo_ctx* ctx, int on) {
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  for (auto& t : ctx->timers) {
    cudaEventDestroy(t.a);
    cudaEventDestroy(t.b);
  }
  ctx->timers.clear();
  ctx->profiling = on != 0;
  return DMO_OK;
}

// "name ms count" lines, one per timer name, summed over the scopes recorded since dmo_profile_enable(1)
int dmo_profile_report(dmo_ctx* ctx, char* buf, uint64_t cap) {
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  std::vector<std::string> names;
  std::vector<double> ms;
  std::vector<int> cnt;
  for (auto& t : ctx->timers) {
    float e = 0.f;
    if (cudaEventElapsedTime(&e, t.a, t.b) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    size_t k = 0;
    for (; k < names.size(); ++k)
      if (names[k] == t.name) break;
    if (k == names.size()) {
      names.push_back(t.name);
      ms.push_back(0.0);
      cnt.push_back(0);
    }
    ms[k] += e;
    cnt[k] += 1;
  }
  std::string out;
  for (size_t k = 0; k < names.size(); ++k) {
    char line[256];
    snprintf(line, sizeof(line), "%s %.6f %d\n", names[k].c_str(), ms[k], cnt[k]);
    out += line;
  }
  if (buf && cap) {
    snprintf(buf, cap, "%s", out.c_str());
  }
  return DMO_OK;
}

__global__ void round_f32_kernel(double* a, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = (double)(float)a[i];
}

// in-place float64 -> float32 -> float64 rounding of a DEVICE array: what storing survivors into the
// reference's float32 state arrays does (dmosopt/NSGA2.py:228-230 with MOASMO.py:64)
int dmo_round_f32(dmo_ctx* ctx, double* a, int64_t n) {
  DMO_CUDA(cudaSetDevice(ctx->device));
  if (n <= 0) return DMO_OK;
  DMO_REQUIRE(a && dmo_is_device_ptr(a), "round_f32: expects a device pointer");
  DMO_LAUNCH(round_f32_kernel, (unsigned)ceil_div(n, 256), 256, 0, a, n);
  DMO_CHECK_LAUNCH();
  return DMO_OK;
}

int dmo_flush_l2(dmo_ctx* ctx) {
  const size_t bytes = (size_t)256 << 20;  // 256 MiB > 126 MB L2
  if (!ctx->flush_buf) {
    DMO_CUDA(cudaMalloc(&ctx->flush_buf, bytes));
    ctx->flush_bytes = bytes;
  }
  DMO_CUDA(cudaMemsetAsync(ctx->flush_buf, 0, ctx->flush_bytes, ctx->stream));
  return DMO_OK;
}

}  // extern "C"
