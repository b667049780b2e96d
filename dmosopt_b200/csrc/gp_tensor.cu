// GP posterior variance on the 5th-generation tensor cores (DMO_GP_TENSOR, and the fast leg of DMO_GP_AUTO).
//
//   ||L^-1 K_*^T||^2 per candidate  ==  row sums of  D^2,   D[p][i] = sum_k K_*[p][k] * Linv[i][k]
//
// D is a dense (candidates x N_train) x N_train contraction, both operands k-contiguous ("TN").  It runs as
// tcgen05.mma kind::f16 with the accumulator in TMEM:
//   * split precision: every float operand x is carried as two fp16 numbers hi + lo (22 significand bits) after an
//     exact power-of-two scaling (per Linv row, per objective for K_*) that keeps both halves in fp16's normal range;
//     D accumulates hi*hi + hi*lo + lo*hi in fp32 (three MMAs per product, the lo*lo term is below fp32 resolution);
//   * A operand = K_* tile (2 x 128 candidates x 32 k), B operand = Linv tile (256 rows x 32 k), so one TMEM lane is
//     one candidate and the epilogue's sum of squares is a private per-thread accumulation (no cross-lane reduction);
//   * Linv is lower triangular: the row block [256 j, 256 j + 256) only needs k < 256 (j + 1) -- half the MMAs skipped;
//   * operand tiles arrive by TMA (cp.async.bulk.tensor, SWIZZLE_64B) into a 3-stage shared-memory ring, completion
//     on mbarriers; one elected thread issues the MMAs; tcgen05.commit releases the ring slots and publishes the
//     accumulator; four epilogue warps drain TMEM with tcgen05.ld;
//   * persistent CTAs (one per SM) walk a list of equal-cost work items in an L2-friendly order (gp_var_tc3_kernel).
//
// K_* itself is produced in fp32 (relative error ~1e-6 on K_*) by kstar_mean_kernel, which accumulates the mean from the same
// kernel values (packed fp32 over 16 training points, then float64, slices added in a fixed order: deterministic);
// kstar_tensor_kernel + mean_split_kernel are the fallback for shapes that kernel does not take.  Predicts without
// variance never write K_*: gp_mean_direct_kernel.
//
// Accuracy contract of this path: |var - var_ref| <= 1e-5 * prior variance and |mean - mean_ref| <= 1e-5 on
// well-conditioned posteriors (tests/test_gpu_parity.py); DMO_GP_AUTO (gp.cu) measures both against the float64 path
// on probe candidates per model and recomputes in float64 what this path cannot hold to 1e-5 relative.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cudaTypedefs.h>

#include "gp.cuh"

namespace {

constexpr int TM = 128;      // candidates per UMMA tile  (UMMA M, TMEM lanes)
constexpr int TN = 256;      // Linv rows per tile        (UMMA N, TMEM columns per accumulator)
constexpr int UK = 16;       // UMMA K for 16-bit inputs
constexpr int NTHREADS = 192;  // warp 0: TMA producer, warp 1: MMA issuer, warps 2..5: epilogue

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait: a protocol bug must not hang the GPU -- after ~2^22 polls the kernel flags an error and every later
// wait falls through immediately (results are then discarded by the host)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, volatile int* abort_flag) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3FFu) == 0u) {
      if (*abort_flag) return;
      if (spins > (1u << 22)) {
        *abort_flag = 1;
        return;
      }
    }
  }
}

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread
__device__ __forceinline__ void tc_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// kind::f16 instruction descriptor (cute::UMMA::InstrDescriptor): fp16 A/B (format 0), fp32 accumulate (c_format 1),
// both K-major, N >> 3 at [17,23), M >> 4 at [24,29)
constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);

// ------------------------------------------------------------------------------------------------ the GEMM
// The 256 candidates of a work item are two M = 128 sub-tiles that share every Linv tile, each with its own TMEM
// accumulator (2 x 256 columns).  k is staged 32 elements at a time (64-byte rows, SWIZZLE_64B), so that three 64 KiB
// stages fit.
//   * A work item is (objective, 256 candidates, PAIR of Linv row blocks {q, n_jt - 1 - q}): every item costs the same
//     n_jt + 1 k-blocks, so a static round-robin over the persistent CTAs has a tail of at most one item in
//     M * n_pb * ceil(n_jt / 2) (6144 at the BASELINE shape, 41.5 rounds on 148 SMs).
//   * Items are ordered (objective, candidate block, pair): the ceil(n_jt / 2) CTAs that hold the same candidate block
//     start together at k = 0 and walk k at the same (MMA-bound) rate, so one of them pulls a K_* tile from DRAM and the
//     others hit it in L2; inside an item the short row block goes first, so its K_* tiles are read again by the long one
//     right away.
namespace v3 {
constexpr int BM = 256, BN = 256, BK = 32, STAGES = 3;  // candidates per item, Linv rows per row block, k per stage
constexpr int TILE_BYTES = 256 * BK * 2;                // 16 KiB: 256 rows x 64 B
constexpr int STAGE_BYTES = 4 * TILE_BYTES;             // K* hi/lo + Linv hi/lo
constexpr size_t GEMM_SMEM = (size_t)STAGES * STAGE_BYTES + 1024 + 256;

// K-major SWIZZLE_64B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, mma_sm100_desc.hpp):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (unused for swizzled K-major: 1)
//   [32,46) stride byte offset >> 4 (8 rows x 64 B = 512 B between 8-row groups) | [46,48) version = 1
//   [61,64) layout type = 4 (SWIZZLE_64B)
__device__ __forceinline__ uint64_t make_sdesc64(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}

struct GemmParams3 {
  int M, n_pb, n_jt, n_q;
  int64_t k_rows, l_rows;
  const float* inv_scale;
  double* vnorm;  // [n_q][M][vn_ld]
  int64_t vn_ld;
  int* abort_flag;
};

__global__ void __launch_bounds__(NTHREADS, 1)
    gp_var_tc3_kernel(const __grid_constant__ CUtensorMap map_kh, const __grid_constant__ CUtensorMap map_kl,
                      const __grid_constant__ CUtensorMap map_lh, const __grid_constant__ CUtensorMap map_ll,
                      const GemmParams3 prm) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* tiles = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(tiles + (size_t)STAGES * STAGE_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* acc_full = bars + 2 * STAGES;
  uint64_t* acc_empty = bars + 2 * STAGES + 1;
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * STAGES + 2);
  volatile int* abort_flag = prm.abort_flag;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int per_m = prm.n_pb * prm.n_q;
  const int n_work = prm.M * per_m;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
        const int m = w / per_m, r = w - m * per_m;
        const int pb = r / prm.n_q, q = r - pb * prm.n_q;
        const int a_row = (int)(m * prm.k_rows + (int64_t)pb * BM);
        const int jhi = prm.n_jt - 1 - q;
        for (int s = 0; s < 2; ++s) {  // short row block first: its K_* tiles are read again right away by the long one
          const int jt = s ? jhi : q;
          if (s && q == jhi) break;
          const int b_row = (int)(m * prm.l_rows + (int64_t)jt * BN);
          const int nkc = (jt + 1) * (BN / BK);
          for (int kc = 0; kc < nkc; ++kc) {
            mbar_wait(&empty[stage], phase ^ 1u, abort_flag);
            uint8_t* st = tiles + (size_t)stage * STAGE_BYTES;
            mbar_expect_tx(&full[stage], STAGE_BYTES);
            tma_load_2d(&map_kh, &full[stage], st, kc * BK, a_row);
            tma_load_2d(&map_kl, &full[stage], st + TILE_BYTES, kc * BK, a_row);
            tma_load_2d(&map_lh, &full[stage], st + 2 * TILE_BYTES, kc * BK, b_row);
            tma_load_2d(&map_ll, &full[stage], st + 3 * TILE_BYTES, kc * BK, b_row);
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, acc_phase = 0;
      for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
        const int r = w % per_m;
        const int q = r % prm.n_q;
        const int jhi = prm.n_jt - 1 - q;
        for (int s = 0; s < 2; ++s) {
          const int jt = s ? jhi : q;
          if (s && q == jhi) break;
          mbar_wait(acc_empty, acc_phase ^ 1u, abort_flag);
          tc_fence_after();
          const int nkc = (jt + 1) * (BN / BK);
          for (int kc = 0; kc < nkc; ++kc) {
            mbar_wait(&full[stage], phase, abort_flag);
            tc_fence_after();
            const uint32_t sa = smem_u32(tiles + (size_t)stage * STAGE_BYTES);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const uint32_t d_tmem = tmem_base + h * BN;
              const uint32_t a_off = h * (128 * BK * 2);  // second sub-tile: rows 128..255 of the K* boxes
              const uint64_t a_hi = make_sdesc64(sa + a_off), a_lo = make_sdesc64(sa + TILE_BYTES + a_off);
              const uint64_t b_hi = make_sdesc64(sa + 2 * TILE_BYTES), b_lo = make_sdesc64(sa + 3 * TILE_BYTES);
#pragma unroll
              for (int ks = 0; ks < BK / UK; ++ks) {
                const uint64_t adv = (uint64_t)((ks * UK * 2) >> 4);
                tc_mma_f16(d_tmem, a_hi + adv, b_hi + adv, IDESC, (kc | ks) ? 1u : 0u);
                tc_mma_f16(d_tmem, a_hi + adv, b_lo + adv, IDESC, 1u);
                tc_mma_f16(d_tmem, a_lo + adv, b_hi + adv, IDESC, 1u);
              }
            }
            tc_commit(&empty[stage]);
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
          tc_commit(acc_full);
          acc_phase ^= 1u;
        }
      }
    }
  } else {
    const int quarter = warp & 3;
    uint32_t acc_phase = 0;
    for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
      const int m = w / per_m, r = w - m * per_m;
      const int pb = r / prm.n_q, q = r - pb * prm.n_q;
      const float* isc = prm.inv_scale + (int64_t)m * prm.l_rows;
      const int jhi = prm.n_jt - 1 - q;
      double total0 = 0.0, total1 = 0.0;
      for (int s = 0; s < 2; ++s) {
        const int jt = s ? jhi : q;
        if (s && q == jhi) break;
        mbar_wait(acc_full, acc_phase, abort_flag);
        tc_fence_after();
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t r0[32], r1[32];
          const uint32_t t_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + c0;
          tc_ld_32x32(t_addr, r0);
          tc_ld_32x32(t_addr + BN, r1);
          tc_wait_ld();
          const float* sc = isc + jt * BN + c0;
          // four independent fp32 partial sums per sub-tile over 8 squares each, folded into float64 every 32 columns:
          // the rounding of the sum of squares stays at the 2^-24 * sqrt(8) level instead of growing with N
          float p0[4] = {0.f, 0.f, 0.f, 0.f}, p1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const float sv = __ldg(sc + e);
            const float t0 = __uint_as_float(r0[e]) * sv, t1 = __uint_as_float(r1[e]) * sv;
            p0[e & 3] = fmaf(t0, t0, p0[e & 3]);
            p1[e & 3] = fmaf(t1, t1, p1[e & 3]);
          }
          total0 += ((double)p0[0] + (double)p0[1]) + ((double)p0[2] + (double)p0[3]);
          total1 += ((double)p1[0] + (double)p1[1]) + ((double)p1[2] + (double)p1[3]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty);
        acc_phase ^= 1u;
      }
      double* out = prm.vnorm + ((int64_t)q * prm.M + m) * prm.vn_ld + (int64_t)pb * BM + quarter * 32 + lane;
      out[0] = total0;
      out[128] = total1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}
}  // namespace v3

// ------------------------------------------------------------------------------------------------ operand preparation
// Linv row -> scaled fp16 hi / lo.  One block per (objective, row).
__global__ void split_linv_kernel(const double* __restrict__ Linv, int64_t Npad, int M, const int* __restrict__ k_exp,
                                  uint16_t* __restrict__ Lh, uint16_t* __restrict__ Ll, float* __restrict__ inv_scale) {
  const int64_t row = blockIdx.x;  // m * Npad + i
  const int m = (int)(row / Npad);
  const double* src = Linv + row * Npad;
  __shared__ double red[256];
  double mx = 0.0;
  for (int64_t k = threadIdx.x; k < Npad; k += blockDim.x) mx = fmax(mx, fabs(src[k]));
  red[threadIdx.x] = mx;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] = fmax(red[threadIdx.x], red[threadIdx.x + o]);
    __syncthreads();
  }
  mx = red[0];
  int e = 0;
  if (mx > 0.0) e = 13 - ilogb(mx);  // scaled row maximum lands in [2^13, 2^14): far from fp16 overflow (65504)
  const double s = scalbn(1.0, e);
  for (int64_t k = threadIdx.x; k < Npad; k += blockDim.x) {
    const float x = (float)(src[k] * s);  // power-of-two scaling is exact; float keeps 24 bits
    const __half h = __float2half_rn(x);
    const __half l = __float2half_rn(x - __half2float(h));
    Lh[row * Npad + k] = __half_as_ushort(h);
    Ll[row * Npad + k] = __half_as_ushort(l);
  }
  if (threadIdx.x == 0) inv_scale[row] = (mx > 0.0) ? (float)scalbn(1.0, -e - k_exp[m]) : 0.f;
}

constexpr int KT_TN = 128, KT_TP = 32;

// c * k(r): hardware approximations (sqrt.approx / ex2.approx, relative error ~2^-22 each) are inside the 2^-22 budget
// the hi + lo fp16 split of K_* has anyway
__device__ __forceinline__ float stationary_f(float s2, int kind) {
  if (kind == DMO_KERNEL_MATERN52) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(s2));
    const float K = r * 2.2360679774997896f;
    return fmaf(K, fmaf(K, 1.0f / 3.0f, 1.0f), 1.0f) * __expf(-K);
  }
  return __expf(-0.5f * s2);
}

// the same for a pair of squared distances, on the packed fp32 pipe (FMUL2 / FFMA2); the two MUFU ops per value stay scalar
__device__ __forceinline__ float2 stationary2_f(float2 s2, int kind) {
  float2 e;
  if (kind == DMO_KERNEL_MATERN52) {
    float2 r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r.x) : "f"(s2.x));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r.y) : "f"(s2.y));
    const float2 K = __fmul2_rn(r, make_float2(2.2360679774997896f, 2.2360679774997896f));
    const float2 one = make_float2(1.0f, 1.0f);
    const float2 p = __ffma2_rn(K, __ffma2_rn(K, make_float2(1.0f / 3.0f, 1.0f / 3.0f), one), one);
    const float2 t = __fmul2_rn(K, make_float2(-1.4426950408889634f, -1.4426950408889634f));  // exp(-K) = 2^(-K log2 e)
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(t.x));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(t.y));
    return __fmul2_rn(p, e);
  }
  const float2 t = __fmul2_rn(s2, make_float2(-0.5f * 1.4426950408889634f, -0.5f * 1.4426950408889634f));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(t.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(t.y));
  return e;
}

// K_* in fp32 -> scaled fp16 hi / lo.  Each thread owns two adjacent training points (their coordinates live in
// registers, results leave as packed half2), a block covers 256 training points x KT_TP candidates; the candidate
// tile is read from shared memory as 16-byte broadcasts (rows padded with zeros to DMAX coordinates, so the
// distance loops need no bounds tests and the LSU pipe carries a quarter of the instructions of scalar loads).
template <bool ISO, int DMAX>
__global__ void __launch_bounds__(KT_TN)
    kstar_tensor_kernel(const double* __restrict__ Xn, int64_t P, int64_t p_base, int64_t Pcpad,
                        const double* __restrict__ Xt, int64_t N, int d, int M, int kind,
                        const double* __restrict__ inv_ls, const double* __restrict__ constant,
                        const int* __restrict__ k_exp, int64_t ldk, int64_t plane, uint16_t* __restrict__ Kh,
                        uint16_t* __restrict__ Kl) {
  extern __shared__ __align__(16) float sxf[];  // [KT_TP][DMAX] candidate tile, then [M][DMAX] 1/l, [M] c * 2^kexp
  float* s_il = sxf + KT_TP * DMAX;
  float* s_c = s_il + M * DMAX;
  const int64_t n0 = ((int64_t)blockIdx.x * KT_TN + threadIdx.x) * 2;
  const int64_t pt0 = (int64_t)blockIdx.y * KT_TP;
  for (int t = threadIdx.x; t < KT_TP * DMAX; t += KT_TN) {
    const int64_t p = p_base + pt0 + t / DMAX;
    const int j = t % DMAX;
    sxf[t] = (p < P && j < d) ? (float)Xn[p * d + j] : 0.f;
  }
  for (int t = threadIdx.x; t < M * DMAX; t += KT_TN) {
    const int m = t / DMAX, j = t % DMAX;
    s_il[t] = j < d ? (float)inv_ls[m * d + j] : 0.f;
  }
  if (threadIdx.x < M) s_c[threadIdx.x] = scalbnf((float)constant[threadIdx.x], k_exp[threadIdx.x]);
  // training coordinates as packed pairs (two coordinates per 64-bit register pair): the distance loop runs on the
  // packed fp32 pipe, FADD2 + FFMA2 per two coordinates and point instead of 2 FADD + 2 FFMA
  float2 xa[DMAX / 2], xb[DMAX / 2];
#pragma unroll
  for (int j = 0; j < DMAX / 2; ++j) {
    const int j0 = 2 * j, j1 = 2 * j + 1;
    xa[j] = make_float2((j0 < d && n0 < N) ? (float)Xt[n0 * d + j0] : 0.f, (j1 < d && n0 < N) ? (float)Xt[n0 * d + j1] : 0.f);
    xb[j] = make_float2((j0 < d && n0 + 1 < N) ? (float)Xt[(n0 + 1) * d + j0] : 0.f,
                        (j1 < d && n0 + 1 < N) ? (float)Xt[(n0 + 1) * d + j1] : 0.f);
  }
  __syncthreads();
  const bool live_a = n0 < N, live_b = n0 + 1 < N;
  uint32_t* Kh32 = reinterpret_cast<uint32_t*>(Kh);
  uint32_t* Kl32 = reinterpret_cast<uint32_t*>(Kl);
  for (int q = 0; q < KT_TP; ++q) {
    const int64_t pl = pt0 + q;
    if (pl >= Pcpad || n0 >= ldk) break;
    const float4* xc = reinterpret_cast<const float4*>(sxf + q * DMAX);
    float sa = 0.f, sb = 0.f;
    if (ISO) {
      float2 acc_a0 = make_float2(0.f, 0.f), acc_a1 = acc_a0, acc_b0 = acc_a0, acc_b1 = acc_a0;  // independent chains
#pragma unroll
      for (int j = 0; j < DMAX / 4; ++j) {
        const float4 c = xc[j];
        const float2 c01 = make_float2(c.x, c.y), c23 = make_float2(c.z, c.w);
        const float2 da0 = __fadd2_rn(c01, make_float2(-xa[2 * j].x, -xa[2 * j].y));
        const float2 db0 = __fadd2_rn(c01, make_float2(-xb[2 * j].x, -xb[2 * j].y));
        const float2 da1 = __fadd2_rn(c23, make_float2(-xa[2 * j + 1].x, -xa[2 * j + 1].y));
        const float2 db1 = __fadd2_rn(c23, make_float2(-xb[2 * j + 1].x, -xb[2 * j + 1].y));
        acc_a0 = __ffma2_rn(da0, da0, acc_a0);
        acc_b0 = __ffma2_rn(db0, db0, acc_b0);
        acc_a1 = __ffma2_rn(da1, da1, acc_a1);
        acc_b1 = __ffma2_rn(db1, db1, acc_b1);
      }
      sa = (acc_a0.x + acc_a0.y) + (acc_a1.x + acc_a1.y);
      sb = (acc_b0.x + acc_b0.y) + (acc_b1.x + acc_b1.y);
    }
    for (int m = 0; m < M; ++m) {
      float2 rr;
      if (ISO) {
        const float il = s_il[m * DMAX];
        const float il2 = il * il;
        rr = __fmul2_rn(make_float2(sa, sb), make_float2(il2, il2));
      } else {
        const float4* il4 = reinterpret_cast<const float4*>(s_il + m * DMAX);
        float2 acc_a = make_float2(0.f, 0.f), acc_b = acc_a;
#pragma unroll
        for (int j = 0; j < DMAX / 4; ++j) {
          const float4 c = xc[j], il = il4[j];
          const float2 c01 = make_float2(c.x, c.y), c23 = make_float2(c.z, c.w);
          const float2 i01 = make_float2(il.x, il.y), i23 = make_float2(il.z, il.w);
          const float2 da0 = __fmul2_rn(__fadd2_rn(c01, make_float2(-xa[2 * j].x, -xa[2 * j].y)), i01);
          const float2 db0 = __fmul2_rn(__fadd2_rn(c01, make_float2(-xb[2 * j].x, -xb[2 * j].y)), i01);
          const float2 da1 = __fmul2_rn(__fadd2_rn(c23, make_float2(-xa[2 * j + 1].x, -xa[2 * j + 1].y)), i23);
          const float2 db1 = __fmul2_rn(__fadd2_rn(c23, make_float2(-xb[2 * j + 1].x, -xb[2 * j + 1].y)), i23);
          acc_a = __ffma2_rn(da0, da0, acc_a);
          acc_b = __ffma2_rn(db0, db0, acc_b);
          acc_a = __ffma2_rn(da1, da1, acc_a);
          acc_b = __ffma2_rn(db1, db1, acc_b);
        }
        rr = make_float2(acc_a.x + acc_a.y, acc_b.x + acc_b.y);
      }
      const float sc = s_c[m];
      const float2 kk = __fmul2_rn(stationary2_f(rr, kind), make_float2(sc, sc));  // c * k(r), scaled by 2^kexp (exact)
      const float ka = live_a ? kk.x : 0.f;
      const float kb = live_b ? kk.y : 0.f;
      const __half2 h = __floats2half2_rn(ka, kb);
      const float2 hf = __half22float2(h);
      const __half2 l = __floats2half2_rn(ka - hf.x, kb - hf.y);
      const int64_t o = (m * plane + pl * ldk + n0) >> 1;
      Kh32[o] = *reinterpret_cast<const uint32_t*>(&h);
      Kl32[o] = *reinterpret_cast<const uint32_t*>(&l);
    }
  }
}

// Mean-only posterior (what MOASMO.optimize asks for every generation: model.evaluate -> mean, MOASMO.py:107-108): K_* is
// never written.  A thread owns two candidates (coordinates in registers), the block walks its share of the training
// points through a shared-memory tile (16-byte broadcast reads, packed fp32 distance loops as in kstar_tensor_kernel),
// k(x, x_n) * (c alpha_n) is accumulated with packed FFMA over 32 training points and then folded into float64; the
// partial sums of the blockIdx.x slices are added in a fixed order by mean_finish_tc_kernel (deterministic).
constexpr int KM_T = 128, KM_Q = 256, KM_NS = 32, KM_D = 32;

__global__ void pad_xt_f32_kernel(const double* __restrict__ Xt, int64_t N, int d, int64_t Npad, float* __restrict__ Xtf) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= Npad * KM_D) return;
  const int64_t n = t / KM_D;
  const int j = (int)(t % KM_D);
  Xtf[t] = (n < N && j < d) ? (float)Xt[n * d + j] : 0.f;
}

__global__ void pad_calpha_f32_kernel(const double* __restrict__ alpha, const double* __restrict__ constant, int64_t N, int M,
                                      int64_t Npad, float* __restrict__ CAf) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)M * Npad) return;
  const int m = (int)(t / Npad);
  const int64_t n = t - (int64_t)m * Npad;
  CAf[t] = n < N ? (float)(constant[m] * alpha[(int64_t)m * N + n]) : 0.f;
}

// NJ: groups of four input dimensions that are evaluated (the tile always carries KM_D = 32 zero-padded coordinates)
template <bool ISO, int MT, int NJ>
__global__ void __launch_bounds__(KM_T, 4)
    gp_mean_direct_kernel(const double* __restrict__ Xn, int64_t P, int64_t p_base, const float* __restrict__ Xtf, int64_t N,
                          int64_t Npad, int64_t n_per_block, int d, int kind, const double* __restrict__ inv_ls,
                          const double* __restrict__ constant, const double* __restrict__ alpha,
                          double* __restrict__ mpart, int64_t mp_ld) {
  __shared__ __align__(16) float s_x[KM_NS * KM_D];
  __shared__ float s_al[MT * KM_NS];  // c_m * alpha_m[n] of the tile (zero beyond N)
  __shared__ __align__(16) float s_il[MT * KM_D];
  const int t = threadIdx.x;
  const int64_t qa = (int64_t)blockIdx.y * KM_Q + t, qb = qa + KM_T;  // candidate rows inside this chunk
  float2 ca[2 * NJ], cb[2 * NJ];
  {
    const int64_t pa = p_base + qa, pb = p_base + qb;
#pragma unroll
    for (int j = 0; j < 2 * NJ; ++j) {
      const int j0 = 2 * j, j1 = 2 * j + 1;
      ca[j] = make_float2((pa < P && j0 < d) ? (float)Xn[pa * d + j0] : 0.f, (pa < P && j1 < d) ? (float)Xn[pa * d + j1] : 0.f);
      cb[j] = make_float2((pb < P && j0 < d) ? (float)Xn[pb * d + j0] : 0.f, (pb < P && j1 < d) ? (float)Xn[pb * d + j1] : 0.f);
    }
  }
  for (int i = t; i < MT * KM_D; i += KM_T) {
    const int m = i / KM_D, j = i % KM_D;
    s_il[i] = j < d ? (float)inv_ls[m * d + j] : 0.f;
  }
  double sum_a[MT], sum_b[MT];
#pragma unroll
  for (int m = 0; m < MT; ++m) sum_a[m] = sum_b[m] = 0.0;
  const int64_t n_begin = (int64_t)blockIdx.x * n_per_block;
  const int64_t n_end = n_begin + n_per_block < Npad ? n_begin + n_per_block : Npad;
  for (int64_t n0 = n_begin; n0 < n_end; n0 += KM_NS) {
    __syncthreads();  // the previous tile has been consumed
    {
      const float4* src = reinterpret_cast<const float4*>(Xtf + n0 * KM_D);
      float4* dst = reinterpret_cast<float4*>(s_x);
      dst[t] = src[t];
      dst[t + KM_T] = src[t + KM_T];
    }
    for (int i = t; i < MT * KM_NS; i += KM_T) {
      const int m = i / KM_NS;
      const int64_t n = n0 + i % KM_NS;
      s_al[i] = n < N ? (float)(constant[m] * alpha[(int64_t)m * N + n]) : 0.f;
    }
    __syncthreads();
    if (ISO) {  // one squared distance per (candidate, training point), scaled per objective
      float2 acc[MT];
#pragma unroll
      for (int m = 0; m < MT; ++m) acc[m] = make_float2(0.f, 0.f);
#pragma unroll 2
      for (int i = 0; i < KM_NS; ++i) {
        const float4* xr = reinterpret_cast<const float4*>(s_x + i * KM_D);
        float2 a0 = make_float2(0.f, 0.f), a1 = a0, b0 = a0, b1 = a0;  // independent chains
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const float4 c = xr[j];
          const float2 c01 = make_float2(c.x, c.y), c23 = make_float2(c.z, c.w);
          const float2 da0 = __fadd2_rn(c01, make_float2(-ca[2 * j].x, -ca[2 * j].y));
          const float2 db0 = __fadd2_rn(c01, make_float2(-cb[2 * j].x, -cb[2 * j].y));
          const float2 da1 = __fadd2_rn(c23, make_float2(-ca[2 * j + 1].x, -ca[2 * j + 1].y));
          const float2 db1 = __fadd2_rn(c23, make_float2(-cb[2 * j + 1].x, -cb[2 * j + 1].y));
          a0 = __ffma2_rn(da0, da0, a0);
          b0 = __ffma2_rn(db0, db0, b0);
          a1 = __ffma2_rn(da1, da1, a1);
          b1 = __ffma2_rn(db1, db1, b1);
        }
        const float2 r2 = make_float2((a0.x + a0.y) + (a1.x + a1.y), (b0.x + b0.y) + (b1.x + b1.y));
#pragma unroll
        for (int m = 0; m < MT; ++m) {
          const float il = s_il[m * KM_D];
          const float il2 = il * il;
          const float al = s_al[m * KM_NS + i];
          acc[m] = __ffma2_rn(stationary2_f(__fmul2_rn(r2, make_float2(il2, il2)), kind), make_float2(al, al), acc[m]);
        }
      }
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        sum_a[m] += (double)acc[m].x;
        sum_b[m] += (double)acc[m].y;
      }
    } else {  // one length scale per dimension and objective: a pass over the tile per objective
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        const float4* il4 = reinterpret_cast<const float4*>(s_il + m * KM_D);
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll 2
        for (int i = 0; i < KM_NS; ++i) {
          const float4* xr = reinterpret_cast<const float4*>(s_x + i * KM_D);
          float2 aa = make_float2(0.f, 0.f), bb = aa;
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            const float4 c = xr[j], il = il4[j];
            const float2 c01 = make_float2(c.x, c.y), c23 = make_float2(c.z, c.w);
            const float2 i01 = make_float2(il.x, il.y), i23 = make_float2(il.z, il.w);
            const float2 da0 = __fmul2_rn(__fadd2_rn(c01, make_float2(-ca[2 * j].x, -ca[2 * j].y)), i01);
            const float2 db0 = __fmul2_rn(__fadd2_rn(c01, make_float2(-cb[2 * j].x, -cb[2 * j].y)), i01);
            const float2 da1 = __fmul2_rn(__fadd2_rn(c23, make_float2(-ca[2 * j + 1].x, -ca[2 * j + 1].y)), i23);
            const float2 db1 = __fmul2_rn(__fadd2_rn(c23, make_float2(-cb[2 * j + 1].x, -cb[2 * j + 1].y)), i23);
            aa = __ffma2_rn(da0, da0, aa);
            bb = __ffma2_rn(db0, db0, bb);
            aa = __ffma2_rn(da1, da1, aa);
            bb = __ffma2_rn(db1, db1, bb);
          }
          const float al = s_al[m * KM_NS + i];
          acc = __ffma2_rn(stationary2_f(make_float2(aa.x + aa.y, bb.x + bb.y), kind), make_float2(al, al), acc);
        }
        sum_a[m] += (double)acc.x;
        sum_b[m] += (double)acc.y;
      }
    }
  }
#pragma unroll
  for (int m = 0; m < MT; ++m) {
    mpart[((int64_t)blockIdx.x * MT + m) * mp_ld + qa] = sum_a[m];
    mpart[((int64_t)blockIdx.x * MT + m) * mp_ld + qb] = sum_b[m];
  }
}

// K_* producer fused with the mean (predicts with variance): the layout of gp_mean_direct_kernel (a thread owns two
// candidates) with 16-point tiles; besides accumulating k * (c alpha) the block stages the scaled hi / lo fp16 split of
// its 256 x 16 tile per objective in shared memory (rows of 10 words: 8-byte stores of four consecutive training points
// are conflict free) and writes it out as full 32-byte sectors.  Replaces kstar_tensor_kernel + mean_split_kernel
// (1.46 + 0.72 ms at the BASELINE shape): K_* is written once and not read back for the mean.
constexpr int KF_NS = 16, KF_LD = 10;

template <bool ISO, int MT>
__global__ void __launch_bounds__(KM_T, 3)
    kstar_mean_kernel(const double* __restrict__ Xn, int64_t P, int64_t p_base, const float* __restrict__ Xtf, int64_t N,
                      int64_t Npad, int64_t n_per_block, int d, int kind, const double* __restrict__ inv_ls,
                      const double* __restrict__ constant, const int* __restrict__ k_exp, const float* __restrict__ CAf,
                      int64_t plane, uint16_t* __restrict__ Kh, uint16_t* __restrict__ Kl, double* __restrict__ mpart,
                      int64_t mp_ld) {
  extern __shared__ __align__(16) uint32_t kf_stage[];  // [MT][2][KM_Q][KF_LD] words: (objective, hi / lo, candidate row)
  __shared__ __align__(16) float s_x[KF_NS * KM_D];
  __shared__ float s_al[MT * KF_NS];  // c_m * alpha_m[n] of the tile (zero beyond N)
  __shared__ float s_live[KF_NS];     // 1 for a training point, 0 for the padding columns (written as zeros)
  __shared__ __align__(16) float s_il[MT * KM_D];
  __shared__ float s_c[MT];           // c_m * 2^kexp_m: scale of the stored K_*
  const int t = threadIdx.x;
  const int64_t q_base = (int64_t)blockIdx.y * KM_Q;
  const int64_t qa = q_base + t, qb = qa + KM_T;
  float2 ca[KM_D / 2], cb[KM_D / 2];
  {
    const int64_t pa = p_base + qa, pb = p_base + qb;
#pragma unroll
    for (int j = 0; j < KM_D / 2; ++j) {
      const int j0 = 2 * j, j1 = 2 * j + 1;
      ca[j] = make_float2((pa < P && j0 < d) ? (float)Xn[pa * d + j0] : 0.f, (pa < P && j1 < d) ? (float)Xn[pa * d + j1] : 0.f);
      cb[j] = make_float2((pb < P && j0 < d) ? (float)Xn[pb * d + j0] : 0.f, (pb < P && j1 < d) ? (float)Xn[pb * d + j1] : 0.f);
    }
  }
  for (int i = t; i < MT * KM_D; i += KM_T) {
    const int m = i / KM_D, j = i % KM_D;
    s_il[i] = j < d ? (float)inv_ls[m * d + j] : 0.f;
  }
  if (t < MT) s_c[t] = scalbnf((float)constant[t], k_exp[t]);
  double sum_a[MT], sum_b[MT];
#pragma unroll
  for (int m = 0; m < MT; ++m) sum_a[m] = sum_b[m] = 0.0;
  const int64_t n_begin = (int64_t)blockIdx.x * n_per_block;
  const int64_t n_end = n_begin + n_per_block < Npad ? n_begin + n_per_block : Npad;
  uint32_t* row_a = kf_stage + (size_t)t * KF_LD;             // + (m * 2 + arr) * KM_Q * KF_LD
  uint32_t* row_b = kf_stage + (size_t)(t + KM_T) * KF_LD;
  // the next tile's training coordinates (one float4 per thread: KF_NS * KM_D / 4 == KM_T) and c * alpha values travel
  // through registers while the current tile is being worked on: no global-load latency between two barriers
  static_assert(KF_NS * KM_D / 4 == KM_T && 6 * KF_NS <= KM_T, "tile prefetch mapping");
  float4 px = reinterpret_cast<const float4*>(Xtf + n_begin * KM_D)[t];
  float pal = t < MT * KF_NS ? CAf[(int64_t)(t / KF_NS) * Npad + n_begin + t % KF_NS] : 0.f;
  __syncthreads();  // s_il, s_c
  reinterpret_cast<float4*>(s_x)[t] = px;
  if (t < MT * KF_NS) s_al[t] = pal;
  if (t < KF_NS) s_live[t] = (n_begin + t < N) ? 1.f : 0.f;
  __syncthreads();
  for (int64_t n0 = n_begin; n0 < n_end; n0 += KF_NS) {
    const bool more = n0 + KF_NS < n_end;
    if (more) {  // in flight during the tile's arithmetic
      px = reinterpret_cast<const float4*>(Xtf + (n0 + KF_NS) * KM_D)[t];
      if (t < MT * KF_NS) pal = CAf[(int64_t)(t / KF_NS) * Npad + n0 + KF_NS + t % KF_NS];
    }
    float2 acc[MT];
#pragma unroll
    for (int m = 0; m < MT; ++m) acc[m] = make_float2(0.f, 0.f);
#pragma unroll 1
    for (int i4 = 0; i4 < KF_NS; i4 += 4) {
      uint32_t wh_a[MT][2], wl_a[MT][2], wh_b[MT][2], wl_b[MT][2];  // four training points -> two half2 words each
#pragma unroll
      for (int u2 = 0; u2 < 2; ++u2) {
        float2 kv[2][MT];  // scaled kernel values of the pair of points (candidates a, b)
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int i = i4 + 2 * u2 + u;
          const float4* xr = reinterpret_cast<const float4*>(s_x + i * KM_D);
          float2 r2 = make_float2(0.f, 0.f);
          if (ISO) {
            float2 a0 = make_float2(0.f, 0.f), a1 = a0, b0 = a0, b1 = a0;
#pragma unroll
            for (int j = 0; j < KM_D / 4; ++j) {
              const float4 c = xr[j];
              const float2 c01 = make_float2(c.x, c.y), c23 = make_float2(c.z, c.w);
              const float2 da0 = __fadd2_rn(c01, make_float2(-ca[2 * j].x, -ca[2 * j].y));
              const float2 db0 = __fadd2_rn(c01, make_float2(-cb[2 * j].x, -cb[2 * j].y));
              const float2 da1 = __fadd2_rn(c23, make_float2(-ca[2 * j + 1].x, -ca[2 * j + 1].y));
              const float2 db1 = __fadd2_rn(c23, make_float2(-cb[2 * j + 1].x, -cb[2 * j + 1].y));
              a0 = __ffma2_rn(da0, da0, a0);
              b0 = __ffma2_rn(db0, db0, b0);
              a1 = __ffma2_rn(da1, da1, a1);
              b1 = __ffma2_rn(db1, db1, b1);
            }
            r2 = make_float2((a0.x + a0.y) + (a1.x + a1.y), (b0.x + b0.y) + (b1.x + b1.y));
          }
          const float live = s_live[i];
#pragma unroll
          for (int m = 0; m < MT; ++m) {
            float2 rr;
            if (ISO) {
              const float il = s_il[m * KM_D];
              const float il2 = il * il;
              rr = __fmul2_rn(r2, make_float2(il2, il2));
            } else {
              const float4* il4 = reinterpret_cast<const float4*>(s_il + m * KM_D);
              float2 aa = make_float2(0.f, 0.f), bb = aa;
#pragma unroll
              for (int j = 0; j < KM_D / 4; ++j) {
                const float4 c = xr[j], il = il4[j];
                const float2 c01 = make_float2(c.x, c.y), c23 = make_float2(c.z, c.w);
                const float2 i01 = make_float2(il.x, il.y), i23 = make_float2(il.z, il.w);
                const float2 da0 = __fmul2_rn(__fadd2_rn(c01, make_float2(-ca[2 * j].x, -ca[2 * j].y)), i01);
                const float2 db0 = __fmul2_rn(__fadd2_rn(c01, make_float2(-cb[2 * j].x, -cb[2 * j].y)), i01);
                const float2 da1 = __fmul2_rn(__fadd2_rn(c23, make_float2(-ca[2 * j + 1].x, -ca[2 * j + 1].y)), i23);
                const float2 db1 = __fmul2_rn(__fadd2_rn(c23, make_float2(-cb[2 * j + 1].x, -cb[2 * j + 1].y)), i23);
                aa = __ffma2_rn(da0, da0, aa);
                bb = __ffma2_rn(db0, db0, bb);
                aa = __ffma2_rn(da1, da1, aa);
                bb = __ffma2_rn(db1, db1, bb);
              }
              rr = make_float2(aa.x + aa.y, bb.x + bb.y);
            }
            const float2 k0 = stationary2_f(rr, kind);
            const float al = s_al[m * KF_NS + i];
            acc[m] = __ffma2_rn(k0, make_float2(al, al), acc[m]);
            const float sc = s_c[m] * live;
            kv[u][m] = __fmul2_rn(k0, make_float2(sc, sc));  // c * k(r), scaled by 2^kexp (exact); padding columns: 0
          }
        }
#pragma unroll
        for (int m = 0; m < MT; ++m) {  // pack (n, n + 1) of one candidate into half2: hi, then lo = value - hi
          const __half2 ha = __floats2half2_rn(kv[0][m].x, kv[1][m].x), hb = __floats2half2_rn(kv[0][m].y, kv[1][m].y);
          const float2 fa = __half22float2(ha), fb = __half22float2(hb);
          const __half2 la = __floats2half2_rn(kv[0][m].x - fa.x, kv[1][m].x - fa.y);
          const __half2 lb = __floats2half2_rn(kv[0][m].y - fb.x, kv[1][m].y - fb.y);
          wh_a[m][u2] = *reinterpret_cast<const uint32_t*>(&ha);
          wl_a[m][u2] = *reinterpret_cast<const uint32_t*>(&la);
          wh_b[m][u2] = *reinterpret_cast<const uint32_t*>(&hb);
          wl_b[m][u2] = *reinterpret_cast<const uint32_t*>(&lb);
        }
      }
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        const size_t oh = (size_t)(m * 2) * KM_Q * KF_LD + (i4 >> 1), ol = oh + (size_t)KM_Q * KF_LD;
        *reinterpret_cast<uint2*>(row_a + oh) = make_uint2(wh_a[m][0], wh_a[m][1]);
        *reinterpret_cast<uint2*>(row_a + ol) = make_uint2(wl_a[m][0], wl_a[m][1]);
        *reinterpret_cast<uint2*>(row_b + oh) = make_uint2(wh_b[m][0], wh_b[m][1]);
        *reinterpret_cast<uint2*>(row_b + ol) = make_uint2(wl_b[m][0], wl_b[m][1]);
      }
    }
#pragma unroll
    for (int m = 0; m < MT; ++m) {
      sum_a[m] += (double)acc[m].x;
      sum_b[m] += (double)acc[m].y;
    }
    __syncthreads();  // the tile is staged, its inputs have been consumed
    // flush: 8-byte units, four per 32-byte row segment (a warp writes eight full sectors per instruction); thread t
    // always moves unit t & 3 of rows (t >> 2) + 32 k, so every offset below is a compile-time constant or one add
    {
      const uint32_t* src = kf_stage + (size_t)(t >> 2) * KF_LD + 2 * (t & 3);
      const int64_t row0 = (q_base + (t >> 2)) * Npad + n0 + 4 * (t & 3);
      const int64_t kstep = (int64_t)32 * Npad;
#pragma unroll
      for (int ma = 0; ma < 2 * MT; ++ma) {
        uint16_t* dst = ((ma & 1) ? Kl : Kh) + (int64_t)(ma >> 1) * plane + row0;
#pragma unroll
        for (int k = 0; k < KM_Q / 32; ++k) {
          const uint2 v = *reinterpret_cast<const uint2*>(src + (size_t)(ma * KM_Q + k * 32) * KF_LD);
          *reinterpret_cast<uint2*>(dst) = v;
          dst += kstep;
        }
      }
    }
    if (more) {  // the next tile's inputs, from the registers filled above
      reinterpret_cast<float4*>(s_x)[t] = px;
      if (t < MT * KF_NS) s_al[t] = pal;
      if (t < KF_NS) s_live[t] = (n0 + KF_NS + t < N) ? 1.f : 0.f;
    }
    __syncthreads();  // stage drained, next inputs in place
  }
#pragma unroll
  for (int m = 0; m < MT; ++m) {
    mpart[((int64_t)blockIdx.x * MT + m) * mp_ld + qa] = sum_a[m];
    mpart[((int64_t)blockIdx.x * MT + m) * mp_ld + qb] = sum_b[m];
  }
}

// mean[p][m] = y_std * sum_n K_*[p][n] alpha[n] + y_mean from the split K_* (hi + lo = 22 bits): HBM-bound pass,
// one warp per (objective, candidate) row, float64 accumulation in a fixed order
__global__ void mean_split_kernel(const uint16_t* __restrict__ Kh, const uint16_t* __restrict__ Kl, int64_t Pc, int64_t N,
                                  int64_t ldk, int64_t plane, int M, const int* __restrict__ k_exp,
                                  const double* __restrict__ alpha, const double* __restrict__ ymean,
                                  const double* __restrict__ ystd, int64_t p_base, double* __restrict__ mean) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= Pc * M) return;
  const int m = (int)(w / Pc);
  const int64_t pl = w - (int64_t)m * Pc;
  const uint32_t* rh = reinterpret_cast<const uint32_t*>(Kh + m * plane + pl * ldk);
  const uint32_t* rl = reinterpret_cast<const uint32_t*>(Kl + m * plane + pl * ldk);
  const double* a = alpha + (int64_t)m * N;
  double s = 0.0;
#pragma unroll 8
  for (int64_t n2 = lane; 2 * n2 < N; n2 += 32) {  // two fp16 values per 32-bit load
    const uint32_t h = rh[n2], l = rl[n2];
    const float k0 = __half2float(__ushort_as_half((uint16_t)(h & 0xFFFFu))) + __half2float(__ushort_as_half((uint16_t)(l & 0xFFFFu)));
    const float k1 = __half2float(__ushort_as_half((uint16_t)(h >> 16))) + __half2float(__ushort_as_half((uint16_t)(l >> 16)));
    const int64_t n = 2 * n2;
    s += (double)k0 * a[n];
    if (n + 1 < N) s += (double)k1 * a[n + 1];
  }
  s = warp_sum(s);
  if (lane == 0) mean[(p_base + pl) * M + m] = ystd[m] * scalbn(s, -k_exp[m]) + ymean[m];
}

// mean[p][m] = y_std * sum over the training-set slices' partial sums of K_* alpha + y_mean (fixed order)
__global__ void mean_finish_tc_kernel(const double* __restrict__ mpart, int nplanes, int64_t Pc, int64_t ld, int M,
                                      const double* __restrict__ ymean, const double* __restrict__ ystd, int64_t p_base,
                                      double* __restrict__ mean) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= Pc * M) return;
  int64_t pl = t / M;
  int m = (int)(t - pl * M);
  double s = 0.0;
  for (int q = 0; q < nplanes; ++q) s += mpart[((int64_t)q * M + m) * ld + pl];
  mean[(p_base + pl) * M + m] = ystd[m] * s + ymean[m];
}

__global__ void var_finish_tc_kernel(const double* __restrict__ vnorm, int nplanes, int64_t Pc, int64_t ld, int M,
                                     const double* __restrict__ constant, const double* __restrict__ noise,
                                     const double* __restrict__ ystd, int64_t p_base, double* __restrict__ var) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= Pc * M) return;
  int64_t pl = t / M;
  int m = (int)(t - pl * M);
  double vn = 0.0;
  for (int q = 0; q < nplanes; ++q) vn += vnorm[((int64_t)q * M + m) * ld + pl];  // partial sums of the work items, fixed order
  double v = (constant[m] + noise[m]) - vn;
  if (v < 0.0) v = 0.0;
  double sd = sqrt(v * (ystd[m] * ystd[m]));
  var[(p_base + pl) * M + m] = sd * sd;
}

// ------------------------------------------------------------------------------------------------ host side
PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (PFN_cuTensorMapEncodeTiled_v12000)p;
  }
  return fn;
}

// 2-D fp16 tensor [rows][cols] (cols contiguous), box = box_rows x box_cols
int make_map(dmo_ctx* ctx, CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
             uint32_t box_cols, CUtensorMapSwizzle swz) {
  auto fn = get_encode_fn();
  if (!fn) return dmo_fail(ctx, DMO_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {cols * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return dmo_fail(ctx, DMO_ERR_CUDA, "cuTensorMapEncodeTiled failed with %d", (int)r);
  return DMO_OK;
}

int prepare_tensor_state(dmo_ctx* ctx, dmo_gp* gp) {
  if (gp->tensor_ready) return DMO_OK;
  const int M = gp->M;
  const int64_t Npad = gp->Npad;
  std::vector<int> kexp(M);
  for (int m = 0; m < M; ++m) {
    double c = gp->h_constant[m];
    kexp[m] = (c > 0.0) ? 13 - ilogb(c) : 13;  // scaled K_* <= 2^14
  }
  DMO_TRY(gp->Kexp.alloc(ctx, M));
  DMO_CUDA(cudaMemcpyAsync(gp->Kexp.p, kexp.data(), M * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));  // kexp is a stack vector
  DMO_TRY(gp->Lhi.alloc(ctx, (size_t)M * Npad * Npad));
  DMO_TRY(gp->Llo.alloc(ctx, (size_t)M * Npad * Npad));
  DMO_TRY(gp->Lscale.alloc(ctx, (size_t)M * Npad));
  DMO_LAUNCH(split_linv_kernel, (unsigned)(M * Npad), 256, 0, gp->Linv.p, Npad, M, gp->Kexp.p, gp->Lhi.p, gp->Llo.p,
             gp->Lscale.p);
  DMO_CHECK_LAUNCH();
  gp->tensor_ready = true;
  return DMO_OK;
}

// float copies of the training inputs and of c * alpha, zero padded to Npad (once per model)
int prepare_direct_state(dmo_ctx* ctx, dmo_gp* gp) {
  if (gp->Xtf.p && gp->CAf.p) return DMO_OK;
  const int64_t N = gp->N, Npad = gp->Npad;
  DMO_TRY(gp->Xtf.alloc(ctx, (size_t)Npad * KM_D));
  DMO_TRY(gp->CAf.alloc(ctx, (size_t)gp->M * Npad));
  DMO_LAUNCH(pad_xt_f32_kernel, (unsigned)ceil_div(Npad * KM_D, 256), 256, 0, gp->Xt.p, N, gp->d, Npad, gp->Xtf.p);
  DMO_LAUNCH(pad_calpha_f32_kernel, (unsigned)ceil_div((int64_t)gp->M * Npad, 256), 256, 0, gp->alpha.p, gp->constant.p, N, gp->M, Npad,
             gp->CAf.p);
  DMO_CHECK_LAUNCH();
  return DMO_OK;
}

// Slices of the training set per candidate block for the two kernels above: the grid (slices x candidate blocks) should
// fill whole waves of `slots` resident CTAs; a slice is a multiple of `tile` points and at least 256 of them.
int64_t pick_slices(int64_t n_qb, int64_t Npad, int tile, int64_t slots, int64_t* n_per_block) {
  int64_t best = 1;
  double best_eff = -1.0;
  *n_per_block = Npad;
  const int64_t smax = Npad / 256 > 1 ? Npad / 256 : 1;
  for (int64_t sp = 1; sp <= smax; ++sp) {
    const int64_t npb = ceil_div(ceil_div(Npad, sp), (int64_t)tile) * tile;
    const int64_t ns = ceil_div(Npad, npb);
    const int64_t blocks = ns * n_qb;
    const double eff = (double)blocks / (double)(ceil_div(blocks, slots) * slots);
    if (eff > best_eff + 0.02) {  // fewer slices (fewer partial sums) unless more of them fill the waves visibly better
      best_eff = eff;
      best = ns;
      *n_per_block = npb;
    }
  }
  return best;
}

// mean-only predict without K_* in memory (d <= 32, M <= 6): see gp_mean_direct_kernel
int gp_mean_direct(dmo_ctx* ctx, dmo_gp* gp, const double* dXn, int64_t P, double* d_mean) {
  const int64_t N = gp->N, Npad = gp->Npad;
  const int M = gp->M, d = gp->d;
  DMO_TRY(prepare_direct_state(ctx, gp));
  const int64_t n_qb = ceil_div(P, KM_Q);
  int64_t n_per_block = Npad;
  const int64_t nsplit = pick_slices(n_qb, Npad, KM_NS, (int64_t)4 * ctx->sm_count, &n_per_block);
  const int64_t ld = n_qb * KM_Q;
  DevBuf<double> mpart;
  DMO_TRY(mpart.alloc(ctx, (size_t)nsplit * M * ld));
  dim3 grid((unsigned)nsplit, (unsigned)n_qb);
  {
    ProfileScope ps_(ctx, "gp_mean_direct");
#define KM_LAUNCH(ISO_, MT_)                                                                                                  \
  do {                                                                                                                      \
    if (d <= 16)                                                                                                            \
      DMO_LAUNCH((gp_mean_direct_kernel<ISO_, MT_, 4>), grid, KM_T, 0, dXn, P, (int64_t)0, gp->Xtf.p, N, Npad, n_per_block, \
                 d, gp->kernel, gp->inv_ls.p, gp->constant.p, gp->alpha.p, mpart.p, ld);                                    \
    else                                                                                                                    \
      DMO_LAUNCH((gp_mean_direct_kernel<ISO_, MT_, 8>), grid, KM_T, 0, dXn, P, (int64_t)0, gp->Xtf.p, N, Npad, n_per_block, \
                 d, gp->kernel, gp->inv_ls.p, gp->constant.p, gp->alpha.p, mpart.p, ld);                                    \
  } while (0)
#define KM_SWITCH(ISO_)        \
  switch (M) {                 \
    case 1: KM_LAUNCH(ISO_, 1); break; \
    case 2: KM_LAUNCH(ISO_, 2); break; \
    case 3: KM_LAUNCH(ISO_, 3); break; \
    case 4: KM_LAUNCH(ISO_, 4); break; \
    case 5: KM_LAUNCH(ISO_, 5); break; \
    default: KM_LAUNCH(ISO_, 6); break; \
  }
    if (gp->isotropic) {
      KM_SWITCH(true)
    } else {
      KM_SWITCH(false)
    }
#undef KM_SWITCH
#undef KM_LAUNCH
  }
  DMO_LAUNCH(mean_finish_tc_kernel, (unsigned)ceil_div(P * M, 256), 256, 0, mpart.p, (int)nsplit, P, ld, M, gp->ymean.p,
             gp->ystd.p, (int64_t)0, d_mean);
  DMO_CHECK_LAUNCH();
  return DMO_OK;  // mpart is released in stream order
}

}  // namespace

int gp_predict_tensor(dmo_ctx* ctx, dmo_gp* gp, const double* dXn, int64_t P, double* d_mean, double* d_var) {
  const int64_t N = gp->N, Npad = gp->Npad;
  const int M = gp->M, d = gp->d;
  DMO_REQUIRE(M <= 16, "gp_predict(tensor): at most 16 objectives per model (got %d)", M);
  DMO_REQUIRE(d <= 64, "gp_predict(tensor): at most 64 input dimensions (got %d); use DMO_GP_FP64", d);
  DMO_REQUIRE(Npad % TN == 0, "gp_predict(tensor): internal padding error");
  if (!d_var && d <= KM_D && M <= 6)
    return gp_mean_direct(ctx, gp, dXn, P, d_mean);  // nothing but the mean is wanted: K_* stays in registers
  DMO_TRY(prepare_tensor_state(ctx, gp));
  constexpr int64_t BM = v3::BM;
  // candidate chunk: K_* hi/lo (2 x M x Pc x Npad fp16) within ~6 GiB
  int64_t Pc_max = ((int64_t)6 << 30) / ((int64_t)M * Npad * 4);
  Pc_max = (Pc_max / BM) * BM;
  if (Pc_max < BM) Pc_max = BM;
  const int64_t Pc_alloc = P < Pc_max ? ceil_div(P, BM) * BM : Pc_max;
  const int n_jt = (int)(Npad / v3::BN);
  const int n_q = (n_jt + 1) / 2;
  DevBuf<uint16_t> Kh, Kl;
  DevBuf<double> vnorm;
  DevBuf<int> abort_flag;
  DMO_TRY(Kh.alloc(ctx, (size_t)M * Pc_alloc * Npad));
  DMO_TRY(Kl.alloc(ctx, (size_t)M * Pc_alloc * Npad));
  DMO_TRY(vnorm.alloc(ctx, (size_t)n_q * M * Pc_alloc));
  DMO_TRY(abort_flag.alloc(ctx, 1));
  DMO_CUDA(cudaMemsetAsync(abort_flag.p, 0, sizeof(int), ctx->stream));
  CUtensorMap map_kh, map_kl, map_lh, map_ll;
  DMO_TRY(make_map(ctx, &map_kh, Kh.p, (uint64_t)M * Pc_alloc, (uint64_t)Npad, 256, v3::BK, CU_TENSOR_MAP_SWIZZLE_64B));
  DMO_TRY(make_map(ctx, &map_kl, Kl.p, (uint64_t)M * Pc_alloc, (uint64_t)Npad, 256, v3::BK, CU_TENSOR_MAP_SWIZZLE_64B));
  DMO_TRY(make_map(ctx, &map_lh, gp->Lhi.p, (uint64_t)M * Npad, (uint64_t)Npad, 256, v3::BK, CU_TENSOR_MAP_SWIZZLE_64B));
  DMO_TRY(make_map(ctx, &map_ll, gp->Llo.p, (uint64_t)M * Npad, (uint64_t)Npad, 256, v3::BK, CU_TENSOR_MAP_SWIZZLE_64B));
  DMO_CUDA(cudaFuncSetAttribute(v3::gp_var_tc3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)v3::GEMM_SMEM));
  const int64_t kplane = Pc_alloc * Npad;
  // K_* producer fused with the mean (d <= 32, M <= 6); per-dimension length scales with more than two objectives spill
  // in the fused kernel, so they take kstar_tensor_kernel + mean_split_kernel like the shapes it does not take at all
  const bool fused = d <= KM_D && M <= 6 && (gp->isotropic || M <= 2);
  DevBuf<double> mpart;
  if (fused) DMO_TRY(prepare_direct_state(ctx, gp));
  for (int64_t p_base = 0; p_base < P; p_base += Pc_alloc) {
    const int64_t Pc = (P - p_base) < Pc_alloc ? (P - p_base) : Pc_alloc;
    const int64_t Pcpad = ceil_div(Pc, BM) * BM;
    if (fused) {
      // K_* and the mean from one kernel (kstar_mean_kernel): K_* is written once and never read back for the mean
      int64_t n_per_block = Npad;
      const int64_t n_qb = Pcpad / KM_Q;
      const int64_t nsplit = pick_slices(n_qb, Npad, KF_NS, (int64_t)3 * ctx->sm_count, &n_per_block);
      DMO_TRY(mpart.alloc(ctx, (size_t)nsplit * M * Pcpad));
      dim3 gf((unsigned)nsplit, (unsigned)n_qb);
      const size_t smem = (size_t)M * 2 * KM_Q * KF_LD * sizeof(uint32_t);
      {
        ProfileScope ps_(ctx, "gp_kstar");
#define KF_LAUNCH(ISO_, MT_)                                                                                               \
  do {                                                                                                                     \
    DMO_CUDA(cudaFuncSetAttribute(kstar_mean_kernel<ISO_, MT_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  \
    DMO_LAUNCH((kstar_mean_kernel<ISO_, MT_>), gf, KM_T, smem, dXn, P, p_base, gp->Xtf.p, N, Npad, n_per_block, d,          \
               gp->kernel, gp->inv_ls.p, gp->constant.p, gp->Kexp.p, gp->CAf.p, kplane, Kh.p, Kl.p, mpart.p, Pcpad);         \
  } while (0)
#define KF_SWITCH(ISO_)                  \
  switch (M) {                           \
    case 1: KF_LAUNCH(ISO_, 1); break;   \
    case 2: KF_LAUNCH(ISO_, 2); break;   \
    case 3: KF_LAUNCH(ISO_, 3); break;   \
    case 4: KF_LAUNCH(ISO_, 4); break;   \
    case 5: KF_LAUNCH(ISO_, 5); break;   \
    default: KF_LAUNCH(ISO_, 6); break;  \
  }
        if (gp->isotropic) {
          KF_SWITCH(true)
        } else {
          KF_SWITCH(false)
        }
#undef KF_SWITCH
#undef KF_LAUNCH
      }
      DMO_LAUNCH(mean_finish_tc_kernel, (unsigned)ceil_div(Pc * M, 256), 256, 0, mpart.p, (int)nsplit, Pc, Pcpad, M, gp->ymean.p,
                 gp->ystd.p, p_base, d_mean);
    } else {
      {
        ProfileScope ps_(ctx, "gp_kstar");
        dim3 gk((unsigned)(Npad / (2 * KT_TN)), (unsigned)ceil_div(Pcpad, KT_TP));
        const int dmax = d <= 32 ? 32 : 64;
        size_t smem = (size_t)(KT_TP * dmax + M * dmax + M) * sizeof(float);
#define KSTAR_LAUNCH(ISO_, DM_)                                                                                 \
  DMO_LAUNCH((kstar_tensor_kernel<ISO_, DM_>), gk, KT_TN, smem, dXn, P, p_base, Pcpad, gp->Xt.p, N, d, M, gp->kernel, \
             gp->inv_ls.p, gp->constant.p, gp->Kexp.p, Npad, kplane, Kh.p, Kl.p)
        if (gp->isotropic) {
          if (d <= 32)
            KSTAR_LAUNCH(true, 32);
          else
            KSTAR_LAUNCH(true, 64);
        } else {
          if (d <= 32)
            KSTAR_LAUNCH(false, 32);
          else
            KSTAR_LAUNCH(false, 64);
        }
#undef KSTAR_LAUNCH
      }
      {
        ProfileScope ps_(ctx, "gp_mean");
        DMO_LAUNCH(mean_split_kernel, (unsigned)ceil_div(Pc * M * 32, 256), 256, 0, Kh.p, Kl.p, Pc, N, Npad, kplane, M,
                   gp->Kexp.p, gp->alpha.p, gp->ymean.p, gp->ystd.p, p_base, d_mean);
      }
    }
    if (d_var) {
      v3::GemmParams3 prm;
      prm.M = M;
      prm.n_pb = (int)(Pcpad / BM);
      prm.n_jt = n_jt;
      prm.n_q = n_q;
      prm.k_rows = Pc_alloc;
      prm.l_rows = Npad;
      prm.inv_scale = gp->Lscale.p;
      prm.vnorm = vnorm.p;
      prm.vn_ld = Pc_alloc;
      prm.abort_flag = abort_flag.p;
      const int n_work = prm.M * prm.n_pb * prm.n_q;
      const int grid = n_work < ctx->sm_count ? n_work : ctx->sm_count;
      {
        ProfileScope ps_(ctx, "gp_var");
        DMO_LAUNCH(v3::gp_var_tc3_kernel, grid, NTHREADS, v3::GEMM_SMEM, map_kh, map_kl, map_lh, map_ll, prm);
      }
      DMO_LAUNCH(var_finish_tc_kernel, (unsigned)ceil_div(Pc * M, 256), 256, 0, vnorm.p, n_q, Pc, Pc_alloc, M,
                 gp->constant.p, gp->noise.p, gp->ystd.p, p_base, d_var);
    }
  }
  DMO_CHECK_LAUNCH();
  int h_abort = 0;
  DMO_CUDA(cudaMemcpyAsync(&h_abort, abort_flag.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  if (h_abort) return dmo_fail(ctx, DMO_ERR_INTERNAL, "gp_predict(tensor): pipeline watchdog tripped (mbarrier wait timed out)");
  return DMO_OK;
}
