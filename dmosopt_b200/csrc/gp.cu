// Exact-GP posterior mean / variance (SURVEY.md section 8a row A18).
// Replaces GPR_Matern.predict / GPR_RBF.predict (dmosopt/model.py:1254-1275, 1343-1364), i.e. per objective
// sklearn GaussianProcessRegressor.predict(return_std=True) with ConstantKernel * Matern(2.5) [RBF] + WhiteKernel:
//     mean = y_std * (K_* alpha) + y_mean
//     var  = y_std^2 * max(0, (c + noise) - || L^-1 K_*^T ||^2_col)
// The variance contraction is evaluated in its triangular "GEMM form": V = L^-1 K_*^T with L^-1 formed once per
// epoch (dmo_gp_create), then a sum of squares per candidate -- all positive terms, so the only cancellation is the
// final subtraction from the prior variance.
//
// This file holds the float64 CUDA-core path (DMO_GP_FP64, the parity anchor, ~1e-10 of sklearn) and the object
// management; the tcgen05 split-precision path lives in gp_tensor.cu.
#include "gp.cuh"

namespace {

// ---- L^-1 (once per epoch, not on the per-generation path): blocked recursive inversion
//   inv([A 0; C B]) = [A^-1 0; -B^-1 C A^-1, B^-1].  The 128 x 128 diagonal blocks are inverted by forward substitution
//   (one thread per column), then log2(N/128) levels of batched float64 GEMMs double the inverted block size.
//   The matrix is embedded in a power-of-two multiple of 128 with an identity tail.
constexpr int TRI_B = 128;

__global__ void tri_embed_kernel(const double* __restrict__ L, int64_t N, int64_t Np, double* __restrict__ Lp) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= Np * Np) return;
  int64_t r = t / Np, c = t - r * Np;
  Lp[t] = (r < N && c < N) ? (c <= r ? L[r * N + c] : 0.0) : (r == c ? 1.0 : 0.0);
}

// one CTA per diagonal block, one thread per column of the block (L entries are warp-uniform loads, X column-coalesced)
__global__ void __launch_bounds__(TRI_B) tri_diag_inverse_kernel(const double* __restrict__ Lp, int64_t Np,
                                                                 double* __restrict__ X) {
  const int64_t base = (int64_t)blockIdx.x * TRI_B;
  const int c = threadIdx.x;
  const double* Lb = Lp + base * Np + base;
  double* Xb = X + base * Np + base;
  for (int i = 0; i < TRI_B; ++i) {
    double s = (i == c) ? 1.0 : 0.0;
    const double* Li = Lb + (int64_t)i * Np;
    for (int k = 0; k < i; ++k) {
      const double l = __ldg(Li + k);
      const double x = (k >= c) ? Xb[(int64_t)k * Np + c] : 0.0;
      s -= l * x;
    }
    Xb[(int64_t)i * Np + c] = (i >= c) ? s / __ldg(Li + i) : 0.0;
  }
}

// C = alpha * A * B, all row-major, batched over blockIdx.z; 64 x 64 tile, 16-wide k step, 256 threads x (4 x 4)
__global__ void __launch_bounds__(256) gemm_nn_f64_kernel(const double* __restrict__ A, int64_t lda, int64_t sA,
                                                          const double* __restrict__ B, int64_t ldb, int64_t sB,
                                                          double* __restrict__ C, int64_t ldc, int64_t sC, int64_t Msz,
                                                          int64_t Nsz, int64_t Ksz, double alpha) {
  __shared__ double As[16][64 + 1];
  __shared__ double Bs[16][64 + 1];
  A += (int64_t)blockIdx.z * sA;
  B += (int64_t)blockIdx.z * sB;
  C += (int64_t)blockIdx.z * sC;
  const int64_t m0 = (int64_t)blockIdx.y * 64, n0 = (int64_t)blockIdx.x * 64;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  double acc[4][4] = {};
  for (int64_t k0 = 0; k0 < Ksz; k0 += 16) {
    for (int t = tid; t < 64 * 16; t += 256) {
      const int r = t >> 4, k = t & 15;  // A tile: 64 rows x 16 k
      As[k][r] = A[(m0 + r) * lda + k0 + k];
      const int kb = t >> 6, cb = t & 63;  // B tile: 16 k x 64 cols
      Bs[kb][cb] = B[(k0 + kb) * ldb + n0 + cb];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      double a[4], b[4];
#pragma unroll
      for (int x = 0; x < 4; ++x) {
        a[x] = As[k][ty * 4 + x];
        b[x] = Bs[k][tx * 4 + x];
      }
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y] = fma(a[x], b[y], acc[x][y]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int x = 0; x < 4; ++x)
#pragma unroll
    for (int y = 0; y < 4; ++y) C[(m0 + ty * 4 + x) * ldc + n0 + tx * 4 + y] = alpha * acc[x][y];
  (void)Msz;
  (void)Nsz;
}

__global__ void tri_extract_kernel(const double* __restrict__ X, int64_t Np, int64_t N, int64_t ldo,
                                   double* __restrict__ out) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= N * N) return;
  int64_t r = t / N, c = t - r * N;
  out[r * ldo + c] = (c <= r) ? X[r * Np + c] : 0.0;
}

__global__ void copy_pad_kernel(const double* __restrict__ src, int64_t rows, int64_t cols, int64_t ldo,
                                double* __restrict__ dst) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows * cols) return;
  int64_t r = t / cols, c = t - r * cols;
  dst[r * ldo + c] = src[t];
}

__global__ void normalise_x_kernel(const double* __restrict__ X, int64_t P, int d, const double* __restrict__ xlb,
                                   const double* __restrict__ xrg, double* __restrict__ Xn) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= P * d) return;
  int j = (int)(t % d);
  Xn[t] = (X[t] - xlb[j]) / xrg[j];  // model.py:1262-1263
}

// ---- K_* tiles: Ks[m][p][n] = c_m * k(||x_p - x_n|| / l_m), float64 ---------------------------------------
constexpr int KS_TN = 128;  // train points per block (one per thread)
constexpr int KS_TP = 32;   // candidates per block
constexpr int KS_DMAX = 64; // input dimensions held in registers

__device__ __forceinline__ double stationary(double s2, int kind) {
  // s2 = squared scaled distance r^2
  if (kind == DMO_KERNEL_MATERN52) {
    double K = sqrt(s2) * 2.23606797749978969641;  // sqrt(5) r
    return (1.0 + K + K * K / 3.0) * exp(-K);
  }
  return exp(-0.5 * s2);
}

template <bool ISO>
__global__ void __launch_bounds__(KS_TN) kstar_kernel(const double* __restrict__ Xn, int64_t P, int64_t p_base,
                                                      int64_t Pc, const double* __restrict__ Xt, int64_t N, int d,
                                                      int M, int kind, const double* __restrict__ inv_ls,
                                                      const double* __restrict__ constant, int64_t ldk,
                                                      int64_t plane, double* __restrict__ Ks) {
  extern __shared__ double sx[];  // [KS_TP][d] candidate tile
  const int64_t n = (int64_t)blockIdx.x * KS_TN + threadIdx.x;
  const int64_t pt0 = (int64_t)blockIdx.y * KS_TP;  // within the chunk
  for (int t = threadIdx.x; t < KS_TP * d; t += KS_TN) {
    int64_t p = p_base + pt0 + t / d;
    sx[t] = (p < P) ? Xn[p * d + (t % d)] : 0.0;
  }
  double xt[KS_DMAX];
#pragma unroll
  for (int j = 0; j < KS_DMAX; ++j) xt[j] = (j < d && n < N) ? Xt[n * d + j] : 0.0;
  __syncthreads();
  if (n >= ldk) return;
  for (int q = 0; q < KS_TP; ++q) {
    const int64_t pl = pt0 + q;
    if (pl >= Pc) break;
    const double* xc = sx + q * d;
    if (ISO) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < KS_DMAX; ++j)
        if (j < d) {
          double df = xc[j] - xt[j];
          s += df * df;
        }
      for (int m = 0; m < M; ++m) {
        double il = inv_ls[m * d];
        double v = (n < N) ? constant[m] * stationary(s * il * il, kind) : 0.0;
        Ks[m * plane + pl * ldk + n] = v;
      }
    } else {
      for (int m = 0; m < M; ++m) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < KS_DMAX; ++j)
          if (j < d) {
            double df = (xc[j] - xt[j]) * inv_ls[m * d + j];
            s += df * df;
          }
        double v = (n < N) ? constant[m] * stationary(s, kind) : 0.0;
        Ks[m * plane + pl * ldk + n] = v;
      }
    }
  }
}

// ---- mean[p][m] = y_std * (Ks[m][p][:] . alpha[m]) + y_mean: one warp per row ---------------------------------
__global__ void mean_kernel(const double* __restrict__ Ks, int64_t Pc, int64_t N, int64_t ldk, int64_t plane, int M,
                            const double* __restrict__ alpha, const double* __restrict__ ymean,
                            const double* __restrict__ ystd, int64_t p_base, double* __restrict__ mean) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= Pc * M) return;
  const int m = (int)(w / Pc);
  const int64_t pl = w - (int64_t)m * Pc;
  const double* row = Ks + m * plane + pl * ldk;
  const double* a = alpha + (int64_t)m * N;
  double s = 0.0;
  for (int64_t n = lane; n < N; n += 32) s += row[n] * a[n];
  s = warp_sum(s);
  if (lane == 0) mean[(p_base + pl) * M + m] = ystd[m] * s + ymean[m];
}

// ---- variance: V = Linv . Ks^T tile by tile, column sums of V^2 -------------------------------------------------
// C[i][p] = sum_k Linv[i][k] Ks[p][k]  (both operands k-contiguous).  128 x 128 tile, 256 threads, 8 x 8 per thread.
// A thread's 8 rows / 8 columns are the interleaved sets {q*32 + t*2 + e : q<4, e<2} so that its double2 shared-memory
// reads are bank-conflict free (consecutive threads read consecutive 16-byte words).
constexpr int VB = 128;           // tile edge (rows of Linv and candidates)
constexpr int VK = 16;            // k step
constexpr int VLD = VB + 2;       // padded shared-memory row (doubles), even => 16-byte aligned rows
constexpr size_t VAR_SMEM = (size_t)2 * 2 * VK * VLD * sizeof(double);

__global__ void __launch_bounds__(256, 1)
    var_kernel(const double* __restrict__ Linv, int64_t ldl, int64_t lplane, const double* __restrict__ Ks, int64_t ldk,
               int64_t kplane, int64_t Npad, double* __restrict__ vnorm, int64_t Pcpad) {
  extern __shared__ __align__(16) double vsm[];
  double* As = vsm;                      // [2][VK][VLD]
  double* Bs = vsm + 2 * VK * VLD;       // [2][VK][VLD]
  const int m = blockIdx.y;
  const int64_t p0 = (int64_t)blockIdx.x * VB;
  const double* A = Linv + (int64_t)m * lplane;
  const double* B = Ks + (int64_t)m * kplane + p0 * ldk;
  const int tid = threadIdx.x;
  const int ti = tid >> 4, tj = tid & 15;  // 16 x 16 thread grid, 8 x 8 elements each
  const int lrow = tid >> 1;               // global->shared: each thread moves 8 doubles of A and of B per k step
  const int lk = (tid & 1) * 8;
  double vsum[8];
#pragma unroll
  for (int x = 0; x < 8; ++x) vsum[x] = 0.0;

  // row blocks of L^-1 are dealt round-robin over gridDim.z CTAs per candidate tile (small candidate sets -- AUTO's probe
  // and refinement calls -- would otherwise run on a handful of SMs); partial sums are combined in a fixed order
  const int64_t ntile = Npad / VB;
  for (int64_t it = blockIdx.z; it < ntile; it += gridDim.z) {
    const int64_t i0 = it * VB;
    const int64_t nk = (i0 + VB) / VK;  // L^-1 is lower triangular: row block `it` only touches k < i0 + VB
    double acc[8][8];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int b = 0; b < 8; ++b) acc[a][b] = 0.0;
    double ra[8], rb[8];
    {
      const double* ap = A + (i0 + lrow) * ldl + lk;
      const double* bp = B + (int64_t)lrow * ldk + lk;
#pragma unroll
      for (int x = 0; x < 8; ++x) {
        ra[x] = ap[x];
        rb[x] = bp[x];
      }
#pragma unroll
      for (int x = 0; x < 8; ++x) {
        As[(lk + x) * VLD + lrow] = ra[x];
        Bs[(lk + x) * VLD + lrow] = rb[x];
      }
    }
    __syncthreads();
    for (int64_t kt = 0; kt < nk; ++kt) {
      const int cur = (int)(kt & 1);
      const double* Ac = As + cur * VK * VLD;
      const double* Bc = Bs + cur * VK * VLD;
      if (kt + 1 < nk) {
        const double* ap = A + (i0 + lrow) * ldl + (kt + 1) * VK + lk;
        const double* bp = B + (int64_t)lrow * ldk + (kt + 1) * VK + lk;
#pragma unroll
        for (int x = 0; x < 8; ++x) {
          ra[x] = ap[x];
          rb[x] = bp[x];
        }
      }
#pragma unroll
      for (int k = 0; k < VK; ++k) {
        double a[8], b[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          double2 av = *reinterpret_cast<const double2*>(Ac + k * VLD + q * 32 + ti * 2);
          double2 bv = *reinterpret_cast<const double2*>(Bc + k * VLD + q * 32 + tj * 2);
          a[2 * q] = av.x;
          a[2 * q + 1] = av.y;
          b[2 * q] = bv.x;
          b[2 * q + 1] = bv.y;
        }
#pragma unroll
        for (int x = 0; x < 8; ++x)
#pragma unroll
          for (int y = 0; y < 8; ++y) acc[x][y] = fma(a[x], b[y], acc[x][y]);
      }
      if (kt + 1 < nk) {
        double* An = As + (cur ^ 1) * VK * VLD;
        double* Bn = Bs + (cur ^ 1) * VK * VLD;
#pragma unroll
        for (int x = 0; x < 8; ++x) {
          An[(lk + x) * VLD + lrow] = ra[x];
          Bn[(lk + x) * VLD + lrow] = rb[x];
        }
      }
      __syncthreads();
    }
#pragma unroll
    for (int y = 0; y < 8; ++y)
#pragma unroll
      for (int x = 0; x < 8; ++x) vsum[y] = fma(acc[x][y], acc[x][y], vsum[y]);
  }
  // reduce the 16 row-groups (ti) that share candidate columns; column of vsum[2q+e] is q*32 + tj*2 + e
  __syncthreads();
  double* red = vsm;  // 16 x 128 doubles
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    red[ti * VB + q * 32 + tj * 2 + 0] = vsum[2 * q];
    red[ti * VB + q * 32 + tj * 2 + 1] = vsum[2 * q + 1];
  }
  __syncthreads();
  if (tid < VB) {
    double s = 0.0;
#pragma unroll
    for (int r = 0; r < 16; ++r) s += red[r * VB + tid];
    vnorm[((int64_t)blockIdx.z * gridDim.y + m) * Pcpad + p0 + tid] = s;
  }
}

__global__ void var_finish_kernel(const double* __restrict__ vnorm, int nplanes, int64_t Pc, int64_t Pcpad, int M,
                                  const double* __restrict__ constant, const double* __restrict__ noise,
                                  const double* __restrict__ ystd, int64_t p_base, double* __restrict__ var) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= Pc * M) return;
  int64_t pl = t / M;
  int m = (int)(t - pl * M);
  double vn = 0.0;
  for (int z = 0; z < nplanes; ++z) vn += vnorm[((int64_t)z * M + m) * Pcpad + pl];  // row-block groups, fixed order
  double v = (constant[m] + noise[m]) - vn;  // kernel_.diag(X) - einsum(V^2)
  if (v < 0.0) v = 0.0;                                                  // sklearn clamps negative variances
  double sd = sqrt(v * (ystd[m] * ystd[m]));                             // sklearn returns the std ...
  var[(p_base + pl) * M + m] = sd * sd;                                  // ... dmosopt squares it (model.py:1267)
}

}  // namespace

int gp_predict_fp64(dmo_ctx* ctx, dmo_gp* gp, const double* dXn, int64_t P, double* d_mean, double* d_var) {
  const int64_t N = gp->N, Npad = gp->Npad;
  const int M = gp->M, d = gp->d;
  // candidate chunk so that Ks (M x Pc x Npad float64) stays within ~8 GiB
  int64_t budget = (int64_t)8 << 30;
  int64_t Pc_max = budget / ((int64_t)M * Npad * 8);
  Pc_max = (Pc_max / VB) * VB;
  if (Pc_max < VB) Pc_max = VB;
  const int64_t Pc_alloc = P < Pc_max ? ceil_div(P, VB) * VB : Pc_max;
  // split the row blocks of L^-1 over gridDim.z so that at least ~2 CTAs per SM exist even for a few hundred candidates
  const int64_t ntile = Npad / VB;
  int64_t nsplit = ceil_div((int64_t)2 * ctx->sm_count, (Pc_alloc / VB) * M);
  if (nsplit > ntile) nsplit = ntile;
  if (nsplit < 1) nsplit = 1;
  DevBuf<double> Ks, vnorm;
  DMO_TRY(Ks.alloc(ctx, (size_t)M * Pc_alloc * Npad));
  DMO_TRY(vnorm.alloc(ctx, (size_t)nsplit * M * Pc_alloc));
  const int64_t kplane = Pc_alloc * Npad;
  for (int64_t p_base = 0; p_base < P; p_base += Pc_alloc) {
    const int64_t Pc = (P - p_base) < Pc_alloc ? (P - p_base) : Pc_alloc;
    const int64_t Pcpad = ceil_div(Pc, VB) * VB;
    dim3 gk((unsigned)ceil_div(Npad, KS_TN), (unsigned)ceil_div(Pcpad, KS_TP));
    size_t smem = (size_t)KS_TP * d * sizeof(double);
    {
      ProfileScope ps(ctx, "gp_kstar");
      if (gp->isotropic)
      DMO_LAUNCH(kstar_kernel<true>, gk, KS_TN, smem, dXn, P, p_base, Pcpad, gp->Xt.p, N, d, M, gp->kernel,
                 gp->inv_ls.p, gp->constant.p, Npad, kplane, Ks.p);
    else
      DMO_LAUNCH(kstar_kernel<false>, gk, KS_TN, smem, dXn, P, p_base, Pcpad, gp->Xt.p, N, d, M, gp->kernel,
                 gp->inv_ls.p, gp->constant.p, Npad, kplane, Ks.p);
    }
    {
      ProfileScope ps(ctx, "gp_mean");
    DMO_LAUNCH(mean_kernel, (unsigned)ceil_div(Pc * M * 32, 256), 256, 0, Ks.p, Pc, N, Npad, kplane, M, gp->alpha.p,
               gp->ymean.p, gp->ystd.p, p_base, d_mean);
    }
    if (d_var) {
      ProfileScope ps(ctx, "gp_var");
      dim3 gv((unsigned)(Pcpad / VB), (unsigned)M, (unsigned)nsplit);
      DMO_CUDA(cudaFuncSetAttribute(var_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VAR_SMEM));
      DMO_LAUNCH(var_kernel, gv, 256, VAR_SMEM, gp->Linv.p, Npad, Npad * Npad, Ks.p, Npad, kplane, Npad, vnorm.p, Pc_alloc);
      DMO_LAUNCH(var_finish_kernel, (unsigned)ceil_div(Pc * M, 256), 256, 0, vnorm.p, (int)nsplit, Pc, Pc_alloc, M,
                 gp->constant.p, gp->noise.p, gp->ystd.p, p_base, d_var);
    }
  }
  DMO_CHECK_LAUNCH();
  return DMO_OK;
}

namespace {

// ---- DMO_GP_AUTO ---------------------------------------------------------------------------------------------
// The tensor path computes K_* in fp32 and the contraction in split-fp16 with fp32 accumulation: its errors are a few
// 1e-7 of the *operands*, so what reaches the posterior depends on the conditioning of the model (alpha and L^-1 of a
// fitted, nearly noise-free GP amplify them by orders of magnitude) and, for the variance, on how much of the prior
// cancels.  AUTO therefore measures instead of assuming: once per model, both paths predict the same 512 probe
// candidates (uniform in the unit cube, and training points displaced by 1e-4 .. 0.3) and
//   * the mean goes through fp32 K_* only if its probe error is <= 2.5e-6 of max(|mean|, y_std)  (bar: 1e-5, 4x margin);
//   * the variance goes through the tensor cores only if its probe error E is <= 4.5e-6 of the prior variance; rows whose
//     variance comes out below theta * prior, theta = max(0.02, 2 E / 1e-5), are then recomputed in float64, so every
//     returned variance is within 1e-5 of its own value (not just of the prior) -- the float64 path is the one that
//     matches scikit-learn to 1e-8.
constexpr int CAL_PROBES = 512;

__global__ void probe_points_kernel(const double* __restrict__ Xt, int64_t N, int d, int n_uniform, int n_total,
                                    double* __restrict__ Xn) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_total) return;
  Philox ph(0x9E3779B97F4A7C15ull);
  const uint4 h = ph((uint64_t)p, 0x51ull);
  const int64_t src = (int64_t)(h.x % (uint32_t)N);
  const double scale = pow(10.0, -4.0 + 3.5 * u01_53(h.y, h.z));
  for (int j = 0; j < d; ++j) {
    const uint4 r = ph((uint64_t)p, (uint64_t)(j + 1) << 8);
    const double u = u01_53(r.x, r.y);
    double x = u;
    if (p >= n_uniform) x = fmin(1.0, fmax(0.0, Xt[src * d + j] + scale * (2.0 * u - 1.0)));
    Xn[(int64_t)p * d + j] = x;
  }
}

__global__ void flag_small_var_kernel(const double* __restrict__ var, int64_t P, int M, const double* __restrict__ constant,
                                      const double* __restrict__ noise, const double* __restrict__ ystd, double theta,
                                      int32_t* __restrict__ flag) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  int f = 0;
  for (int m = 0; m < M; ++m) {
    const double prior = (constant[m] + noise[m]) * ystd[m] * ystd[m];
    if (!(var[p * M + m] >= theta * prior)) f = 1;  // NaN counts as small
  }
  flag[p] = f;
}

__global__ void compact_rows_kernel(const int32_t* __restrict__ flag, const int32_t* __restrict__ pos, int64_t P, int d,
                                    const double* __restrict__ Xn, int32_t* __restrict__ idx, double* __restrict__ Xsub) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P || !flag[p]) return;
  const int32_t o = pos[p];
  idx[o] = (int32_t)p;
  for (int j = 0; j < d; ++j) Xsub[(int64_t)o * d + j] = Xn[p * d + j];
}

__global__ void scatter_rows_kernel(const int32_t* __restrict__ idx, int64_t n, int M, const double* __restrict__ msub,
                                    const double* __restrict__ vsub, double* __restrict__ mean, double* __restrict__ var) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * M) return;
  const int64_t r = t / M;
  const int m = (int)(t - r * M);
  const int64_t p = idx[r];
  mean[p * M + m] = msub[t];
  var[p * M + m] = vsub[t];
}

int gp_calibrate(dmo_ctx* ctx, dmo_gp* gp) {
  if (gp->calibrated) return DMO_OK;
  const int M = gp->M, d = gp->d;
  const int P = CAL_PROBES;
  gp->auto_mean_tensor = gp->auto_var_tensor = gp->auto_mean_only = false;
  gp->cal_mean_err = gp->cal_var_err = gp->cal_mean_err_only = INFINITY;
  gp->refine_theta = 1.0;
  if (M > 16 || d > 64) {  // outside the tensor path's shape limits: float64 only
    gp->calibrated = true;
    return DMO_OK;
  }
  DevBuf<double> xn, m64, v64, mt, vt;
  DMO_TRY(xn.alloc(ctx, (size_t)P * d));
  DMO_TRY(m64.alloc(ctx, (size_t)P * M));
  DMO_TRY(v64.alloc(ctx, (size_t)P * M));
  DMO_TRY(mt.alloc(ctx, (size_t)P * M));
  DMO_TRY(vt.alloc(ctx, (size_t)P * M));
  DMO_LAUNCH(probe_points_kernel, (unsigned)ceil_div(P, 128), 128, 0, gp->Xt.p, gp->N, d, P / 2, P, xn.p);
  DMO_CHECK_LAUNCH();
  const bool prof = ctx->profiling;
  ctx->profiling = false;  // calibration launches are not part of any timed step
  DevBuf<double> mo;
  DMO_TRY(mo.alloc(ctx, (size_t)P * M));
  int rc = gp_predict_fp64(ctx, gp, xn.p, P, m64.p, v64.p);
  if (rc == DMO_OK) rc = gp_predict_tensor(ctx, gp, xn.p, P, mt.p, vt.p);
  if (rc == DMO_OK) rc = gp_predict_tensor(ctx, gp, xn.p, P, mo.p, nullptr);  // the mean-only call takes its own kernel
  ctx->profiling = prof;
  if (rc != DMO_OK) return rc;
  std::vector<double> h((size_t)4 * P * M), ho((size_t)P * M);
  DMO_CUDA(cudaMemcpyAsync(ho.data(), mo.p, (size_t)P * M * 8, cudaMemcpyDeviceToHost, ctx->stream));
  DMO_CUDA(cudaMemcpyAsync(h.data(), m64.p, (size_t)P * M * 8, cudaMemcpyDeviceToHost, ctx->stream));
  DMO_CUDA(cudaMemcpyAsync(h.data() + (size_t)P * M, v64.p, (size_t)P * M * 8, cudaMemcpyDeviceToHost, ctx->stream));
  DMO_CUDA(cudaMemcpyAsync(h.data() + (size_t)2 * P * M, mt.p, (size_t)P * M * 8, cudaMemcpyDeviceToHost, ctx->stream));
  DMO_CUDA(cudaMemcpyAsync(h.data() + (size_t)3 * P * M, vt.p, (size_t)P * M * 8, cudaMemcpyDeviceToHost, ctx->stream));
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  const double *a64 = h.data(), *b64 = a64 + (size_t)P * M, *at = b64 + (size_t)P * M, *bt = at + (size_t)P * M;
  double em = 0.0, ev = 0.0, eo = 0.0;
  for (int p = 0; p < P; ++p)
    for (int m = 0; m < M; ++m) {
      const double ys = gp->h_ystd[m];
      const double prior = (gp->h_constant[m] + gp->h_noise[m]) * ys * ys;
      const double dm = fabs(at[p * M + m] - a64[p * M + m]) / fmax(fabs(a64[p * M + m]), ys);
      const double dv = fabs(bt[p * M + m] - b64[p * M + m]) / prior;
      em = (dm > em || dm != dm) ? (dm != dm ? INFINITY : dm) : em;
      ev = (dv > ev || dv != dv) ? (dv != dv ? INFINITY : dv) : ev;
      const double dq = fabs(ho[p * M + m] - a64[p * M + m]) / fmax(fabs(a64[p * M + m]), ys);
      eo = (dq > eo || dq != dq) ? (dq != dq ? INFINITY : dq) : eo;
    }
  gp->cal_mean_err = em;
  gp->cal_mean_err_only = eo;
  gp->cal_var_err = ev;
  gp->auto_mean_tensor = em <= 2.5e-6;
  gp->auto_mean_only = eo <= 2.5e-6;
  gp->auto_var_tensor = gp->auto_mean_tensor && ev <= 4.5e-6;
  gp->refine_theta = fmax(0.02, 2.0 * ev / 1e-5);
  gp->calibrated = true;
  if (getenv("DMO_GP_VERBOSE"))
    fprintf(stderr, "dmosopt_b200: GP calibration (N=%lld d=%d M=%d): mean err K*alpha %.3e, mean-only kernel %.3e, var err/prior %.3e -> mean %s, var %s, theta %.3f\n",
            (long long)gp->N, d, M, em, eo, ev, gp->auto_mean_tensor ? "K*alpha pass" : "float64",
            gp->auto_var_tensor ? "tensor" : "float64", gp->refine_theta);
  return DMO_OK;
}

// AUTO predict on normalised inputs: tensor path where the calibration allows it, float64 for the rest
int gp_predict_auto(dmo_ctx* ctx, dmo_gp* gp, const double* dXn, int64_t P, double* d_mean, double* d_var) {
  DMO_TRY(gp_calibrate(ctx, gp));
  gp->last_refined = 0;
  if (d_var ? !gp->auto_var_tensor : !gp->auto_mean_only) {
    gp->last_refined = P;
    return gp_predict_fp64(ctx, gp, dXn, P, d_mean, d_var);
  }
  DMO_TRY(gp_predict_tensor(ctx, gp, dXn, P, d_mean, d_var));
  if (!d_var) return DMO_OK;
  const int M = gp->M, d = gp->d;
  DevBuf<int32_t> flag, pos;
  DMO_TRY(flag.alloc(ctx, (size_t)P + 1));
  DMO_TRY(pos.alloc(ctx, (size_t)P + 1));
  DMO_CUDA(cudaMemsetAsync(flag.p + P, 0, sizeof(int32_t), ctx->stream));
  DMO_LAUNCH(flag_small_var_kernel, (unsigned)ceil_div(P, 256), 256, 0, d_var, P, M, gp->constant.p, gp->noise.p, gp->ystd.p,
             gp->refine_theta, flag.p);
  DMO_TRY(prim_exclusive_sum_i32(ctx, flag.p, pos.p, P + 1));
  int32_t n_ref = 0;
  DMO_CUDA(cudaMemcpyAsync(&n_ref, pos.p + P, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  gp->last_refined = n_ref;
  if (n_ref == 0) return DMO_OK;
  DevBuf<int32_t> idx;
  DevBuf<double> xs, ms, vs;
  DMO_TRY(idx.alloc(ctx, (size_t)n_ref));
  DMO_TRY(xs.alloc(ctx, (size_t)n_ref * d));
  DMO_TRY(ms.alloc(ctx, (size_t)n_ref * M));
  DMO_TRY(vs.alloc(ctx, (size_t)n_ref * M));
  DMO_LAUNCH(compact_rows_kernel, (unsigned)ceil_div(P, 256), 256, 0, flag.p, pos.p, P, d, dXn, idx.p, xs.p);
  {
    ProfileScope ps(ctx, "gp_refine_fp64");
    DMO_TRY(gp_predict_fp64(ctx, gp, xs.p, n_ref, ms.p, vs.p));
  }
  DMO_LAUNCH(scatter_rows_kernel, (unsigned)ceil_div((int64_t)n_ref * M, 256), 256, 0, idx.p, (int64_t)n_ref, M, ms.p, vs.p,
             d_mean, d_var);
  DMO_CHECK_LAUNCH();
  return DMO_OK;
}

}  // namespace

extern "C" {

int dmo_gp_create(dmo_ctx* ctx, int64_t N, int d, int M, int kernel, const double* X_train, const double* alpha,
                  const double* factor, int factor_is_inverse, const double* constant, const double* length_scale,
                  const double* noise, const double* y_mean, const double* y_std, const double* xlb, const double* xub,
                  dmo_gp** out) {
  if (!ctx) return DMO_ERR_ARG;
  DMO_CUDA(cudaSetDevice(ctx->device));
  DMO_REQUIRE(out, "gp_create: null output");
  *out = nullptr;
  DMO_REQUIRE(N >= 1 && d >= 1 && d <= KS_DMAX && M >= 1 && M <= 16, "gp_create: unsupported shape N=%lld d=%d M=%d",
              (long long)N, d, M);
  DMO_REQUIRE(kernel == DMO_KERNEL_MATERN52 || kernel == DMO_KERNEL_RBF, "gp_create: unknown kernel %d", kernel);
  DMO_REQUIRE(X_train && alpha && factor && constant && length_scale && noise && y_mean && y_std && xlb && xub,
              "gp_create: null pointer");
  // host copies of the small parameter vectors (needed to derive 1/l, ranges, isotropy)
  std::vector<double> h_ls((size_t)M * d), h_lb(d), h_ub(d);
  DMO_CUDA(cudaMemcpy(h_ls.data(), length_scale, h_ls.size() * sizeof(double), cudaMemcpyDefault));
  DMO_CUDA(cudaMemcpy(h_lb.data(), xlb, d * sizeof(double), cudaMemcpyDefault));
  DMO_CUDA(cudaMemcpy(h_ub.data(), xub, d * sizeof(double), cudaMemcpyDefault));
  dmo_gp* gp = new dmo_gp();
  gp->N = N;
  gp->d = d;
  gp->M = M;
  gp->kernel = kernel;
  gp->Npad = ceil_div(N, 256) * 256;  // multiple of the fp64 tile (128) and of the tensor path's Linv tile (256)
  gp->isotropic = true;
  std::vector<double> h_inv((size_t)M * d), h_rg(d);
  for (int m = 0; m < M; ++m)
    for (int j = 0; j < d; ++j) {
      h_inv[(size_t)m * d + j] = 1.0 / h_ls[(size_t)m * d + j];
      if (h_ls[(size_t)m * d + j] != h_ls[(size_t)m * d]) gp->isotropic = false;
    }
  for (int j = 0; j < d; ++j) h_rg[j] = h_ub[j] - h_lb[j];
  int st = DMO_OK;
  auto fail = [&](int s) {
    delete gp;
    return s;
  };
#define GP_TRY(e)                    \
  do {                               \
    st = (e);                        \
    if (st != DMO_OK) return fail(st); \
  } while (0)
#define GP_CUDA(call)                                                                                 \
  do {                                                                                                \
    cudaError_t e__ = (call);                                                                         \
    if (e__ != cudaSuccess)                                                                           \
      return fail(dmo_fail(ctx, DMO_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__)));      \
  } while (0)
  const int64_t Npad = gp->Npad;
  GP_TRY(gp->Xt.alloc(ctx, (size_t)N * d));
  GP_TRY(gp->alpha.alloc(ctx, (size_t)M * N));
  GP_TRY(gp->Linv.alloc(ctx, (size_t)M * Npad * Npad));
  GP_TRY(gp->inv_ls.alloc(ctx, (size_t)M * d));
  GP_TRY(gp->constant.alloc(ctx, M));
  GP_TRY(gp->noise.alloc(ctx, M));
  GP_TRY(gp->ymean.alloc(ctx, M));
  GP_TRY(gp->ystd.alloc(ctx, M));
  GP_TRY(gp->xlb.alloc(ctx, d));
  GP_TRY(gp->xrg.alloc(ctx, d));
  GP_CUDA(cudaMemcpyAsync(gp->Xt.p, X_train, (size_t)N * d * sizeof(double), cudaMemcpyDefault, ctx->stream));
  GP_CUDA(cudaMemcpyAsync(gp->alpha.p, alpha, (size_t)M * N * sizeof(double), cudaMemcpyDefault, ctx->stream));
  GP_CUDA(cudaMemcpyAsync(gp->inv_ls.p, h_inv.data(), h_inv.size() * sizeof(double), cudaMemcpyDefault, ctx->stream));
  GP_CUDA(cudaMemcpyAsync(gp->constant.p, constant, M * sizeof(double), cudaMemcpyDefault, ctx->stream));
  GP_CUDA(cudaMemcpyAsync(gp->noise.p, noise, M * sizeof(double), cudaMemcpyDefault, ctx->stream));
  GP_CUDA(cudaMemcpyAsync(gp->ymean.p, y_mean, M * sizeof(double), cudaMemcpyDefault, ctx->stream));
  GP_CUDA(cudaMemcpyAsync(gp->ystd.p, y_std, M * sizeof(double), cudaMemcpyDefault, ctx->stream));
  GP_CUDA(cudaMemcpyAsync(gp->xlb.p, h_lb.data(), d * sizeof(double), cudaMemcpyDefault, ctx->stream));
  GP_CUDA(cudaMemcpyAsync(gp->xrg.p, h_rg.data(), d * sizeof(double), cudaMemcpyDefault, ctx->stream));
  GP_CUDA(cudaMemsetAsync(gp->Linv.p, 0, (size_t)M * Npad * Npad * sizeof(double), ctx->stream));
  {
    In<double> f;
    GP_TRY(f.init(ctx, factor, (size_t)M * N * N));
    for (int m = 0; m < M; ++m) {
      const double* src = f.d + (size_t)m * N * N;
      double* dst = gp->Linv.p + (size_t)m * Npad * Npad;
      if (factor_is_inverse) {
        DMO_LAUNCH(copy_pad_kernel, (unsigned)ceil_div(N * N, 256), 256, 0, src, N, N, Npad, dst);
      } else {
        int64_t Np = TRI_B;
        while (Np < N) Np *= 2;
        DevBuf<double> Lp, X, T;
        GP_TRY(Lp.alloc(ctx, (size_t)Np * Np));
        GP_TRY(X.alloc(ctx, (size_t)Np * Np));
        GP_TRY(T.alloc(ctx, (size_t)Np * Np / 2));
        GP_CUDA(cudaMemsetAsync(X.p, 0, (size_t)Np * Np * sizeof(double), ctx->stream));
        DMO_LAUNCH(tri_embed_kernel, (unsigned)ceil_div(Np * Np, 256), 256, 0, src, N, Np, Lp.p);
        DMO_LAUNCH(tri_diag_inverse_kernel, (unsigned)(Np / TRI_B), TRI_B, 0, Lp.p, Np, X.p);
        for (int64_t sz = TRI_B; sz < Np; sz *= 2) {
          const int64_t pairs = Np / (2 * sz);
          const int64_t stride = 2 * sz * Np + 2 * sz;  // next diagonal 2s x 2s block
          dim3 grid((unsigned)(sz / 64), (unsigned)(sz / 64), (unsigned)pairs);
          // T = C * A^-1        (C = Lp[s:2s, 0:s], A^-1 = X[0:s, 0:s])
          DMO_LAUNCH(gemm_nn_f64_kernel, grid, 256, 0, Lp.p + sz * Np, Np, stride, X.p, Np, stride, T.p, sz, sz * sz, sz, sz,
                     sz, 1.0);
          // X[s:2s, 0:s] = -B^-1 * T   (B^-1 = X[s:2s, s:2s])
          DMO_LAUNCH(gemm_nn_f64_kernel, grid, 256, 0, X.p + sz * Np + sz, Np, stride, T.p, sz, sz * sz, X.p + sz * Np, Np,
                     stride, sz, sz, sz, -1.0);
        }
        DMO_LAUNCH(tri_extract_kernel, (unsigned)ceil_div(N * N, 256), 256, 0, X.p, Np, N, Npad, dst);
        GP_CUDA(cudaGetLastError());
        GP_CUDA(cudaStreamSynchronize(ctx->stream));
      }
    }
    GP_CUDA(cudaGetLastError());
    GP_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  // host copies used by the tensor path's scaling
  gp->h_constant.resize(M);
  gp->h_noise.resize(M);
  gp->h_ystd.resize(M);
  GP_CUDA(cudaMemcpy(gp->h_constant.data(), constant, M * sizeof(double), cudaMemcpyDefault));
  GP_CUDA(cudaMemcpy(gp->h_noise.data(), noise, M * sizeof(double), cudaMemcpyDefault));
  GP_CUDA(cudaMemcpy(gp->h_ystd.data(), y_std, M * sizeof(double), cudaMemcpyDefault));
#undef GP_TRY
#undef GP_CUDA
  *out = gp;
  return DMO_OK;
}

int dmo_gp_destroy(dmo_ctx* ctx, dmo_gp* gp) {
  if (!ctx) return DMO_ERR_ARG;
  if (!gp) return DMO_OK;
  DMO_CUDA(cudaSetDevice(ctx->device));
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  delete gp;
  return DMO_OK;
}

// mean[p][m] += y_std[m] * (w_m . xn_p + b_m): the prior mean of a gpytorch ExactGP with LinearMean
__global__ void linear_mean_add_kernel(const double* __restrict__ Xn, int64_t P, int d, int M,
                                       const double* __restrict__ w, const double* __restrict__ b,
                                       const double* __restrict__ ystd, double* __restrict__ mean) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= P * M) return;
  const int64_t p = t / M;
  const int m = (int)(t - p * M);
  double s = b[m];
  for (int j = 0; j < d; ++j) s = fma(w[m * d + j], Xn[p * d + j], s);
  mean[t] += ystd[m] * s;
}

int dmo_gp_set_linear_mean(dmo_ctx* ctx, dmo_gp* gp, const double* weight, const double* bias) {
  if (!ctx) return DMO_ERR_ARG;
  DMO_CUDA(cudaSetDevice(ctx->device));
  DMO_REQUIRE(gp, "gp_set_linear_mean: null model");
  if (!weight && !bias) {
    gp->has_linear_mean = false;
    return DMO_OK;
  }
  DMO_REQUIRE(weight && bias, "gp_set_linear_mean: weight and bias must both be given (or both NULL)");
  In<double> w, b;
  DMO_TRY(w.init(ctx, weight, (size_t)gp->M * gp->d));
  DMO_TRY(b.init(ctx, bias, (size_t)gp->M));
  DMO_TRY(gp->lin_w.alloc(ctx, (size_t)gp->M * gp->d));
  DMO_TRY(gp->lin_b.alloc(ctx, (size_t)gp->M));
  DMO_CUDA(cudaMemcpyAsync(gp->lin_w.p, w.d, (size_t)gp->M * gp->d * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  DMO_CUDA(cudaMemcpyAsync(gp->lin_b.p, b.d, (size_t)gp->M * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  gp->has_linear_mean = true;
  return DMO_OK;
}

int dmo_gp_auto_info(dmo_ctx* ctx, dmo_gp* gp, int* mean_tensor, int* var_tensor, double* mean_err, double* var_err,
                     double* theta, int64_t* last_refined) {
  if (!ctx) return DMO_ERR_ARG;
  DMO_CUDA(cudaSetDevice(ctx->device));
  DMO_REQUIRE(gp, "gp_auto_info: null model");
  DMO_TRY(gp_calibrate(ctx, gp));
  if (mean_tensor) *mean_tensor = (gp->auto_mean_tensor ? 1 : 0) | (gp->auto_mean_only ? 4 : 0);
  if (var_tensor) *var_tensor = gp->auto_var_tensor ? 1 : 0;
  if (mean_err) *mean_err = gp->cal_mean_err;
  if (var_err) *var_err = gp->cal_var_err;
  if (theta) *theta = gp->refine_theta;
  if (last_refined) *last_refined = gp->last_refined;
  return DMO_OK;
}

int dmo_gp_predict(dmo_ctx* ctx, dmo_gp* gp, const double* X, int64_t P, double* mean, double* var, int precision) {
  if (!ctx) return DMO_ERR_ARG;
  DMO_CUDA(cudaSetDevice(ctx->device));
  DMO_REQUIRE(gp, "gp_predict: null model");
  if (P == 0) return DMO_OK;
  DMO_REQUIRE(P > 0 && X && mean, "gp_predict: bad arguments");
  In<double> x;
  Out<double> om, ov;
  DMO_TRY(x.init(ctx, X, (size_t)P * gp->d));
  DMO_TRY(om.init(ctx, mean, (size_t)P * gp->M));
  DMO_TRY(ov.init(ctx, var, (size_t)P * gp->M));
  DevBuf<double> xn;
  DMO_TRY(xn.alloc(ctx, (size_t)P * gp->d));
  DMO_LAUNCH(normalise_x_kernel, (unsigned)ceil_div(P * gp->d, 256), 256, 0, x.d, P, gp->d, gp->xlb.p, gp->xrg.p, xn.p);
  if (precision == DMO_GP_FP64) {
    DMO_TRY(gp_predict_fp64(ctx, gp, xn.p, P, om.d, ov.d));
  } else if (precision == DMO_GP_TENSOR) {
    DMO_TRY(gp_predict_tensor(ctx, gp, xn.p, P, om.d, ov.d));
  } else if (precision == DMO_GP_AUTO) {
    DMO_TRY(gp_predict_auto(ctx, gp, xn.p, P, om.d, ov.d));
  } else {
    return dmo_fail(ctx, DMO_ERR_ARG, "gp_predict: unknown precision %d", precision);
  }
  if (gp->has_linear_mean) {
    DMO_LAUNCH(linear_mean_add_kernel, (unsigned)ceil_div(P * gp->M, 256), 256, 0, xn.p, P, gp->d, gp->M, gp->lin_w.p,
               gp->lin_b.p, gp->ystd.p, om.d);
    DMO_CHECK_LAUNCH();
  }
  DMO_TRY(om.finish(ctx));
  DMO_TRY(ov.finish(ctx));
  DMO_CUDA(cudaStreamSynchronize(ctx->stream));
  return DMO_OK;
}

}  // extern "C"
