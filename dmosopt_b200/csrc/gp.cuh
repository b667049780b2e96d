// GP posterior state shared by gp.cu (float64 path) and gp_tensor.cu (tcgen05 path).
#pragma once
#include <vector>

#include "common.cuh"

struct dmo_gp {
  int64_t N = 0, Npad = 0;  // training points; padded to the variance tile edge
  int d = 0, M = 0, kernel = 0;
  bool isotropic = true;
  DevBuf<double> Xt;        // (N, d) normalised training inputs
  DevBuf<double> alpha;     // (M, N)
  DevBuf<double> Linv;      // (M, Npad, Npad) lower-triangular inverse Cholesky factors, zero padded
  DevBuf<double> inv_ls;    // (M, d) 1 / length_scale
  DevBuf<double> constant, noise, ymean, ystd;  // (M,)
  DevBuf<double> xlb, xrg;  // (d,)
  std::vector<double> h_constant, h_noise, h_ystd;
  // optional linear prior mean m(x) = w . x_n + b in the normalised-output space (gpytorch LinearMean, A19)
  bool has_linear_mean = false;
  DevBuf<double> lin_w, lin_b;  // (M, d), (M,)
  // tensor path (built lazily on first DMO_GP_TENSOR predict)
  bool tensor_ready = false;
  DevBuf<uint16_t> Lhi, Llo;  // (M, Npad, Npad) fp16 split of the row-scaled L^-1
  DevBuf<float> Lscale;       // (M, Npad) 1 / (row scale * K_* scale), powers of two
  DevBuf<int> Kexp;           // (M,) K_* scaling exponents
  DevBuf<float> Xtf;          // (Npad, 32) float copy of Xt, zero padded (mean-only direct kernel, d <= 32); built lazily
  DevBuf<float> CAf;          // (M, Npad) c_m * alpha_m as float, zero padded (fused K_* + mean kernel); built with Xtf
  // DMO_GP_AUTO: per-model calibration of the tensor path against the float64 path on probe candidates (gp.cu)
  bool calibrated = false;
  bool auto_mean_tensor = false;  // the tensor-path mean of predicts with variance holds 1e-5 on the probes (with margin)
  bool auto_var_tensor = false;   // split-fp16 variance holds 1e-5 * prior on the probes (with margin)
  double cal_mean_err = 0.0;      // max |mean_t - mean_64| / max(|mean_64|, y_std) over the probes
  bool auto_mean_only = false;    // the mean-only tensor-path call (direct kernel where it applies) holds 1e-5 on the probes
  double cal_mean_err_only = 0.0; // its probe error
  double cal_var_err = 0.0;       // max |var_t - var_64| / prior over the probes
  double refine_theta = 1.0;      // rows with var_t < theta * prior are recomputed in float64
  int64_t last_refined = 0;       // rows recomputed by the last DMO_GP_AUTO predict
};

int gp_predict_fp64(dmo_ctx* ctx, dmo_gp* gp, const double* dXn, int64_t P, double* d_mean, double* d_var);
int gp_predict_tensor(dmo_ctx* ctx, dmo_gp* gp, const double* dXn, int64_t P, double* d_mean, double* d_var);
