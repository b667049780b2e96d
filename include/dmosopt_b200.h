/*
 * dmosopt_b200 -- C ABI of the B200-native surrogate-generation hot path.
 *
 * The reference (dmosopt @ 5cd63e4c) is pure Python and has NO foreign-function
 * interface; this header is new surface that sits directly under the Python
 * plugin classes (dmosopt_b200.NSGA2 / AGEMOEA / SMPSO / CMAES, GPR_Matern ...)
 * which dmosopt loads by import path (dmosopt/config.py:5-11,
 * dmosopt/MOASMO.py:256-259,516-519).  Every entry point names the reference
 * function it replaces (file:line relative to the reference checkout).
 *
 * Conventions
 *   - plain C, no C++ / torch types; every function returns an int status
 *     (DMO_OK == 0) and never throws; dmo_last_error(ctx) gives the message.
 *   - matrices are row-major (C order), double unless stated; index outputs
 *     are int64 (numpy intp), ranks int32.
 *   - every array pointer may be HOST memory (pageable or pinned) or DEVICE
 *     memory of the context's GPU; the library detects which
 *     (cudaPointerGetAttributes) and stages host buffers through the
 *     context's stream.  The caller owns all buffers; the library owns only
 *     its context, its stream-ordered scratch memory and the objects it
 *     creates (dmo_gp).
 *   - one context per GPU and per calling thread (not re-entrant); all work is
 *     issued on the context's own stream and calls return after the results
 *     are in the caller's buffers (host outputs) or enqueued (device outputs;
 *     call dmo_synchronize before reading them from another stream).
 */
#ifndef DMOSOPT_B200_H
#define DMOSOPT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMO_OK 0
#define DMO_ERR_CUDA 1        /* a CUDA runtime call or kernel failed           */
#define DMO_ERR_ARG 2         /* bad shape / null pointer / unsupported size    */
#define DMO_ERR_STATE 3       /* object used before it was initialised          */
#define DMO_ERR_UNSUPPORTED 4 /* valid request that this build does not cover   */
#define DMO_ERR_INTERNAL 5    /* watchdog / consistency check tripped           */

/* distance metrics of MOEA.sortMO (dmosopt/MOEA.py:256-266) */
#define DMO_METRIC_NONE 0
#define DMO_METRIC_CROWDING 1  /* indicators.crowding_distance_metric  */
#define DMO_METRIC_EUCLIDEAN 2 /* indicators.euclidean_distance_metric */

/* stationary kernels of the sklearn surrogates (dmosopt/model.py:1227-1229, 1318-1320) */
#define DMO_KERNEL_MATERN52 0
#define DMO_KERNEL_RBF 1

/* arithmetic used for the GP posterior variance contraction */
#define DMO_GP_FP64 0   /* CUDA-core float64 everywhere: matches sklearn to ~1e-10               */
#define DMO_GP_TENSOR 1 /* tcgen05 split-fp16 (3 MMAs / product), fp32 accumulate in TMEM        */
#define DMO_GP_AUTO 2   /* tensor path where a per-model calibration against the float64 path   *
                         * holds 1e-5, float64 for the rest (rows with small variance, badly   *
                         * conditioned models): see dmo_gp_auto_info                            */

typedef struct dmo_ctx dmo_ctx;
typedef struct dmo_gp dmo_gp;

/* ---- context ----------------------------------------------------------- */
int dmo_version(void);
int dmo_create(int device, dmo_ctx** out);
int dmo_destroy(dmo_ctx* ctx);
const char* dmo_last_error(dmo_ctx* ctx);
int dmo_synchronize(dmo_ctx* ctx);
void* dmo_stream(dmo_ctx* ctx);             /* the context's cudaStream_t */
int64_t dmo_launch_count(dmo_ctx* ctx);     /* kernels launched by this context so far */
int dmo_sm_count(dmo_ctx* ctx);
/* CUDA-event stopwatch on the context's stream (bench.py times kernels with it) */
int dmo_timer_begin(dmo_ctx* ctx);
int dmo_timer_end(dmo_ctx* ctx, float* elapsed_ms);
/* pinned host memory for callers that want asynchronous staging */
int dmo_host_alloc(void** out, uint64_t bytes);
int dmo_host_free(void* p);
/* device memory for callers that keep populations resident */
int dmo_device_alloc(dmo_ctx* ctx, void** out, uint64_t bytes);
int dmo_device_free(dmo_ctx* ctx, void* p);
int dmo_memcpy(dmo_ctx* ctx, void* dst, const void* src, uint64_t bytes); /* any direction, stream ordered + sync */
/* bytes staged so far between host buffers and the GPU by this context */
int dmo_transfer_bytes(dmo_ctx* ctx, uint64_t* h2d, uint64_t* d2h);
/* per-kernel CUDA-event timers: enable(1) clears and starts recording, report() writes "name ms count" lines */
int dmo_profile_enable(dmo_ctx* ctx, int on);
int dmo_profile_report(dmo_ctx* ctx, char* buf, uint64_t cap);
/* in-place float64 -> float32 -> float64 rounding of a device array (the reference's float32 state arrays,
 * dmosopt/NSGA2.py:228-230 + dmosopt/MOASMO.py:64), for callers that keep the population resident */
int dmo_round_f32(dmo_ctx* ctx, double* a, int64_t n);
/* writes zeros through a scratch buffer larger than L2 (bench L2 flush) */
int dmo_flush_l2(dmo_ctx* ctx);

/* ---- A1/A2: non-dominated rank ------------------------------------------
 * replaces dda.dda_ens (dmosopt/dda.py:97-152), the rank used by every sortMO.
 * Y (n, M) -> rank (n,), the canonical Pareto front index; identical vectors are
 * mutually non-dominating (dda.py:108-115).  Equal to dda_ens whenever
 * objective 0 is tie-free.  1 <= M <= 8. */
int dmo_rank_nd(dmo_ctx* ctx, const double* Y, int64_t n, int M, int32_t* rank);

/* ---- A3/A4: distance metrics ---------------------------------------------
 * replace indicators.crowding_distance_metric (dmosopt/indicators.py:12-51) and
 * indicators.euclidean_distance_metric (:54-62).  Bit-identical float64. */
int dmo_crowding_distance(dmo_ctx* ctx, const double* Y, int64_t n, int M, double* D);
int dmo_euclidean_distance(dmo_ctx* ctx, const double* Y, int64_t n, int M, double* D);

/* ---- A5: sortMO / orderMO / remove_worst ----------------------------------
 * dmosopt/MOEA.py:242-347, 398-423.
 * dmo_order_mo: perm = np.lexsort((-extra_k..., -ydist, rank)); outputs are in sorted
 *   order.  extra_desc_keys: n_extra host-evaluated x-metrics (feasibility rank,
 *   NSGA2.py:47-49), each (n,), least-significant first; may be NULL.
 *   rank_sorted / dist_sorted may be NULL.
 * dmo_remove_worst: the first `keep` rows of that order gathered from X (n,d) / Y (n,M). */
int dmo_order_mo(dmo_ctx* ctx, const double* Y, int64_t n, int M, int metric,
                 const double* const* extra_desc_keys, int n_extra,
                 int64_t* perm, int32_t* rank_sorted, double* dist_sorted);
int dmo_remove_worst(dmo_ctx* ctx, const double* X, const double* Y, int64_t n, int d, int M,
                     int metric, const double* const* extra_desc_keys, int n_extra, int64_t keep,
                     double* X_out, double* Y_out, int32_t* rank_out, int64_t* perm_out);

/* dmo_remove_worst on the row-wise concatenation [A (na rows); B (nb rows)] without building it on the host
 * (NSGA2.update_strategy stacks the children over the parents, dmosopt/NSGA2.py:205-214). Outputs may alias B. */
int dmo_remove_worst_pair(dmo_ctx* ctx, const double* Xa, const double* Ya, int64_t na, const double* Xb,
                          const double* Yb, int64_t nb, int d, int M, int metric, int64_t keep,
                          double* X_out, double* Y_out, int32_t* rank_out, int64_t* perm_out);

/* ---- A6: tournament selection ---------------------------------------------
 * replaces MOEA.tournament_selection (dmosopt/MOEA.py:375-395): candidates ordered by
 * lexsort(metrics) (rank primary; AGE-MOEA adds -crowd_dist as secondary,
 * AGEMOEA.py:140-142), P(i-th best) ~ p (1-p)^i, poolsize draws WITHOUT replacement.
 * Implemented in log space (Gumbel-top-k), so it does not underflow for pop > 2150.
 * crowd may be NULL.  u_out (pop,) optionally receives the uniforms used, in candidate
 * order position (for distribution / replay tests). */
int dmo_tournament(dmo_ctx* ctx, const int32_t* rank, const double* crowd, int64_t pop,
                   int64_t poolsize, uint64_t seed, uint64_t stream_id,
                   int64_t* pool_idx, double* u_out);

/* ---- A7/A8: variation operators with explicit uniforms (kernel-level parity) ----
 * MOEA.mutation (dmosopt/MOEA.py:191-212) and MOEA.crossover_sbx (:215-239) applied
 * row-wise: parents / u / children (n, d); di_* / xlb / xub (d,). */
int dmo_mutation_u(dmo_ctx* ctx, const double* parents, const double* u, int64_t n, int d,
                   const double* di_mutation, const double* xlb, const double* xub,
                   double mutation_rate, double* children);
int dmo_sbx_u(dmo_ctx* ctx, const double* parent1, const double* parent2, const double* u,
              int64_t n, int d, const double* di_crossover, const double* xlb, const double* xub,
              double* child1, double* child2);

/* ---- A9: NSGA-II / AGE-MOEA offspring generation ----------------------------
 * replaces the serial loop of NSGA2.generate_strategy (dmosopt/NSGA2.py:142-178; same
 * loop in AGEMOEA.py:144-180): iteration t emits an SBX pair w.p. crossover_prob and
 * then a mutant w.p. mutation_prob, until count >= popsize-1.  The control flow is
 * planned in parallel from counter-based Philox4x32-10 draws (seed, stream_id).
 * pop_x (npop, d); pool_idx (poolsize,) rows of pop_x forming the mating pool.
 * x_gen has room for popsize+1 rows; child_kind (popsize+1,) gets 0/1 = SBX child 1/2,
 * 2 = mutant; n_children the number of rows produced.
 * draws (optional, may be NULL): receives the random draws actually used so the CPU
 * oracle can replay them: T * (5 + 2 d) doubles, T = dmo_nsga2_plan_length(...) planned
 * iterations, layout documented in dmosopt_b200/_lib.py (nsga2_generate).
 * dmo_nsga2_plan_length: the number of loop iterations planned for the given rates
 * (>= 2 popsize + 64; grows as 1 / (2 crossover_prob + mutation_prob) so that mutation-only
 * and low-rate configurations terminate like the reference's while-loop); -1 if the rates
 * are too small to plan. */
int64_t dmo_nsga2_plan_length(int64_t popsize, double crossover_prob, double mutation_prob);
int dmo_nsga2_generate(dmo_ctx* ctx, const double* pop_x, int64_t npop, int d,
                       const int64_t* pool_idx, int64_t poolsize, int64_t popsize,
                       double crossover_prob, double mutation_prob, double mutation_rate,
                       const double* di_crossover, const double* di_mutation,
                       const double* xlb, const double* xub, uint64_t seed, uint64_t stream_id,
                       double* x_gen, int32_t* child_kind, int64_t* n_children, double* draws);

/* ---- A10 + A20: one resident NSGA-II surrogate generation ----------------------
 * the body of MOASMO.optimize's loop (dmosopt/MOASMO.py:105-116) for NSGA2 (dmosopt/NSGA2.py:116-236) with a
 * GP surrogate, population resident in HBM: tournament -> variation -> GP posterior mean [+ variance] ->
 * vstack(children, parents) -> rank + stable truncation -> float32 rounding of the stored objectives
 * (NSGA2.py:228-230) -> optional hypervolume of the survivors (hv_ref / hv_out host pointers, may be NULL).
 * pop_x (pop,d), pop_y (pop,M), rank (pop,) are DEVICE buffers, updated in place; Philox streams
 * stream_id (tournament) and stream_id + 1 (variation) are consumed; n_children (host) receives P.
 * distance_metric: DMO_METRIC_* used to break rank ties in the truncation (NSGA2's own default is
 * "crowding", NSGA2.py:25; MOASMO.epoch constructs it with distance_metric=None, MOASMO.py:370). */
int dmo_nsga2_step(dmo_ctx* ctx, dmo_gp* gp, double* pop_x, double* pop_y, int32_t* rank, int64_t pop,
                   int d, int M, double crossover_prob, double mutation_prob, double mutation_rate,
                   const double* di_crossover, const double* di_mutation, const double* xlb,
                   const double* xub, uint64_t seed, uint64_t stream_id, int precision,
                   int distance_metric, int with_variance, int round_to_f32, const double* hv_ref,
                   int64_t* n_children, double* hv_out);

/* ---- A18: exact-GP posterior (GPR_Matern / GPR_RBF predict) -------------------
 * replaces GPR_Matern.predict / .evaluate (dmosopt/model.py:1254-1275; GPR_RBF :1343-1364),
 * i.e. per objective sklearn GaussianProcessRegressor.predict(return_std=True) ** 2.
 * dmo_gp_create uploads the posterior state once per epoch:
 *   X_train (N,d) normalised inputs; alpha (M,N); L (M,N,N) lower Cholesky factors of
 *   K + noise I (factor_is_inverse = 0) or their inverses L^-1 (factor_is_inverse = 1);
 *   constant (M,), length_scale (M,d) (isotropic = the scalar repeated), noise (M,),
 *   y_mean (M,), y_std (M,), xlb / xub (d,) raw input bounds.
 * dmo_gp_predict: X (P,d) raw inputs -> mean (P,M), var (P,M) (var may be NULL). */
int dmo_gp_create(dmo_ctx* ctx, int64_t N, int d, int M, int kernel, const double* X_train,
                  const double* alpha, const double* factor, int factor_is_inverse,
                  const double* constant, const double* length_scale, const double* noise,
                  const double* y_mean, const double* y_std, const double* xlb, const double* xub,
                  dmo_gp** out);
int dmo_gp_destroy(dmo_ctx* ctx, dmo_gp* gp);
/* N1: the exact-GP fit for given hyper-parameters, per objective m: K = c_m k(X, X; l_m) + (noise_m + jitter) I,
 * L = chol(K), alpha = K^-1 y_m, lml = log p(y_m | theta) -- what GaussianProcessRegressor.fit /
 * .log_marginal_likelihood compute behind GPR_Matern.__init__ (dmosopt/model.py:1214-1251) and what every trial of the
 * SCE-UA hyper-parameter search evaluates (dmosopt/model.py:1419-1753).  X_train (N,d) normalised inputs, y (M,N)
 * normalised targets; scikit-learn's jitter is 1e-10 (its alpha parameter).  L_out (M,N,N), alpha_out (M,N), lml_out (M,)
 * may each be NULL (an SCE-UA trial needs lml only).  Fails with DMO_ERR_ARG when K is not positive definite. */
int dmo_gp_fit(dmo_ctx* ctx, int64_t N, int d, int M, int kernel, const double* X_train, const double* y,
               const double* constant, const double* length_scale, const double* noise, double jitter,
               double* L_out, double* alpha_out, double* lml_out);
/* A19: prior mean of the gpytorch exact GPs (model_gpytorch.EGP_Matern.predict,
 * dmosopt/model_gpytorch.py:2188-2228; GPyTorchExactGPModelMatern with LinearMean, :455-508):
 * after this call dmo_gp_predict returns y_std * (K_* alpha + weight_m . x_n + bias_m) + y_mean,
 * x_n the normalised input; alpha must then be (K + noise I)^-1 (y_n - X_n weight - bias).
 * weight (M,d), bias (M,); both NULL removes the term.  The variance is unaffected. */
int dmo_gp_set_linear_mean(dmo_ctx* ctx, dmo_gp* gp, const double* weight, const double* bias);
int dmo_gp_predict(dmo_ctx* ctx, dmo_gp* gp, const double* X, int64_t P, double* mean,
                   double* var, int precision);
/* What DMO_GP_AUTO decided for this model (runs the one-off calibration if it has not run yet):
 * both arithmetic paths predict 512 probe candidates; mean_tensor bit 0 = the fp32-K_* alpha pass is
 * admitted (predicts with variance), bit 1 is reserved (always 0), bit 2 = the mean-only kernel (K_* never
 * written, fp32 kernel values, float64 partial sums) is admitted for predicts without variance;
 * var_tensor = 1 when the tcgen05 variance is admitted; errors relative to max(|mean|, y_std) and to
 * the prior variance, margins documented in csrc/gp.cu; theta: rows whose tensor variance is
 * below theta * prior are recomputed in float64; last_refined: rows the last AUTO predict recomputed
 * (= P when the whole call ran in float64).  Any output pointer may be NULL. */
int dmo_gp_auto_info(dmo_ctx* ctx, dmo_gp* gp, int* mean_tensor, int* var_tensor, double* mean_err,
                     double* var_err, double* theta, int64_t* last_refined);

/* ---- A16: exact hypervolume ---------------------------------------------------
 * replaces hv.AdaptiveHyperVolume.compute_hypervolume(..., 'box') (dmosopt/hv.py:123-189)
 * -> HyperVolumeBoxDecomposition.compute_hypervolume (dmosopt/hv_box_decomposition.py:86-304)
 * and indicators.Hypervolume._do (dmosopt/indicators.py:244-256).  Minimisation; points not
 * strictly inside ref are ignored (hv.py:159).  True hypervolume (see DESIGN.md for the
 * reference's <=0-coordinate defect).  1 <= M <= 8: chain sums for M <= 5 (M >= 4 is
 * O(n^(M-1))), limit-set recursion for 6 .. 8 objectives (fronts of up to 2048 points; exponential in the worst case, as
 * every exact algorithm, cheap on the mostly non-dominated fronts an optimizer produces). */
int dmo_hypervolume(dmo_ctx* ctx, const double* F, int64_t n, int M, const double* ref, double* out);
/* The same for a set that carries its non-dominated ranks within the superset it was selected from by rank
 * (the survivors of dmo_remove_worst / MOEA.remove_worst, dmosopt/MOEA.py:398-423): rows with rank > 0 are dominated
 * by a rank-0 row of the same set and add no volume, so the non-dominated filter pass is skipped.  rank (n,) int32. */
int dmo_hypervolume_ranked(dmo_ctx* ctx, const double* F, int64_t n, int M, const double* ref,
                           const int32_t* rank, double* out);

/* ---- A17: HV-improvement (EHVI) candidate selection -----------------------------
 * replaces indicators.HypervolumeImprovement._do (dmosopt/indicators.py:295-313) ->
 * HyperVolumeBoxDecomposition.select_candidates / _compute_batch_ehvi /
 * _decompose_dominated_space (dmosopt/hv_box_decomposition.py:306-437).
 * F (nf,M): the chosen set (its rank-0 subset is taken when nds != 0); means / variances (nc,M);
 * sel (k,) indices of the k largest scores (ties by index); score (nc,) may be NULL. */
int dmo_ehvi_select(dmo_ctx* ctx, const double* F, int64_t nf, const double* means,
                    const double* variances, int64_t nc, int M, const double* ref, int nds,
                    int64_t k, int64_t* sel, double* score);

/* ---- A21: duplicate rows ---------------------------------------------------------
 * replaces MOEA.get_duplicates (dmosopt/MOEA.py:426-437) at its default eps = 1e-16:
 * is_dup[i] = 1 iff an earlier row j < i has ||x_i - x_j||_2 <= eps. */
int dmo_get_duplicates(dmo_ctx* ctx, const double* X, int64_t n, int d, double eps, uint8_t* is_dup);
/* the two-set form MOASMO's resample step uses (dmosopt/MOASMO.py:442, MOEA.get_duplicates(best_x, x_0)):
 * is_dup[i] = 1 when some row j < i of Y (ny, d) lies within eps of row i of X (n, d) -- the reference masks
 * the upper triangle of cdist(X, Y) including the diagonal (MOEA.py:430). */
int dmo_get_duplicates_pair(dmo_ctx* ctx, const double* X, int64_t n, const double* Y, int64_t ny, int d,
                            double eps, uint8_t* is_dup);

/* ---- A11: AGE-MOEA survival score (greedy part) -------------------------------------
 * replaces the O(m^2) greedy loop of AGEMOEA.survival_score (dmosopt/AGEMOEA.py:398-428):
 * yn (m,M) normalised front, nn (m,) = ||yn_i||_p, extreme (n_ext,) pre-selected corner solutions;
 * crowd (m,): inf for the extremes, else the sum of the two smallest distances
 * ||yn_s - yn_r||_p / nn[s] to the already selected set at the moment r is selected. */
int dmo_age_survival(dmo_ctx* ctx, const double* yn, const double* nn, int64_t m, int M, double p,
                     const int32_t* extreme, int n_ext, double* crowd);

/* ---- A12: SMPSO --------------------------------------------------------------------------
 * dmo_smpso_velocity: SMPSO.velocity_vector (dmosopt/SMPSO.py:316-348) for one swarm given its scalar
 *   draws: position (n,d) float32 state, velocity (n,d), the two leader rows (d,) -> out (n,d);
 *   f32_difference != 0 forms (leader - position) in float32 (both operands float32 in NumPy), else float64.
 * dmo_mutate_groups: per_group polynomial mutants per group (swarm), parents drawn uniformly inside each
 *   group of group_size rows of pop_x (SMPSO.py:167-182; MOEA.mutation, MOEA.py:191-212), Philox draws.
 *   children (n_groups*per_group, d); parent_rows (n_groups*per_group,) may be NULL. */
int dmo_smpso_velocity(dmo_ctx* ctx, const float* position, const double* velocity, const double* leader1,
                       const double* leader2, int f32_difference, int64_t n, int d, double w, double c1,
                       double r1, double c2, double r2, double chi, const double* xlb, const double* xub,
                       double* out);
int dmo_mutate_groups(dmo_ctx* ctx, const double* pop_x, int64_t group_size, int64_t n_groups,
                      int64_t per_group, int d, const double* di_mutation, const double* xlb,
                      const double* xub, double mutation_rate, uint64_t seed, uint64_t stream_id,
                      double* children, int64_t* parent_rows);
/* SMPSO with the swarm state resident in HBM: one call per generate / update instead of per-swarm host loops.
 * parm (swarms*pop, d), obj (swarms*pop, M), vel (swarms*pop, d): DEVICE float64 arrays owned by the caller; position and
 * objective values are float32-representable (the reference's state arrays are float32, SMPSO.py:107-113).
 * dmo_smpso_generate (SMPSO.py:143-185): x_gen (2*swarms*pop, d) float32, swarm-major, per swarm pop moved positions
 *   clip(x + v) then pop polynomial mutants of uniformly drawn particles of that swarm (Philox seed / stream_id);
 *   x_gen_f64 (optional, host or device) receives the same float32 values widened to float64 -- what MOEA.generate
 *   hands on after its np.clip (MOEA.py:155).  Either output may be NULL.
 * dmo_smpso_update (SMPSO.py:187-238): consumes rows [0, swarms*pop) of x_gen (float32 when x_is_f32, else float64) and
 *   y_gen (float64) exactly as the reference slices them; scalars (swarms, 8) HOST doubles per swarm = w, c1, r1, c2, r2,
 *   chi, ind1, ind2 drawn by the caller in the reference's order (velocity_vector, SMPSO.py:316-335; ind < 0 = no draw);
 *   the leader with the larger crowding distance of y_gen[swarm slice] goes first.  All velocities are updated against
 *   the old positions, then every swarm keeps the best pop of vstack(offspring slice, particles) (MOEA.remove_worst).
 *   ranks (swarms*pop,) int32 and perm (swarms*pop,) int64 (indices into the swarm's stacked 2*pop rows) are returned;
 *   parm_f32 / obj_f32 (optional) receive the new state as float32 host arrays. */
int dmo_smpso_generate(dmo_ctx* ctx, const double* parm, const double* vel, int swarms, int64_t pop, int d,
                       const double* di_mutation, const double* xlb, const double* xub, double mutation_rate,
                       uint64_t seed, uint64_t stream_id, float* x_gen, double* x_gen_f64);
int dmo_smpso_update(dmo_ctx* ctx, double* parm, double* obj, double* vel, const void* x_gen, int x_is_f32,
                     const double* y_gen, int swarms, int64_t pop, int d, int M, int metric, const double* scalars,
                     const double* xlb, const double* xub, int32_t* ranks, int64_t* perm, float* parm_f32,
                     float* obj_f32);

/* ---- A13 / A15: MO-CMA-ES ----------------------------------------------------------------
 * dmo_cmaes_sample: individuals[i] = x_p + sigma_p * (A_p @ z_i), p = p_idx[i] (dmosopt/CMAES.py:263-267);
 *   sigmas (n_parents, sigma_cols) with sigma_cols = 1 or d, A (n_parents,d,d), z (n,d).
 * dmo_cmaes_update_cholesky: CMAES.updateCholesky (dmosopt/CMAES.py:489-537) for n individuals at once,
 *   in place on A / Ainv (n,d,d) and pc (n,d); z (n,d), psucc (n,). */
int dmo_cmaes_sample(dmo_ctx* ctx, const double* parents_x, const double* sigmas, int sigma_cols,
                     const double* A, int64_t n_parents, const int64_t* p_idx, const double* z, int64_t n,
                     int d, double* individuals);
int dmo_cmaes_update_cholesky(dmo_ctx* ctx, double* A, double* Ainv, double* pc, const double* z,
                              const double* psucc, int64_t n, int d, double cc, double ccov, double pthresh);
/* Device-resident MO-CMA-ES generation / update steps (parents_x, sigmas, factors stay in HBM between generations):
 * dmo_cmaes_generate: dmo_cmaes_sample followed by the reference's global rescale and MOEA.generate's clip,
 *   x = clip((individual / max|individuals|) * (xub - xlb) + xlb, xlb, xub)   (dmosopt/CMAES.py:265-270, MOEA.py:155);
 *   x_out (n, d) host or device.
 * dmo_cmaes_step_z: z[i] = ((x_gen[cand_idx[i]] - parents_x[par_idx[i]]) / (xub - xlb)) / steps[i]  (CMAES.py:359), the
 *   argument of updateCholesky for the chosen offspring; x_gen, parents_x, steps (n, d), z_out (n, d) are DEVICE arrays.
 * dmo_scale_rows: rows[seg_row[s], :] *= factors[e], e = seg_start[s] .. seg_start[s+1]-1, one rounded multiplication
 *   after the other (the per-parent step-size recurrences, CMAES.py:330-383, are sequential); seg_row NULL: row s,
 *   seg_start NULL: factors[s] only.  rows is a DEVICE array of row_elems doubles per row. */
int dmo_cmaes_generate(dmo_ctx* ctx, const double* parents_x, const double* sigmas, int sigma_cols, const double* A,
                       int64_t n_parents, const int64_t* p_idx, const double* z, int64_t n, int d, const double* xlb,
                       const double* xub, double* x_out);
int dmo_cmaes_step_z(dmo_ctx* ctx, const double* x_gen, const int64_t* cand_idx, const double* parents_x,
                     const int64_t* par_idx, const double* xlb, const double* xub, const double* steps, int64_t n, int d,
                     double* z_out);
int dmo_scale_rows(dmo_ctx* ctx, double* rows, int64_t row_elems, int64_t n_seg, const int64_t* seg_row,
                   const int64_t* seg_start, const double* factors, int64_t n_factors);
/* Row gather between DEVICE-resident per-individual state arrays (the (n, d, d) Cholesky factors and (n, d) paths of
 * MO-CMA-ES stay in HBM across generations; CMAES.py:385-411 re-assembles the next parent set from old parents and
 * updated offspring): dst[i, :] = (sel && sel[i] ? alt : src)[idx[i], :], rows of row_elems doubles.  idx (n,) int64 and
 * sel (n,) uint8 (may be NULL, then alt is ignored) may be host arrays. */
int dmo_gather_rows(dmo_ctx* ctx, const double* src, const double* alt, const uint8_t* sel, const int64_t* idx,
                    int64_t n, int64_t row_elems, double* dst);

/* ---- N4: vectorised benchmark objective functions --------------------------------------------
 * replaces the row-at-a-time Python functions of dmosopt/benchmarks/moo_benchmarks.py (dtlz1 :21, dtlz2 :59,
 * dtlz3 :97, dtlz4 :136, dtlz5 :174, dtlz7 :218, wfg4 :335) and the example objectives ZDT1 / ZDT3
 * (examples/example_dmosopt_zdt1.py:9-20, examples/example_dmosopt_zdt3.py:9-21): X (n, n_var) -> Y (n, n_obj).
 * alpha is DTLZ4's bias exponent (the reference's default is 100), ignored elsewhere. */
#define DMO_BM_ZDT1 0
#define DMO_BM_ZDT3 1
#define DMO_BM_DTLZ1 10
#define DMO_BM_DTLZ2 11
#define DMO_BM_DTLZ3 12
#define DMO_BM_DTLZ4 13
#define DMO_BM_DTLZ5 14
#define DMO_BM_DTLZ7 16
#define DMO_BM_WFG4 24
int dmo_benchmark_eval(dmo_ctx* ctx, int problem, const double* X, int64_t n, int n_var, int n_obj, double alpha,
                       double* Y);

#ifdef __cplusplus
}
#endif
#endif /* DMOSOPT_B200_H */
