/*
 * gpboost_b200 — device-engine C ABI (plain pointers and sizes, no C++/torch types).
 *
 * This is the seam the host-side REModel (gpboost_b200/csrc/host) calls; each entry cites the
 * reference function(s) whose work it replaces (paths relative to fabsig/GPBoost @ c93fa49).
 * All functions return 0 on success, non-zero on failure; the message is available from
 * gpbdev_last_error() (thread-local, like LGBM_GetLastError — include/LightGBM/c_api.h:1837-1849).
 * There is NO CPU fallback: without a CUDA device every compute entry fails.
 */
#ifndef GPBOOST_B200_DEV_H_
#define GPBOOST_B200_DEV_H_
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define GPBDEV_EXPORT __attribute__((visibility("default")))

/* covariance function ids (closed forms of include/GPBoost/cov_fcts.h:2100-2118, :2154) */
enum { GPBDEV_COV_EXPONENTIAL = 0, GPBDEV_COV_MATERN15 = 1, GPBDEV_COV_MATERN25 = 2, GPBDEV_COV_GAUSSIAN = 3 };
/* evaluation modes of gpbdev_vecchia_eval */
enum { GPBDEV_MODE_NLL = 0, GPBDEV_MODE_STORE = 1, GPBDEV_MODE_GRAD = 2 };
/* sums returned by gpbdev_vecchia_eval (out[GPBDEV_NUM_SUMS]) */
enum {
  GPBDEV_SUM_QUAD = 0,    /* y^T Psi^-1 y = sum (By)_i^2 / D_i      re_model_template.h:9957-9964 */
  GPBDEV_SUM_LOGDET = 1,  /* log|Psi| = sum log D_i                  re_model_template.h:2947      */
  GPBDEV_SUM_NBAD = 2,    /* #(D_i <= 0)                             Vecchia_utils.cpp:1685-1698   */
  GPBDEV_SUM_UKU0 = 3, GPBDEV_SUM_UKU1 = 4,   /* sum (dB_k y)_i u_i, u = D^-1 B y   re_model_template.h:2002-2004 */
  GPBDEV_SUM_UDU0 = 5, GPBDEV_SUM_UDU1 = 6,   /* sum u_i^2 dD_k,i                                               */
  GPBDEV_SUM_TR0 = 7, GPBDEV_SUM_TR1 = 8,     /* sum dD_k,i / D_i                                               */
  GPBDEV_NUM_SUMS = 9
};

typedef struct gpbdev_vecchia* gpbdev_vecchia_t;

GPBDEV_EXPORT const char* gpbdev_last_error(void);
/* number of visible CUDA devices (0 when none / driver missing) */
GPBDEV_EXPORT int gpbdev_device_count(void);

/*
 * Create the device-resident state of one Vecchia-approximated GP: ordered coordinates, neighbour sets,
 * the CSC view of B's sparsity pattern and work buffers.
 *   coords_ordered : host, n x d ROW-major, already in Vecchia order
 *   perm           : host, n; ordered position i holds original observation perm[i]
 *                    (data_indices_per_cluster after Vecchia_utils.cpp:1129-1131)
 *   nn             : host n x m int32 (-1 padded) or NULL to run the device neighbour search
 *                    (replaces find_nearest_neighbors_Vecchia_fast, Vecchia_utils.cpp:733-985)
 *   row_begin/end  : shard [row_begin,row_end) of ordered observations this engine evaluates
 *                    (whole range on one GPU); coordinates are replicated (SURVEY §8e)
 */
GPBDEV_EXPORT int gpbdev_vecchia_create(gpbdev_vecchia_t* out, int device, int64_t n, int d, int m,
                                        const double* coords_ordered, const int32_t* perm,
                                        const int32_t* nn, int64_t row_begin, int64_t row_end);
GPBDEV_EXPORT int gpbdev_vecchia_free(gpbdev_vecchia_t h);

/* copy the neighbour sets back (n x m int32, -1 padded) — parity tests */
GPBDEV_EXPORT int gpbdev_vecchia_get_nn(gpbdev_vecchia_t h, int32_t* nn_host);

/* y in ORIGINAL observation order; host pointer (H2D inside) or device pointer. Replaces SetY
 * (re_model_template.h:6185-6200) incl. the per-cluster re-ordering. */
GPBDEV_EXPORT int gpbdev_vecchia_set_y(gpbdev_vecchia_t h, const double* y_host);
GPBDEV_EXPORT int gpbdev_vecchia_set_y_device(gpbdev_vecchia_t h, const double* y_dev);

/*
 * One pass of the hot path at transformed parameters (var = sigma1^2/sigma^2, range per
 * cov_fcts.h:485-552). Replaces CalcCovFactorVecchia (re_model_template.h:9471) /
 * CalcCovFactorGradientVecchia (Vecchia_utils.cpp:1367-1699) + CalcYTPsiIInvY (:9938) + the log-det
 * (:2947) and, in GRAD mode, CalcGradientVecchia (:9601) + the gradient assembly (:1988-2010).
 *   mode NLL   : sums 0..2
 *   mode STORE : sums 0..2 and keeps A (= -B off-diagonal), D^-1 and u = D^-1 B y on the device
 *   mode GRAD  : sums 0..8
 * Synchronous: returns after the sums reached `out` (host, GPBDEV_NUM_SUMS doubles; shard-local sums).
 */
GPBDEV_EXPORT int gpbdev_vecchia_eval(gpbdev_vecchia_t h, int cov_type, double var, double range, int mode,
                                      double* out);
/* same, asynchronous on the engine's stream and without the D2H of the sums (bench: device-only timing) */
GPBDEV_EXPORT int gpbdev_vecchia_eval_async(gpbdev_vecchia_t h, int cov_type, double var, double range, int mode);
/* the sums of the last evaluation (GPBDEV_NUM_SUMS doubles into a host buffer; waits for the engine's stream) */
GPBDEV_EXPORT int gpbdev_vecchia_get_sums(gpbdev_vecchia_t h, double* out);

/* After a STORE eval: y_aux = Psi^-1 y = B^T D^-1 B y (CalcYAux, re_model_template.h:9772) returned in
 * ORIGINAL observation order into a host buffer of n doubles. */
GPBDEV_EXPORT int gpbdev_vecchia_yaux(gpbdev_vecchia_t h, double* yaux_host);
/* Same as gpbdev_vecchia_yaux but the result (times `scale`) stays on the device, original order, written to out_dev
 * (may alias the engine-external gradient buffer of the boosting driver). */
GPBDEV_EXPORT int gpbdev_vecchia_yaux_device(gpbdev_vecchia_t h, double* out_dev, double scale);
/* bench hook (after gpbdev_vecchia_laplace_eval): mean device time of one operator application and of one VADU preconditioner
 * application on t columns (t = 1 or the probe count); out_ms = {operator, preconditioner} */
GPBDEV_EXPORT int gpbdev_vecchia_laplace_time_ops(gpbdev_vecchia_t h, int t, int reps, float* out_ms);
/* Vecchia prediction at new locations (SURVEY §8 f1): CalcPredVecchiaObservedFirstOrder with CondObsOnly = true
 * (src/GPBoost/Vecchia_utils.cpp:1701-2100), Gaussian likelihood, responses of the last gpbdev_vecchia_set_y*. coords_pred_host: np x d
 * row-major. num_neighbors_pred <= 60 (the reference's default is twice the model's num_neighbors, re_model_template.h:299).
 * mean_out_host[p] = A_p y_N(p); var_out_host[p] = D_p on the transformed scale (times sigma^2 = latent predictive variance). */
GPBDEV_EXPORT int gpbdev_vecchia_predict(gpbdev_vecchia_t h, int cov_type, double var, double range, const double* coords_pred_host,
                                         int64_t np, int num_neighbors_pred, double* mean_out_host, double* var_out_host);
/* Newton update of the leaf values in GPBoost (SURVEY §8 f2; REModelTemplate::NewtonUpdateLeafValues, Vecchia branch,
 * include/GPBoost/re_model_template.h:4982-5063). After a STORE pass at the current parameters: M_host (L x L row-major) =
 * H^T B^T D^-1 B H and rhs_host (L) = H^T g for the leaf incidence H given by leaf_of_row_dev (n int32, original row order, device)
 * and g = grad_dev (n doubles, original order, device). The caller solves M x = -sigma^2 rhs (L <= 256). */
GPBDEV_EXPORT int gpbdev_vecchia_newton_system(gpbdev_vecchia_t h, const int32_t* leaf_of_row_dev, int num_leaves, const double* grad_dev,
                                               double* M_host, double* rhs_host);
/* Latent factor (non-Gaussian likelihood) and its derivative w.r.t. log(range) — B_grad[1] = -dA, D_grad[1] = dD of
 * CalcCovFactorGradientVecchia (src/GPBoost/Vecchia_utils.cpp:1636-1652) — copied to host buffers (A, dA: n x m row-major in
 * Vecchia order; Dinv, dD: n). Diagnostics / test entry of the factor kernel's MODE_STORE_GRAD. */
GPBDEV_EXPORT int gpbdev_vecchia_latent_factor_grad(gpbdev_vecchia_t h, int cov_type, double var, double range, double* A_host,
                                                    double* Dinv_host, double* dA_host, double* dD_host);
/* After a STORE eval: copy A (n x m) and D^-1 (n) to the host — parity tests against the oracle's B, D^-1 */
GPBDEV_EXPORT int gpbdev_vecchia_get_factor(gpbdev_vecchia_t h, double* A_host, double* Dinv_host);

/* CUDA-event timing on the engine's stream (bench.py): start, run work, stop -> milliseconds */
GPBDEV_EXPORT int gpbdev_vecchia_timer_start(gpbdev_vecchia_t h);
GPBDEV_EXPORT int gpbdev_vecchia_timer_stop(gpbdev_vecchia_t h, float* ms);
GPBDEV_EXPORT int gpbdev_vecchia_sync(gpbdev_vecchia_t h);
/* number of kernels this engine has launched so far (bench.py's gpu_launches) */
GPBDEV_EXPORT int64_t gpbdev_vecchia_launch_count(gpbdev_vecchia_t h);
/* number of queries of the device neighbour search that were re-derived by the exact replay of the reference's
 * pruned walk (rounding-decided ties, typically only on lattice data) */
GPBDEV_EXPORT int gpbdev_vecchia_knn_replayed(gpbdev_vecchia_t h);
/* measured FP64 FMA peak (TFLOP/s, 2 flops per FMA) of `device`: a register-only DFMA microbenchmark.
 * The Vecchia factor kernel is FP64-pipe bound (SURVEY §8d), so this is its roofline denominator. */
/* Device collective hook (multi-GPU): in-place sum over all ranks of `count` fp64 values at DEVICE pointer `dev_buf`, enqueued on
 * `stream` (cudaStream_t). With a hook installed the engine all-reduces its 9 sums (and the Psi^-1 y vector) on its own stream
 * before they leave the device; without one the caller reduces the host copies (the injected collective of GPB200_SetCollective). */
typedef int (*gpbdev_allreduce_fn)(void* ctx, double* dev_buf, int64_t count, void* stream);
GPBDEV_EXPORT int gpbdev_vecchia_set_allreduce(gpbdev_vecchia_t h, gpbdev_allreduce_fn fn, void* ctx);
GPBDEV_EXPORT int gpbdev_fp64_peak(int device, double* tflops);
/* write > L2-size bytes to evict the L2 between timed iterations */
GPBDEV_EXPORT int gpbdev_vecchia_flush_l2(gpbdev_vecchia_t h);

/* ---- Laplace approximation, latent Vecchia GP + bernoulli_logit likelihood (SURVEY §8 a12) -----------------------
 * Replaces FindModePostRandEffCalcMLLVecchia (include/GPBoost/likelihoods.h:3773-4059) with
 * matrix_inversion_method = "iterative", cg_preconditioner_type = "vadu": Newton mode finding with PCG solves
 * (CGVecchiaLaplaceVec, src/GPBoost/CG_utils.cpp:21-108) and the log-determinant by stochastic Lanczos quadrature
 * (CalcLogDetStochVecchia likelihoods.h:16376-16521, CGTridiagVecchiaLaplace CG_utils.cpp:110-229).
 * Labels (0/1 as doubles) are set with gpbdev_vecchia_set_y. */
/* probe vectors r_i ~ N(0, I): n x t COLUMN-major, rows in the Vecchia order (GenRandVecNormalParallel, CG_utils.cpp:978) */
GPBDEV_EXPORT int gpbdev_vecchia_laplace_set_probes(gpbdev_vecchia_t h, const double* probes_colmajor, int t);
/* cfg[8]: 0 maxit_mode_newton, 1 delta_conv_mode_finding, 2 max step halvings, 3 cg_max_num_it, 4 cg_max_num_it_tridiag,
 *         5 cg_delta_conv, 6 calculate the log-determinant (0/1), 7 c_armijo.  var = sigma_1^2, range transformed.
 * out[6]: 0 approximate NEGATIVE marginal log-likelihood, 1 Newton iterations, 2 CG iterations, 3 SLQ iterations,
 *         4 log det(Sigma W + I), 5 objective at the mode. fixed_effects_host: original data order or NULL. */
GPBDEV_EXPORT int gpbdev_vecchia_laplace_eval(gpbdev_vecchia_t h, int cov_type, double var, double range,
                                              const double* fixed_effects_host, const double* cfg, double* out);
GPBDEV_EXPORT int gpbdev_vecchia_laplace_get_mode(gpbdev_vecchia_t h, double* mode_host);
/* Gradient of the Laplace-approximated negative log-likelihood w.r.t. (log variance, log range) — the covariance-parameter part of
 * CalcGradNegMargLikelihoodLaplaceApproxVecchia (include/GPBoost/likelihoods.h:6521-7044, iterative branch, VADU). Call
 * gpbdev_vecchia_laplace_keep_solutions(h, 1), then gpbdev_vecchia_laplace_eval, then this with the same covariance parameters
 * and cfg. out[0..1] = gradient (scale of the reference's optimiser: log of the original parameters), out[2] = CG iterations. */
GPBDEV_EXPORT int gpbdev_vecchia_laplace_keep_solutions(gpbdev_vecchia_t h, int keep);
GPBDEV_EXPORT int gpbdev_vecchia_laplace_grad(gpbdev_vecchia_t h, int cov_type, double var, double range, const double* cfg, double* out);
/* multi-GPU: this process holds t of the job's t_total probe columns; allreduce_sum sums `count` doubles over the ranks */
GPBDEV_EXPORT int gpbdev_vecchia_laplace_set_collective(gpbdev_vecchia_t h, void (*allreduce_sum)(double*, int), int t_total);

/* ------------------------------------------------------------------------------------------------------------------
 * Exact (dense) Gaussian process, Gaussian likelihood (SURVEY §8 a6, BASELINE config 1). coords: host n x d row-major in the
 * original observation order. Replaces RECompGP::CalcSigma (re_comp.h:1273), CalcZSigmaZt (re_model_template.h:9273),
 * CalcChol (:6492), the solves of CalcYAux (:9894) / CalcYTPsiIInvY (:10002) and the log-determinant (:3127).
 */
typedef struct gpbdev_dense* gpbdev_dense_t;
GPBDEV_EXPORT const char* gpbdev_dense_last_error(void);
GPBDEV_EXPORT int gpbdev_dense_create(gpbdev_dense_t* out, int device, int n, int d, const double* coords_rowmajor);
GPBDEV_EXPORT int gpbdev_dense_free(gpbdev_dense_t h);
GPBDEV_EXPORT int gpbdev_dense_set_y(gpbdev_dense_t h, const double* y_host);
/* Gram build + blocked Cholesky of [[I + Sigma, y],[y^T, *]] at transformed (var, range):
 * out3 = { y^T Psi^-1 y, log|Psi|, #non-positive pivots } */
GPBDEV_EXPORT int gpbdev_dense_eval(gpbdev_dense_t h, int cov_type, double var, double range, double* out3);
/* after an eval: Psi^-1 y * scale (host, n doubles) */
GPBDEV_EXPORT int gpbdev_dense_yaux(gpbdev_dense_t h, double scale, double* yaux_host);
/* gradient sums at the parameters of the last gpbdev_dense_eval (CalcPsiInv re_model_template.h:6586-6617 + the dense branch of
 * CalcGradPars :2018-2039): out4 = {tr(Psi^-1 Sigma), tr(Psi^-1 dSigma/dlog range), alpha^T Sigma alpha, alpha^T dSigma/dlog range alpha} */
GPBDEV_EXPORT int gpbdev_dense_grad(gpbdev_dense_t h, double* out4);
GPBDEV_EXPORT int64_t gpbdev_dense_launch_count(gpbdev_dense_t h);

/* ------------------------------------------------------------------------------------------------------------------
 * Single-level grouped random effect, Gaussian likelihood (SURVEY §8 a7). group_index: host, n int32 in [0, num_groups).
 * Replaces InitializeMatricesForUseWoodburyIdentity / CalcZtY / CalcCovFactor single-RE branch / CalcYtilde / CalcYAux /
 * the Woodbury gradient (re_model_template.h:7174-7308, :6326, :9417-9420, :9907-9918, :9843-9891, :2462-2529).
 */
typedef struct gpbdev_grouped* gpbdev_grouped_t;
GPBDEV_EXPORT const char* gpbdev_grouped_last_error(void);
GPBDEV_EXPORT int gpbdev_grouped_create(gpbdev_grouped_t* out, int device, int64_t n, const int32_t* group_index, int num_groups);
GPBDEV_EXPORT int gpbdev_grouped_free(gpbdev_grouped_t h);
/* y in original order (host): H2D + per-group sums Z^T y (SetY / CalcZtY) */
GPBDEV_EXPORT int gpbdev_grouped_set_y(gpbdev_grouped_t h, const double* y_host);
/* sums at variance ratio v = sigma_1^2/sigma^2: out5 = { y'y, sum s_g^2/(1/v+n_g), sum log(1+v n_g),
 * sum s_g^2 v/(1+v n_g)^2, sum v n_g/(1+v n_g) } */
GPBDEV_EXPORT int gpbdev_grouped_eval(gpbdev_grouped_t h, double var_ratio, double* out5);
/* y_aux = Psi^-1 y * scale in original order (CalcYAux single-RE branch) */
GPBDEV_EXPORT int gpbdev_grouped_yaux(gpbdev_grouped_t h, double var_ratio, double scale, double* yaux_host);
/* Device-resident forms (the boosting loop keeps F - y and its gradient in HBM): y_dev / out_dev are device pointers to n doubles
 * in original order. set_y_device is enqueued on the engine's stream (the caller has synchronised the producer);
 * yaux_device returns after the result is complete. */
GPBDEV_EXPORT int gpbdev_grouped_set_y_device(gpbdev_grouped_t h, const double* y_dev);
GPBDEV_EXPORT int gpbdev_grouped_yaux_device(gpbdev_grouped_t h, double var_ratio, double scale, double* out_dev);
GPBDEV_EXPORT int64_t gpbdev_grouped_launch_count(gpbdev_grouped_t h);

/* ------------------------------------------------------------------------------------------------------------------
 * Device tree learner (dense uint8 bins, numerical features, no missing values, constant hessian).
 * Seam: the reference's TreeLearner interface (include/LightGBM/tree_learner.h:29-117: Init / Train / AddPredictionToScore /
 * GetDataLeafIndices), selected there by device_type (src/LightGBM/treelearner/tree_learner.cpp:15-52).
 */
typedef struct gpbdev_tree* gpbdev_tree_t;
typedef struct {
  int num_leaves;                 /* config.h: num_leaves            */
  int min_data_in_leaf;           /*           min_data_in_leaf      */
  double min_sum_hessian_in_leaf; /*           min_sum_hessian_in_leaf */
  double lambda_l2;               /*           lambda_l2             */
  double min_gain_to_split;       /*           min_gain_to_split     */
  int max_depth;                  /*           max_depth (<= 0: unlimited) */
} gpbdev_tree_config;

GPBDEV_EXPORT const char* gpbdev_tree_last_error(void);
/* bins_feature_major: host, F x n uint8 (the reference's dense-bin layout: one column per feature); num_bin[f] <= 256.
 * Replaces TreeLearner::Init (serial_tree_learner.cpp:38-85). */
GPBDEV_EXPORT int gpbdev_tree_create(gpbdev_tree_t* out, int device, int64_t n, int F, const uint8_t* bins_feature_major,
                                     const int32_t* num_bin, const gpbdev_tree_config* cfg);
/* Same learner on a bin matrix that is already in HBM (gpbdev_bin_matrix below): bins_dev is row-major n x Fpad uint8 on `device`
 * (Fpad a multiple of 32, padding bytes 0); the learner reads it in place and does NOT own it — a row shard is just an offset. */
GPBDEV_EXPORT int gpbdev_tree_create_on_device_bins(gpbdev_tree_t* out, int device, int64_t n, int F, int Fpad, const uint8_t* bins_dev,
                                                    const int32_t* num_bin, const gpbdev_tree_config* cfg);
GPBDEV_EXPORT int gpbdev_tree_free(gpbdev_tree_t h);

/* ------------------------------------------------------------------------------------------------------------------
 * Device binning (SURVEY §8 f3). Replaces the n x F value -> bin pass of LGBM_DatasetCreateFromMat
 * (src/LightGBM/c_api.cpp:1134-1232 -> BinMapper::ValueToBin, include/LightGBM/bin.h:465-503; numerical, MissingType::None).
 * data_host: nrow x ncol matrix in host memory, data_type 0 = float32 / 1 = float64 (C_API_DTYPE_*), row- or column-major.
 * real_feature[f] = column of used feature f; upper_bounds[f * upper_bounds_stride + b], b < num_bin[f] = the feature's strictly
 * increasing bin upper bounds (last one +inf). Output: *bins_dev_out = device buffer, row-major nrow x Fpad uint8 (Fpad multiple of 32,
 * >= F; padding 0), released with gpbdev_bin_free. No CPU fallback: fails without a CUDA device. */
GPBDEV_EXPORT const char* gpbdev_bin_last_error(void);
GPBDEV_EXPORT int gpbdev_bin_matrix(int device, const void* data_host, int data_type, int64_t nrow, int ncol, int is_row_major, int F,
                                    const int32_t* real_feature, const int32_t* num_bin, const double* upper_bounds,
                                    int upper_bounds_stride, int Fpad, uint8_t** bins_dev_out);
GPBDEV_EXPORT int gpbdev_bin_free(int device, uint8_t* bins_dev);
/* test hook: the bin matrix back on the host (nrow x Fpad bytes) */
GPBDEV_EXPORT int gpbdev_bin_download(int device, const uint8_t* bins_dev, int64_t nrow, int Fpad, uint8_t* out_host);
/* Grow one tree from gradients (n doubles; host pointer, or device pointer when grad_on_device != 0) with hessian == hess_const.
 * Replaces SerialTreeLearner::Train (serial_tree_learner.cpp:159-209). Output arrays are caller-allocated with num_leaves entries:
 * per internal node split_feature / threshold_bin / left_child / right_child (~leaf for leaves, Tree convention) / split_gain;
 * per leaf leaf_value (unshrunk) / leaf_count. */
GPBDEV_EXPORT int gpbdev_tree_train(gpbdev_tree_t h, const double* grad, int grad_on_device, double hess_const, int* num_leaves,
                                    int* split_feature, int* threshold_bin, int* left_child, int* right_child, float* split_gain,
                                    double* leaf_value, int* leaf_count);
/* score_dev[row] += leaf_values[leaf(row)] over the partition of the last trained tree (ScoreUpdater::AddScore(tree_learner, tree),
 * score_updater.hpp); optionally also writes the leaf index of every row (GetDataLeafIndices). Either pointer may be NULL. */
GPBDEV_EXPORT int gpbdev_tree_add_score(gpbdev_tree_t h, const double* leaf_values, int num_leaves, double* score_dev,
                                        int32_t* leaf_of_row_dev);
/* bench hook: mean device time (CUDA events on the learner's stream, L2 flushed before every launch) of the root-pass histogram kernel
 * over all n rows; algorithmic bytes per launch n * (Fpad + 8) */
GPBDEV_EXPORT int gpbdev_tree_time_root_hist(gpbdev_tree_t h, const double* grad_dev, int reps, float* mean_ms);
/* leaf index of every row of the last trained tree (TreeLearner::GetDataLeafIndices, serial_tree_learner.cpp:818): device pointer to n
 * int32 owned by the learner, valid until the next call / tree */
GPBDEV_EXPORT int gpbdev_tree_leaf_indices(gpbdev_tree_t h, const int32_t** leaf_of_row_dev);
/* device vectors of the boosting driver (training score, label, gradient) on the learner's device/stream */
GPBDEV_EXPORT int gpbdev_vec_alloc(gpbdev_tree_t h, double** out, int64_t n);
GPBDEV_EXPORT int gpbdev_vec_free(gpbdev_tree_t h, double* p);
GPBDEV_EXPORT int gpbdev_vec_upload(gpbdev_tree_t h, double* dst_dev, const double* src_host, int64_t n);
GPBDEV_EXPORT int gpbdev_vec_download(gpbdev_tree_t h, double* dst_host, const double* src_dev, int64_t n);
/* out = a - b: the L2 objective's gradient score - label (regression_objective.hpp:158-162) */
GPBDEV_EXPORT int gpbdev_vec_sub(gpbdev_tree_t h, const double* a_dev, const double* b_dev, double* out_dev, int64_t n);
GPBDEV_EXPORT int gpbdev_vec_add_const(gpbdev_tree_t h, double* a_dev, double c, int64_t n);
/* a . b in a fixed summation order (the line search's two inner products: re_model_template.h:1165-1178), zero fill, copy */
GPBDEV_EXPORT int gpbdev_vec_dot(gpbdev_tree_t h, const double* a_dev, const double* b_dev, int64_t n, double* out_host);
GPBDEV_EXPORT int gpbdev_vec_zero(gpbdev_tree_t h, double* a_dev, int64_t n);
GPBDEV_EXPORT int gpbdev_vec_copy(gpbdev_tree_t h, double* dst_dev, const double* src_dev, int64_t n);
/* data-parallel mode: this learner holds a contiguous shard of the rows; the root gradient sum and the smaller child's histogram of
 * every split are summed over the ranks through `fn` on the learner's stream (DataParallelTreeLearner,
 * src/LightGBM/treelearner/data_parallel_tree_learner.cpp:155-175). n_global = rows over all ranks. */
GPBDEV_EXPORT int gpbdev_tree_set_allreduce(gpbdev_tree_t h, gpbdev_allreduce_fn fn, void* ctx, int64_t n_global);
/* replicated n-vector of which this rank keeps rows [b, e) current: bring the whole vector up to date on every rank */
GPBDEV_EXPORT int gpbdev_vec_allgather_rows(gpbdev_tree_t h, double* vec_dev, int64_t n, int64_t b, int64_t e);
GPBDEV_EXPORT int gpbdev_tree_sync(gpbdev_tree_t h);
GPBDEV_EXPORT int64_t gpbdev_tree_launch_count(gpbdev_tree_t h);
GPBDEV_EXPORT void* gpbdev_tree_stream(gpbdev_tree_t h);

#ifdef __cplusplus
}
#endif
#endif /* GPBOOST_B200_DEV_H_ */
