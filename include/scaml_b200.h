/* scaml_b200.h -- C ABI of the B200-native ScaML-GP hot path (libscaml_b200.so).
 *
 * The reference (boschresearch/Scalable-Meta-Learning-with-Gaussian-Processes) is pure
 * Python: it has no FFI.  The interfaces these entry points replace are therefore the
 * Python call sites at which the reference hands the arithmetic to botorch/gpytorch
 * (cited per function as reference file:line).  INTEGRATION.md shows the ctypes stubs a
 * maintainer of the reference would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (torch tensors' data_ptr());
 *    the library never allocates, frees or retains memory;
 *  - all floating point data is IEEE binary64, row-major, dense;
 *  - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); calls are
 *    asynchronous w.r.t. the host and re-entrant;
 *  - return value: 0 = launched; <0 = bad argument (SCAML_E_*); >0 = cudaError_t.
 *  - per-evaluation numerical failures never abort a batch: they are reported through
 *    `info` (LAPACK style: k > 0 = first non-positive pivot, 1-based) with NaN outputs,
 *    mirroring the NotPSD -> NaN-loss behaviour of the reference's fit closure
 *    (scamlgp/utils.py:174-198).
 *
 * Layouts
 *   X          [M][n_max][d]     inputs in [0,1]^d, rows >= n_valid[m] ignored
 *   y          [M][n_max]        per-task standardised targets (botorch Standardize)
 *   n_valid    [M] int32         points of task m (1..n_max); NULL = n_max everywhere
 *   theta_raw  [M][R][P]         P = d + 2: raw (pre-sigmoid) lengthscales, outputscale, noise
 *   "packed factor" (scaml_factorize output, scaml_predict_* input):
 *       n_pad = 64*ceil(n_max/64), NB = n_pad/32, lower 32x32 tiles (bi >= bj) of L^-1 at
 *       tile index bi*(bi+1)/2 + bj, each tile 1024 doubles COLUMN-major; stride per task
 *       = NB*(NB+1)/2*1024 doubles.
 */
#ifndef SCAML_B200_H
#define SCAML_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCAML_KERNEL_RBF 0
#define SCAML_KERNEL_MATERN12 1
#define SCAML_KERNEL_MATERN32 2
#define SCAML_KERNEL_MATERN52 3

#define SCAML_PRIOR_NONE 0
#define SCAML_PRIOR_GAMMA 1     /* p1 = concentration, p2 = rate   */
#define SCAML_PRIOR_LOGNORMAL 2 /* p1 = mu,            p2 = sigma  */

#define SCAML_E_ARG (-1)      /* null pointer / non-positive size            */
#define SCAML_E_WORKSPACE (-2) /* workspace smaller than scaml_fit_workspace_bytes */
#define SCAML_E_UNSUPPORTED (-3) /* d or n_max beyond what the kernels are built for */
#define SCAML_E_SMEM (-4)     /* configuration does not fit 227 KB shared memory */

/* Kernel family + gpytorch `Interval` constraints + priors of one GP
 * (reference scamlgp/model.py:25-33 likelihood, :36-70 source kernel, :73-105 target kernel). */
typedef struct scaml_hyper_spec {
  int32_t kernel;      /* SCAML_KERNEL_*                                   */
  int32_t ls_prior;    /* SCAML_PRIOR_* on each lengthscale                */
  int32_t os_prior;    /* ... on the outputscale                           */
  int32_t noise_prior; /* ... on the noise variance                        */
  double ls_lo, ls_hi; /* Interval(lower, upper) of the lengthscales       */
  double os_lo, os_hi;
  double noise_lo, noise_hi;
  double ls_p1, ls_p2;
  double os_p1, os_p2;
  double noise_p1, noise_p2;
} scaml_hyper_spec;

/* Library / build identification ("scaml_b200 <version> sm_100a"). */
const char* scaml_version(void);

/* Largest n_max / d the fit kernels accept (shared-memory budget), and the number of
 * workspace bytes scaml_lml_grad / scaml_factorize need for M tasks x R rows of (n_max, d)
 * on this device: the per-CTA tile workspaces plus the scheduling block (work counter and
 * the list of active rows, most expensive first).  The workspace is scratch: contents are
 * undefined between calls.  scaml_factorize: R = 1. */
int scaml_fit_limits(int* n_max_limit, int* d_limit);
size_t scaml_fit_workspace_bytes(int M, int R, int n_max, int d);

/* K1 standalone: K[m] = s_m * kappa(X_m / l_m) + noise_m * I for every task, written dense
 * [M][n_max][n_max] (rows/cols >= n_valid are the identity).  `theta` holds CONSTRAINED
 * values [M][P].  Replaces `covar_module(X)` + likelihood noise evaluated inside
 * `mll(model(X), y)` (reference scamlgp/utils.py:175-177; kernels model.py:44-70). */
int scaml_kernel_matrix(const double* X, const int32_t* n_valid, const double* theta,
                        double* K, int M, int n_max, int d, int kernel, void* stream);

/* K1-K5 fused: (LML + log priors)/n and its gradient w.r.t. the RAW parameters for
 * M tasks x R hyper-parameter rows in ONE launch.  Replaces one evaluation of the
 * closure scipy drives inside `fit.fit_gpytorch_mll(mll)` and of
 * `mll(model(*model.train_inputs), model.train_targets)` (reference
 * scamlgp/utils.py:171-177,190-192; loop over tasks model.py:176-188).
 *   jitter [M][R] or NULL : added to the diagonal (psd_safe_cholesky ladder is driven
 *                           by the host: 1e-8, 1e-7, 1e-6)
 *   skip   [M][R] or NULL : non-zero entries are not evaluated and not written
 *   lml    [M][R], grad [M][R][P], info [M][R]                                    */
int scaml_lml_grad(const double* X, const double* y, const int32_t* n_valid,
                   const double* theta_raw, const double* jitter, const int32_t* skip,
                   double* lml, double* grad, int32_t* info, void* workspace,
                   size_t workspace_bytes, int M, int R, int n_max, int d,
                   const scaml_hyper_spec* spec, void* stream);

/* The same evaluation with linear_operator's psd_safe_cholesky jitter ladder applied INSIDE the
 * kernel: a row whose factorisation meets a non-positive pivot is repeated with 1e-8, 1e-7, 1e-6
 * added to the diagonal of the original matrix; info > 0 / NaN only when 1e-6 fails too.  No
 * device -> host read of `info` is needed between the rounds of an optimiser (the reference gets
 * this behaviour from gpytorch inside the closure, scamlgp/utils.py:171-177). */
int scaml_lml_grad_ladder(const double* X, const double* y, const int32_t* n_valid,
                          const double* theta_raw, const int32_t* skip, double* lml, double* grad,
                          int32_t* info, void* workspace, size_t workspace_bytes, int M, int R,
                          int n_max, int d, const scaml_hyper_spec* spec, void* stream);

/* K1-K3 for prediction: factorise K_y of every task at its fitted parameters
 * (theta_raw [M][P]) and emit the packed L^-1 tiles, alpha = K_y^-1 y~ [M][n_pad], and
 * the constrained parameters theta [M][P].  Replaces the prediction-strategy caches
 * gpytorch builds on the first `gp.posterior(x)` (reference scamlgp/model.py:128,281). */
int scaml_factorize(const double* X, const double* y, const int32_t* n_valid,
                    const double* theta_raw, const double* jitter, double* linv_packed,
                    double* alpha, double* theta, int32_t* info, void* workspace,
                    size_t workspace_bytes, int M, int n_max, int d,
                    const scaml_hyper_spec* spec, void* stream);
/* scaml_factorize with the in-kernel jitter ladder (see scaml_lml_grad_ladder). */
int scaml_factorize_ladder(const double* X, const double* y, const int32_t* n_valid,
                           const double* theta_raw, double* linv_packed, double* alpha,
                           double* theta, int32_t* info, void* workspace, size_t workspace_bytes,
                           int M, int n_max, int d, const scaml_hyper_spec* spec, void* stream);


/* Largest n_max the prediction kernel (scaml_predict_weighted, scaml_predict_conditioned) accepts at input
 * dimension d: its k* tiles, the L^-1 ring and the staged inputs must fit 227 KB (576 for d <= 6, 512 at
 * d = 10, 320 at d = 16, 256 at d = 32); 0 for d outside 1..32. */
int scaml_predict_max_points(int d);

/* Bytes of partial-sum scratch scaml_predict_weighted needs for B candidates. */
size_t scaml_predict_workspace_bytes(int M, int n_max, int d, int B);

/* K6-K9 fused: weighted ScaML-GP prior prediction at B candidates (q = 1),
 *   mean[b] = sum_m w_m (ybar_m + ystd_m * k*_m(b)^T alpha_m)
 *   var[b]  = sum_m w_m^2 ystd_m^2 (s_m - || L_m^-1 k*_m(b) ||^2)
 * reduced over the M tasks inside the kernel in a fixed order (deterministic).
 * Tasks with w_m == 0 are skipped (weight pruning, reference model.py:192-215,365-372).
 * Replaces `_compute_target_prior` (reference scamlgp/model.py:108-135).
 *   theta [M][P] constrained (from scaml_factorize), Xc [B][d], mean [B], var [B].     */
int scaml_predict_weighted(const double* X, const int32_t* n_valid, const double* theta,
                           const double* linv_packed, const double* alpha,
                           const double* ybar, const double* ystd, const double* w,
                           const double* Xc, double* mean, double* var, void* workspace,
                           size_t workspace_bytes, int M, int n_max, int d, int B,
                           int kernel, void* stream);

/* K6/K7 with q > 1: source posteriors at two point sets A (nA) and B (nB),
 *   mean_m(A),  Sigma_m(A,B) = ystd_m^2 (K_m(A,B) - V_m(A)^T V_m(B)),  V_m(.) = L_m^-1 K_m(X_m, .)
 * reduce = 0: per task, mean [nA][M] and cov [nA][nB][M] in raw-Y units -- the `source_means` /
 *             `source_covs` caches of `ScaMLGP.__init__` (reference scamlgp/model.py:278-289);
 * reduce = 1: mean [nA] = sum_m w_m mean_m, cov [nA][nB] = sum_m w_m^2 Sigma_m in a fixed order --
 *             the joint prior blocks `ScaMLGP.forward` builds in eval mode
 *             (reference scamlgp/model.py:364-375 via _compute_target_prior :108-135).
 * n_max <= scaml_predict_cross_max_points(d) (k(X,A), k(X,B) are held in shared memory: 256 for d <= 24,
 * 192 above). */
int scaml_predict_cross_max_points(int d);
size_t scaml_predict_cross_workspace_bytes(int M, int nA, int nB, int reduce);
int scaml_predict_cross(const double* X, const int32_t* n_valid, const double* theta,
                        const double* linv_packed, const double* alpha, const double* ybar,
                        const double* ystd, const double* w, const double* XA, const double* XB,
                        double* mean, double* cov, void* workspace, size_t workspace_bytes, int M,
                        int n_max, int d, int nA, int nB, int kernel, int reduce, void* stream);

/* a7: ScaML-GP target objective in training mode, R rows (restarts) per call:
 *   mean = (S w - mu_all)/s_all,  K = (sum_i w_i^2 C_i)/s_all^2 + s k(X_t) + (noise + jitter) I
 *   lml[r] = ( log N(y_t | mean, K) + log p(theta_t) + sum_i log p(w_i) ) / n_t
 * and its gradient w.r.t. the weights (grad_w [R][M]) and the RAW kernel parameters
 * (grad_theta [R][P]).  S = source_means [n_t][M], C = source_covs [n_t][n_t][M] (outputs of
 * scaml_predict_cross, reduce = 0), y_t standardised with the frozen all-data transform.
 * Replaces `mll(model(X_t), y_t)` + backward on the `ScaMLGP.forward` training branch
 * (reference scamlgp/model.py:359-363,376-383; weights prior :325-330).  n_t <= 116. */
size_t scaml_target_workspace_bytes(int n_t, int R);
/* Largest n_t the shared-memory target-GP kernels accept at input dimension d (their n_t x n_t system plus the
 * d x n_t scaled inputs must fit 227 KB: 116 for small d); the host mirrors raise above it
 * (scamlgp_b200/model.py: ScaMLGP.__init__) where the reference (model.py:359-384) has no limit. */
int scaml_target_max_points(int d);
int scaml_target_lml_grad(const double* source_means, const double* source_covs, const double* Xt,
                          const double* yt, const double* w, const double* theta_raw,
                          const double* jitter, double mu_all, double s_all, double* lml,
                          double* grad_w, double* grad_theta, int32_t* info, void* workspace,
                          size_t workspace_bytes, int M, int n_t, int d, int R,
                          const scaml_hyper_spec* spec, int w_prior, double w_p1, double w_p2,
                          void* stream);

/* scaml_target_lml_grad with linear_operator's psd_safe_cholesky jitter ladder applied INSIDE the kernel: a row whose
 * factorisation fails is retried with +1e-8, +1e-7, +1e-6 on the diagonal before it is reported (info > 0, NaN
 * outputs).  Same results as re-running the failed rows from the host with those jitters, without reading `info`
 * back between the rounds of the L-BFGS driver (reference call site scamlgp/utils.py:171-177,190-192). */
int scaml_target_lml_grad_ladder(const double* source_means, const double* source_covs, const double* Xt,
                                 const double* yt, const double* w, const double* theta_raw, double mu_all,
                                 double s_all, double* lml, double* grad_w, double* grad_theta, int32_t* info,
                                 void* workspace, size_t workspace_bytes, int M, int n_t, int d, int R,
                                 const scaml_hyper_spec* spec, int w_prior, double w_p1, double w_p2, void* stream);

/* Target-GP prediction state at the fitted parameters (R = 1): row-major L_t^-1 [n_t][n_t] of
 * K = (sum_i w_i^2 C_i)/s_all^2 + s k(X_t) + (noise + jitter) I, alpha_t = K^-1 (y_t - mean) [n_t], the
 * constrained kernel parameters theta [P] and the objective value lml[1].  Replaces the prediction
 * strategy gpytorch builds on the first `ScaMLGP.posterior` call in eval mode (exact_prediction over the
 * training-branch prior, reference scamlgp/model.py:359-363,376-383).  Workspace:
 * scaml_target_workspace_bytes(n_t, 1) + 8 * (d + 3) bytes. */
int scaml_target_factorize(const double* source_means, const double* source_covs, const double* Xt,
                           const double* yt, const double* w, const double* theta_raw,
                           double jitter_value, double mu_all, double s_all, double* linv_t,
                           double* alpha_t, double* theta, double* lml, int32_t* info,
                           void* workspace, size_t workspace_bytes, int M, int n_t, int d,
                           const scaml_hyper_spec* spec, void* stream);

/* ScaML-GP posterior at B candidates (q = 1) conditioned on the n_t target points:
 *   k_s[j]  = cross[b][j]/s_all^2 + s k(x_b, X_t[j])
 *   mean[b] = mu_all + s_all ((prior_mean[b] - mu_all)/s_all + k_s . alpha_t)
 *   var[b]  = s_all^2 (prior_var[b]/s_all^2 + s - ||L_t^-1 k_s||^2)
 * prior_mean / prior_var [B] come from scaml_predict_weighted and cross [B][n_t] from
 * scaml_predict_cross (reduce = 1, A = candidates, B = X_t), all with the pruned weights.  Replaces the
 * eval branch of `ScaMLGP.forward` + gpytorch exact prediction + un-standardisation
 * (reference scamlgp/model.py:364-383); consumer: UpperConfidenceBound, scamlgp/utils.py:215-224. */
int scaml_target_posterior(const double* prior_mean, const double* prior_var, const double* cross,
                           const double* Xc, const double* Xt, const double* theta,
                           const double* linv_t, const double* alpha_t, double mu_all, double s_all,
                           double* mean, double* var, int B, int n_t, int d, int kernel, void* stream);

/* Analytic candidate gradients of the ScaML-GP posterior (q = 1), the quantity botorch's optimize_acqf obtains by
 * autograd through `ScaMLGP.forward` (eval branch, reference scamlgp/model.py:364-375) + gpytorch's exact prediction
 * while L-BFGS-B maximises the acquisition function (consumer: UpperConfidenceBound, scamlgp/utils.py:215-224).
 *   scaml_target_posterior_beta : scaml_target_posterior plus beta[b][:] = K_t^-1 k_s(x_b)   [B][n_tp], n_tp = 8*ceil(n_t/8)
 *   scaml_posterior_grad        : dmean [B][d] = d mean / d x_b,  dvar [B][d] = d var / d x_b  (un-standardised, as
 *                                 scaml_target_posterior returns them; for n_t = 0 the gradient of the weighted prior
 *                                 of scaml_predict_weighted).
 * U [M][n_pad][B_p] = K_m^-1 K_m(X_m, Xc) is the output of scaml_cond_prepare called with the candidates in the place
 * of the target inputs (B_p = 8*ceil(B/8), B <= 128 per call); A [M][n_pad][n_tp] is scaml_cond_prepare at X_t;
 * theta_t [P] / alpha_t [n_t] are the outputs of scaml_target_factorize.  For n_t = 0 pass NULL for Xt, A, alpha_t,
 * beta, theta_t.  U is CONSUMED when n_t > 0: a DMMA pass replaces it by U - A beta(x_b) in place before the
 * contraction.  Tasks with w == 0 are skipped (pruning).  The sum over tasks runs in a fixed order
 * (deterministic).  kernel_t = -1 leaves out the terms of the target kernel itself: with the tasks sharded over
 * GPUs every rank contracts its block and exactly one rank adds those terms before the all-reduce(sum). */
int scaml_target_posterior_beta(const double* prior_mean, const double* prior_var, const double* cross,
                                const double* Xc, const double* Xt, const double* theta, const double* linv_t,
                                const double* alpha_t, double mu_all, double s_all, double* mean, double* var,
                                double* beta, int B, int n_t, int d, int kernel, void* stream);
size_t scaml_posterior_grad_workspace_bytes(int M, int n_max, int d, int B);
int scaml_posterior_grad(const double* X, const int32_t* n_valid, const double* theta, const double* alpha,
                         const double* ystd, const double* w, const double* Xc, double* U, const double* Xt,
                         const double* A, const double* alpha_t, const double* beta, const double* theta_t,
                         double s_all, double* dmean, double* dvar, void* workspace, size_t workspace_bytes, int M,
                         int n_max, int d, int B, int n_t, int kernel, int kernel_t, void* stream);

/* Joint posterior of q-point blocks (batch acquisition, q > 1: botorch's optimize_acqf over q candidates jointly, by
 * autograd through `ScaMLGP.forward`, eval branch, reference scamlgp/model.py:364-375).  Xc [B][d] holds B / q blocks
 * of q consecutive points, 1 <= q <= 16, B % q == 0, B <= 128 per call.  U is the output of scaml_cond_prepare_pruned
 * at Xc (as for scaml_posterior_grad); with c_m = w_m^2 ystd_m^2:
 *   scaml_qblock_cov : weighted prior block of every block, cov [B / q][q][q],
 *                        cov[b][i][j] = sum_m c_m ( s_m kappa_m(x_i, x_j) - k*_m(x_i)^T K_m^-1 k*_m(x_j) )
 *                      (exactly symmetric; its diagonal is the variance of scaml_predict_weighted).  U is read only.
 *                      The conditioning on the target points, Sigma = cov + s_all^2 (s_t kappa_t(x_i, x_j) -
 *                      k_s(x_i)^T beta(x_j)), is n_t-dimensional and left to the caller.
 *   scaml_qblock_vjp : vector-Jacobian product of the conditioned posterior (mean [B], Sigma [B / q][q][q], the
 *                      quantities of scaml_target_posterior_beta / scaml_qblock_cov): given g_mean [B] = da/dmean and
 *                      g_cov [B / q][q][q] = da/dSigma, dX [B][d] = da/dXc.  Same inputs as scaml_posterior_grad
 *                      (beta from scaml_target_posterior_beta; NULL Xt, A, alpha_t, beta for n_t = 0) plus theta_t,
 *                      which is required for every n_t (s_t kappa_t(x_i, x_j) is part of Sigma).  U is CONSUMED.
 *                      kernel_t = 0..3 (no task-sharded partial sums).
 * Tasks with w == 0 are skipped; every sum over tasks runs in a fixed order (deterministic). */
size_t scaml_qblock_cov_workspace_bytes(int M, int B, int q);
int scaml_qblock_cov(const double* X, const int32_t* n_valid, const double* theta, const double* ystd,
                     const double* w, const double* Xc, const double* U, double* cov, void* workspace,
                     size_t workspace_bytes, int M, int n_max, int d, int B, int q, int kernel, void* stream);
size_t scaml_qblock_vjp_workspace_bytes(int M, int n_max, int d, int B, int n_t);
int scaml_qblock_vjp(const double* X, const int32_t* n_valid, const double* theta, const double* alpha,
                     const double* ystd, const double* w, const double* Xc, double* U, const double* Xt,
                     const double* A, const double* alpha_t, const double* beta, const double* theta_t,
                     double s_all, const double* g_mean, const double* g_cov, double* dX, void* workspace,
                     size_t workspace_bytes, int M, int n_max, int d, int B, int q, int n_t, int kernel,
                     int kernel_t, void* stream);

/* The same quantities as scaml_predict_conditioned (weighted prior mean [B], variance [B], cross-covariance with the
 * target inputs [B][n_t]; reference scamlgp/model.py:364-375, q = 1) computed from U = K_m^-1 K_m(X_m, Xc) instead of a
 * second pass over the packed factors: mean = sum w (ybar + ystd k*^T alpha), var = sum c (s - k*^T u),
 * cross = sum c (K_m(x, x_tj) - k*^T A_m[:, j]).  The value half of a value-and-gradient evaluation (call it BEFORE
 * scaml_posterior_grad, which consumes U).  B <= 128; n_t = 0: pass NULL for Xt, A, cross. */
size_t scaml_posterior_values_from_u_workspace_bytes(int M, int B, int n_t);
int scaml_posterior_values_from_u(const double* X, const int32_t* n_valid, const double* theta, const double* alpha,
                                  const double* ybar, const double* ystd, const double* w, const double* Xc,
                                  const double* U, const double* Xt, const double* A, double* mean, double* var,
                                  double* cross, void* workspace, size_t workspace_bytes, int M, int n_max, int d,
                                  int B, int n_t, int kernel, void* stream);

/* Conditioning at scale.  scaml_cond_prepare: A_m = K_m^-1 K_m(X_m, X_t) for every source task, A [M][n_pad][n_tp]
 * with n_pad = 64*ceil(n_max/64), n_tp = 8*ceil(n_t/8) (rows >= n_valid and columns >= n_t are zero; the caller
 * zero-initialises A).  It depends only on the fitted source GPs and the target inputs: once per
 * `ScaMLGPBO.report`.  scaml_predict_conditioned: weighted prior mean / variance at B candidates as
 * scaml_predict_weighted PLUS the weighted prior cross-covariance with the target inputs
 *   cross[b][j] = sum_m w_m^2 ystd_m^2 ( K_m(x_b, x_tj) - k*_m(x_b)^T A_m[:, j] )          [B][n_t]
 * with the k*^T A contraction fused into the prediction kernel (the k* tile is already in shared memory).
 * Together with scaml_target_posterior this replaces the eval branch of `ScaMLGP.forward` for q = 1 candidate
 * batches (reference scamlgp/model.py:364-375 evaluates every source posterior at [X_t; x] jointly).
 * scaml_cond_caches: the per-task caches `source_means` [n_t][M] / `source_covs` [n_t][n_t][M] of
 * `ScaMLGP.__init__` (reference scamlgp/model.py:278-289) from A:
 *   source_covs[t][t'][m] = ystd_m^2 ( K_m(x_t, x_t') - K_m(x_t, X_m) A_m[:, t'] ).
 * n_max <= 512 (whatever scaml_predict_weighted accepts), n_t <= 128. */
int scaml_cond_caches(const double* X, const int32_t* n_valid, const double* theta, const double* alpha,
                      const double* ybar, const double* ystd, const double* Xt, const double* A, double* mean,
                      double* cov, int M, int n_max, int d, int n_t, int kernel, void* stream);
int scaml_cond_prepare(const double* X, const int32_t* n_valid, const double* theta, const double* linv_packed,
                       const double* Xt, double* A, int M, int n_max, int d, int n_t, int kernel, void* stream);
/* scaml_cond_prepare restricted to the tasks with w[m] != 0 (the pruned tasks of `significant_weights_mask`,
 * reference scamlgp/model.py:192-215,365-372, are skipped; their slices of A are left untouched).  Used for
 * U = K_m^-1 K_m(X_m, Xc) of scaml_posterior_grad. */
int scaml_cond_prepare_pruned(const double* X, const int32_t* n_valid, const double* theta,
                              const double* linv_packed, const double* Xt, const double* w, double* A, int M,
                              int n_max, int d, int n_t, int kernel, void* stream);
/* Number of task splits the direct term sum_m c_m K_m(x_b, x_tj) of the cross-covariance is summed over (> 1 for
 * small candidate batches, where one CTA per 256 (b, j) pairs would leave the GPU idle; one more launch then). */
int scaml_cond_combine_task_splits(int M, int B, int n_t);
size_t scaml_predict_conditioned_workspace_bytes(int M, int n_max, int d, int B, int n_t);
int scaml_predict_conditioned(const double* X, const int32_t* n_valid, const double* theta,
                              const double* linv_packed, const double* alpha, const double* ybar,
                              const double* ystd, const double* w, const double* Xc, const double* Xt,
                              const double* A, double* mean, double* var, double* cross, void* workspace,
                              size_t workspace_bytes, int M, int n_max, int d, int B, int n_t, int kernel,
                              void* stream);

/* Device-side batched projected L-BFGS (m = history, E independent rows of dimension D, one warp per row).
 * One call consumes the objective values ft [E] / gradients gt [E][D] at the trial points xt [E][D] and
 * overwrites xt with the next trial points of the rows that are still active; flags [E]: bit 0 active, bit 1
 * converged (gtol / ftol / line search at the resolution of the objective), bit 2 failed (objective not finite
 * at the start).  init != 0: xt holds the starting points (already clamped to `lower`), state is initialised.
 * `lower` [D] or NULL (-inf = free variable).  The caller owns every buffer; state buffers must persist between
 * calls.  Replaces the scipy L-BFGS-B loop behind `fit_gpytorch_mll` (reference scamlgp/utils.py:175,190), for
 * all tasks x restarts at once. */
typedef struct scaml_lbfgs_state {
  double* x;         /* [E][D] accepted iterates            */
  double* f;         /* [E]    objective at x               */
  double* g;         /* [E][D] gradient at x                */
  double* d;         /* [E][D] search directions            */
  double* t;         /* [E]    step lengths                 */
  double* S;         /* [E][m][D] iterate differences       */
  double* Y;         /* [E][m][D] gradient differences      */
  double* rho;       /* [E][m]                              */
  int32_t* count;    /* [E] stored pairs                    */
  int32_t* head;     /* [E] next history slot               */
  int32_t* iters;    /* [E] accepted steps                  */
  int32_t* ls_count; /* [E] consecutive rejected trials     */
  int32_t* flags;    /* [E]                                 */
} scaml_lbfgs_state;
int scaml_lbfgs_step(const scaml_lbfgs_state* state, double* xt, const double* ft, const double* gt,
                     const double* lower, int E, int D, int m, int init, double gtol, double ftol,
                     int maxiter, int max_ls, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SCAML_B200_H */
