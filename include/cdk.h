/* cdk.h -- C ABI of the B200-native continuous-discrete Gaussian filtering kernels ("cdk").
 *
 * This is the drop-in boundary for ONE hot path of hd-UQ/cd_dynamax: batched continuous-discrete Kalman / extended /
 * unscented / ensemble Kalman filtering and RTS-type smoothing over N independent, irregularly sampled trajectories.
 * Plain pointers and sizes only; no torch / jax / C++ types.  Every entry point only enqueues work on the given CUDA
 * stream (no host synchronisation, no allocation, no global state) and returns 0 or a negative CDK_E* code for an
 * invalid descriptor.  Numerical failure (non-PD covariance, max_steps exceeded) is not an error: that trajectory's
 * outputs become NaN and status[n] != 0, which is the reference's own "NaNs propagate" behaviour.
 *
 * Reference interface each entry point replaces (paths relative to the reference repository root):
 *   cdk_kf_filter_*    cdlgssm_filter              src/continuous_discrete_linear_gaussian_ssm/inference.py:555-632
 *   cdk_kf_smooth_*    cdlgssm_smoother backward   src/continuous_discrete_linear_gaussian_ssm/inference.py:694-823
 *                      scan (types 1 and 2)          (+ _smooth :636-690)
 *   cdk_ekf_filter_*   extended_kalman_filter      src/continuous_discrete_nonlinear_gaussian_ssm/inference_ekf.py:202-326
 *   cdk_ekf_smooth_*   extended_kalman_smoother    .../inference_ekf.py:450-539 (+ _smooth :363-448)
 *   cdk_ukf_filter_*   unscented_kalman_filter     .../inference_ukf.py:206-308
 *   cdk_enkf_filter_*  ensemble_kalman_filter      .../inference_enkf.py:151-276
 *   cdk_ll_sum_f64     vmap(marginal_log_prob)(...).sum()      src/ssm_temissions.py:555-567
 *   cdk_ll_allreduce   the same sum across GPUs (the reference has no multi-device path)
 * The predict step inside each filter restates diffrax 0.4.0 `diffeqsolve` with `ConstantStepSize`
 * (src/utils/diffrax_utils.py:40-165); the update restates dynamax `psd_solve`/`symmetrize`
 * (dynamax/utils/utils.py:202-211) and TFP `MultivariateNormalFullCovariance.log_prob`.
 *
 * Layout: all arrays row-major, contiguous, last axis fastest (the JAX default), element type = the entry point's
 * dtype (times and parameters too); status is int32.  A leading N axis is present on an input iff its bit is set in
 * cdk_desc.batched_mask (Y and T normally are; parameters are when the caller vmaps over parameter samples).
 */
#ifndef CDK_H_
#define CDK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CDK_VERSION 1

typedef struct CUstream_st* cdk_stream_t; /* == cudaStream_t */

/* error codes (host-side, synchronous) */
enum {
  CDK_OK = 0,
  CDK_E_NULL = -1,        /* a required pointer is NULL */
  CDK_E_SIZE = -2,        /* descriptor size / dimension out of the supported range */
  CDK_E_ENUM = -3,        /* unknown solver / drift / emission / order / smoother type */
  CDK_E_UNSUPPORTED = -4, /* valid request that this build does not implement */
  CDK_E_CUDA = -5,        /* a CUDA runtime call failed; see cdk_last_error() */
  CDK_E_NCCL = -6
};

/* fixed-step explicit solvers (diffrax names; RK4 is the classical tableau the north star names) */
enum { CDK_EULER = 0, CDK_HEUN = 1, CDK_MIDPOINT = 2, CDK_RALSTON = 3, CDK_BOSH3 = 4, CDK_RK4 = 5, CDK_DOPRI5 = 6 };

/* drift registry: a CUDA kernel cannot take the reference's Python callable (cdnlgssm_utils.py:13-36).
 * theta layout:  LINEAR    W[n*n] row-major, bias[n]          (LearnableLinear   cdnlgssm_utils.py:50-61)
 *                LORENZ63  sigma, rho, beta                   (LearnableLorenz63 cdnlgssm_utils.py:63-83)
 *                LORENZ96  forcing F                          (BASELINE configs 4-5; not in the reference)
 *                QUADRATIC a[n], B[n*n], C[n*n*n]: f_i = a_i + B_ij x_j + C_ijk x_j x_k                      */
enum { CDK_DRIFT_LINEAR = 0, CDK_DRIFT_LORENZ63 = 1, CDK_DRIFT_LORENZ96 = 2, CDK_DRIFT_QUADRATIC = 3,
       /* USER: a drift compiled INTO a variant of this library (SURVEY 8f rank 4; the reference takes any Python callable,
        * cdnlgssm_utils.py:13-36).  The caller supplies CUDA device code for f_i(x; theta) and dJ_ij(x; theta) (and,
        * for EKF state_order 'second', g_k = sum_i d2 f_i / dx_i dx_k); cd_dynamax_b200.build.build_user_drift() compiles
        * csrc/ with -DCDK_USER_DRIFT_HEADER=<that code> into lib/user/libcdk_user_<hash>.so, which exports this same ABI.
        * theta: any n_theta >= 0 doubles; with n_theta = 0, in[CDK_IN_F] is not read (may be NULL).  The stock libcdk.so
        * rejects this id. */
       CDK_DRIFT_USER = 4 };
/* emission registry.  LINEAR: h(x) = H x + d (LearnableLinear); in[CDK_IN_H] = H [m,n], in[CDK_IN_D] = d [m].
 * USER: an emission compiled INTO a variant of this library (the reference takes any LearnableFunction.f as emission,
 *   cdnlgssm_utils.py:13-36).  The caller supplies CUDA device code for n_phi = num_params(n, m), h_a(x; phi) and
 *   d h_a / d x_j; cd_dynamax_b200.build.build_variant(drift_code, emission_code) compiles csrc/ with
 *   -DCDK_USER_EMISSION_HEADER=<that code> (a variant may hold a user drift as well).  in[CDK_IN_H] then holds phi
 *   ([n_phi], or [N, n_phi] with its batched_mask bit: the batched stride is n_phi) and in[CDK_IN_D] is not read (may be
 *   NULL).  num_params may be 0 (an emission with no parameters, e.g. a fixed sensor geometry compiled in): in[CDK_IN_H]
 *   is then not read either and may be NULL.  The EKF linearises h at the running mean of every update iteration (H = jac(mu), residual y - h(mu)), the UKF
 *   pushes its 2n + 1 sigma points through h, the EnKF every member, and cdk_sample_path emits h(x_k) + chol(R) z.
 *   The stock library and a variant without a user emission reject this id with CDK_E_UNSUPPORTED, and so do every
 *   gradient entry point and cdk_emission_moments_*. */
enum { CDK_EMISSION_LINEAR = 0, CDK_EMISSION_USER = 1 };
/* EKFHyperParams.state_order (inference_ekf.py:40) */
enum { CDK_ORDER_ZEROTH = 0, CDK_ORDER_FIRST = 1, CDK_ORDER_SECOND = 2 };

/* input slots: in[CDK_NUM_IN] */
enum {
  CDK_IN_Y = 0,   /* emissions            [N,K,m]                                                   */
  CDK_IN_T,       /* observation times    [N,K]   (the reference's [K,1] column, squeezed)         */
  CDK_IN_U,       /* inputs               [N,K,d_u] or NULL (linear model only)                     */
  CDK_IN_M0,      /* initial mean         [n]                                                       */
  CDK_IN_P0,      /* initial covariance   [n,n]                                                     */
  CDK_IN_F,       /* kf: dynamics weights F [n,n];  ekf/ukf/enkf: drift parameter vector theta     */
  CDK_IN_B,       /* kf: dynamics bias b  [n] (added after the pushforward, cd_linear/inference.py:204) */
  CDK_IN_BU,      /* kf: dynamics input weights B [n,d_u] or NULL                                   */
  CDK_IN_L,       /* diffusion coefficient L [n,n]                                                  */
  CDK_IN_QC,      /* diffusion covariance Qc [n,n]                                                  */
  CDK_IN_H,       /* emission weights H   [m,n]   (CDK_EMISSION_USER: emission parameters phi [n_phi]) */
  CDK_IN_D,       /* emission bias d      [m]     (CDK_EMISSION_USER: not read, may be NULL)         */
  CDK_IN_DU,      /* kf: emission input weights D [m,d_u] or NULL                                   */
  CDK_IN_R,       /* emission covariance R [m,m] ([m] with CDK_FLAG_DIAG_R)                         */
  CDK_IN_FM,      /* smooth: filtered means        [N,K,n]                                          */
  CDK_IN_FP,      /* smooth: filtered covariances  [N,K,n,n]                                        */
  CDK_NUM_IN
};

/* output slots: out[CDK_NUM_OUT]; a NULL pointer means "do not write this output" (the reference's output_fields) */
enum {
  CDK_OUT_LL = 0, /* marginal log-likelihood per trajectory [N]                                    */
  CDK_OUT_FM,     /* filtered means        [N,K,n]                                                  */
  CDK_OUT_FP,     /* filtered covariances  [N,K,n,n]                                                */
  CDK_OUT_PM,     /* predicted means       [N,K,n]   (entry k is the prediction for t_{k+1})       */
  CDK_OUT_PP,     /* predicted covariances [N,K,n,n]                                                */
  CDK_OUT_LLCUM,  /* cumulative log-likelihood [N,K] ("marginal_loglik" listed in output_fields)   */
  CDK_OUT_SM,     /* smoothed means        [N,K,n]                                                  */
  CDK_OUT_SP,     /* smoothed covariances  [N,K,n,n]                                                */
  CDK_OUT_SCROSS, /* smoothed cross terms  [N,K-1,n,n] (type 1; NaN for type 2)                    */
  CDK_OUT_STATUS, /* int32 [N]: 0 ok, 1 non-finite result (non-PD / NaN), 2 max_steps exceeded      */
  CDK_OUT_SCRATCH,/* device scratch of cdk_scratch_bytes() bytes (CD-KF pushforward cache), else NULL */
  CDK_OUT_GRAD,   /* d marginal log-likelihood / d parameters: cdk_ekf_grad_f64 [N, CDK_GRAD_COLS_L63],
                   * cdk_kf_grad_f64 [N, CDK_GRAD_COLS_KF(n, m)],
                   * cdk_ekf_grad_dense_f64 / cdk_ukf_grad_dense_f64 / cdk_ukf_grad_sigma_f64 [N, CDK_GRAD_COLS_EKF] */
  CDK_NUM_OUT
};

typedef struct cdk_desc {
  int32_t struct_size;    /* sizeof(cdk_desc), checked */
  int32_t K;              /* observations per trajectory, >= 1 */
  int64_t N;              /* trajectories, >= 0 */
  int32_t n;              /* state dimension   1..CDK_MAX_N */
  int32_t m;              /* emission dimension 1..CDK_MAX_M */
  int32_t d_u;            /* input dimension, 0 = no inputs */
  int32_t E;              /* EnKF ensemble size */
  int32_t solver;         /* CDK_EULER .. CDK_DOPRI5 */
  int32_t max_steps;      /* diffrax max_steps (default 100000) */
  double dt0;             /* solver step (diffrax dt0, default 0.01) */
  double dt_final;        /* length of the gap after the last observation (default 1e-10) */
  int32_t state_order;    /* ekf */
  int32_t num_iter;       /* ekf: re-linearisations in the update (>= 1) */
  int32_t smoother_type;  /* kf smooth: 1 or 2 */
  int32_t drift_id;
  int32_t emission_id;
  int32_t n_theta;        /* length of the drift parameter vector */
  uint32_t batched_mask;  /* bit i set: in[i] has a leading N axis */
  int32_t perturb_measurements; /* enkf */
  double cov_rescaling;   /* ekf zeroth order (inference_ekf.py:135) */
  double alpha, beta, kappa;    /* ukf (inference_ukf.py:31-33) */
  uint64_t rng_seed;      /* enkf: Philox4x32-10 key */
  uint64_t rng_offset;    /* enkf: added to the trajectory index in the counter (sharding across GPUs) */
  int32_t reserved[4];    /* [0], [1]: absent-slot masks of the XLA adaptor; [2]: CDK_FLAG_* bits; [3]: cdk_ekf_grad groups (0 for cdk_kf_grad) */
} cdk_desc;

/* reserved[2] bit 0: keep the pushforward.  cdk_kf_filter_f64 then also writes (A_k, Q_k) of every gap k < K-1 into
 * out[CDK_OUT_SCRATCH] ([N][K-1][2][n][n], cdk_scratch_bytes() bytes) and cdk_kf_smooth_f64 (smoother_type 1) called with
 * the same flag and buffer reads them back instead of re-integrating them (cd_linear/inference.py:753 recomputes; the
 * values are bit-identical).  cdk_scratch_bytes() returns 0 when the request is not served by the warp kernels. */
#define CDK_FLAG_KEEP_PUSHFORWARD 1
/* reserved[2] bit 1: cdk_ukf_filter_* evaluates the 2n + 1 sigma points literally (Cholesky factor of P at every RK stage,
 * inference_ukf.py:45-60, :130-152).  By default the unscented predict runs in closed form -- every registry drift is a
 * polynomial of degree <= 2 and the emission is linear, for which the sigma-point sums are exactly f(m) + tr(Hess P)/2 and
 * J P (cdk_generic.cu, ODE_UKFC) -- which gives the same moments up to rounding at a fraction of the cost. */
#define CDK_FLAG_UKF_SIGMA_POINTS 2
/* reserved[2] bit 2: cdk_kf_filter_*: in[CDK_IN_R] is the DIAGONAL of the emission covariance, [m] (a 1-D emissions.cov):
 * the update takes the reference's Woodbury branch (cd_linear/inference.py:240-254) and the log-likelihood its broadcast
 * of the vector over H P H^T (:613), both restated literally (csrc/cdk_generic.cu: condition_on_diag_r). */
#define CDK_FLAG_DIAG_R 4
/* reserved[2] bit 3: FORECAST (cdk_ekf_filter_*, cdk_ukf_filter_*, cdk_enkf_filter_*, cdk_kf_filter_*): no measurement
 * updates.  in[CDK_IN_T] is [N, K+1] -- t_init followed by the K forecast times --, in[CDK_IN_Y] is ignored (may be NULL),
 * (M0, P0) is the distribution at t_init and out[CDK_OUT_PM] / out[CDK_OUT_PP] [N, K, ...] receive the forecasted moments
 * (forecast_extended_kalman_filter inference_ekf.py:679-761 and its UKF / EnKF twins: the same _predict, scanned). */
#define CDK_FLAG_PREDICT_ONLY 8
/* reserved[2] bit 4: cdk_sample_path_*: start from the given state in[CDK_IN_M0] at t_init instead of sampling
 * x_0 ~ N(m0, P0); in[CDK_IN_T] is then [N, K+1] (t_init, then the K output times) and no emission is drawn at t_init
 * (the point-estimate branch of cdnlgssm_forecast, cd_nonlinear/models.py:840-936). */
#define CDK_FLAG_FIXED_INIT 16

/* Upper bounds of the ABI.  The real limit of the shared-memory kernels (any n > 3 EKF / UKF, KF with n > 16 or m > 8,
 * smoothers) is the 227 KB of one CTA, which holds the whole per-trajectory working set: in fp64 with m = n, KF n <= 38
 * (30 with dopri5, whose seven stages are all kept), EKF n <= 45 (37), UKF n <= 50-55; more with m << n (KF n <= 43 at
 * m = 4), about 1.4x in fp32.  Larger requests return CDK_E_SIZE with a message, never a wrong answer. */
#define CDK_MAX_N 64
#define CDK_MAX_M 64

/* Fill a descriptor with the reference's defaults (KFHyperParams / EKFHyperParams / UKFHyperParams / diffeqsolve). */
void cdk_desc_init(cdk_desc* d);

#define CDK_DECL(name) \
  int name(const cdk_desc* d, const void* const* in, void* const* out, cdk_stream_t stream)

CDK_DECL(cdk_kf_filter_f64);
CDK_DECL(cdk_kf_filter_f32);
CDK_DECL(cdk_kf_smooth_f64);
CDK_DECL(cdk_kf_smooth_f32);
CDK_DECL(cdk_ekf_filter_f64);
CDK_DECL(cdk_ekf_filter_f32);
CDK_DECL(cdk_ekf_smooth_f64);
CDK_DECL(cdk_ekf_smooth_f32);
CDK_DECL(cdk_ukf_filter_f64);
CDK_DECL(cdk_ukf_filter_f32);
CDK_DECL(cdk_enkf_filter_f64);
CDK_DECL(cdk_enkf_filter_f32);
/* The gradient entry points below (cdk_ekf_grad_f64, cdk_kf_grad_f64, cdk_ekf_grad_dense_f64, cdk_ukf_grad_dense_f64,
 * cdk_ukf_grad_sigma_f64) differentiate the linear emission.  cdk_ekf_grad_dense_f64 also differentiates CDK_EMISSION_USER
 * in a variant whose gradient unit was compiled with the emission (build_variant(..., emission_grad=True)); everywhere
 * else the nonlinear entry points return CDK_E_UNSUPPORTED for CDK_EMISSION_USER before any other check.
 *
 * Log-likelihood (out[CDK_OUT_LL]) and its gradient with respect to the model parameters (out[CDK_OUT_GRAD],
 * [N, CDK_GRAD_COLS_L63]) of the CD-EKF: what jax.value_and_grad(marginal_log_prob) hands the reference's fit_sgd
 * (src/utils/optimize_utils.py:102, src/ssm_temissions.py:550-568).  Forward-mode derivative of exactly the discrete filter
 * cdk_ekf_filter_f64 runs, one launch per direction.  Columns: theta = sigma, rho, beta (3) | L Qc L^T, packed upper
 * triangle 00 01 02 11 12 22 (6) | R | d | H (3) | m0 (3) | P0, packed upper triangle (6).  Symmetric matrices are
 * differentiated along SYMMETRIC directions (an off-diagonal column moves both mirror entries).  desc.reserved[3] is a
 * bit mask of the column groups to compute, in that order (0 = theta only); other columns are left untouched.  Today:
 * Lorenz-63 drift, scalar emission, num_iter = 1, state_order first / second; anything else returns CDK_E_UNSUPPORTED. */
#define CDK_GRAD_COLS_L63 23
/* desc.reserved[3] bit 7: REVERSE mode -- all 23 columns from ONE backward launch behind a forward filter pass whose moments
 * go to out[CDK_OUT_SCRATCH] (cdk_scratch_bytes(desc, "cdk_ekf_grad") = N*K*24*8 bytes); ~4 filter passes in total instead
 * of ~2.2 per column.  Without the bit (or without scratch) the forward-mode kernels run, one launch per requested column. */
#define CDK_GRAD_REVERSE 128
CDK_DECL(cdk_ekf_grad_f64);
/* Log-likelihood (out[CDK_OUT_LL]), status (out[CDK_OUT_STATUS]) and reverse-mode gradient (out[CDK_OUT_GRAD],
 * [N, CDK_GRAD_COLS_KF(n, m)]) of the linear CD Kalman filter, for the same descriptor and inputs as cdk_kf_filter_f64:
 * what jax.value_and_grad(marginal_log_prob) hands the reference's fit_sgd for ContDiscreteLinearGaussianSSM.  The forward
 * pass IS cdk_kf_filter_f64 (the log-likelihood is bit-identical), its moments go to out[CDK_OUT_SCRATCH] (required,
 * cdk_scratch_bytes(desc, "cdk_kf_grad") bytes, linear in N), then one backward launch re-integrates every gap and steps
 * back through it.  Columns, row-major blocks in this order: F (n*n, entry-wise) | b (n) | Sigma = L Qc L^T (n*n) |
 * H (m*n) | d (m) | R (m*m) | m0 (n) | P0 (n*n).  Symmetric parameters (Sigma, R, P0) get the symmetric part (G + G^T)/2
 * of the entry-wise gradient G, i.e. the derivative along symmetric directions.  A trajectory whose status is not 0 gets
 * a NaN row.  Coverage: fp64, n <= 16, m <= 8, every solver, shared or batched parameters; d_u > 0, CDK_FLAG_DIAG_R,
 * CDK_FLAG_PREDICT_ONLY, n > 16 or m > 8 return CDK_E_UNSUPPORTED, a NULL out[CDK_OUT_GRAD] or out[CDK_OUT_SCRATCH]
 * CDK_E_NULL (host-side checks, before any CUDA call).  desc.reserved[3] must be 0. */
#define CDK_GRAD_COLS_KF(n, m) (3 * (n) * (n) + (m) * (n) + (m) * (m) + 2 * (n) + (m))
CDK_DECL(cdk_kf_grad_f64);
/* Log-likelihood (out[CDK_OUT_LL]), status (out[CDK_OUT_STATUS]) and reverse-mode gradient (out[CDK_OUT_GRAD],
 * [N, CDK_GRAD_COLS_EKF(n, m, n_theta)]) of the CD-EKF for every registry drift (LINEAR, LORENZ63, LORENZ96, QUADRATIC)
 * and emission size, for the same descriptor and inputs as cdk_ekf_filter_f64.  The forward pass IS the launch
 * cdk_ekf_filter_f64 makes (the log-likelihood is bit-identical), its moments go to out[CDK_OUT_SCRATCH] (required), then
 * one backward launch (one CTA per trajectory) re-integrates every gap and steps back through it.  Columns, row-major
 * blocks in this order: theta (n_theta) | Sigma = L Qc L^T (n*n) | H (m*n) | d (m) | R (m*m) | m0 (n) | P0 (n*n); for a
 * LINEAR drift theta = W | bias is the F | b of CDK_GRAD_COLS_KF.  Sigma, R and P0 get the symmetric part (G + G^T)/2.
 * A trajectory whose status is not 0 gets a NaN row.  The gap after the last observation does not enter the
 * log-likelihood and is not differentiated.
 * Scratch, cdk_scratch_bytes(desc, "cdk_ekf_grad_dense") = 8 N (K (2 n + 2 n^2) + (64 + 2 S) st + 1) bytes with
 * st = 2 ceil(n / 2) + n (n | 1) (one moment state) and S the solver's stage count: the forward moments, two levels of
 * 32 checkpoints and the stage inputs and cotangents of one substep.
 * Coverage: fp64, state_order first / second, num_iter = 1, full R, every solver, shared or batched parameters, and
 * CDK_DRIFT_USER in a variant built with build_user_drift(code, grad=True), whose backward pass takes the drift's
 * derivatives from dual-number evaluations of the user's f / jac / graddiv (the
 * scratch formula is the same; the shared memory adds a dual copy of [x | theta], and an n_theta that does not fit
 * returns CDK_E_SIZE).  The stock library and a filter-only variant reject CDK_DRIFT_USER with CDK_E_UNSUPPORTED.
 * state_order zeroth, num_iter > 1, CDK_FLAG_DIAG_R, CDK_FLAG_PREDICT_ONLY, d_u > 0 and a non-zero
 * desc.reserved[3] return CDK_E_UNSUPPORTED, a NULL out[CDK_OUT_GRAD] or out[CDK_OUT_SCRATCH] CDK_E_NULL, a shape whose
 * backward working set exceeds the 227 KB of one CTA CDK_E_SIZE (with m = n, n <= 36 for RK4; n = 40, m = 20
 * fits with every solver) -- all host-side checks, before any CUDA call.
 * CDK_GRAD_COLS_EKF is shared with cdk_ukf_grad_dense_f64, whose rows have the same layout. */
#define CDK_GRAD_COLS_EKF(n, m, n_theta) ((n_theta) + 2 * (n) * (n) + (m) * (n) + (m) * (m) + (n) + (m))
/* CDK_EMISSION_USER in a variant built with build_variant(..., emission_grad=True) (LearnableUserEmission(...,
 * differentiable=True)): the emission is re-linearised at every step's predicted mean, as the filter does, and the
 * second derivatives of the user's h / jac come from dual-number evaluations of its own code (DESIGN 4.2h).  The row is
 * theta | Sigma | phi (n_phi) | R | m0 | P0: phi takes the place of H | d (for the linear emission written as user
 * code, phi = [H | d] and the row has the stock layout).  The shared memory adds phi, its cotangent and the dual copies
 * of [x | phi] (aliasing the moment buffers when they fit there); an n_phi that does not fit returns CDK_E_SIZE naming
 * n_phi (registry drifts; n = 40, m = 20: n_phi <= 1,099; n = 2, m = 1: n_phi <= 4,070).  A drift may be a registry drift or a
 * differentiable CDK_DRIFT_USER.  The stock library and a variant whose gradient unit lacks the emission reject
 * CDK_EMISSION_USER with CDK_E_UNSUPPORTED before any other check. */
#define CDK_GRAD_COLS_EKF_UE(n, m, n_theta, n_phi) ((n_theta) + 2 * (n) * (n) + (n_phi) + (m) * (m) + (n))
CDK_DECL(cdk_ekf_grad_dense_f64);
/* Log-likelihood (out[CDK_OUT_LL]), status (out[CDK_OUT_STATUS]) and reverse-mode gradient (out[CDK_OUT_GRAD],
 * [N, CDK_GRAD_COLS_EKF(n, m, n_theta)], the row layout of cdk_ekf_grad_dense_f64) of the CD-UKF for every registry
 * drift and emission size, for the same descriptor and inputs as cdk_ukf_filter_f64: what jax.value_and_grad of
 * marginal_log_prob with UKFHyperParams hands the reference's fit_sgd.  The forward pass IS the launch cdk_ukf_filter_f64
 * makes, in closed form (the log-likelihood is bit-identical on the register-resident and the shared-memory moment ODE
 * alike), its moments go to out[CDK_OUT_SCRATCH] (required, cdk_scratch_bytes(desc, "cdk_ukf_grad_dense") bytes: the
 * formula of cdk_ekf_grad_dense_f64), then the backward launch of cdk_ekf_grad_dense_f64 runs with the unscented mean
 * term 0.5 tr(Hess f . P).  Sigma, R and P0 get the symmetric part (G + G^T)/2; a trajectory whose status is not 0 gets
 * a NaN row.  alpha, beta and kappa do not enter the closed form and get no gradient; state_order and num_iter do not
 * apply and are ignored, as by the filter.
 * Coverage: fp64, full R, every solver, shared or batched parameters, the same shapes as cdk_ekf_grad_dense_f64.
 * CDK_DRIFT_USER and CDK_FLAG_UKF_SIGMA_POINTS (literal sigma points: cdk_ukf_grad_sigma_f64 differentiates those),
 * CDK_FLAG_DIAG_R, CDK_FLAG_PREDICT_ONLY, d_u > 0 and a non-zero desc.reserved[3] return CDK_E_UNSUPPORTED, a NULL
 * out[CDK_OUT_GRAD] or out[CDK_OUT_SCRATCH] CDK_E_NULL, a backward working set beyond the 227 KB of one CTA CDK_E_SIZE --
 * all host-side checks, before any CUDA call. */
CDK_DECL(cdk_ukf_grad_dense_f64);
/* Log-likelihood (out[CDK_OUT_LL]), status (out[CDK_OUT_STATUS]) and reverse-mode gradient (out[CDK_OUT_GRAD],
 * [N, CDK_GRAD_COLS_EKF(n, m, n_theta)], the row layout of cdk_ekf_grad_dense_f64) of the CD-UKF with LITERAL sigma
 * points, for the same descriptor and inputs as cdk_ukf_filter_f64.  The entry point sets CDK_FLAG_UKF_SIGMA_POINTS on
 * its own copy of the descriptor, so the forward pass IS the launch cdk_ukf_filter_f64 makes with that flag (the
 * log-likelihood is bit-identical to it) whatever the caller's flags say.  Its moments go to out[CDK_OUT_SCRATCH]
 * (required, cdk_scratch_bytes(desc, "cdk_ukf_grad_sigma") bytes: the formula of cdk_ekf_grad_dense_f64 -- the sigma
 * points of the backward pass live in shared memory), then one backward launch (ukf_sigma_grad_kernel) steps back
 * through the sigma-point moment ODE: a Cholesky factor of P, 2n + 1 drift evaluations and their VJPs, and the Cholesky
 * VJP at every stage.  Its shared memory is that of cdk_ekf_grad_dense_f64 plus one n x (n | 1) block (n = 40, m = 20
 * fits with every solver).  Sigma, R and P0 get the symmetric part (G + G^T)/2; a trajectory whose status is not 0 gets a
 * NaN row.  alpha, beta and kappa get no gradient (beta does not enter the predict; alpha and kappa are hyper-parameters).
 * Coverage: fp64, full R, every solver, shared or batched parameters, every registry drift, and CDK_DRIFT_USER in a
 * variant built with build_user_drift(code, grad=True) (the theta-derivatives of f from dual numbers; an n_theta that
 * does not fit returns CDK_E_SIZE).  The stock library and a filter-only variant reject CDK_DRIFT_USER with
 * CDK_E_UNSUPPORTED.  CDK_FLAG_DIAG_R, CDK_FLAG_PREDICT_ONLY, d_u > 0 and a non-zero desc.reserved[3] return
 * CDK_E_UNSUPPORTED, a NULL out[CDK_OUT_GRAD] or out[CDK_OUT_SCRATCH] CDK_E_NULL, a backward working set beyond the
 * 227 KB of one CTA CDK_E_SIZE -- all host-side checks, before any CUDA call. */
CDK_DECL(cdk_ukf_grad_sigma_f64);

/* Forward sample paths of the model (cdnlgssm_path_sample, cd_nonlinear/models.py:525-656; what
 * SSM.sample_batch(..., transition_type="path") vmaps, src/ssm_temissions.py:187-225): x_0 ~ N(m0, P0), x_k = SDE solve of
 * dx = f(x) dt + L chol(Qc) dW over [t_{k-1}, t_k] (desc.solver = CDK_HEUN, the reference default for SDEs, or CDK_EULER =
 * Euler-Maruyama; diffrax stepping rule with desc.dt0), y_k ~ N(H x_k + d, R) (CDK_EMISSION_USER: y_k ~ N(h(x_k), R), the same
 * deviates).  out[CDK_OUT_FM] = states [N, K, n],
 * out[CDK_OUT_PM] = emissions [N, K, m] (either may be NULL), out[CDK_OUT_STATUS].  Philox4x32-10 stream keyed by
 * desc.rng_seed / rng_offset (the reference's jax.random stream is not reproducible outside JAX).  Model parameters must
 * not be batched (in[CDK_IN_M0] may be). */
CDK_DECL(cdk_sample_path_f64);
CDK_DECL(cdk_sample_path_f32);
/* Emission moments of Gaussian state estimates under the linear emission (CDK_EMISSION_USER returns CDK_E_UNSUPPORTED;
 * emissions_extended_kalman_filter,
 * inference_ekf.py:762-855, and its unscented twin): in[CDK_IN_FM] [N, K, n], in[CDK_IN_FP] [N, K, n, n] or NULL (point
 * estimates) -> out[CDK_OUT_PM] = H m + d [N, K, m], out[CDK_OUT_PP] = H P H^T + R [N, K, m, m]. */
CDK_DECL(cdk_emission_moments_f64);
CDK_DECL(cdk_emission_moments_f32);

/* Bytes of device scratch the given entry point needs in out[CDK_OUT_SCRATCH] (0 for most). algo: "kf_filter", ... */
size_t cdk_scratch_bytes(const cdk_desc* d, const char* entry_point);

/* Deterministic sum of ll[N] into *ll_sum (one double / float on the device): the reference's `.sum()` over the
 * vmapped axis (src/ssm_temissions.py:567). */
int cdk_ll_sum_f64(const double* ll, int64_t N, double* ll_sum, cdk_stream_t stream);
int cdk_ll_sum_f32(const float* ll, int64_t N, double* ll_sum, cdk_stream_t stream);

/* Sum *ll_sum (one double on the device) across the ranks of an NCCL communicator, in place.
 * `nccl_comm` is an ncclComm_t created by the caller; libnccl is resolved at run time (dlopen). */
int cdk_ll_allreduce(void* nccl_comm, double* ll_sum, cdk_stream_t stream);

/* Legacy XLA GPU custom-call target (jax 0.4.13: xla_client.register_custom_call_target(name, capsule, "CUDA")).
 * opaque = a cdk_xla_opaque blob: {char entry_point[32]; cdk_desc desc;}.  buffers = in[0..CDK_NUM_IN) followed by
 * out[0..CDK_NUM_OUT) with absent slots passed as zero-size dummies flagged in desc.reserved[0] (absent-input mask)
 * and desc.reserved[1] (absent-output mask). */
typedef struct cdk_xla_opaque {
  char entry_point[32];
  cdk_desc desc;
} cdk_xla_opaque;
void cdk_xla_custom_call(cdk_stream_t stream, void** buffers, const char* opaque, size_t opaque_len);
/* The same target with XLA's status-returning signature (CustomCallApiVersion API_VERSION_STATUS_RETURNING; register with
 * api_version=1 in jax 0.4.13's xla_client).  A non-zero CDK_E_* code from descriptor validation or the launch is
 * reported with XlaCustomCallStatusSetFailure(status, "cdk (<code>): <cdk_last_error()>"), resolved from the calling XLA
 * runtime at run time, so a rejected request fails the XLA executable instead of passing silently.  `status` may be NULL. */
void cdk_xla_custom_call_status(cdk_stream_t stream, void** buffers, const char* opaque, size_t opaque_len, void* status);
/* Return code of the last cdk_xla_custom_call* on this thread (the legacy signature has no way to report it). */
int cdk_xla_last_rc(void);

/* FP64/FP32 FMA-pipe probe used by bench.py for the roofline denominator: runs `iters` dependent-chain-free FMAs per
 * thread on `blocks` x 256 threads and writes one value per thread to sink (so the work is not eliminated).
 * flops = 2 * 16 * iters * blocks * 256.  Returns 0 / CDK_E_CUDA. */
int cdk_fma_probe_f64(int blocks, int iters, double* sink, cdk_stream_t stream);
int cdk_fma_probe_f32(int blocks, int iters, float* sink, cdk_stream_t stream);
/* The same FMA probe with three DISTINCT vector-register operands per FMA (seed: 256 finite doubles on the device):
 * flops = 2 * 16 * iters * blocks * 256.  On B200 this runs at 2/3 of cdk_fma_probe_f64 (register-file read bandwidth:
 * a three-register DFMA issues every 3 cycles per SM sub-partition, not 2) -- the attainable rate of filter arithmetic. */
int cdk_fma3_probe_f64(int blocks, int iters, double* sink, const double* seed, cdk_stream_t stream);
/* FP64 tensor-core probe (mma.sync m8n8k4 f64, the path the EnKF ensemble contractions use): 8 independent
 * accumulator tiles per warp; flops = 2 * 8*8*4 * 8 * iters * blocks * 8 warps. */
int cdk_dmma_probe_f64(int blocks, int iters, double* sink, cdk_stream_t stream);

/* The library's normal deviates (the counter-based stream of the EnKF and the path sampler, csrc/cdk_rng.cuh): writes the
 * four deviates of counter (member = i, traj, step, c3 = c3_base + (i & 0xff)) for i < count to out[4 i .. 4 i + 3].
 * Test hook: the CPU oracle reproduces the stream bit for bit (oracle/cd_oracle.py:philox_normal_quad). */
int cdk_rng_probe_f64(int64_t count, uint32_t traj, uint32_t step, uint32_t c3_base, uint64_t seed, double* out,
                      cdk_stream_t stream);

/* Diagnostics: register (or clear, with NULL) a device buffer of 4 x uint64 per warp of 32 trajectories; the Lorenz-63
 * EKF kernel then records {globaltimer at entry, at exit, %smid, %warpid} per warp (scripts/trace_lw.py). */
int cdk_debug_set_trace(void* devbuf);

/* Number of kernels this library has launched since load (for bench.py's gpu_launches accounting). */
int64_t cdk_launch_count(void);

/* 1 when this library is a variant compiled with a user-defined drift (CDK_DRIFT_USER), 0 for the stock build. */
int cdk_has_user_drift(void);
/* 1 when this library is a variant compiled with a user-defined emission (CDK_EMISSION_USER), 0 otherwise. */
int cdk_has_user_emission(void);
/* Length n_phi of the user emission's parameter vector for state dimension n and emission dimension m (its num_params),
 * or -1 in a library without a user emission. */
int cdk_user_emission_params(int n, int m);
int cdk_version(void);
const char* cdk_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* CDK_H_ */
