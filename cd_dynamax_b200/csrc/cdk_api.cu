// cdk_api.cu -- extern "C" entry points: descriptor validation, dispatch, reductions, XLA adaptor, NCCL hook.
#include <dlfcn.h>
#include <stdio.h>
#include <string.h>

#include <atomic>

#include "cdk_common.cuh"
#include "cdk_rng.cuh"

namespace cdk {

static std::atomic<long long> g_launches{0};
static thread_local char g_err[256] = "";

void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int check_launch(const char* what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    cudaGetLastError();
    return CDK_E_CUDA;
  }
  return CDK_OK;
}

static int fail(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}

// elements per trajectory of every input slot
static long long slot_elems(const cdk_desc& d, int slot, int algo) {
  const long long n = d.n, m = d.m, K = d.K, du = d.d_u;
  switch (slot) {
    case CDK_IN_Y: return K * m;
    case CDK_IN_T: return (d.reserved[2] & (CDK_FLAG_PREDICT_ONLY | CDK_FLAG_FIXED_INIT)) ? K + 1 : K;
    case CDK_IN_U: return K * du;
    case CDK_IN_M0: return n;
    case CDK_IN_P0: return n * n;
    case CDK_IN_F: return (algo == ALGO_KF_FILTER || algo == ALGO_KF_SMOOTH) ? n * n : d.n_theta;
    case CDK_IN_B: return n;
    case CDK_IN_BU: return n * du;
    case CDK_IN_L: return n * n;
    case CDK_IN_QC: return n * n;
    case CDK_IN_H:  // phi of a user emission (the linear model has no emission registry)
      return (algo != ALGO_KF_FILTER && algo != ALGO_KF_SMOOTH && d.emission_id == CDK_EMISSION_USER)
                 ? cdk::user_emission_params(d.n, d.m) : m * n;
    case CDK_IN_D: return m;
    case CDK_IN_DU: return m * du;
    case CDK_IN_R: return ((algo == ALGO_KF_FILTER || algo == ALGO_KF_SMOOTH) && (d.reserved[2] & CDK_FLAG_DIAG_R)) ? m : m * m;
    case CDK_IN_FM: return K * n;
    case CDK_IN_FP: return K * n * n;
  }
  return 0;
}

static int expected_theta(const cdk_desc& d) {
  switch (d.drift_id) {
    case CDK_DRIFT_LINEAR: return d.n * d.n + d.n;
    case CDK_DRIFT_LORENZ63: return 3;
    case CDK_DRIFT_LORENZ96: return 1;
    case CDK_DRIFT_QUADRATIC: return d.n + d.n * d.n + d.n * d.n * d.n;
    case CDK_DRIFT_USER: return d.n_theta >= 0 ? d.n_theta : -1;
  }
  return -1;
}

static int validate(const cdk_desc* d, const void* const* in, void* const* out, int algo) {
  if (!d || !in || !out) return fail(CDK_E_NULL, "descriptor / in / out is NULL");
  if (d->struct_size != (int)sizeof(cdk_desc)) return fail(CDK_E_SIZE, "cdk_desc.struct_size mismatch");
  if (d->N < 0 || d->K < 1) return fail(CDK_E_SIZE, "need N >= 0 and K >= 1");
  if (d->n < 1 || d->n > CDK_MAX_N || d->m < 1 || d->m > CDK_MAX_M) return fail(CDK_E_SIZE, "n or m out of range");
  if (d->d_u < 0 || d->d_u > 64) return fail(CDK_E_SIZE, "d_u out of range");
  if (d->solver < CDK_EULER || d->solver > CDK_DOPRI5) return fail(CDK_E_ENUM, "unknown solver");
  if (!(d->dt0 > 0.0)) return fail(CDK_E_SIZE, "dt0 must be positive");
  if (d->max_steps < 1) return fail(CDK_E_SIZE, "max_steps must be >= 1");
  const bool linear = algo == ALGO_KF_FILTER || algo == ALGO_KF_SMOOTH;
  const bool smooth = algo == ALGO_KF_SMOOTH || algo == ALGO_EKF_SMOOTH;
  const bool user_emission = !linear && d->emission_id == CDK_EMISSION_USER;  // in[CDK_IN_D] is not read
  // a parameter-free user emission (num_params = 0) or user drift (n_theta = 0) reads nothing from in[CDK_IN_H] /
  // in[CDK_IN_F]: the caller may pass NULL there (an empty array has no data pointer)
  const bool no_phi = user_emission && cdk::user_emission_params(d->n, d->m) == 0;
  const bool no_theta = !linear && d->drift_id == CDK_DRIFT_USER && d->n_theta == 0;
  auto optional_input = [&](int s) {
    return (user_emission && s == CDK_IN_D) || (no_phi && s == CDK_IN_H) || (no_theta && s == CDK_IN_F);
  };
  if (!linear && algo != ALGO_EMISSIONS) {
    if (d->drift_id < CDK_DRIFT_LINEAR || d->drift_id > CDK_DRIFT_USER) return fail(CDK_E_ENUM, "unknown drift_id");
    if (d->drift_id == CDK_DRIFT_USER && !cdk::has_user_drift())
      return fail(CDK_E_UNSUPPORTED, "CDK_DRIFT_USER needs a variant library built with the user's device code (build_user_drift)");
    if (d->emission_id != CDK_EMISSION_LINEAR && d->emission_id != CDK_EMISSION_USER) return fail(CDK_E_ENUM, "unknown emission_id");
    if (d->emission_id == CDK_EMISSION_USER && !cdk::has_user_emission())
      return fail(CDK_E_UNSUPPORTED, "CDK_EMISSION_USER needs a variant library built with the user's emission code (build_variant)");
    if (d->n_theta != expected_theta(*d)) return fail(CDK_E_SIZE, "n_theta does not match drift_id / n");
    if (d->drift_id == CDK_DRIFT_LORENZ63 && d->n != 3) return fail(CDK_E_SIZE, "lorenz63 needs n == 3");
    if (d->drift_id == CDK_DRIFT_LORENZ96 && d->n < 4) return fail(CDK_E_SIZE, "lorenz96 needs n >= 4");
    if (d->drift_id == CDK_DRIFT_QUADRATIC && d->n > 16) return fail(CDK_E_SIZE, "quadratic drift needs n <= 16");
  }
  if (algo == ALGO_EKF_FILTER || algo == ALGO_EKF_SMOOTH) {
    if (d->state_order < CDK_ORDER_ZEROTH || d->state_order > CDK_ORDER_SECOND) return fail(CDK_E_ENUM, "unknown state_order");
    if (d->num_iter < 1) return fail(CDK_E_SIZE, "num_iter must be >= 1");
  }
  if (algo == ALGO_KF_SMOOTH && d->smoother_type != 1 && d->smoother_type != 2) return fail(CDK_E_ENUM, "smoother_type must be 1 or 2");
  if (!linear && (d->reserved[2] & CDK_FLAG_DIAG_R)) return fail(CDK_E_UNSUPPORTED, "CDK_FLAG_DIAG_R applies to the linear model only");
  if (algo == ALGO_ENKF_FILTER) {
    if (d->E < 2 || d->E > 65536) return fail(CDK_E_SIZE, "E out of range");
    if (d->solver != CDK_EULER && d->solver != CDK_HEUN) return fail(CDK_E_UNSUPPORTED, "EnKF supports solver euler (Euler-Maruyama) or heun");
  }
  if (algo == ALGO_EMISSIONS) {
    if (d->emission_id == CDK_EMISSION_USER)
      return fail(CDK_E_UNSUPPORTED, "cdk_emission_moments: the emission moments of a user-defined emission are not implemented");
    if (d->N > 0 && (!in[CDK_IN_FM] || !in[CDK_IN_H] || !in[CDK_IN_D] || !in[CDK_IN_R]))
      return fail(CDK_E_NULL, "emission moments need the state means, H, d and R");
    return CDK_OK;
  }
  if (algo == ALGO_SAMPLE) {
    if (d->solver != CDK_EULER && d->solver != CDK_HEUN) return fail(CDK_E_UNSUPPORTED, "the sampler supports solver euler (Euler-Maruyama) or heun");
    static const int req_s[] = {CDK_IN_T, CDK_IN_M0, CDK_IN_F, CDK_IN_L, CDK_IN_QC, CDK_IN_H, CDK_IN_D, CDK_IN_R};
    if (d->N > 0) {
      for (int s : req_s)
        if (!in[s] && !optional_input(s)) return fail(CDK_E_NULL, "a required input of the sampler is NULL");
      if (!(d->reserved[2] & CDK_FLAG_FIXED_INIT) && !in[CDK_IN_P0]) return fail(CDK_E_NULL, "sampling x_0 needs P0");
    }
    return CDK_OK;
  }
  const bool ponly = (d->reserved[2] & CDK_FLAG_PREDICT_ONLY) != 0;
  if (ponly && smooth) return fail(CDK_E_UNSUPPORTED, "CDK_FLAG_PREDICT_ONLY applies to the filter entry points");
  if (ponly && d->N > 0 && (out[CDK_OUT_FM] || out[CDK_OUT_FP] || out[CDK_OUT_LLCUM]))
    return fail(CDK_E_UNSUPPORTED, "a forecast produces predicted moments only (PM / PP)");
  static const int req_lin[] = {CDK_IN_Y, CDK_IN_T, CDK_IN_M0, CDK_IN_P0, CDK_IN_F, CDK_IN_B, CDK_IN_L, CDK_IN_QC, CDK_IN_H, CDK_IN_D, CDK_IN_R};
  static const int req_nl[] = {CDK_IN_Y, CDK_IN_T, CDK_IN_M0, CDK_IN_P0, CDK_IN_F, CDK_IN_L, CDK_IN_QC, CDK_IN_H, CDK_IN_D, CDK_IN_R};
  if (d->N > 0) {
    if (linear) {
      for (int s : req_lin)
        if (!in[s] && !(ponly && s == CDK_IN_Y)) return fail(CDK_E_NULL, "a required input of the linear model is NULL");
      if (d->d_u > 0 && (!in[CDK_IN_U] || !in[CDK_IN_BU] || !in[CDK_IN_DU])) return fail(CDK_E_NULL, "d_u > 0 needs U, BU and DU");
    } else {
      for (int s : req_nl)
        if (!in[s] && !(ponly && s == CDK_IN_Y) && !optional_input(s))
          return fail(CDK_E_NULL, "a required input of the nonlinear model is NULL");
    }
    if (smooth && (!in[CDK_IN_FM] || !in[CDK_IN_FP])) return fail(CDK_E_NULL, "smoothing needs the filtered moments");
    if (smooth && (!out[CDK_OUT_SM] || !out[CDK_OUT_SP])) return fail(CDK_E_NULL, "smoothing needs SM and SP outputs");
  }
  return CDK_OK;
}

template <typename T>
static KArgs<T> make_args(const cdk_desc* d, const void* const* in, void* const* out, int algo) {
  KArgs<T> a;
  a.d = *d;
  for (int i = 0; i < CDK_NUM_IN; ++i) {
    a.in[i] = static_cast<const T*>(in[i]);
    a.in_stride[i] = (d->batched_mask >> i) & 1u ? slot_elems(*d, i, algo) : 0;
  }
  for (int i = 0; i < CDK_NUM_OUT; ++i) a.out[i] = out[i];
  return a;
}

template <typename T>
static int run(int algo, const cdk_desc* d, const void* const* in, void* const* out, cdk_stream_t stream) {
  int rc = validate(d, in, out, algo);
  if (rc != CDK_OK) return rc;
  if (d->N == 0) return CDK_OK;
  KArgs<T> a = make_args<T>(d, in, out, algo);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (algo == ALGO_EKF_FILTER) {
    rc = launch_ekf_small<T>(a, s);
    if (rc != CDK_E_UNSUPPORTED) return rc;
  }
  if (algo == ALGO_EKF_SMOOTH) {
    rc = launch_eks_small<T>(a, s);
    if (rc != CDK_E_UNSUPPORTED) return rc;
  }
  if (algo == ALGO_KF_FILTER || algo == ALGO_KF_SMOOTH) {
    rc = launch_kf_warp<T>(algo, a, s);
    if (rc != CDK_E_UNSUPPORTED) return rc;
  }
  if (algo == ALGO_ENKF_FILTER) {
    rc = launch_enkf<T>(a, s);
    if (rc == CDK_E_SIZE && d->emission_id == CDK_EMISSION_USER)
      return fail(rc, "enkf: the ensemble, the members' user-emission outputs and the model do not fit the shared memory of "
                      "an 8-CTA cluster (8 x 227 KB; roughly (n + m) * E * sizeof(T) / 8 + 12 n^2 sizeof(T) per CTA)");
    return rc == CDK_E_SIZE ? fail(rc, "enkf: the ensemble and its model do not fit the shared memory of an 8-CTA cluster "
                                       "(8 x 227 KB; roughly n * E * sizeof(T) / 8 + 12 n^2 sizeof(T) per CTA)")
                            : rc;
  }
  if (algo == ALGO_SAMPLE) {
    rc = launch_sample_path<T>(a, s);
    return rc == CDK_E_UNSUPPORTED ? fail(rc, "cdk_sample_path: model parameters must not be batched; solver euler or heun") : rc;
  }
  if (algo == ALGO_EMISSIONS) {
    rc = launch_emission_moments<T>(a, s);
    return rc == CDK_E_UNSUPPORTED ? fail(rc, "cdk_emission_moments: H, d, R must not be batched") : rc;
  }
  rc = launch_generic<T>(algo, a, s);
  if (rc == CDK_E_SIZE) {
    static thread_local char msg[256];
    snprintf(msg, sizeof(msg),
             "n = %d, m = %d: the per-trajectory working set of the shared-memory kernels exceeds the 227 KB of one CTA "
             "(fp64, m = n: KF n <= 38 / 30, EKF 45 / 37, UKF 50-55 with a chain tableau (euler, heun, rk4) / dopri5; see cdk.h)",
             d->n, d->m);
    return fail(rc, msg);
  }
  return rc;
}

// ---- deterministic ll reduction ------------------------------------------------------------------------------------
template <typename T>
__global__ void ll_sum_kernel(const T* __restrict__ ll, long long N, double* __restrict__ out) {
  // single CTA, fixed traversal order => bit-reproducible for a given N
  __shared__ double part[1024];
  double acc = 0.0;
  for (long long i = threadIdx.x; i < N; i += blockDim.x) acc += (double)ll[i];
  part[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) part[threadIdx.x] += part[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = part[0];
}

template <typename T>
static int ll_sum(const T* ll, int64_t N, double* out, cdk_stream_t stream) {
  if (!out || (N > 0 && !ll)) return fail(CDK_E_NULL, "ll_sum: NULL pointer");
  ll_sum_kernel<T><<<1, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(ll, N, out);
  note_launch();
  return check_launch("ll_sum_kernel");
}

// ---- FMA pipe probe ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) fma_probe_kernel(int iters, T* sink) {
  T x[16];
  const T a = T(1.0000001), b = T(1e-9) * T(threadIdx.x + 1);
#pragma unroll
  for (int i = 0; i < 16; ++i) x[i] = T(i) + T(blockIdx.x) * T(1e-3);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = fma(x[i], a, b);
  }
  T s = T(0);
#pragma unroll
  for (int i = 0; i < 16; ++i) s += x[i];
  sink[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// Same probe with THREE DISTINCT vector-register operands per FMA (what a filter's arithmetic looks like: state times
// state plus state).  On B200 such a DFMA issues every 3 cycles per sub-partition instead of 2 (register-file read
// bandwidth), so the attainable FP64 rate of register-operand code is 2/3 of the nominal peak.
__global__ void __launch_bounds__(256) fma3_probe_kernel(int iters, double* sink, const double* __restrict__ seed) {
  double x[8], y[8], z[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    x[i] = seed[(threadIdx.x + i) & 255];
    y[i] = 1.0 + 1e-9 * seed[(threadIdx.x + 8 + i) & 255];
    z[i] = 1e-9 * seed[(threadIdx.x + 16 + i) & 255];
  }
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = fma(y[(i + u) & 7], z[(i + 3 + u) & 7], x[i]);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += x[i] + y[i] + z[i];
  sink[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <typename T>
static int fma_probe(int blocks, int iters, T* sink, cdk_stream_t stream) {
  if (!sink || blocks < 1 || iters < 1) return fail(CDK_E_NULL, "fma_probe: bad arguments");
  fma_probe_kernel<T><<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(iters, sink);
  note_launch();
  return check_launch("fma_probe_kernel");
}

// ---- normal-deviate probe (tests: bit equality with the oracle's stream) ------------------------------------------
__global__ void __launch_bounds__(256) rng_probe_kernel(long long count, uint32_t traj, uint32_t step, uint32_t c3_base,
                                                        uint64_t seed, double* out) {
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= count) return;
  double z[4];
  normal_quad((uint32_t)i, traj, step, c3_base + ((uint32_t)i & 0xffu), seed, z);
#pragma unroll
  for (int u = 0; u < 4; ++u) out[4 * i + u] = z[u];
}

// ---- FP64 tensor-core (DMMA m8n8k4) probe -------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dmma_probe_kernel(int iters, double* sink) {
  double c[8][2];
  const double a = 1.0 + 1e-9 * threadIdx.x, b = 1.0 - 1e-9 * threadIdx.x;
#pragma unroll
  for (int i = 0; i < 8; ++i) c[i][0] = c[i][1] = 1e-3 * i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c[i][0]), "+d"(c[i][1])
                   : "d"(a), "d"(b));
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
  sink[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace cdk

using namespace cdk;

extern "C" {

void cdk_desc_init(cdk_desc* d) {
  if (!d) return;
  memset(d, 0, sizeof(*d));
  d->struct_size = (int32_t)sizeof(cdk_desc);
  d->K = 1;
  d->n = 1;
  d->m = 1;
  d->E = 2000;              // EnKFHyperParams.N_particles (inference_enkf.py:34)
  d->solver = CDK_DOPRI5;   // diffrax_utils.py:121-124
  d->max_steps = 100000;    // diffrax_utils.py:52
  d->dt0 = 0.01;            // diffrax_utils.py:50
  d->dt_final = 1e-10;      // KFHyperParams / EKFHyperParams / UKFHyperParams / EnKFHyperParams
  d->state_order = CDK_ORDER_SECOND;  // EKFHyperParams.state_order (inference_ekf.py:40)
  d->num_iter = 1;
  d->smoother_type = 1;
  d->batched_mask = (1u << CDK_IN_Y) | (1u << CDK_IN_T) | (1u << CDK_IN_U) | (1u << CDK_IN_FM) | (1u << CDK_IN_FP);
  d->perturb_measurements = 1;
  d->cov_rescaling = 1.0;
  d->alpha = 1.7320508075688772;  // sqrt(3), UKFHyperParams (inference_ukf.py:31-33)
  d->beta = 2.0;
  d->kappa = 1.0;
}

#define CDK_DEF(name, T, algo) \
  int name(const cdk_desc* d, const void* const* in, void* const* out, cdk_stream_t stream) { return run<T>(algo, d, in, out, stream); }

CDK_DEF(cdk_kf_filter_f64, double, ALGO_KF_FILTER)
CDK_DEF(cdk_kf_filter_f32, float, ALGO_KF_FILTER)
CDK_DEF(cdk_kf_smooth_f64, double, ALGO_KF_SMOOTH)
CDK_DEF(cdk_kf_smooth_f32, float, ALGO_KF_SMOOTH)
CDK_DEF(cdk_ekf_filter_f64, double, ALGO_EKF_FILTER)
CDK_DEF(cdk_ekf_filter_f32, float, ALGO_EKF_FILTER)
CDK_DEF(cdk_ekf_smooth_f64, double, ALGO_EKF_SMOOTH)
CDK_DEF(cdk_ekf_smooth_f32, float, ALGO_EKF_SMOOTH)
CDK_DEF(cdk_ukf_filter_f64, double, ALGO_UKF_FILTER)
CDK_DEF(cdk_ukf_filter_f32, float, ALGO_UKF_FILTER)
CDK_DEF(cdk_enkf_filter_f64, double, ALGO_ENKF_FILTER)
CDK_DEF(cdk_enkf_filter_f32, float, ALGO_ENKF_FILTER)
CDK_DEF(cdk_sample_path_f64, double, ALGO_SAMPLE)
CDK_DEF(cdk_sample_path_f32, float, ALGO_SAMPLE)
CDK_DEF(cdk_emission_moments_f64, double, ALGO_EMISSIONS)
CDK_DEF(cdk_emission_moments_f32, float, ALGO_EMISSIONS)

// Every gradient entry point reads in[CDK_IN_H] as the m x n matrix of a linear emission: a user emission is refused
// before any other check or launch.
static bool user_emission_grad(const cdk_desc* d) { return d && d->emission_id == CDK_EMISSION_USER; }
static const char* const kUserEmissionGrad = "a user-defined emission (CDK_EMISSION_USER) has no gradient";

int cdk_ekf_grad_f64(const cdk_desc* d, const void* const* in, void* const* out, cdk_stream_t stream) {
  if (user_emission_grad(d)) return fail(CDK_E_UNSUPPORTED, "cdk_ekf_grad_f64: a user-defined emission (CDK_EMISSION_USER) has no gradient");
  int rc = validate(d, in, out, ALGO_EKF_FILTER);
  if (rc != CDK_OK) return rc;
  if (d->N == 0) return CDK_OK;
  if (!out[CDK_OUT_GRAD]) return fail(CDK_E_NULL, "cdk_ekf_grad_f64 needs out[CDK_OUT_GRAD]");
  KArgs<double> a = make_args<double>(d, in, out, ALGO_EKF_FILTER);
  rc = launch_ekf_l63_grad(a, static_cast<double*>(out[CDK_OUT_GRAD]), reinterpret_cast<cudaStream_t>(stream));
  if (rc == CDK_E_UNSUPPORTED)
    return fail(rc, "cdk_ekf_grad_f64: only the Lorenz-63 drift with a scalar emission, num_iter = 1, order first/second");
  return rc;
}

int cdk_kf_grad_f64(const cdk_desc* d, const void* const* in, void* const* out, cdk_stream_t stream) {
  if (d && (d->reserved[2] & CDK_FLAG_PREDICT_ONLY))
    return fail(CDK_E_UNSUPPORTED, "cdk_kf_grad_f64: CDK_FLAG_PREDICT_ONLY has no log-likelihood to differentiate");
  int rc = validate(d, in, out, ALGO_KF_FILTER);
  if (rc != CDK_OK) return rc;
  if (d->d_u > 0) return fail(CDK_E_UNSUPPORTED, "cdk_kf_grad_f64: inputs (d_u > 0) are not supported");
  if (d->reserved[2] & CDK_FLAG_DIAG_R) return fail(CDK_E_UNSUPPORTED, "cdk_kf_grad_f64: CDK_FLAG_DIAG_R is not supported");
  if (d->n > 16 || d->m > 8) return fail(CDK_E_UNSUPPORTED, "cdk_kf_grad_f64: needs n <= 16 and m <= 8");
  if (d->reserved[3] != 0) return fail(CDK_E_UNSUPPORTED, "cdk_kf_grad_f64: desc.reserved[3] must be 0");
  if (d->N == 0) return CDK_OK;
  if (!out[CDK_OUT_GRAD]) return fail(CDK_E_NULL, "cdk_kf_grad_f64 needs out[CDK_OUT_GRAD]");
  if (!out[CDK_OUT_SCRATCH]) return fail(CDK_E_NULL, "cdk_kf_grad_f64 needs out[CDK_OUT_SCRATCH] (cdk_scratch_bytes)");
  KArgs<double> a = make_args<double>(d, in, out, ALGO_KF_FILTER);
  rc = launch_kf_grad(a, static_cast<double*>(out[CDK_OUT_GRAD]), reinterpret_cast<cudaStream_t>(stream));
  if (rc == CDK_E_UNSUPPORTED) return fail(rc, "cdk_kf_grad_f64: the forward pass needs the warp filter (CDK_KF_WARP=0 disables it)");
  return rc;
}

// The part of cdk_ekf_grad_dense_f64 / cdk_ukf_grad_dense_f64 / cdk_ukf_grad_sigma_f64 after their own checks: the
// shared-memory budget, the output buffers, then the forward filter launch of `algo` with its moments in the scratch and the
// dense backward launch (`sigma`: through the literal sigma-point predict; d has CDK_FLAG_UKF_SIGMA_POINTS set then).
static int dense_grad(int algo, const cdk_desc* d, const void* const* in, void* const* out, cdk_stream_t stream, const char* me,
                      bool sigma = false) {
  char msg[256];
  auto reject = [&](int code, const char* why) {
    snprintf(msg, sizeof(msg), "%s: %s", me, why);
    return fail(code, msg);
  };
  if (!cdk::ekf_grad_dense_fits(*d, sigma)) {
    if (d->drift_id == CDK_DRIFT_USER)
      snprintf(msg, sizeof(msg), "%s: n = %d, m = %d, n_theta = %d: the backward working set with the user drift's dual "
               "copy of [x | theta] exceeds the 227 KB of one CTA (see cdk.h)", me, d->n, d->m, d->n_theta);
    else
      snprintf(msg, sizeof(msg), "%s: n = %d, m = %d: the backward working set exceeds the 227 KB of one CTA (see cdk.h)", me,
               d->n, d->m);
    return fail(CDK_E_SIZE, msg);
  }
  if (d->N == 0) return CDK_OK;
  if (!out[CDK_OUT_GRAD]) return reject(CDK_E_NULL, "needs out[CDK_OUT_GRAD]");
  if (!out[CDK_OUT_SCRATCH]) return reject(CDK_E_NULL, "needs out[CDK_OUT_SCRATCH] (cdk_scratch_bytes)");
  KArgs<double> a = make_args<double>(d, in, out, algo);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  double* sc = static_cast<double*>(out[CDK_OUT_SCRATCH]);
  const long long NK = d->N * (long long)d->K;
  const int n = d->n;
  int* status = out[CDK_OUT_STATUS] ? static_cast<int*>(out[CDK_OUT_STATUS])
                                    : reinterpret_cast<int*>(sc + cdk::ekf_grad_dense_scratch_doubles(*d) - d->N);
  // the forward pass: the launch cdk_ekf_filter_f64 / cdk_ukf_filter_f64 makes (run()), its moments into the scratch
  KArgs<double> f = a;
  f.out[CDK_OUT_FM] = sc;
  f.out[CDK_OUT_FP] = sc + NK * n;
  f.out[CDK_OUT_PM] = sc + NK * (n + n * n);
  f.out[CDK_OUT_PP] = sc + NK * (2 * n + n * n);
  f.out[CDK_OUT_LLCUM] = nullptr;
  f.out[CDK_OUT_STATUS] = status;
  f.out[CDK_OUT_SCRATCH] = nullptr;
  f.out[CDK_OUT_GRAD] = nullptr;
  int rc = algo == ALGO_EKF_FILTER ? launch_ekf_small<double>(f, s) : CDK_E_UNSUPPORTED;
  if (rc == CDK_E_UNSUPPORTED) rc = launch_generic<double>(algo, f, s);
  if (rc == CDK_E_SIZE) return reject(rc, "the forward filter's working set exceeds the 227 KB of one CTA");
  if (rc != CDK_OK) return rc;
  return launch_ekf_grad_dense(a, status, static_cast<double*>(out[CDK_OUT_GRAD]), algo == ALGO_UKF_FILTER && !sigma, sigma, s);
}

int cdk_ekf_grad_dense_f64(const cdk_desc* d, const void* const* in, void* const* out, cdk_stream_t stream) {
  static const char* me = "cdk_ekf_grad_dense_f64";
  char msg[256];
  auto reject = [&](int code, const char* why) {
    snprintf(msg, sizeof(msg), "%s: %s", me, why);
    return fail(code, msg);
  };
  if (user_emission_grad(d)) return reject(CDK_E_UNSUPPORTED, kUserEmissionGrad);
  if (d && (d->reserved[2] & CDK_FLAG_PREDICT_ONLY)) return reject(CDK_E_UNSUPPORTED, "CDK_FLAG_PREDICT_ONLY has no log-likelihood to differentiate");
  if (d && (d->reserved[2] & CDK_FLAG_DIAG_R)) return reject(CDK_E_UNSUPPORTED, "CDK_FLAG_DIAG_R is not supported");
  if (d && d->drift_id == CDK_DRIFT_USER && !cdk::ekf_grad_has_user_drift())
    return reject(CDK_E_UNSUPPORTED, "a user-defined drift is differentiated only by a variant library built with its "
                                     "gradient unit: build_user_drift(code, grad=True), i.e. LearnableUserDrift(..., "
                                     "differentiable=True)");
  int rc = validate(d, in, out, ALGO_EKF_FILTER);
  if (rc != CDK_OK) return rc;
  if (d->state_order == CDK_ORDER_ZEROTH) return reject(CDK_E_UNSUPPORTED, "state_order zeroth is not supported");
  if (d->num_iter != 1) return reject(CDK_E_UNSUPPORTED, "num_iter must be 1 (the iterated EKF is not supported)");
  if (d->d_u > 0) return reject(CDK_E_UNSUPPORTED, "inputs (d_u > 0) are not supported");
  if (d->reserved[3] != 0) return reject(CDK_E_UNSUPPORTED, "desc.reserved[3] must be 0");
  return dense_grad(ALGO_EKF_FILTER, d, in, out, stream, me);
}

int cdk_ukf_grad_dense_f64(const cdk_desc* d, const void* const* in, void* const* out, cdk_stream_t stream) {
  static const char* me = "cdk_ukf_grad_dense_f64";
  char msg[192];
  auto reject = [&](int code, const char* why) {
    snprintf(msg, sizeof(msg), "%s: %s", me, why);
    return fail(code, msg);
  };
  if (user_emission_grad(d)) return reject(CDK_E_UNSUPPORTED, kUserEmissionGrad);
  if (d && (d->reserved[2] & CDK_FLAG_PREDICT_ONLY)) return reject(CDK_E_UNSUPPORTED, "CDK_FLAG_PREDICT_ONLY has no log-likelihood to differentiate");
  if (d && (d->reserved[2] & CDK_FLAG_DIAG_R)) return reject(CDK_E_UNSUPPORTED, "CDK_FLAG_DIAG_R is not supported");
  if (d && (d->reserved[2] & CDK_FLAG_UKF_SIGMA_POINTS))
    return reject(CDK_E_UNSUPPORTED, "CDK_FLAG_UKF_SIGMA_POINTS: differentiated by cdk_ukf_grad_sigma_f64");
  if (d && d->drift_id == CDK_DRIFT_USER)
    return reject(CDK_E_UNSUPPORTED, "a user-defined drift runs literal sigma points: differentiated by cdk_ukf_grad_sigma_f64");
  int rc = validate(d, in, out, ALGO_UKF_FILTER);
  if (rc != CDK_OK) return rc;
  if (d->d_u > 0) return reject(CDK_E_UNSUPPORTED, "inputs (d_u > 0) are not supported");
  if (d->reserved[3] != 0) return reject(CDK_E_UNSUPPORTED, "desc.reserved[3] must be 0");
  return dense_grad(ALGO_UKF_FILTER, d, in, out, stream, me);
}

int cdk_ukf_grad_sigma_f64(const cdk_desc* d, const void* const* in, void* const* out, cdk_stream_t stream) {
  static const char* me = "cdk_ukf_grad_sigma_f64";
  char msg[256];
  auto reject = [&](int code, const char* why) {
    snprintf(msg, sizeof(msg), "%s: %s", me, why);
    return fail(code, msg);
  };
  if (user_emission_grad(d)) return reject(CDK_E_UNSUPPORTED, kUserEmissionGrad);
  if (d && (d->reserved[2] & CDK_FLAG_PREDICT_ONLY)) return reject(CDK_E_UNSUPPORTED, "CDK_FLAG_PREDICT_ONLY has no log-likelihood to differentiate");
  if (d && (d->reserved[2] & CDK_FLAG_DIAG_R)) return reject(CDK_E_UNSUPPORTED, "CDK_FLAG_DIAG_R is not supported");
  if (d && d->drift_id == CDK_DRIFT_USER && !cdk::ekf_grad_has_user_drift())
    return reject(CDK_E_UNSUPPORTED, "a user-defined drift is differentiated only by a variant library built with its "
                                     "gradient unit: build_user_drift(code, grad=True), i.e. LearnableUserDrift(..., "
                                     "differentiable=True)");
  if (!d) return validate(d, in, out, ALGO_UKF_FILTER);
  cdk_desc sd = *d;  // the forward pass is the sigma-point filter whatever the caller's flags say
  sd.reserved[2] |= CDK_FLAG_UKF_SIGMA_POINTS;
  int rc = validate(&sd, in, out, ALGO_UKF_FILTER);
  if (rc != CDK_OK) return rc;
  if (sd.d_u > 0) return reject(CDK_E_UNSUPPORTED, "inputs (d_u > 0) are not supported");
  if (sd.reserved[3] != 0) return reject(CDK_E_UNSUPPORTED, "desc.reserved[3] must be 0");
  return dense_grad(ALGO_UKF_FILTER, &sd, in, out, stream, me, true);
}

size_t cdk_scratch_bytes(const cdk_desc* d, const char* entry_point) {
  if (!d || !entry_point) return 0;
  // the EnKF keeps its ensemble in (distributed) shared memory; the only device scratch is the optional pushforward
  // cache shared by the CD-KF filter and its type-1 smoother (CDK_FLAG_KEEP_PUSHFORWARD)
  const bool kf = strstr(entry_point, "kf_filter") != nullptr && strstr(entry_point, "ekf") == nullptr &&
                  strstr(entry_point, "ukf") == nullptr && strstr(entry_point, "enkf") == nullptr;
  const bool ks = strstr(entry_point, "kf_smooth") != nullptr && strstr(entry_point, "ekf") == nullptr;
  // the dense gradients first: "cdk_ukf_grad_dense" and "cdk_ukf_grad_sigma" also contain "kf_grad" and not "ekf_grad"
  if (strstr(entry_point, "ekf_grad_dense") != nullptr || strstr(entry_point, "ukf_grad_dense") != nullptr ||
      strstr(entry_point, "ukf_grad_sigma") != nullptr)
    return (size_t)cdk::ekf_grad_dense_scratch_doubles(*d) * sizeof(double);
  if (strstr(entry_point, "kf_grad") != nullptr && strstr(entry_point, "ekf_grad") == nullptr)
    return (size_t)cdk::kf_grad_scratch_doubles(*d) * sizeof(double);
  if (strstr(entry_point, "ekf_grad") != nullptr)
    return (d->reserved[3] & CDK_GRAD_REVERSE) ? (size_t)d->N * (size_t)d->K * 24u * sizeof(double) : 0;
  if ((kf || ks) && (d->reserved[2] & CDK_FLAG_KEEP_PUSHFORWARD) && cdk::kf_warp_eligible(*d, ks) && d->K > 1)
    return (size_t)d->N * (size_t)(d->K - 1) * 2u * (size_t)d->n * (size_t)d->n * sizeof(double);
  return 0;
}

int cdk_ll_sum_f64(const double* ll, int64_t N, double* ll_sum_out, cdk_stream_t stream) { return ll_sum<double>(ll, N, ll_sum_out, stream); }
int cdk_ll_sum_f32(const float* ll, int64_t N, double* ll_sum_out, cdk_stream_t stream) { return ll_sum<float>(ll, N, ll_sum_out, stream); }

int cdk_ll_allreduce(void* nccl_comm, double* ll_sum, cdk_stream_t stream) {
  // ncclAllReduce(sendbuff, recvbuff, count, ncclFloat64 = 8, ncclSum = 0, comm, stream); resolved lazily so that the
  // library has no link-time NCCL dependency (torch bundles libnccl.so.2).
  typedef int (*allreduce_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
  static allreduce_fn fn = nullptr;
  if (!nccl_comm || !ll_sum) return fail(CDK_E_NULL, "ll_allreduce: NULL pointer");
  if (!fn) {
    void* sym = dlsym(RTLD_DEFAULT, "ncclAllReduce");
    if (!sym) {
      void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
      if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
      if (h) sym = dlsym(h, "ncclAllReduce");
    }
    if (!sym) return fail(CDK_E_NCCL, "ncclAllReduce not found (libnccl not loaded)");
    fn = reinterpret_cast<allreduce_fn>(sym);
  }
  int rc = fn(ll_sum, ll_sum, 1, /*ncclFloat64*/ 8, /*ncclSum*/ 0, nccl_comm, reinterpret_cast<cudaStream_t>(stream));
  if (rc != 0) return fail(CDK_E_NCCL, "ncclAllReduce failed");
  return CDK_OK;
}

// Shared body of the two XLA adaptors: unpack the opaque blob, rebuild the in[] / out[] slot arrays, dispatch by name.
static int xla_dispatch(cdk_stream_t stream, void** buffers, const char* opaque, size_t opaque_len) {
  if (!buffers || !opaque || opaque_len < sizeof(cdk_xla_opaque)) return fail(CDK_E_SIZE, "xla custom call: bad opaque");
  cdk_xla_opaque op;
  memcpy(&op, opaque, sizeof(op));
  op.entry_point[sizeof(op.entry_point) - 1] = 0;
  const void* in[CDK_NUM_IN];
  void* out[CDK_NUM_OUT];
  const uint32_t absent_in = (uint32_t)op.desc.reserved[0], absent_out = (uint32_t)op.desc.reserved[1];
  for (int i = 0; i < CDK_NUM_IN; ++i) in[i] = (absent_in >> i) & 1u ? nullptr : buffers[i];
  for (int i = 0; i < CDK_NUM_OUT; ++i) out[i] = (absent_out >> i) & 1u ? nullptr : buffers[CDK_NUM_IN + i];
  struct { const char* name; int (*fn)(const cdk_desc*, const void* const*, void* const*, cdk_stream_t); } table[] = {
      {"cdk_kf_filter_f64", cdk_kf_filter_f64},   {"cdk_kf_filter_f32", cdk_kf_filter_f32},
      {"cdk_kf_smooth_f64", cdk_kf_smooth_f64},   {"cdk_kf_smooth_f32", cdk_kf_smooth_f32},
      {"cdk_ekf_filter_f64", cdk_ekf_filter_f64}, {"cdk_ekf_filter_f32", cdk_ekf_filter_f32},
      {"cdk_ekf_smooth_f64", cdk_ekf_smooth_f64}, {"cdk_ekf_smooth_f32", cdk_ekf_smooth_f32},
      {"cdk_ukf_filter_f64", cdk_ukf_filter_f64}, {"cdk_ukf_filter_f32", cdk_ukf_filter_f32},
      {"cdk_enkf_filter_f64", cdk_enkf_filter_f64}, {"cdk_enkf_filter_f32", cdk_enkf_filter_f32},
      {"cdk_ekf_grad_f64", cdk_ekf_grad_f64},     {"cdk_kf_grad_f64", cdk_kf_grad_f64},
      {"cdk_ekf_grad_dense_f64", cdk_ekf_grad_dense_f64}, {"cdk_ukf_grad_dense_f64", cdk_ukf_grad_dense_f64},
      {"cdk_ukf_grad_sigma_f64", cdk_ukf_grad_sigma_f64},
      {"cdk_sample_path_f64", cdk_sample_path_f64}, {"cdk_sample_path_f32", cdk_sample_path_f32},
      {"cdk_emission_moments_f64", cdk_emission_moments_f64}, {"cdk_emission_moments_f32", cdk_emission_moments_f32}};
  for (auto& e : table)
    if (strcmp(e.name, op.entry_point) == 0) return e.fn(&op.desc, in, out, stream);
  return fail(CDK_E_ENUM, "xla custom call: unknown entry point");
}

static thread_local int g_xla_rc = 0;

void cdk_xla_custom_call(cdk_stream_t stream, void** buffers, const char* opaque, size_t opaque_len) {
  g_xla_rc = xla_dispatch(stream, buffers, opaque, opaque_len);
}

void cdk_xla_custom_call_status(cdk_stream_t stream, void** buffers, const char* opaque, size_t opaque_len, void* status) {
  g_xla_rc = xla_dispatch(stream, buffers, opaque, opaque_len);
  if (g_xla_rc == CDK_OK || !status) return;
  // XlaCustomCallStatusSetFailure(XlaCustomCallStatus*, const char* message, size_t message_len) lives in the XLA
  // runtime (jaxlib) that called us; resolved at run time so libcdk.so has no link-time dependency on it.
  typedef void (*set_failure_fn)(void*, const char*, size_t);
  static set_failure_fn set_failure = reinterpret_cast<set_failure_fn>(dlsym(RTLD_DEFAULT, "XlaCustomCallStatusSetFailure"));
  if (!set_failure) set_failure = reinterpret_cast<set_failure_fn>(dlsym(RTLD_DEFAULT, "XlaCustomCallStatusSetFailure"));
  if (set_failure) {
    char msg[320];
    const int len = snprintf(msg, sizeof(msg), "cdk (%d): %s", g_xla_rc, g_err);
    set_failure(status, msg, (size_t)(len < (int)sizeof(msg) ? len : (int)sizeof(msg) - 1));
  }
}

int cdk_xla_last_rc(void) { return g_xla_rc; }

int cdk_fma_probe_f64(int blocks, int iters, double* sink, cdk_stream_t stream) { return fma_probe<double>(blocks, iters, sink, stream); }
int cdk_fma_probe_f32(int blocks, int iters, float* sink, cdk_stream_t stream) { return fma_probe<float>(blocks, iters, sink, stream); }
int cdk_fma3_probe_f64(int blocks, int iters, double* sink, const double* seed, cdk_stream_t stream) {
  if (!sink || !seed || blocks < 1 || iters < 1) return fail(CDK_E_NULL, "fma3_probe: bad arguments");
  fma3_probe_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(iters, sink, seed);
  note_launch();
  return check_launch("fma3_probe_kernel");
}

int cdk_rng_probe_f64(int64_t count, uint32_t traj, uint32_t step, uint32_t c3_base, uint64_t seed, double* out,
                      cdk_stream_t stream) {
  if (!out || count < 1) return fail(CDK_E_NULL, "rng_probe: bad arguments");
  rng_probe_kernel<<<(unsigned)((count + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(count, traj, step, c3_base,
                                                                                                   seed, out);
  note_launch();
  return check_launch("rng_probe_kernel");
}

int cdk_dmma_probe_f64(int blocks, int iters, double* sink, cdk_stream_t stream) {
  if (!sink || blocks < 1 || iters < 1) return fail(CDK_E_NULL, "dmma_probe: bad arguments");
  dmma_probe_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(iters, sink);
  note_launch();
  return check_launch("dmma_probe_kernel");
}

int cdk_debug_set_trace(void* devbuf) { return cdk::set_lw_trace(devbuf); }
int64_t cdk_launch_count(void) { return (int64_t)g_launches.load(); }
int cdk_has_user_drift(void) { return cdk::has_user_drift() ? 1 : 0; }
int cdk_has_user_emission(void) { return cdk::has_user_emission() ? 1 : 0; }
int cdk_user_emission_params(int n, int m) { return cdk::user_emission_params(n, m); }
int cdk_version(void) { return CDK_VERSION; }
const char* cdk_last_error(void) { return g_err; }

}  // extern "C"
