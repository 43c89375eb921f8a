// cdk_aux.cu -- the callers either side of the filters (SURVEY section 8f ranks 2 and 3):
//
//  * sample_path_kernel     cdnlgssm_path_sample         src/continuous_discrete_nonlinear_gaussian_ssm/models.py:525-656
//                           (what SSM.sample_batch(..., transition_type="path") vmaps, src/ssm_temissions.py:187-225) and the
//                           point-estimate branch of cdnlgssm_forecast (models.py:840-936): x_0 ~ N(m0, P0) (or a given
//                           state), x_k = SDE solve of dx = f(x) dt + L chol(Qc) dW over [t_{k-1}, t_k] with the diffrax
//                           stepping rule (Heun by default, Euler-Maruyama on request), y_k ~ N(H x_k + d, R).
//  * emission_moments_kernel  emissions_extended_kalman_filter (inference_ekf.py:762-855) and its unscented twin for the
//                           linear emission: E[y] = H m + d, cov[y] = H P H^T + R for every (trajectory, step).
//
// Randomness: the reference draws from jax.random and a diffrax VirtualBrownianTree, not reproducible outside JAX; the
// sampler uses the Philox4x32-10 + Box-Muller stream of cdk_rng.cuh (shared bit-for-bit with oracle/cd_oracle.py), so it is
// checked against the oracle to rounding and against the model in distribution.
//
// Mapping: ONE THREAD PER TRAJECTORY (a path is a serial chain; N is the parallel axis), the state in registers for the
// compile-time drifts (Lorenz-63: n = 3) and in thread-private arrays otherwise; the model constants (drift parameters,
// G = L chol(Qc), chol(R), chol(P0), H, d) are prepared once per CTA in shared memory.
#include "cdk_dense.cuh"
#include "cdk_rng.cuh"

namespace cdk {
namespace {

constexpr int SP_TPB = 128;

struct SLay {
  int n, m, ldn, ldm;
  size_t TH, G, CR, CP, H, DV, W1, W2, total;  // element offsets
  // nphi >= 0: a user emission (cdk.h CDK_EMISSION_USER) whose phi [nphi] takes the place of H (and d is not read)
  __host__ __device__ SLay(int n_, int m_, int nth, int nphi = -1) {
    n = n_; m = m_; ldn = ldp(n); ldm = ldp(m);
    size_t o = 0;
    auto take = [&](size_t c) { size_t r = o; o += (c + 1) & ~size_t(1); return r; };
    TH = take(nth > 0 ? nth : 1); G = take((size_t)n * ldn); CR = take((size_t)m * ldm); CP = take((size_t)n * ldn);
    H = take(nphi >= 0 ? (size_t)(nphi > 0 ? nphi : 1) : (size_t)m * ldn); DV = take(m); W1 = take((size_t)(n > m ? n : m) * ldp(n > m ? n : m));
    W2 = take((size_t)(n > m ? n : m) * ldp(n > m ? n : m));
    total = o;
  }
};

template <typename T, int NX>
__device__ __forceinline__ T path_f(int drift_id, const T* th, int n, int i, const T* x) {
  if (NX == 3) {
    if (i == 0) return th[0] * (x[1] - x[0]);
    if (i == 1) return x[0] * (th[1] - x[2]) - x[1];
    return x[0] * x[1] - th[2] * x[2];
  }
  return drift_f<T>(drift_id, th, n, i, [&](int j) { return x[j]; });
}

// in[CDK_IN_T]: [N, K] time stamps, or -- CDK_FLAG_FIXED_INIT -- [N, K + 1]: t_init followed by the K output times.
// out[CDK_OUT_FM]: states [N, K, n]; out[CDK_OUT_PM]: emissions [N, K, m] (either may be NULL).
template <typename T, int NX>
__global__ void __launch_bounds__(SP_TPB) sample_path_kernel(const KArgs<T> a) {
  constexpr int NXA = NX > 0 ? NX : CDK_MAX_N;
  extern __shared__ __align__(16) unsigned char sp_raw[];
  T* sh = reinterpret_cast<T*>(sp_raw);
  const cdk_desc& d = a.d;
  const int n = NX > 0 ? NX : d.n, m = d.m, K = d.K;
  const bool ue = user_emission(d);
  const SLay L(n, m, d.n_theta, ue ? emission_params(d) : -1);
  const int ldn = L.ldn, ldm = L.ldm;
  T* th = sh + L.TH;
  T* G = sh + L.G;
  T* chR = sh + L.CR;
  T* chP = sh + L.CP;
  T* H = sh + L.H;
  T* dv = sh + L.DV;
  const bool fixed = (d.reserved[2] & CDK_FLAG_FIXED_INIT) != 0;
  // ---- model constants (shared by the CTA; the launcher refuses per-trajectory model parameters) ----
  FOR_T(i, d.n_theta) th[i] = a.in[CDK_IN_F][i];
  {
    T* Lm = sh + L.W1;
    T* Qc = sh + L.W2;
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      Lm[i * ldn + j] = a.in[CDK_IN_L][e];
      Qc[i * ldn + j] = a.in[CDK_IN_QC][e];
    }
    if (ue) {
      FOR_T(i, emission_params(d)) H[i] = a.in[CDK_IN_H][i];  // phi
    } else {
      FOR_T(e, m * n) H[(e / n) * ldn + (e % n)] = a.in[CDK_IN_H][e];
      FOR_T(i, m) dv[i] = a.in[CDK_IN_D][i];
    }
    __syncthreads();
    chol<T>(Qc, chP, n, ldn, T(0));  // chol(Qc), parked in CP
    FOR_T(e, n * n) {                // G = L chol(Qc)  (models.py:583-588)
      const int i = e / n, j = e - i * n;
      T s = T(0);
      for (int q = j; q < n; ++q) s += Lm[i * ldn + q] * chP[q * ldn + j];
      G[i * ldn + j] = s;
    }
    __syncthreads();
    T* Rm = sh + L.W1;
    FOR_T(e, m * m) Rm[(e / m) * ldm + (e % m)] = a.in[CDK_IN_R][e];
    __syncthreads();
    chol<T>(Rm, chR, m, ldm, T(0));
    if (!fixed) {
      T* P0 = sh + L.W2;
      FOR_T(e, n * n) P0[(e / n) * ldn + (e % n)] = a.in[CDK_IN_P0][e];  // P0 shared; m0 may be per trajectory
      __syncthreads();
      chol<T>(P0, chP, n, ldn, T(0));
    }
    __syncthreads();
  }
  int offd = 0;
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    if (i != j && G[i * ldn + j] != T(0)) offd = 1;
  }
  const bool diagG = __syncthreads_or(offd) == 0;

  const long long traj = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (traj >= d.N) return;
  const uint32_t ctr = (uint32_t)(((unsigned long long)traj + d.rng_offset) & 0xffffffffull);
  const uint64_t seed = d.rng_seed;
  const T* Tm = a.in[CDK_IN_T] + traj * a.in_stride[CDK_IN_T];
  const T* m0 = a.in[CDK_IN_M0] + traj * a.in_stride[CDK_IN_M0];
  T* XS = static_cast<T*>(a.out[CDK_OUT_FM]);
  T* YS = static_cast<T*>(a.out[CDK_OUT_PM]);
  const T dt0 = T(d.dt0);
  T x[NXA], xe[NXA], z[NXA];
  int status = 0;

  auto normals = [&](int stream, int step, int substep, int dim, T* out) {
    for (int j = 0; j < dim; j += 4) {
      double z4[4];
      normal_quad(0u, ctr, (uint32_t)step, rng_c3(stream, substep, j >> 2), seed, z4);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (j + u < dim) out[j + u] = (T)z4[u];
    }
  };
  auto emit = [&](int row, int step) {  // y ~ N(h(x), R), h(x) = H x + d or the user's, and the state -> row `row`
    if (XS)
      for (int i = 0; i < n; ++i) XS[(traj * (long long)K + row) * n + i] = x[i];
    if (YS) {
      T r[CDK_MAX_M];
      normals(RNG_OBS, step, 0, m, r);
      for (int p = m - 1; p >= 0; --p) {  // r <- chol(R) z, in place from the bottom row up
        T s = T(0);
        for (int q = 0; q <= p; ++q) s += chR[p * ldm + q] * r[q];
        r[p] = s;
      }
      for (int p = 0; p < m; ++p) {
        T hx;
        if (ue) {
          hx = user_h<T>(H, n, m, p, [&](int j) { return x[j]; });
        } else {
          hx = dv[p];
#pragma unroll(NX > 0 ? NX : 1)
          for (int i = 0; i < NXA; ++i)
            if (i < n) hx += H[p * ldn + i] * x[i];
        }
        YS[(traj * (long long)K + row) * m + p] = hx + r[p];
      }
    }
  };

  // ---- initial state (models.py:545-571): x_0 = m0 + chol(P0) z, emission at t_0; or the given point (forecast) ----
  if (fixed) {
#pragma unroll(NX > 0 ? NX : 1)
    for (int i = 0; i < NXA; ++i)
      if (i < n) x[i] = m0[i];
  } else {
    normals(RNG_INIT, 0, 0, n, z);
#pragma unroll(NX > 0 ? NX : 1)
    for (int i = 0; i < NXA; ++i)
      if (i < n) {
        T s = T(0);
        for (int j = 0; j <= i; ++j) s += chP[i * ldn + j] * z[j];
        x[i] = m0[i] + s;
      }
    emit(0, 0);
  }
  const int first = fixed ? 0 : 1;  // first output row produced by a transition
  for (int k = first; k < K; ++k) {
    // transition over [t_{k-1}, t_k] (fixed: [T[k], T[k+1]])
    const T t0 = fixed ? Tm[k] : Tm[k - 1], t1 = fixed ? Tm[k + 1] : Tm[k];
    StepClock<T> clk(t0, t1, dt0);
    while (clk.running()) {
      if (clk.n >= d.max_steps) {
        status = 2;
        for (int i = 0; i < n; ++i) x[i] = T(NAN);
        break;
      }
      const T dt = clk.dt(), sqdt = sqrt(dt);
      normals(RNG_DYN, k, clk.n, n, z);
      if (diagG) {
#pragma unroll(NX > 0 ? NX : 1)
        for (int i = 0; i < NXA; ++i)
          if (i < n) xe[i] = G[i * ldn + i] * (sqdt * z[i]);
      } else {
#pragma unroll(NX > 0 ? NX : 1)
        for (int i = 0; i < NXA; ++i)
          if (i < n) {
            T s = T(0);
            for (int j = 0; j < n; ++j) s += G[i * ldn + j] * (sqdt * z[j]);
            xe[i] = s;
          }
      }
      T f0[NXA];
#pragma unroll(NX > 0 ? NX : 1)
      for (int i = 0; i < NXA; ++i)
        if (i < n) f0[i] = path_f<T, NX>(d.drift_id, th, n, i, x);
#pragma unroll(NX > 0 ? NX : 1)
      for (int i = 0; i < NXA; ++i)
        if (i < n) xe[i] = fma(dt, f0[i], x[i]) + xe[i];  // Euler-Maruyama state
      if (d.solver == CDK_HEUN) {
        // x + dt/2 (f(x) + f(xe)) + noise, written as xe + dt/2 (f(xe) - f(x)) (the form the EnKF kernel and the oracle use)
        const T hdt = T(0.5) * dt;
        T xn[NXA];
#pragma unroll(NX > 0 ? NX : 1)
        for (int i = 0; i < NXA; ++i)
          if (i < n) xn[i] = xe[i] + hdt * (path_f<T, NX>(d.drift_id, th, n, i, xe) - f0[i]);
#pragma unroll(NX > 0 ? NX : 1)
        for (int i = 0; i < NXA; ++i)
          if (i < n) x[i] = xn[i];
      } else {
#pragma unroll(NX > 0 ? NX : 1)
        for (int i = 0; i < NXA; ++i)
          if (i < n) x[i] = xe[i];
      }
      clk.advance();
    }
    emit(k, fixed ? k + 1 : k);
  }
  if (a.out[CDK_OUT_STATUS]) {
    bool bad = false;
    for (int i = 0; i < n; ++i) bad |= !isfinite(x[i]);
    static_cast<int*>(a.out[CDK_OUT_STATUS])[traj] = final_status(status, !bad);
  }
}

// in[CDK_IN_FM] / in[CDK_IN_FP]: state means [N, K, n] and covariances [N, K, n, n] (FP may be NULL: point estimates);
// out[CDK_OUT_PM]: emission means [N, K, m]; out[CDK_OUT_PP]: emission covariances [N, K, m, m] (H P H^T + R, or R alone).
template <typename T>
__global__ void __launch_bounds__(128) emission_moments_kernel(const KArgs<T> a) {
  extern __shared__ __align__(16) unsigned char em_raw[];
  T* sh = reinterpret_cast<T*>(em_raw);
  const cdk_desc& d = a.d;
  const int n = d.n, m = d.m;
  T* H = sh;                // [m][n]
  T* R = H + m * n;         // [m][m]
  T* dv = R + m * m;        // [m]
  T* W = dv + m;            // per warp: P [n][n] + HP [m][n]
  FOR_T(e, m * n) H[e] = a.in[CDK_IN_H][e];
  FOR_T(e, m * m) R[e] = a.in[CDK_IN_R][e];
  FOR_T(e, m) dv[e] = a.in[CDK_IN_D][e];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  T* P = W + (size_t)warp * (n * n + m * n + n);
  T* HP = P + n * n;
  T* mu = HP + m * n;
  const long long rows = d.N * (long long)d.K;
  T* EM = static_cast<T*>(a.out[CDK_OUT_PM]);
  T* EC = static_cast<T*>(a.out[CDK_OUT_PP]);
  for (long long row = (long long)blockIdx.x * nw + warp; row < rows; row += (long long)gridDim.x * nw) {
    const T* ms = a.in[CDK_IN_FM] + row * n;
    for (int i = lane; i < n; i += 32) mu[i] = ms[i];
    if (a.in[CDK_IN_FP])
      for (int e = lane; e < n * n; e += 32) P[e] = a.in[CDK_IN_FP][row * n * n + e];
    __syncwarp();
    if (EM)
      for (int p = lane; p < m; p += 32) {
        T s = dv[p];
        for (int q = 0; q < n; ++q) s += H[p * n + q] * mu[q];
        EM[row * m + p] = s;
      }
    if (EC) {
      if (a.in[CDK_IN_FP]) {
        for (int e = lane; e < m * n; e += 32) {
          const int p = e / n, j = e - p * n;
          T s = T(0);
          for (int q = 0; q < n; ++q) s += H[p * n + q] * P[q * n + j];
          HP[e] = s;
        }
        __syncwarp();
        for (int e = lane; e < m * m; e += 32) {
          const int p = e / m, q2 = e - p * m;
          T s = T(0);
          for (int q = 0; q < n; ++q) s += HP[p * n + q] * H[q2 * n + q];
          EC[row * m * m + e] = s + R[e];
        }
      } else {
        for (int e = lane; e < m * m; e += 32) EC[row * m * m + e] = R[e];
      }
    }
    __syncwarp();
  }
}

}  // namespace

template <typename T>
int launch_sample_path(const KArgs<T>& a, cudaStream_t s) {
  const cdk_desc& d = a.d;
  if (d.N == 0) return CDK_OK;
  if (d.solver != CDK_EULER && d.solver != CDK_HEUN) return CDK_E_UNSUPPORTED;
  const uint32_t model_mask = (1u << CDK_IN_F) | (1u << CDK_IN_L) | (1u << CDK_IN_QC) | (1u << CDK_IN_H) | (1u << CDK_IN_D) |
                              (1u << CDK_IN_R) | (1u << CDK_IN_P0);
  if (d.batched_mask & model_mask) return CDK_E_UNSUPPORTED;  // per-trajectory model parameters: not in the sampler
  const SLay L(d.n, d.m, d.n_theta, user_emission(d) ? emission_params(d) : -1);
  const size_t smem = L.total * sizeof(T);
  const long long blocks = (d.N + SP_TPB - 1) / SP_TPB;
  if (blocks > 2147483647LL) return CDK_E_SIZE;
  auto kern = (d.n == 3 && d.drift_id == CDK_DRIFT_LORENZ63) ? sample_path_kernel<T, 3> : sample_path_kernel<T, 0>;
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("cudaFuncSetAttribute(sample_path_kernel)");
  kern<<<(unsigned)blocks, SP_TPB, smem, s>>>(a);
  note_launch();
  return check_launch("sample_path_kernel");
}

template <typename T>
int launch_emission_moments(const KArgs<T>& a, cudaStream_t s) {
  const cdk_desc& d = a.d;
  const long long rows = d.N * (long long)d.K;
  if (rows == 0) return CDK_OK;
  const uint32_t model_mask = (1u << CDK_IN_H) | (1u << CDK_IN_D) | (1u << CDK_IN_R);
  if (d.batched_mask & model_mask) return CDK_E_UNSUPPORTED;
  const int nw = 4;
  const size_t smem = sizeof(T) * ((size_t)d.m * d.n + (size_t)d.m * d.m + d.m + (size_t)nw * (d.n * d.n + d.m * d.n + d.n));
  long long blocks = (rows + nw - 1) / nw;
  if (blocks > 148 * 16) blocks = 148 * 16;
  auto kern = emission_moments_kernel<T>;
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("cudaFuncSetAttribute(emission_moments_kernel)");
  kern<<<(unsigned)blocks, 32 * nw, smem, s>>>(a);
  note_launch();
  return check_launch("emission_moments_kernel");
}

template int launch_sample_path<double>(const KArgs<double>&, cudaStream_t);
template int launch_sample_path<float>(const KArgs<float>&, cudaStream_t);
template int launch_emission_moments<double>(const KArgs<double>&, cudaStream_t);
template int launch_emission_moments<float>(const KArgs<float>&, cudaStream_t);

}  // namespace cdk
