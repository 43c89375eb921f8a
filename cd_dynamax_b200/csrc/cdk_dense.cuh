// cdk_dense.cuh -- block-cooperative small dense helpers and the drift registry, shared by the shared-memory kernels.
#pragma once
#include "cdk_common.cuh"

namespace cdk {

#define FOR_T(i, cnt) for (int i = threadIdx.x; i < (cnt); i += blockDim.x)

__host__ __device__ inline int ldp(int c) { return c | 1; }


// ---- user-defined drift (CDK_DRIFT_USER): only in a variant library built with -DCDK_USER_DRIFT_HEADER="file" --------
// The header defines, in namespace cdk_user:
//   template <typename T, class XF> __device__ T f(const T* th, int n, int i, XF x);     // f_i; x(j) reads component j
//   template <typename T> __device__ T jac(const T* th, int n, int i, int j, const T* x); // d f_i / d x_j
//   template <typename T> __device__ T graddiv(const T* th, int n, int k, const T* x);    // sum_i d2 f_i / dx_i dx_k (or 0)
// A differentiable drift (build_user_drift(code, grad=True)) is also instantiated with T = cdk_dual::Dual<W>
// (cdk_dual.cuh) by the dense EKF gradient, so it must use only T arithmetic and the UNQUALIFIED functions sqrt exp log
// sin cos tan tanh sinh cosh atan fabs pow(T, double); ::sin, std::exp or __expf do not compile with the dual type.
#ifdef CDK_USER_DRIFT_HEADER
#include CDK_USER_DRIFT_HEADER
#define CDK_HAS_USER_DRIFT 1
#else
#define CDK_HAS_USER_DRIFT 0
#endif

// ---- user-defined emission (CDK_EMISSION_USER): only in a variant built with -DCDK_USER_EMISSION_HEADER="file" ----------
// The header defines, in namespace cdk_user_emission:
//   __host__ __device__ int num_params(int n, int m);                                       // length of phi
//   template <typename T, class XF> __device__ T h(const T* phi, int n, int m, int a, XF x);   // h_a(x; phi); x(j) = x_j
//   template <typename T> __device__ T jac(const T* phi, int n, int m, int a, int j, const T* x); // d h_a / d x_j
// for T = float and double.  Nothing differentiates it (the gradient entry points reject the id).
#ifdef CDK_USER_EMISSION_HEADER
#include CDK_USER_EMISSION_HEADER
#define CDK_HAS_USER_EMISSION 1
#else
#define CDK_HAS_USER_EMISSION 0
#endif

// True iff the request takes the user emission; a compile-time false in a library without one, so the callers' user-emission
// branches vanish from those objects.
__host__ __device__ static inline bool user_emission(const cdk_desc& d) {
  return CDK_HAS_USER_EMISSION && d.emission_id == CDK_EMISSION_USER;
}
// n_phi of the user emission (0 when the request does not take it)
__host__ __device__ static inline int emission_params(const cdk_desc& d) {
#if CDK_HAS_USER_EMISSION
  if (d.emission_id == CDK_EMISSION_USER) return cdk_user_emission::num_params(d.n, d.m);
#endif
  return 0;
}
template <typename T, class XF>
__device__ __forceinline__ T user_h(const T* phi, int n, int m, int a, XF x) {
#if CDK_HAS_USER_EMISSION
  return cdk_user_emission::h<T>(phi, n, m, a, x);
#else
  return T(0);
#endif
}
template <typename T>
__device__ __forceinline__ T user_h_jac(const T* phi, int n, int m, int a, int j, const T* x) {
#if CDK_HAS_USER_EMISSION
  return cdk_user_emission::jac<T>(phi, n, m, a, j, x);
#else
  return T(0);
#endif
}

// ---- drift registry, element-wise, on an arbitrary accessor x(j) ---------------------------------------------------
template <typename T, class XF>
__device__ __forceinline__ T drift_f(int id, const T* th, int n, int i, XF x) {
  switch (id) {
    case CDK_DRIFT_LINEAR: {
      T s = T(0);
      for (int k = 0; k < n; ++k) s += th[i * n + k] * x(k);
      return s + th[n * n + i];
    }
    case CDK_DRIFT_LORENZ63:
      if (i == 0) return th[0] * (x(1) - x(0));
      if (i == 1) return x(0) * (th[1] - x(2)) - x(1);
      return x(0) * x(1) - th[2] * x(2);
    case CDK_DRIFT_LORENZ96: {
      const int ip = i + 1 == n ? 0 : i + 1, im1 = i == 0 ? n - 1 : i - 1, im2 = im1 == 0 ? n - 1 : im1 - 1;
      return (x(ip) - x(im2)) * x(im1) - x(i) + th[0];
    }
#if CDK_HAS_USER_DRIFT
    case CDK_DRIFT_USER: return cdk_user::f<T>(th, n, i, x);
#endif
    default: {  // quadratic
      const T* B = th + n;
      const T* C = th + n + n * n;
      T s = th[i];
      for (int j = 0; j < n; ++j) {
        const T xj = x(j);
        T c = B[i * n + j];
        for (int k = 0; k < n; ++k) c += C[(i * n + j) * n + k] * x(k);
        s += c * xj;
      }
      return s;
    }
  }
}

template <typename T>
__device__ __forceinline__ T drift_jac(int id, const T* th, int n, int i, int j, const T* x) {
  switch (id) {
    case CDK_DRIFT_LINEAR: return th[i * n + j];
    case CDK_DRIFT_LORENZ63: {
      if (i == 0) return j == 0 ? -th[0] : (j == 1 ? th[0] : T(0));
      if (i == 1) return j == 0 ? th[1] - x[2] : (j == 1 ? T(-1) : -x[0]);
      return j == 0 ? x[1] : (j == 1 ? x[0] : -th[2]);
    }
    case CDK_DRIFT_LORENZ96: {
      const int ip = i + 1 == n ? 0 : i + 1, im1 = i == 0 ? n - 1 : i - 1, im2 = im1 == 0 ? n - 1 : im1 - 1;
      T v = T(0);
      if (j == ip) v += x[im1];
      if (j == im2) v -= x[im1];
      if (j == im1) v += x[ip] - x[im2];
      if (j == i) v -= T(1);
      return v;
    }
#if CDK_HAS_USER_DRIFT
    case CDK_DRIFT_USER: return cdk_user::jac<T>(th, n, i, j, x);
#endif
    default: {
      const T* B = th + n;
      const T* C = th + n + n * n;
      T s = B[i * n + j];
      for (int k = 0; k < n; ++k) s += (C[(i * n + j) * n + k] + C[(i * n + k) * n + j]) * x[k];
      return s;
    }
  }
}

// g_k = sum_i d2 f_i / dx_i dx_k: the only Hessian contraction the reference's 'second' order uses
// (0.5*jnp.trace(H_t @ P) traces axes (0,1): inference_ekf.py:111-114, SURVEY F8).  Zero unless quadratic.
template <typename T>
__device__ __forceinline__ T drift_graddiv(int id, const T* th, int n, int k) {
  if (id != CDK_DRIFT_QUADRATIC) return T(0);
  const T* C = th + n + n * n;
  T s = T(0);
  for (int i = 0; i < n; ++i) s += C[(i * n + i) * n + k] + C[(i * n + k) * n + i];
  return s;
}

// 0.5 * trace(Hess f_r(x) P) for the registry drifts (all polynomials of degree <= 2, so the Hessian is constant):
// the exact second-order term of the unscented mean (NOT the reference EKF's 'second' order, whose trace runs over the
// wrong axes -- SURVEY F8 -- and which drift_graddiv restates).
template <typename T>
__device__ __forceinline__ T drift_half_trhp(int id, const T* th, int n, int r, const T* P, int ld) {
  auto ps = [&](int i, int j) { return T(0.5) * (P[i * ld + j] + P[j * ld + i]); };
  switch (id) {
    case CDK_DRIFT_LINEAR: return T(0);
    case CDK_DRIFT_LORENZ63: return r == 0 ? T(0) : (r == 1 ? -ps(0, 2) : ps(0, 1));  // f1 = x (rho - z) - y, f2 = x y - b z
    case CDK_DRIFT_LORENZ96: {  // f_r = (x_{r+1} - x_{r-2}) x_{r-1} - x_r + F
      const int ip = r + 1 == n ? 0 : r + 1, im1 = r == 0 ? n - 1 : r - 1, im2 = im1 == 0 ? n - 1 : im1 - 1;
      return ps(ip, im1) - ps(im2, im1);
    }
    default: {  // f_r = a_r + B_rj x_j + C_rjk x_j x_k
      const T* C = th + n + n * n;
      T s = T(0);
      for (int j = 0; j < n; ++j)
        for (int k = 0; k < n; ++k) s += C[(r * n + j) * n + k] * ps(j, k);
      return s;
    }
  }
}

// ---- reverse-mode contractions of the registry (cdk_ekf_grad_dense_f64) --------------------------------------------
// Every registry drift is a polynomial of degree <= 2, so dJ_ik/dx_l is constant.  For the cotangent ab of the mean
// right-hand side and Jb of the Jacobian J(x) (Jb = (Pb + Pb^T) P^T for the cotangent Pb of J P + (J P)^T):
//   x-contraction      sum_ik Jb_ik dJ_ik/dx_l                 (the caller adds J^T ab)
//   theta-contraction  sum_i ab_i df_i/dtheta_e + sum_ik Jb_ik dJ_ik/dtheta_e
//                      + for 'second' order: sum_l ab_l 0.5 sum_k P_kl dg_k/dtheta_e, g = drift_graddiv (quadratic only)
template <typename T>
__device__ __forceinline__ T drift_jac_vjp_x(int id, const T* th, int n, int l, const T* Jb, int ld) {
  switch (id) {
    case CDK_DRIFT_LORENZ63:  // J10 = rho - z, J12 = -x, J20 = y, J21 = x
      if (l == 0) return Jb[2 * ld + 1] - Jb[ld + 2];
      if (l == 1) return Jb[2 * ld];
      return -Jb[ld];
    case CDK_DRIFT_LORENZ96: {
      // x_l is x_{i-1} of row i = l+1 (J_{i,i+1} = x_{i-1}, J_{i,i-2} = -x_{i-1}), x_{i+1} of row l-1 and x_{i-2} of row
      // l+2 (J_{i,i-1} = x_{i+1} - x_{i-2})
      auto w = [&](int q) { return q < 0 ? q + n : (q >= n ? q - n : q); };
      const int a = w(l + 1), b = w(l - 1), c = w(l + 2);
      return Jb[a * ld + c] - Jb[a * ld + b] + Jb[b * ld + w(l - 2)] - Jb[c * ld + a];
    }
    case CDK_DRIFT_QUADRATIC: {  // dJ_ij/dx_l = C_ijl + C_ilj
      const T* C = th + n + n * n;
      T s = T(0);
      for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) s += Jb[i * ld + j] * (C[(i * n + j) * n + l] + C[(i * n + l) * n + j]);
      return s;
    }
    default: return T(0);  // linear: J = W
  }
}

// JB = false: the f-part sum_i ab_i df_i/dtheta_e alone (Jb, P and second unused) -- all the theta-contraction the
// sigma-point UKF gradient needs, its sigma points entering f only (drift_theta_vjp_f).
template <typename T, bool JB = true>
__device__ __forceinline__ T drift_theta_vjp(int id, const T* th, int n, int e, const T* x, const T* ab, const T* Jb, int ld,
                                             const T* P, bool second) {
  switch (id) {
    case CDK_DRIFT_LINEAR:
      if (e < n * n) return JB ? ab[e / n] * x[e % n] + Jb[(e / n) * ld + e % n] : ab[e / n] * x[e % n];
      return ab[e - n * n];
    case CDK_DRIFT_LORENZ63:  // J00 = -sigma, J01 = sigma, J10 = rho - z, J22 = -beta
      if (e == 0) return JB ? ab[0] * (x[1] - x[0]) - Jb[0] + Jb[1] : ab[0] * (x[1] - x[0]);
      if (e == 1) return JB ? ab[1] * x[0] + Jb[ld] : ab[1] * x[0];
      return JB ? -ab[2] * x[2] - Jb[2 * ld + 2] : -ab[2] * x[2];
    case CDK_DRIFT_LORENZ96: {
      T s = T(0);
      for (int i = 0; i < n; ++i) s += ab[i];
      return s;
    }
    default: {  // quadratic: a | B | C
      if (e < n) return ab[e];
      if (e < n + n * n) {
        const int q = e - n, i = q / n, j = q % n;
        return JB ? ab[i] * x[j] + Jb[i * ld + j] : ab[i] * x[j];
      }
      const int q = e - n - n * n, i = q / (n * n), j = (q / n) % n, k = q % n;
      if (!JB) return ab[i] * x[j] * x[k];
      T s = ab[i] * x[j] * x[k] + Jb[i * ld + j] * x[k] + Jb[i * ld + k] * x[j];
      if (second) {  // g_k = sum_i (C_iik + C_iki)
        if (i == j) {
          T v = T(0);
          for (int l = 0; l < n; ++l) v += ab[l] * P[k * ld + l];
          s += T(0.5) * v;
        }
        if (i == k) {
          T v = T(0);
          for (int l = 0; l < n; ++l) v += ab[l] * P[j * ld + l];
          s += T(0.5) * v;
        }
      }
      return s;
    }
  }
}

template <typename T>
__device__ __forceinline__ T drift_theta_vjp_f(int id, int n, int e, const T* x, const T* ab) {
  return drift_theta_vjp<T, false>(id, nullptr, n, e, x, ab, nullptr, 0, nullptr, false);
}

// Reverse-mode contractions of drift_half_trhp (cdk_ukf_grad_dense_f64) for the cotangent ab of the mean right-hand side.
// The term is linear in sym(P) and the Hessians are constant, so
//   P-contraction      P_bar_jk += 0.5 sum_r ab_r (Hess f_r)_jk    (symmetric in j, k)
//   theta-contraction  quadratic only (Hess f_r = C_r + C_r^T): C_bar_rjk += ab_r sym(P)_jk; the other Hessians are fixed
template <typename T>
__device__ __forceinline__ T drift_half_trhp_vjp_p(int id, const T* th, int n, int j, int k, const T* ab) {
  switch (id) {
    case CDK_DRIFT_LORENZ63: {  // Hess f_1 = -(e0 e2^T + e2 e0^T), Hess f_2 = e0 e1^T + e1 e0^T
      const int lo = j < k ? j : k, hi = j < k ? k : j;
      if (lo == 0 && hi == 2) return T(-0.5) * ab[1];
      if (lo == 0 && hi == 1) return T(0.5) * ab[2];
      return T(0);
    }
    case CDK_DRIFT_LORENZ96: {
      // Hess f_r: +1 at (r+1, r-1) and (r-1, r+1), -1 at (r-2, r-1) and (r-1, r-2); for row j these are the rows
      // r = j-1, j+1 (+1, columns j-2, j+2) and r = j+2, j+1 (-1, columns j+1, j-1).  n = 4 folds j-2 onto j+2: both add.
      auto w = [&](int q) { return q < 0 ? q + n : (q >= n ? q - n : q); };
      T v = T(0);
      if (k == w(j - 2)) v += ab[w(j - 1)];
      if (k == w(j + 2)) v += ab[w(j + 1)];
      if (k == w(j + 1)) v -= ab[w(j + 2)];
      if (k == w(j - 1)) v -= ab[w(j + 1)];
      return T(0.5) * v;
    }
    case CDK_DRIFT_QUADRATIC: {
      const T* C = th + n + n * n;
      T s = T(0);
      for (int r = 0; r < n; ++r) s += ab[r] * (C[(r * n + j) * n + k] + C[(r * n + k) * n + j]);
      return T(0.5) * s;
    }
    default: return T(0);  // linear: no second-order term
  }
}

template <typename T>
__device__ __forceinline__ T drift_half_trhp_vjp_theta(int id, int n, int e, const T* ab, const T* P, int ld) {
  if (id != CDK_DRIFT_QUADRATIC || e < n + n * n) return T(0);
  const int q = e - n - n * n, r = q / (n * n), j = (q / n) % n, k = q % n;
  return ab[r] * (T(0.5) * (P[j * ld + k] + P[k * ld + j]));
}

// ---- block-cooperative dense helpers (all end WITHOUT a barrier unless noted) ---------------------------------------
// L = chol(A + boost I) (lower; reads the lower triangle of A; A != L). Upper triangle of L zeroed. Ends with a barrier.
// BLOCKED right-looking, panels of 8 columns, in place in L.  The critical path of a Cholesky is the dependent chain
// dot product -> pivot -> scale of every column; the UKF factors P at every RK stage, so this chain was 62 % of its time
// (profiles/r01_generic_ukf_n40*.txt).  History: one thread per row with two CTA barriers per column and a scalar k-loop,
// ~1,400 cycles per column; one warp (lane = rows r and r + 32, __syncwarp between columns, left-looking over all
// previous columns), ~1,000; + rsqrt pivots, ~750.  Now warp 0 factors an 8-column panel IN REGISTERS (dot products over
// the panel's own <= 7 columns, pivot rows broadcast with shuffles), then the whole CTA subtracts panel * panel^T from the
// trailing matrix on the FP64 tensor cores (mm_dmma) -- two CTA barriers per PANEL.  The pivot is one rsqrt (<= 2 ulp from sqrt + divide; NaN for a
// negative pivot, as the reference's non-PD behaviour).  mm_dmma is declared below.
template <typename T, bool TRANSA, bool TRANSB, class Epi>
__device__ __forceinline__ void mm_dmma(const T* __restrict__ A, int lda, const T* __restrict__ B, int ldb, int M, int N,
                                        int Kd, Epi epi);
template <typename T, bool TRANSA, bool TRANSB, bool LOWER = false, class Epi>
__device__ __forceinline__ void mm_dmma_w(int warp, int nwarp, const T* __restrict__ A, int lda, const T* __restrict__ B,
                                          int ldb, int M, int N, int Kd, Epi epi);

template <typename T>
__device__ void chol(const T* A, T* L, int n, int ld, T boost) {
  FOR_T(e, n * ld) {
    const int i = e / ld, j = e - i * ld;
    L[e] = j < i ? A[e] : (j == i ? A[e] + boost : T(0));  // working copy of the lower triangle
  }
  __syncthreads();
  for (int j0 = 0; j0 < n; j0 += 8) {
    const int bs = n - j0 < 8 ? n - j0 : 8;
    if (threadIdx.x < 32) {
      // The panel lives in REGISTERS while it is factored: lane r holds the 8 panel entries of rows j0 + r and
      // j0 + r + 32; the pivot row of column jj is lane jj's, broadcast entry by entry with shuffles -- no shared-memory
      // round trip and no __syncwarp inside the panel.
      const int lane = threadIdx.x;
      const int r0 = j0 + lane, r1 = r0 + 32;
      const bool v0 = r0 < n, v1 = r1 < n;
      T x[8], y[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        x[q] = (v0 && q < bs) ? L[r0 * ld + j0 + q] : T(0);
        y[q] = (v1 && q < bs) ? L[r1 * ld + j0 + q] : T(0);
      }
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        if (jj < bs) {
          T a = x[jj], b = y[jj];
#pragma unroll
          for (int q = 0; q < jj; ++q) {
            const T pq = __shfl_sync(0xffffffffu, x[q], jj);  // L[j0 + jj][j0 + q]
            a -= x[q] * pq;
            b -= y[q] * pq;
          }
          const T sjj = __shfl_sync(0xffffffffu, a, jj);  // the pivot row's own dot product
          const T rinv = rsqrt(sjj);
          x[jj] = lane == jj ? sjj * rinv : (lane > jj ? a * rinv : T(0));
          y[jj] = b * rinv;
        }
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        if (q < bs) {
          if (v0) L[r0 * ld + j0 + q] = x[q];
          if (v1) L[r1 * ld + j0 + q] = y[q];
        }
      }
    }
    __syncthreads();
    const int M = n - j0 - bs;
    if (M > 0) {  // trailing update: W[j0+bs.., j0+bs..] -= panel * panel^T (lower triangle only)
      const T* Pn = L + (j0 + bs) * ld + j0;
      T* W = L + (j0 + bs) * ld + (j0 + bs);
      mm_dmma<T, false, true>(Pn, ld, Pn, ld, M, M, bs, [&](int i, int c, double v) {
        if (c <= i) W[i * ld + c] -= (T)v;
      });
      __syncthreads();
    }
  }
}

// The same factorisation run by ONE WARP (warp `w` of the CTA; the others return at once): register panels as above, the
// trailing update on that warp's tensor-core tiles, __syncwarp instead of CTA barriers.  For the m x m innovation covariance
// (m ~ 20) a CTA-wide trailing update buys nothing and its 2 barriers per panel park seven warps behind one; and the two
// factorisations every measurement update needs -- chol(S) for the log-density, chol(sym(S) + 1e-9 I) for psd_solve -- are
// independent, so two warps run them side by side (condition_on).
//
// Working copy for chol_warp, written by the whole CTA (no barrier inside): the lower triangle of A, or of
// 0.5 (A + A^T) (SYM), plus boost on the diagonal, zeros above.
template <typename T, bool SYM>
__device__ __forceinline__ void chol_prep(const T* A, T* L, int n, int ld, T boost) {
  FOR_T(e, n * ld) {
    const int i = e / ld, j = e - i * ld;
    T v = T(0);
    if (j < i) v = SYM ? T(0.5) * (A[e] + A[j * ld + i]) : A[e];
    if (j == i) v = A[e] + boost;
    L[e] = v;
  }
}

// 1 / sqrt(x): hardware seed (MUFU.RSQ64H) and two Newton steps, without the exception branches of rsqrt(); <= 2 ulp.
// NaN for x < 0 -- the reference's behaviour for a non-PD matrix -- and for x = 0.
__device__ __forceinline__ double fast_rsqrt(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double h = 0.5 * x;
  double e = fma(-h * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-h * y, y, 0.5);
  return fma(y, e, y);
}
__device__ __forceinline__ float fast_rsqrt(float x) { return rsqrtf(x); }

template <typename T, bool TWO>
__device__ __forceinline__ void chol_warp_impl(T* L, int n, int ld) {
  const int lane = threadIdx.x & 31;
  for (int j0 = 0; j0 < n; j0 += 8) {
    const int bs = n - j0 < 8 ? n - j0 : 8;
    const int r0 = j0 + lane, r1 = r0 + 32;
    const bool v0 = r0 < n, v1 = TWO && r1 < n;
    T x[8], y[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      x[q] = (v0 && q < bs) ? L[r0 * ld + j0 + q] : T(0);
      y[q] = (v1 && q < bs) ? L[r1 * ld + j0 + q] : T(0);
    }
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
      if (jj < bs) {
        T a = x[jj], b = y[jj];
#pragma unroll
        for (int q = 0; q < jj; ++q) {
          const T pq = __shfl_sync(0xffffffffu, x[q], jj);
          a -= x[q] * pq;
          if (TWO) b -= y[q] * pq;
        }
        const T sjj = __shfl_sync(0xffffffffu, a, jj);
        const T rinv = fast_rsqrt(sjj);
        x[jj] = lane == jj ? sjj * rinv : (lane > jj ? a * rinv : T(0));
        if (TWO) y[jj] = b * rinv;
      }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      if (q < bs) {
        if (v0) L[r0 * ld + j0 + q] = x[q];
        if (v1) L[r1 * ld + j0 + q] = y[q];
      }
    }
    __syncwarp();
    const int M = n - j0 - bs;
    if (M > 0) {
      const T* Pn = L + (j0 + bs) * ld + j0;
      T* W = L + (j0 + bs) * ld + (j0 + bs);
      mm_dmma_w<T, false, true, true>(0, 1, Pn, ld, Pn, ld, M, M, bs, [&](int i, int c, double v) {
        if (c <= i) W[i * ld + c] -= (T)v;
      });
      __syncwarp();
    }
  }
}

// In-place factorisation of a chol_prep working copy by warp `w` alone (the other warps return at once); the caller
// synchronises the CTA before (the copy) and after (other warps reading L).
template <typename T>
__device__ void chol_warp(int w, T* L, int n, int ld) {
  if ((threadIdx.x >> 5) != w) return;
  if (n <= 32) {
    chol_warp_impl<T, false>(L, n, ld);
  } else {
    chol_warp_impl<T, true>(L, n, ld);
  }
}

// Solve (L L^T) X = B, B is [n x c] with leading dimension ldb, X written to `X` (may alias B).  Ends with a barrier.
// Each warp takes chunks of CB right-hand sides and keeps them in registers (lane r: rows r and r + 32); the substitutions
// are column-oriented: at step i the lane owning row i scales its entries by the reciprocal pivot (all reciprocals formed up
// front), CB shuffles broadcast them, and every lane below (forward) / above (backward) subtracts its L entry times the
// broadcast values -- one shared-memory load and CB FMAs per lane and step, no barrier until the end.  (History: one
// THREAD per right-hand side with serial dot products, ~21k cycles for m = 20, n = 40 with six of eight warps parked at
// the barrier -- 17 % of the UKF observation-step, profiles/r02_generic_ukf_rowseg*.)  Chunks are dealt from the LAST warp
// down so that warp 0, which evaluates the log-density first (mvn_ll_warp), gets the fewest.  FWD = false skips the forward
// substitution: then X solves L^T X = B alone (the Cholesky VJP of the sigma-point UKF gradient).
template <typename T, bool TWO, bool FWD = true>
__device__ __forceinline__ void chol_solve_chunks(const T* L, int n, int ld, const T* B, T* X, int c, int ldb) {
  constexpr int CB = 5;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int r0 = lane, r1 = lane + 32;
  const bool v0 = r0 < n, v1 = TWO && r1 < n;
  const T ri0 = v0 ? T(1) / L[r0 * ld + r0] : T(0);
  const T ri1 = v1 ? T(1) / L[r1 * ld + r1] : T(0);
  const int nchunk = (c + CB - 1) / CB;
  for (int ch = nwarp - 1 - warp; ch < nchunk; ch += nwarp) {
    const int col0 = ch * CB;
    T x0[CB], x1[CB];
#pragma unroll
    for (int q = 0; q < CB; ++q) {
      x0[q] = (v0 && col0 + q < c) ? B[r0 * ldb + col0 + q] : T(0);
      x1[q] = (v1 && col0 + q < c) ? B[r1 * ldb + col0 + q] : T(0);
    }
    for (int i = 0; FWD && i < n; ++i) {  // L z = b
      const int src = i & 31;
      const bool hi = TWO && i >= 32;
      const T l0 = (v0 && r0 > i) ? L[r0 * ld + i] : T(0);
      const T l1 = (v1 && r1 > i) ? L[r1 * ld + i] : T(0);
#pragma unroll
      for (int q = 0; q < CB; ++q) {
        const T z = __shfl_sync(0xffffffffu, hi ? x1[q] * ri1 : x0[q] * ri0, src);
        if (lane == src) {
          if (hi) x1[q] = z; else x0[q] = z;
        }
        x0[q] -= l0 * z;
        if (TWO) x1[q] -= l1 * z;
      }
    }
    for (int i = n - 1; i >= 0; --i) {  // L^T x = z
      const int src = i & 31;
      const bool hi = TWO && i >= 32;
      const T l0 = r0 < i ? L[i * ld + r0] : T(0);
      const T l1 = (TWO && r1 < i) ? L[i * ld + r1] : T(0);
#pragma unroll
      for (int q = 0; q < CB; ++q) {
        const T z = __shfl_sync(0xffffffffu, hi ? x1[q] * ri1 : x0[q] * ri0, src);
        if (lane == src) {
          if (hi) x1[q] = z; else x0[q] = z;
        }
        x0[q] -= l0 * z;
        if (TWO) x1[q] -= l1 * z;
      }
    }
#pragma unroll
    for (int q = 0; q < CB; ++q) {
      if (col0 + q < c) {
        if (v0) X[r0 * ldb + col0 + q] = x0[q];
        if (v1) X[r1 * ldb + col0 + q] = x1[q];
      }
    }
  }
}

template <typename T>
__device__ void chol_solve(const T* L, int n, int ld, const T* B, T* X, int c, int ldb) {
  if (n <= 32) {
    chol_solve_chunks<T, false>(L, n, ld, B, X, c, ldb);
  } else {
    chol_solve_chunks<T, true>(L, n, ld, B, X, c, ldb);
  }
  __syncthreads();
}

template <typename T>
__device__ void chol_solve(const T* L, int n, int ld, T* B, int c, int ldb) {
  chol_solve<T>(L, n, ld, B, B, c, ldb);
}

// Solve L^T X = B in place (B [n x c], leading dimension ldb): the backward phase of chol_solve.  Ends with a barrier.
template <typename T>
__device__ void chol_solve_lt(const T* L, int n, int ld, T* B, int c, int ldb) {
  if (n <= 32) {
    chol_solve_chunks<T, false, false>(L, n, ld, B, B, c, ldb);
  } else {
    chol_solve_chunks<T, true, false>(L, n, ld, B, B, c, ldb);
  }
  __syncthreads();
}

// log N(r; 0, L L^T) = -0.5 |L^-1 r|^2 - sum_i log L_ii - (m / 2) log(2 pi) for m <= 64, by WARP 0 (the MVN.log_prob of every
// update: TFP's Cholesky-based formula).  Lane j holds r_j and r_{j+32}; column-oriented forward substitution: at step i
// lane i scales its entry by the reciprocal pivot (all reciprocals and logs are computed up front, in parallel), one shuffle
// broadcasts z_i and the lanes below subtract L_ji z_i.  ~45 cycles per step instead of one thread's serial dot products,
// divisions and logarithms (that single thread was ~9k cycles of every observation-step, with the whole CTA waiting).
// Call from every thread of the CTA; threads outside warp 0 return immediately; the result is written to *out by lane 0
// (no barrier inside).
template <typename T>
__device__ __forceinline__ void mvn_ll_warp(const T* __restrict__ L, int ld, const T* __restrict__ r, int m, T* out) {
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  const bool v0 = lane < m, v1 = lane + 32 < m;
  const T d0 = v0 ? L[lane * ld + lane] : T(1), d1 = v1 ? L[(lane + 32) * ld + lane + 32] : T(1);
  const T ri0 = T(1) / d0, ri1 = T(1) / d1;
  T logdet = (v0 ? log(d0) : T(0)) + (v1 ? log(d1) : T(0));
  T x0 = v0 ? r[lane] : T(0), x1 = v1 ? r[lane + 32] : T(0);
  T quad = T(0);
  for (int i = 0; i < m; ++i) {
    const int src = i & 31;
    const T mine = i < 32 ? x0 * ri0 : x1 * ri1;  // meaningful on lane `src` only
    const T zi = __shfl_sync(0xffffffffu, mine, src);
    if (lane == src) quad += zi * zi;
    if (v0 && lane > i) x0 -= L[lane * ld + i] * zi;
    if (v1 && lane + 32 > i) x1 -= L[(lane + 32) * ld + i] * zi;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    quad += __shfl_xor_sync(0xffffffffu, quad, o);
    logdet += __shfl_xor_sync(0xffffffffu, logdet, o);
  }
  if (lane == 0) *out = T(-0.5) * quad - logdet - T(m) * half_log_2pi<T>();
}


// ---- block-cooperative small GEMM on the FP64 tensor cores ----------------------------------------------------------
// C(i, j) = sum_k opA(i, k) * opB(k, j), i < M, j < N, k < Kd, operands in shared memory (any T, converted to double in
// the fragment loads), result handed element-wise to `epi(i, j, double value)`.
//   TRANSA = false: opA(i, k) = A[i * lda + k];   true: opA(i, k) = A[k * lda + i]
//   TRANSB = false: opB(k, j) = B[k * ldb + j];   true: opB(k, j) = B[j * ldb + k]
// mma.sync.m8n8k4.f64 (SASS DMMA): each warp owns whole 8x8 output tiles and sweeps k in steps of 4 with two interleaved
// accumulator sets.  Fragment layout: A (8x4) lane -> (row lane/4, col lane%4); B (4x8) lane -> (row lane%4, col lane/4);
// C (8x8) lane -> (row lane/4, cols 2*(lane%4), +1).  Compared with one output element per thread (two shared-memory
// operand loads per FMA) this needs 2 loads per 256 FMAs and 1/16 of the instructions.  Every thread of the CTA must
// call it; no barrier inside (callers synchronise before the operands are read and after the epilogue writes).
// mm_dmma_w: the tiles are dealt to `nwarp` warps, the caller being number `warp` (mm_dmma: all warps of the CTA).
template <typename T, bool TRANSA, bool TRANSB, class Epi>
__device__ __forceinline__ void mm_dmma(const T* __restrict__ A, int lda, const T* __restrict__ B, int ldb, int M, int N,
                                        int Kd, Epi epi) {
  mm_dmma_w<T, TRANSA, TRANSB>(threadIdx.x >> 5, blockDim.x >> 5, A, lda, B, ldb, M, N, Kd, epi);
}

// LOWER: only the tiles that touch the lower triangle (row block >= column block).
template <typename T, bool TRANSA, bool TRANSB, bool LOWER, class Epi>
__device__ __forceinline__ void mm_dmma_w(int warp, int nwarp, const T* __restrict__ A, int lda, const T* __restrict__ B,
                                          int ldb, int M, int N, int Kd, Epi epi) {
  const int lane = threadIdx.x & 31;
  const int gid = lane >> 2, tig = lane & 3;
  const int tm = (M + 7) >> 3, tn = (N + 7) >> 3;
  for (int t = warp; t < tm * tn; t += nwarp) {
    const int r0 = (t / tn) << 3, c0 = (t % tn) << 3;
    if (LOWER && c0 > r0) continue;
    const int ia = r0 + gid, jb = c0 + gid;
    const bool va = ia < M, vb = jb < N;
    double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0;
    for (int k0 = 0; k0 < Kd; k0 += 8) {
      {
        const int k = k0 + tig;
        const bool vk = k < Kd;
        const double av = (va && vk) ? (double)(TRANSA ? A[k * lda + ia] : A[ia * lda + k]) : 0.0;
        const double bv = (vb && vk) ? (double)(TRANSB ? B[jb * ldb + k] : B[k * ldb + jb]) : 0.0;
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                     : "+d"(d0), "+d"(d1)
                     : "d"(av), "d"(bv));
      }
      {
        const int k = k0 + 4 + tig;
        const bool vk = k < Kd;
        const double av = (va && vk) ? (double)(TRANSA ? A[k * lda + ia] : A[ia * lda + k]) : 0.0;
        const double bv = (vb && vk) ? (double)(TRANSB ? B[jb * ldb + k] : B[k * ldb + jb]) : 0.0;
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                     : "+d"(e0), "+d"(e1)
                     : "d"(av), "d"(bv));
      }
    }
    const int i = r0 + gid, j = c0 + 2 * tig;
    if (i < M) {
      if (j < N) epi(i, j, d0 + e0);
      if (j + 1 < N) epi(i, j + 1, d1 + e1);
    }
  }
}

// C(i, j) = sum_k opA(i, k) * B[k * ldb + j] for a WIDE result (N >> M: a small matrix applied to every member of an
// ensemble): each warp takes strips of 8 columns and keeps the accumulators of ALL row tiles (M <= 64) in registers, so a
// B fragment is loaded once per k-step and reused by every row tile, and the per-tile bookkeeping of mm_dmma (index
// arithmetic, bounds, accumulator setup: ~130 instructions around the 5-10 DMMAs of a short k loop) is paid once per strip.
template <typename T, bool TRANSA, class Epi>
__device__ __forceinline__ void mm_dmma_strip(const T* __restrict__ A, int lda, const T* __restrict__ B, int ldb, int M, int N,
                                              int Kd, Epi epi) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int gid = lane >> 2, tig = lane & 3;
  const int tm = (M + 7) >> 3, ts = (N + 7) >> 3;
  for (int sidx = warp; sidx < ts; sidx += nwarp) {
    const int jb = (sidx << 3) + gid;
    const bool vb = jb < N;
    double acc[8][2];
#pragma unroll
    for (int t = 0; t < 8; ++t) acc[t][0] = acc[t][1] = 0.0;
    for (int k0 = 0; k0 < Kd; k0 += 4) {
      const int k = k0 + tig;
      const bool vk = k < Kd;
      const double bv = (vb && vk) ? (double)B[(size_t)k * ldb + jb] : 0.0;
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        if (t < tm) {
          const int ia = (t << 3) + gid;
          const double av = (ia < M && vk) ? (double)(TRANSA ? A[k * lda + ia] : A[ia * lda + k]) : 0.0;
          asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                       : "+d"(acc[t][0]), "+d"(acc[t][1])
                       : "d"(av), "d"(bv));
        }
      }
    }
    const int j = (sidx << 3) + 2 * tig;
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int i = (t << 3) + gid;
      if (t < tm && i < M) {
        if (j < N) epi(i, j, acc[t][0]);
        if (j + 1 < N) epi(i, j + 1, acc[t][1]);
      }
    }
  }
}

// ---- the literal sigma-point unscented moment ODE (cdk_ukf_filter with CDK_FLAG_UKF_SIGMA_POINTS, cdk_ukf_grad_sigma) ----
// lambda = alpha^2 (n + kappa) - n;  c = sqrt(n + lambda);  w = 1 / (2 (n + lambda));  w0 = lambda / (n + lambda)
template <typename T>
struct UkfSigmaWeights {
  T lam, cs, w, w0;
  __device__ explicit UkfSigmaWeights(const cdk_desc& d) {
    lam = T(d.alpha * d.alpha * (d.n + d.kappa) - d.n);
    cs = sqrt(T(d.n) + lam);
    w = T(1) / (T(2) * (T(d.n) + lam));
    w0 = lam / (T(d.n) + lam);
  }
};

// k = dt * rhs(m, P) of Sarkka eq. 3.183 (inference_ukf.py:130-152).  With X = [m, m + c L_i, m - c L_i], Lc = chol(P):
//   dm = w0 f(m) + w sum_i (f(X_i^+) + f(X_i^-))
//   f_X^T W X = sum_k w_c[k] (f_k - fbar)(x_k - xbar)^T = w c sum_i (f_i^+ - f_i^-) L_i^T     (xbar = m)
//   dP = w c (D Lc^T + Lc D^T) + Sigma,  D[:, i] = f(X_i^+) - f(X_i^-)
// m, P, lql (Sigma), Lc, dF (D) and the outputs km, kP are n x ld blocks in shared memory; Lc and dF are left holding
// chol(P) and D.  Ends with a barrier.
template <typename T>
__device__ void ukf_sigma_rhs(const cdk_desc& d, const T* th, int n, int ld, const T* mm, const T* P, const T* lql, T* Lc,
                              T* dF, T* km, T* kP, T dt) {
  T* sF = kP;  // sF[j*ld + i] = f_j(X_i^+) + f_j(X_i^-): parked in the output block until the row sums are taken
  chol<T>(P, Lc, n, ld, T(0));
  const UkfSigmaWeights<T> u(d);
  const T cs = u.cs, w = u.w, w0 = u.w0;
  FOR_T(e, n * n) {
    const int j = e / n, i = e - j * n;
    const T fp = drift_f<T>(d.drift_id, th, n, j, [&](int q) { return mm[q] + cs * Lc[q * ld + i]; });
    const T fm = drift_f<T>(d.drift_id, th, n, j, [&](int q) { return mm[q] - cs * Lc[q * ld + i]; });
    dF[j * ld + i] = fp - fm;
    sF[j * ld + i] = fp + fm;
  }
  __syncthreads();
  FOR_T(j, n) {
    T s = T(0);
    for (int i = 0; i < n; ++i) s += sF[j * ld + i];
    const T f0 = drift_f<T>(d.drift_id, th, n, j, [&](int q) { return mm[q]; });
    km[j] = dt * (w0 * f0 + w * s);
  }
  __syncthreads();  // the row sums are taken: the output block may be overwritten
  const T wc = w * cs;
  T* DL = kP;  // dF Lc^T, symmetrised in place below
  mm_dmma<T, false, true>(dF, ld, Lc, ld, n, n, n, [&](int i, int j, double v) { DL[i * ld + j] = (T)v; });
  __syncthreads();
  FOR_T(e, n * n) {
    const int a = e / n, b = e - a * n;
    if (a <= b) {  // one thread owns the pair (a, b), (b, a)
      const T dab = DL[a * ld + b], dba = DL[b * ld + a];
      kP[a * ld + b] = dt * (wc * (dab + dba) + lql[a * ld + b]);
      if (a != b) kP[b * ld + a] = dt * (wc * (dba + dab) + lql[b * ld + a]);
    }
  }
  __syncthreads();
}

}  // namespace cdk
