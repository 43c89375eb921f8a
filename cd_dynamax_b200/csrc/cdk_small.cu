// cdk_small.cu -- register-arithmetic CD-EKF for tiny state dimensions (Lorenz-63: m[3] + symmetric P[6]).
//
// Replaces extended_kalman_filter (src/continuous_discrete_nonlinear_gaussian_ssm/inference_ekf.py:202-326) with its
// _predict (:46-148, moment ODE dm = f(m), dP = F P + P F^T + L Qc L^T) and _condition_on (:153-199) for the
// registry drifts whose whole filter state fits in registers.
//
// B200 mapping (BASELINE config 3: N = 65,536, K = 1,000, n = 3, m = 1) -- kernel `ekf_small_lw` below: one warp keeps 32
// trajectories for the whole kernel, all arithmetic in registers (FP64 FMA pipe bound), warps never synchronise with each
// other.  `eks_small_lw` is the matching backward (smoothing) pass.  Earlier variants -- thread per trajectory with a
// flattened substep stream, CTA-wide per-step regrouping by substep count with a helper I/O warp, a trajectory pool per
// warp -- were measured slower and removed; DESIGN.md section 4.1 and profiles/ keep their numbers.
#include <type_traits>

#include "cdk_common.cuh"

#include <cuda.h>
#include <stdlib.h>
#include <string.h>

namespace cdk {
namespace {

// ---- symmetric packed storage: upper triangle, row-major ----------------------------------------------------------
template <int NX>
__host__ __device__ constexpr int pidx(int i, int j) {
  return i <= j ? i * NX - (i * (i - 1)) / 2 + (j - i) : j * NX - (j * (j - 1)) / 2 + (i - j);
}

template <typename T, int NX>
struct St {
  static constexpr int NP = NX * (NX + 1) / 2;
  T m[NX];
  T P[NP];
};

// ---- drift policies: f(x), G = J(x) P (P symmetric packed) ---------------------------------------------------------
struct DriftL63 {
  static constexpr int NX = 3;
  static constexpr int NTHETA = 3;
  template <typename T>
  __device__ __forceinline__ static void f(const T* th, const T (&x)[3], T (&o)[3]) {
    // LearnableLorenz63.f, cdnlgssm_utils.py:77-83
    o[0] = th[0] * (x[1] - x[0]);
    o[1] = x[0] * (th[1] - x[2]) - x[1];
    o[2] = x[0] * x[1] - th[2] * x[2];
  }
  template <typename T>
  __device__ __forceinline__ static void jac(const T* th, const T (&x)[3], T (&J)[3][3]) {
    J[0][0] = -th[0]; J[0][1] = th[0]; J[0][2] = T(0);
    J[1][0] = th[1] - x[2]; J[1][1] = T(-1); J[1][2] = -x[0];
    J[2][0] = x[1]; J[2][1] = x[0]; J[2][2] = -th[2];
  }
  template <typename T>
  __device__ __forceinline__ static void jp(const T* th, const T (&x)[3], const T (&P)[6], T (&G)[3][3]) {
    // J = [[-s, s, 0], [r - z, -1, -x], [y, x, -b]]  (jacfwd(f), inference_ekf.py:95)
    const T rz = th[1] - x[2];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const T p0 = P[pidx<3>(0, j)], p1 = P[pidx<3>(1, j)], p2 = P[pidx<3>(2, j)];
      G[0][j] = th[0] * (p1 - p0);
      G[1][j] = rz * p0 - p1 - x[0] * p2;
      G[2][j] = x[1] * p0 + x[0] * p1 - th[2] * p2;
    }
  }
};

// rhs of the EKF moment ODE, WITHOUT the dt factor (orders 'first' and 'second'; the reference's second-order term
// 0.5*einsum('iik,kl->l', Hess, P) is identically zero for every drift handled here -- SURVEY F8).
// Lorenz-63: the six entries of J P + P J^T + L Qc L^T written out for the sparse Jacobian
//   J = [[-s, s, 0], [rz, -1, -x], [y, x, -b]],  rz = rho - z,
// with like terms merged (s P11 - (1 + s) P01, ...): 22 FP64 instructions instead of the 30 of forming G = J P (21) and then
// G + G^T + L Qc L^T (9) -- 16 % of the substep, which is the FP64-pipe-bound part of the kernel.
template <typename T, class Drift>
__device__ __forceinline__ void ekf_rhs(const T* th, const T* lql, const St<T, Drift::NX>& y, St<T, Drift::NX>& k) {
  constexpr int NX = Drift::NX;
  if constexpr (std::is_same<Drift, DriftL63>::value) {
    const T s = th[0], b = th[2], x = y.m[0], yy = y.m[1], z = y.m[2];
    const T rz = th[1] - z;
    const T P00 = y.P[0], P01 = y.P[1], P02 = y.P[2], P11 = y.P[3], P12 = y.P[4], P22 = y.P[5];
    k.m[0] = s * (yy - x);
    k.m[1] = fma(x, rz, -yy);
    k.m[2] = fma(x, yy, -(b * z));
    const T s1 = T(1) + s, sb = s + b, b1 = T(1) + b;  // loop-invariant: hoisted out of the substep loop by the compiler
    // (0,0): 2 (J P)_00 = 2 s (P01 - P00)
    k.P[0] = fma(s + s, P01 - P00, lql[0]);
    // (0,1): (J P)_01 + (J P)_10 = s (P11 - P01) + rz P00 - P01 - x P02
    k.P[1] = fma(-x, P02, fma(rz, P00, fma(-s1, P01, fma(s, P11, lql[1]))));
    // (0,2): s (P12 - P02) + y P00 + x P01 - b P02
    k.P[2] = fma(x, P01, fma(yy, P00, fma(-sb, P02, fma(s, P12, lql[2]))));
    // (1,1): 2 (rz P01 - P11 - x P12)
    k.P[3] = fma(T(2), fma(-x, P12, fma(rz, P01, -P11)), lql[3]);
    // (1,2): rz P02 - P12 - x P22 + y P01 + x P11 - b P12
    k.P[4] = fma(x, P11, fma(yy, P01, fma(-x, P22, fma(-b1, P12, fma(rz, P02, lql[4])))));
    // (2,2): 2 (y P02 + x P12 - b P22)
    k.P[5] = fma(T(2), fma(-b, P22, fma(x, P12, yy * P02)), lql[5]);
  } else {
    Drift::f(th, y.m, k.m);
    T G[NX][NX];
    Drift::jp(th, y.m, y.P, G);
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int j = i; j < NX; ++j)
        k.P[pidx<NX>(i, j)] = (i == j) ? fma(T(2), G[i][i], lql[pidx<NX>(i, i)]) : (G[i][j] + G[j][i]) + lql[pidx<NX>(i, j)];
  }
}

// One explicit RK step y <- y + dt * sum_i b_i f(y_i), y_i = y + dt * sum_j a_ij f(y_j)  (diffrax stores k_i = dt f;
// folding dt into the coefficients is the same arithmetic up to rounding and saves one multiply per state element).
template <typename T, class Drift, int SOLVER>
__device__ __forceinline__ void rk_step(const T* th, const T* lql, St<T, Drift::NX>& y, T dt) {
  using TB = Tab<SOLVER>;
  constexpr int NX = Drift::NX;
  constexpr int NP = St<T, NX>::NP;
  // The weighted stage sum is accumulated relative to the first non-zero weight, ksum = sum_i (b_i / b_i0) k_i, and added
  // with ONE in-place fma y += (b_i0 dt) ksum: the same operation count as accumulating y + dt b_i k_i stage by stage, but
  // the new state is written straight into the registers of the old one (no register copies at the loop back-edge).
  constexpr int I0 = TB::b(0) != 0.0 ? 0 : (TB::S > 1 && TB::b(1) != 0.0 ? 1 : (TB::S > 2 && TB::b(2) != 0.0 ? 2 : 3));
  St<T, NX> k[TB::S];
  St<T, NX> ksum;
#pragma unroll
  for (int i = 0; i < TB::S; ++i) {
    St<T, NX> yi = y;
#pragma unroll
    for (int j = 0; j < i; ++j) {
      if (TB::a(i, j) != 0.0) {
        const T c = T(TB::a(i, j)) * dt;
#pragma unroll
        for (int e = 0; e < NX; ++e) yi.m[e] = fma(c, k[j].m[e], yi.m[e]);
#pragma unroll
        for (int e = 0; e < NP; ++e) yi.P[e] = fma(c, k[j].P[e], yi.P[e]);
      }
    }
    ekf_rhs<T, Drift>(th, lql, yi, k[i]);
    if (i == I0) {
      ksum = k[i];
    } else if (TB::b(i) != 0.0) {
      const T c = T(TB::b(i) / TB::b(I0));
      if (TB::b(i) == TB::b(I0)) {
#pragma unroll
        for (int e = 0; e < NX; ++e) ksum.m[e] += k[i].m[e];
#pragma unroll
        for (int e = 0; e < NP; ++e) ksum.P[e] += k[i].P[e];
      } else {
#pragma unroll
        for (int e = 0; e < NX; ++e) ksum.m[e] = fma(c, k[i].m[e], ksum.m[e]);
#pragma unroll
        for (int e = 0; e < NP; ++e) ksum.P[e] = fma(c, k[i].P[e], ksum.P[e]);
      }
    }
  }
  const T w = T(TB::b(I0)) * dt;
#pragma unroll
  for (int e = 0; e < NX; ++e) y.m[e] = fma(w, ksum.m[e], y.m[e]);
#pragma unroll
  for (int e = 0; e < NP; ++e) y.P[e] = fma(w, ksum.P[e], y.P[e]);
}

// 1 / x for a positive, normal x without the IEEE slow path: MUFU.RCP64H seed (rcp.approx.ftz.f64, ~20 bits) and two
// Newton steps (error e -> e^2: below 2^-53 after the second).  The compiler's own double division carries two
// data-dependent branches and a call to a fix-up routine per division; the scalar-emission update needs two reciprocals
// per observation, of innovation variances that are positive and nowhere near the ends of the exponent range (anything
// else -- zero, negative, NaN -- gives inf / NaN here and the trajectory is flagged, as in the reference).
__device__ __forceinline__ double fast_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  return fma(r, e, r);
}
__device__ __forceinline__ float fast_rcp(float x) { return 1.0f / x; }

// Measurement update + log-likelihood increment (inference_ekf.py:285-289, :153-199; psd_solve utils.py:202-207).
// sh: H[NY*NX], d[NY], R[NY*NY] in shared memory.
template <typename T, int NX, int NY>
__device__ __forceinline__ T ekf_update(const T* H, const T* dvec, const T* R, St<T, NX>& s, const T (&y)[NY],
                                        int num_iter, T* s_defer = nullptr) {
  // s_defer (scalar emission only): the caller accumulates log S itself (as the log of a running product, one log per
  // 8 steps instead of one per step); the returned increment then omits the -log(S)/2 term and *s_defer = S.
  T ll = T(0);
  if constexpr (NY == 1) {
    // Scalar emission: the 1x1 Cholesky / triangular solves collapse to two independent reciprocals and one log, which
    // the scheduler can overlap (the generic path below is one long sqrt -> rcp -> log dependency chain).
    //   log N(y; h(m), S) = -r^2 / (2 S) - log(S) / 2 - log(2 pi) / 2;   K = P H^T / (S + 1e-9);   P -= K S K^T
    for (int it = 0; it < num_iter; ++it) {
      T HP[NX];
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        T acc = T(0);
#pragma unroll
        for (int k = 0; k < NX; ++k) acc += H[k] * s.P[pidx<NX>(k, j)];
        HP[j] = acc;
      }
      T S = R[0], hm = dvec[0];
#pragma unroll
      for (int k = 0; k < NX; ++k) {
        S += HP[k] * H[k];
        hm += H[k] * s.m[k];
      }
      const T r = y[0] - hm;
      const T rb = T(1) / (S + T(1e-9));
      if (it == 0) {
        if (s_defer) {
          *s_defer = S;
          ll = T(-0.5) * (r * r / S) - half_log_2pi<T>();
        } else {
          ll = T(-0.5) * (r * r / S) - T(0.5) * log(S) - half_log_2pi<T>();
        }
      }
      T Kt[NX];
#pragma unroll
      for (int j = 0; j < NX; ++j) Kt[j] = HP[j] * rb;
#pragma unroll
      for (int i = 0; i < NX; ++i) {
        const T ks = Kt[i] * S;
#pragma unroll
        for (int j = i; j < NX; ++j) s.P[pidx<NX>(i, j)] -= ks * Kt[j];
        s.m[i] += Kt[i] * r;
      }
    }
    return ll;
  } else {
  for (int it = 0; it < num_iter; ++it) {
    T HP[NY][NX];
#pragma unroll
    for (int a = 0; a < NY; ++a)
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        T acc = T(0);
#pragma unroll
        for (int k = 0; k < NX; ++k) acc += H[a * NX + k] * s.P[pidx<NX>(k, j)];
        HP[a][j] = acc;
      }
    T S[NY][NY];
#pragma unroll
    for (int a = 0; a < NY; ++a)
#pragma unroll
      for (int b = 0; b < NY; ++b) {
        T acc = T(0);
#pragma unroll
        for (int k = 0; k < NX; ++k) acc += HP[a][k] * H[b * NX + k];
        S[a][b] = R[a * NY + b] + acc;
      }
    T r[NY];
#pragma unroll
    for (int a = 0; a < NY; ++a) {
      T acc = dvec[a];
#pragma unroll
      for (int k = 0; k < NX; ++k) acc += H[a * NX + k] * s.m[k];
      r[a] = y[a] - acc;
    }
    if (it == 0) {
      // MVN(h(m), H P H^T + R).log_prob(y): Cholesky of S without jitter (TFP)
      T Lc[NY][NY];
      T z[NY];
      T logdet = T(0), quad = T(0);
#pragma unroll
      for (int j = 0; j < NY; ++j) {
        T dsum = S[j][j];
#pragma unroll
        for (int k = 0; k < j; ++k) dsum -= Lc[j][k] * Lc[j][k];
        const T ljj = sqrt(dsum);
        Lc[j][j] = ljj;
        const T inv = T(1) / ljj;
#pragma unroll
        for (int i = j + 1; i < NY; ++i) {
          T v = S[i][j];
#pragma unroll
          for (int k = 0; k < j; ++k) v -= Lc[i][k] * Lc[j][k];
          Lc[i][j] = v * inv;
        }
        T zz = r[j];
#pragma unroll
        for (int k = 0; k < j; ++k) zz -= Lc[j][k] * z[k];
        z[j] = zz * inv;
        quad += z[j] * z[j];
        logdet += log(ljj);
      }
      ll = T(-0.5) * quad - logdet - T(NY) * half_log_2pi<T>();
    }
    // K = psd_solve(S, H P)^T : Cholesky of sym(S) + 1e-9 I
    T Lb[NY][NY];
    T inv_d[NY];
#pragma unroll
    for (int j = 0; j < NY; ++j) {
      T dsum = S[j][j] + T(1e-9);
#pragma unroll
      for (int k = 0; k < j; ++k) dsum -= Lb[j][k] * Lb[j][k];
      const T ljj = sqrt(dsum);
      Lb[j][j] = ljj;
      inv_d[j] = T(1) / ljj;
#pragma unroll
      for (int i = j + 1; i < NY; ++i) {
        T v = T(0.5) * (S[i][j] + S[j][i]);
#pragma unroll
        for (int k = 0; k < j; ++k) v -= Lb[i][k] * Lb[j][k];
        Lb[i][j] = v * inv_d[j];
      }
    }
    T Kt[NY][NX];  // Kt = (S + boost)^-1 H P, K = Kt^T
#pragma unroll
    for (int c = 0; c < NX; ++c) {
      T w[NY];
#pragma unroll
      for (int i = 0; i < NY; ++i) {
        T v = HP[i][c];
#pragma unroll
        for (int k = 0; k < i; ++k) v -= Lb[i][k] * w[k];
        w[i] = v * inv_d[i];
      }
#pragma unroll
      for (int i = NY - 1; i >= 0; --i) {
        T v = w[i];
#pragma unroll
        for (int k = i + 1; k < NY; ++k) v -= Lb[k][i] * Kt[k][c];
        Kt[i][c] = v * inv_d[i];
      }
    }
    // P <- P - K S K^T (un-boosted S), m <- m + K (y - h(m))
    T KS[NX][NY];
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int b = 0; b < NY; ++b) {
        T acc = T(0);
#pragma unroll
        for (int a = 0; a < NY; ++a) acc += Kt[a][i] * S[a][b];
        KS[i][b] = acc;
      }
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int j = i; j < NX; ++j) {
        T acc = T(0);
#pragma unroll
        for (int b = 0; b < NY; ++b) acc += KS[i][b] * Kt[b][j];
        s.P[pidx<NX>(i, j)] -= acc;
      }
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      T acc = T(0);
#pragma unroll
      for (int a = 0; a < NY; ++a) acc += Kt[a][i] * r[a];
      s.m[i] += acc;
    }
  }
  return ll;
  }
}


// ---- cp.async (LDGSTS) element copies: sizeof(T) in {4, 8} is always naturally aligned -----------------------------
template <typename T>
__device__ __forceinline__ void cp_async_elem(T* smem_dst, const T* gsrc) {
  const unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(d), "l"(gsrc), "n"(sizeof(T)) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// TMA descriptors of the per-step output arrays viewed as 2-D tensors [N][K*len] (len = NX or NX*NX): one box is
// {2 steps x len elements, 32 trajectories}, so ONE cp.async.bulk.tensor store per array writes a warp's two steps.
struct alignas(64) V5Maps {
  CUtensorMap m[4];  // FM, FP, PM, PP
  int use_tma;
};

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_src));
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(map), "r"(c0), "r"(c1),
               "r"(s)
               : "memory");
}

// ======================================================================================================================
// INDEPENDENT WARPS.  One warp = 32 trajectories kept for the whole kernel (the 14 warps of a CTA share it only for
// placement: they never synchronise with each other); the filter state never leaves registers, every gap runs to the
// warp-wide maximum substep count (predicated lanes, 4.5/6 = 75 % lane efficiency on the benchmark grid), and the
// latency-bound measurement update of one warp hides behind the FP64-bound substeps of the others.  Inputs come through a
// private 4-deep cp.async ring; each warp stores its own 2-step output block with four TMA tensor stores.
// ======================================================================================================================
constexpr int LW_RING = 4;

// Diagnostics (scripts/trace_lw.py): when a device buffer is registered with cdk_debug_set_trace(), lane 0 of every warp
// records {globaltimer at entry, at exit, %smid, %warpid} -- used to see how warp run times spread over SM sub-partitions.
__device__ unsigned long long* g_lw_trace = nullptr;
__device__ __forceinline__ unsigned long long globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

template <typename T, int NX, int NY>
struct alignas(128) LWSmem {
  T fm[32][2][NX];
  alignas(128) T fp[32][2][NX * NX];
  alignas(128) T pm[32][2][NX];
  alignas(128) T pp[32][2][NX * NX];
  T inY[LW_RING][NY][32];
  T inT[LW_RING][32];
  // followed by the model constants: NPAR values (shared) or 32 * NPAR (one block per lane when batched)
};

// Time-sliced mode (see ekf_small_lw): the filter state of a group of 32 trajectories between two K-segments.
template <typename T, int NX>
struct alignas(128) LWGroup {
  T m[NX][32];
  T P[NX * (NX + 1) / 2][32];
  T ll[32], sprod[32];
  int esum[32], flags[32];  // flags: bit 0 sbad, bits 8.. status
};

// Write one staging row (LEN elements of step parity ROW) of this lane's [2][LEN] block.  fp64: the block starts 16-byte
// aligned (lane stride 16 LEN bytes), so all but at most one element go out as 128-bit stores (conflict-free per quarter
// warp) -- 14 shared-memory stores per step instead of 24.
template <int ROW, int LEN, typename T>
__device__ __forceinline__ void stage_row(T* lane_block, const T (&v)[LEN]) {
  T* p = lane_block + ROW * LEN;
  if constexpr (sizeof(T) == 8) {
    constexpr int FIRST = (ROW * LEN) & 1;
    if (FIRST) p[0] = v[0];
#pragma unroll
    for (int e = FIRST; e + 1 < LEN; e += 2) *reinterpret_cast<double2*>(p + e) = make_double2(v[e], v[e + 1]);
    if ((LEN - FIRST) & 1) p[LEN - 1] = v[LEN - 1];
  } else {
#pragma unroll
    for (int e = 0; e < LEN; ++e) p[e] = v[e];
  }
}

// Warps per CTA: 7 (two CTAs per SM, <= 128 registers) or 14 (ONE CTA per SM, <= 144 registers: the drift parameters and
// L Qc L^T then live in registers instead of being re-read from shared memory every substep).  Either way 65,536
// trajectories are one wave of 2,048 warps over 148 SMs.  CDK_LW_WPC selects.
template <typename T, class Drift, int NY, int SOLVER, int WPC, bool SLICED = false>
__global__ void __launch_bounds__(SLICED ? 32 * 12 : 32 * WPC, WPC == 7 ? 2 : 1)
    ekf_small_lw(const KArgs<T> a, const __grid_constant__ V5Maps maps, const int warp_bytes, const int use_token, const int G,
                 const int segk) {
  constexpr int NX = Drift::NX;
  constexpr int NP = St<T, NX>::NP;
  constexpr int NTH = Drift::NTHETA;
  constexpr int NPAR = NTH + NP + NY * NX + NY + NY * NY;  // theta | lql (packed) | H | d | R
  using S = LWSmem<T, NX, NY>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5;
  S& sm = *reinterpret_cast<S*>(smem_raw + (size_t)warp * warp_bytes);  // every warp owns a private slice
  T* parbase = reinterpret_cast<T*>(smem_raw + (size_t)warp * warp_bytes + sizeof(S));

  const long long N = a.d.N;
  const int K = a.d.K;
  const int lane = threadIdx.x & 31;
  // the CTA may be launched with FEWER warps than WPC (launch_one picks the count from N so that a small batch still
  // spreads over every SM and sub-partition): the trajectory map only depends on the run-time block size
  //
  // TIME SLICING (G groups of 32 trajectories per CTA, K cut into segments of `segk` steps; the launcher enables it when the
  // batch is more than one balanced wave): the CTA's W resident warps work through the items (segment, group) in rounds of W,
  // item i = segment i / G, group i % G, with a CTA barrier between rounds -- item i - G (the same group's previous segment)
  // always lies in an earlier round because W <= G.  A group's state crosses segments through an LWGroup block in shared
  // memory.  Why: 2,048 warps on 148 SMs are 13.84 per SM, i.e. (4, 4, 3, 3) per sub-partition, and the pass takes as long
  // as the sub-partitions with four; with W = 12 (or 8) resident warps every sub-partition carries three (two) at any time
  // and the 14 groups of an SM take 14 / 12 passes of a balanced SM instead of 4 / 3 (measured balanced rates:
  // profiles/r02_c3_outputs_probe.jsonl).  Without slicing G = W, one segment: warp w keeps group w for the whole kernel.
  // (SLICED is its own instantiation with at most 12 resident warps and 170 registers: the bookkeeping that stays live
  // across the step loop costs the 128-register 14-warp kernel spills inside the loop.)
  const int W = blockDim.x >> 5;
  const long long ngroups = (N + 31) >> 5;
  const int Gq = SLICED ? G : W;
  const long long gfirst = (long long)blockIdx.x * Gq;
  const int Gc = (int)(ngroups - gfirst < (long long)Gq ? ngroups - gfirst : (long long)Gq);  // groups of this CTA
  const int nseg = SLICED ? (K + segk - 1) / segk : 1;
  const int Wr = W < Gc ? W : Gc;  // items per round
  const int nitems = SLICED ? Gc * nseg : 1;
  long long traj0 = (gfirst + warp) * 32;  // first item (the only one without slicing); reset per item below
  // Optional FP64-pipe semaphore (CDK_LW_TOKEN = permits, default off): at most `permits` warps of an SM sub-partition are
  // inside the RK substep loop at a time (FIFO tickets), the others update / stage / store.  Built to break the convoy
  // that forms because warps sharing a pipe equally re-synchronise their phases; measured no gain (7.2-7.5 ms with 2-3
  // permits, 8.1 ms with 1, 7.3 ms without), because the loop is bound by register-file bandwidth, not latency: a DFMA
  // with three distinct register operands issues every 3 cycles, not 2 (scripts/micro/fp64_regs.cu), and the update phase
  // of one warp already hides behind the substeps of the others.  Kept for experiments.
  __shared__ unsigned lw_token[4][2];  // [sub-partition][next ticket, tenures completed]
  if (threadIdx.x < 8) (&lw_token[0][0])[threadIdx.x] = 0u;
  __syncthreads();
  if (!SLICED && warp >= Gc) return;  // whole warp out of range (without slicing nobody ever waits for it)
  unsigned hw_warp;
  asm volatile("mov.u32 %0, %warpid;" : "=r"(hw_warp));
  volatile unsigned* const tok = &lw_token[hw_warp & 3][0];
  long long traj = traj0 + lane;
  bool live = traj < N;
  // A lane past the end of the batch (ragged last warp) shadows the last trajectory: it computes, never stores (its
  // staging rows fall outside the tensor map and TMA clips them; the cooperative flush copies `nlive` rows).  The step
  // body therefore has no per-lane `live` branch at all.
  long long trc = live ? traj : N - 1;
  int nlive = (int)((N - traj0) < 32 ? (N - traj0) : 32);
  const uint32_t par_mask = (1u << CDK_IN_F) | (1u << CDK_IN_L) | (1u << CDK_IN_QC) | (1u << CDK_IN_H) |
                            (1u << CDK_IN_D) | (1u << CDK_IN_R);
  const bool par_batched = (a.d.batched_mask & par_mask) != 0;
  // log-likelihood-only calls (output_fields = []) skip the staging stores and the output flush altogether
  const bool any_out = a.out[CDK_OUT_FM] || a.out[CDK_OUT_FP] || a.out[CDK_OUT_PM] || a.out[CDK_OUT_PP];
  const bool use_tma = sizeof(T) == 8 && maps.use_tma != 0 && any_out;
  unsigned long long* const trace = g_lw_trace;
  const unsigned long long t_entry = trace ? globaltimer() : 0ull;
  if (par_batched || lane == 0) {
    T* par = par_batched ? parbase + lane * NPAR : parbase;
    const long long tj = par_batched ? trc : 0;
    const T* th = a.in[CDK_IN_F] + tj * a.in_stride[CDK_IN_F];
    const T* Lm = a.in[CDK_IN_L] + tj * a.in_stride[CDK_IN_L];
    const T* Qc = a.in[CDK_IN_QC] + tj * a.in_stride[CDK_IN_QC];
    const T* H = a.in[CDK_IN_H] + tj * a.in_stride[CDK_IN_H];
    const T* dv = a.in[CDK_IN_D] + tj * a.in_stride[CDK_IN_D];
    const T* R = a.in[CDK_IN_R] + tj * a.in_stride[CDK_IN_R];
    for (int i = 0; i < NTH; ++i) par[i] = th[i];
    for (int i = 0; i < NX; ++i)
      for (int j = i; j < NX; ++j) {
        T acc = T(0);
        for (int p = 0; p < NX; ++p) {
          T lq = T(0);
          for (int q = 0; q < NX; ++q) lq += Lm[i * NX + q] * Qc[q * NX + p];
          acc += lq * Lm[j * NX + p];
        }
        par[NTH + pidx<NX>(i, j)] = acc;
      }
    for (int i = 0; i < NY * NX; ++i) par[NTH + NP + i] = H[i];
    for (int i = 0; i < NY; ++i) par[NTH + NP + NY * NX + i] = dv[i];
    for (int i = 0; i < NY * NY; ++i) par[NTH + NP + NY * NX + NY + i] = R[i];
  }
  const T* Yg = a.in[CDK_IN_Y] ? a.in[CDK_IN_Y] + trc * a.in_stride[CDK_IN_Y] : nullptr;
  const T* Tg = a.in[CDK_IN_T] + trc * a.in_stride[CDK_IN_T];
  // forecast (CDK_FLAG_PREDICT_ONLY): no updates, no observations; Tg holds K + 1 stamps per trajectory, t_init first
  const bool ponly = (a.d.reserved[2] & CDK_FLAG_PREDICT_ONLY) != 0;
  const int KT = ponly ? K + 1 : K;
  int kb = 0, ke = K, kpre = KT;  // the item's step range [kb, ke) and the end of its input prefetches
  auto prefetch = [&](int kk) {
    if (kk < kpre) {
      if (!ponly) {
#pragma unroll
        for (int c = 0; c < NY; ++c) cp_async_elem(&sm.inY[kk & (LW_RING - 1)][c][lane], Yg + (long long)kk * NY + c);
      }
      cp_async_elem(&sm.inT[kk & (LW_RING - 1)][lane], Tg + kk);
    }
    cp_async_commit();
  };
  St<T, NX> s;
  __syncwarp();
  const T* par = par_batched ? parbase + lane * NPAR : parbase;
  // WPC == 14: theta and L Qc L^T stay in registers for the whole kernel; WPC == 7: re-read from shared memory
  T th_r[NTH], lql_r[NP];
#pragma unroll
  for (int i = 0; i < NTH; ++i) th_r[i] = par[i];
#pragma unroll
  for (int i = 0; i < NP; ++i) lql_r[i] = par[NTH + i];
  const T* th = WPC == 7 ? par : th_r;
  const T* lql = WPC == 7 ? par + NTH : lql_r;
  const T* Hs = par + NTH + NP;
  const T* ds = Hs + NY * NX;
  const T* Rs = ds + NY;
  // scalar emission, WPC == 14: the emission row, bias and variance live in registers too (the step body then reads
  // shared memory only for the observation and the two time stamps)
  constexpr bool EM_REGS = NY == 1 && WPC == 14;
  T Hr[NX], dr = T(0), Rr = T(0);
#pragma unroll
  for (int i = 0; i < NX; ++i) Hr[i] = EM_REGS ? Hs[i] : T(0);
  if (EM_REGS) {
    dr = ds[0];
    Rr = Rs[0];
  }
  const T dt0 = T(a.d.dt0);
  const T dtf = T(a.d.dt_final);
  const int max_steps = a.d.max_steps;
  const int num_iter = a.d.num_iter;
  T* __restrict__ LLC = static_cast<T*>(a.out[CDK_OUT_LLCUM]);
  // Scalar emission, one update per observation, no cumulative output: the LEAN update.  sum_k log S_k is kept as
  // (esum, sprod) with prod_k S_k = sprod * 2^esum, sprod renormalised into [1, 2) by integer operations on its exponent
  // field every step, so the whole pass takes ONE log per trajectory (at the end); r^2 / S and the gain use fast_rcp.
  const bool lean = NY == 1 && !LLC && num_iter == 1;
  T ll = T(0), sprod = T(1);
  int esum = 0;
  bool sbad = false;
  int status = 0;
  auto tma_pair = [&](int first, int k0) {  // lane 0: store arrays {first, first + 1} of the block starting at step k0
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    const int c1 = (int)traj0;
    if (first == 0) {
      if (a.out[CDK_OUT_FM]) tma_store_2d(&maps.m[0], &sm.fm[0][0][0], k0 * NX, c1);
      if (a.out[CDK_OUT_FP]) tma_store_2d(&maps.m[1], &sm.fp[0][0][0], k0 * NX * NX, c1);
    } else {
      if (a.out[CDK_OUT_PM]) tma_store_2d(&maps.m[2], &sm.pm[0][0][0], k0 * NX, c1);
      if (a.out[CDK_OUT_PP]) tma_store_2d(&maps.m[3], &sm.pp[0][0][0], k0 * NX * NX, c1);
    }
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  };
  auto poison = [&]() {
    status = 2;
#pragma unroll
    for (int i = 0; i < NX; ++i) s.m[i] = T(NAN);
#pragma unroll
    for (int i = 0; i < NP; ++i) s.P[i] = T(NAN);
  };

  // current mean / full covariance -> this lane's staging rows of step parity `row`
  auto stage = [&](auto rowc, T* mrow, T* prow) {
    constexpr int row = decltype(rowc)::value;
    T full[NX * NX];
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int j = 0; j < NX; ++j) full[i * NX + j] = s.P[pidx<NX>(i, j)];
    stage_row<row, NX>(mrow, s.m);
    stage_row<row, NX * NX>(prow, full);
  };
  // one observation step; `row` (= k & 1, the staging row) is a compile-time constant: the k loop is unrolled by two
  auto step = [&](auto rowc, const int k) {
    constexpr int row = decltype(rowc)::value;
    asm volatile("cp.async.wait_group 1;" ::: "memory");  // own loads of steps <= k+1 have landed
    T y[NY];
#pragma unroll
    for (int c = 0; c < NY; ++c) y[c] = sm.inY[k & (LW_RING - 1)][c][lane];
    const T t0 = sm.inT[k & (LW_RING - 1)][lane];
    const T t1 = k + 1 < KT ? sm.inT[(k + 1) & (LW_RING - 1)][lane] : t0 + dtf;
    if (ponly) {
      // forecast: the state is propagated, never updated
    } else if constexpr (NY == 1) {
      if (lean) {
        // log N(y; H m + d, S) = -r^2 / (2 S) - log(S) / 2 - log(2 pi) / 2,  K = P H^T / (S + 1e-9),  P -= K S K^T
        // (inference_ekf.py:285-289, :153-199; psd_solve boost utils.py:204); the constant is added after the loop
        const T* Hp = EM_REGS ? Hr : Hs;
        const T dd = EM_REGS ? dr : ds[0], RR = EM_REGS ? Rr : Rs[0];
        T HP[NX];
#pragma unroll
        for (int j = 0; j < NX; ++j) {
          T acc = Hp[0] * s.P[pidx<NX>(0, j)];
#pragma unroll
          for (int q = 1; q < NX; ++q) acc = fma(Hp[q], s.P[pidx<NX>(q, j)], acc);
          HP[j] = acc;
        }
        T Sk = RR, hm = dd;
#pragma unroll
        for (int q = 0; q < NX; ++q) {
          Sk = fma(HP[q], Hp[q], Sk);
          hm = fma(Hp[q], s.m[q], hm);
        }
        const T r = y[0] - hm;
        const T iS = fast_rcp(Sk), rb = fast_rcp(Sk + T(1e-9));
        const T rr = r * r;
        T quad = rr * iS;
        quad = fma(fma(-Sk, quad, rr), iS, quad);  // one residual correction: r^2 / S to the last bit or two
        ll = fma(T(-0.5), quad, ll);
        if (!(Sk > T(0)) || !(Sk < T(INFINITY))) sbad = true;  // log() of a non-PD innovation variance is NaN
        sprod *= Sk;
        if constexpr (sizeof(T) == 8) {
          const int hi = __double2hiint(sprod);
          esum += (hi >> 20) - 1023;
          sprod = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(sprod));
        } else {
          const int bits = __float_as_int(sprod);
          esum += (bits >> 23) - 127;
          sprod = __int_as_float((bits & 0x007fffff) | 0x3f800000);
        }
        T Kt[NX];
#pragma unroll
        for (int j = 0; j < NX; ++j) Kt[j] = HP[j] * rb;
#pragma unroll
        for (int i = 0; i < NX; ++i) {
          const T ks = Kt[i] * Sk;
#pragma unroll
          for (int j = i; j < NX; ++j) s.P[pidx<NX>(i, j)] = fma(-ks, Kt[j], s.P[pidx<NX>(i, j)]);
          s.m[i] = fma(Kt[i], r, s.m[i]);
        }
      } else {
        ll += ekf_update<T, NX, NY>(Hs, ds, Rs, s, y, num_iter);
        if (LLC && live) LLC[traj * (long long)K + k] = ll;
      }
    } else {
      ll += ekf_update<T, NX, NY>(Hs, ds, Rs, s, y, num_iter);
      if (LLC && live) LLC[traj * (long long)K + k] = ll;
    }
    prefetch(k + 3);
    if (use_tma && row == 0 && k > kb) {  // the FM/FP store of the previous block was issued ~6 substeps ago
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      __syncwarp();
    }
    if (any_out) stage(rowc, &sm.fm[lane][0][0], &sm.fp[lane][0][0]);
    if (use_tma && row == 1) {  // the filtered rows of this block are complete: store them while the gap is integrated
      __syncwarp();
      if (lane == 0) tma_pair(0, k - 1);
    }
    unsigned ticket = 0;
    if (use_token) {  // warp-uniform spin: every lane polls the same shared-memory word (a broadcast read)
      if (lane == 0) ticket = atomicAdd(const_cast<unsigned*>(tok), 1u);
      ticket = __shfl_sync(0xffffffffu, ticket, 0);
      while ((int)(ticket - tok[1]) >= use_token) {  // use_token = permits: warps inside the substep loop at a time
      }
    }
    {
      // A lane whose gap is already complete takes substeps of length 0, which leave its state bit-identical
      // (y + 0 * ksum), so the substep loop needs no per-lane predication -- its trip count is warp-uniform (vote).
      StepClock<T> clk(t0, t1, dt0);
      while (__any_sync(0xffffffffu, clk.running()) && clk.n < max_steps) {
        rk_step<T, Drift, SOLVER>(th, lql, s, clk.dt());
        clk.advance();
      }
      if (clk.running()) poison();  // diffrax max_steps exceeded: the reference result is NaN
    }
    if (use_token) {
      __syncwarp();
      if (lane == 0) atomicAdd(const_cast<unsigned*>(tok + 1), 1u);
    }
    if (use_tma && row == 0 && k > kb) {  // the PM/PP store of the previous block was issued one whole step ago
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      __syncwarp();
    }
    if (any_out) stage(rowc, &sm.pm[lane][0][0], &sm.pp[lane][0][0]);
    if (any_out && (row == 1 || k == ke - 1)) {
      __syncwarp();
      if (use_tma) {
        if (lane == 0) tma_pair(2, k - 1);
      } else {
        const int k0 = k - row, nrow = row + 1;
#pragma unroll
        for (int arr = 0; arr < 4; ++arr) {
          T* __restrict__ G = static_cast<T*>(
              a.out[arr == 0 ? CDK_OUT_FM : arr == 1 ? CDK_OUT_FP : arr == 2 ? CDK_OUT_PM : CDK_OUT_PP]);
          if (!G) continue;
          const int len = (arr & 1) ? NX * NX : NX;
          const T* src = arr == 0 ? &sm.fm[0][0][0] : arr == 1 ? &sm.fp[0][0][0] : arr == 2 ? &sm.pm[0][0][0] : &sm.pp[0][0][0];
          const int per = nrow * len;
          for (int u = lane; u < nlive * per; u += 32) {
            const int slot = u / per, e = u - slot * per;
            G[((traj0 + slot) * (long long)K + k0) * len + e] = src[slot * 2 * len + e];
          }
        }
        __syncwarp();
      }
    }
  };

  LWGroup<T, NX>* const groups = reinterpret_cast<LWGroup<T, NX>*>(smem_raw + (size_t)W * warp_bytes);  // nseg > 1 only
  for (int base = 0; base < nitems; base += SLICED ? Wr : 1) {
    const int item = SLICED ? base + warp : warp;
    if (!SLICED || (warp < Wr && item < nitems)) {  // (!SLICED: out-of-range warps have returned above)
      const int seg = SLICED ? item / Gc : 0, g = SLICED ? item - seg * Gc : warp;
      traj0 = (gfirst + g) * 32;
      traj = traj0 + lane;
      live = traj < N;
      trc = live ? traj : N - 1;
      nlive = (int)((N - traj0) < 32 ? (N - traj0) : 32);
      Yg = a.in[CDK_IN_Y] ? a.in[CDK_IN_Y] + trc * a.in_stride[CDK_IN_Y] : nullptr;
      Tg = a.in[CDK_IN_T] + trc * a.in_stride[CDK_IN_T];
      kb = seg * segk;
      ke = kb + segk < K ? kb + segk : K;
      kpre = ke + 1 < KT ? ke + 1 : KT;  // step ke - 1 reads the stamp of step ke
      if (SLICED && use_tma && base > 0) {  // this warp's staging rows may still be read by the stores of its previous item
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncwarp();
      }
      prefetch(kb);
      prefetch(kb + 1);
      prefetch(kb + 2);
      if (seg == 0) {
        const T* m0 = a.in[CDK_IN_M0] + trc * a.in_stride[CDK_IN_M0];
        const T* P0 = a.in[CDK_IN_P0] + trc * a.in_stride[CDK_IN_P0];
#pragma unroll
        for (int i = 0; i < NX; ++i) s.m[i] = m0[i];
#pragma unroll
        for (int i = 0; i < NX; ++i)
#pragma unroll
          for (int j = i; j < NX; ++j) s.P[pidx<NX>(i, j)] = P0[i * NX + j];
        ll = T(0);
        sprod = T(1);
        esum = 0;
        sbad = false;
        status = 0;
      } else {
        const LWGroup<T, NX>& gs = groups[g];
#pragma unroll
        for (int i = 0; i < NX; ++i) s.m[i] = gs.m[i][lane];
#pragma unroll
        for (int i = 0; i < NP; ++i) s.P[i] = gs.P[i][lane];
        ll = gs.ll[lane];
        sprod = gs.sprod[lane];
        esum = gs.esum[lane];
        sbad = (gs.flags[lane] & 1) != 0;
        status = gs.flags[lane] >> 8;
      }
      for (int k = kb; k < ke; k += 2) {
        step(std::integral_constant<int, 0>{}, k);
        if (k + 1 < ke) step(std::integral_constant<int, 1>{}, k + 1);
      }
      asm volatile("cp.async.wait_group 0;" ::: "memory");  // the input ring is refilled from the next item's range
      if (seg + 1 < nseg) {
        LWGroup<T, NX>& gs = groups[g];
#pragma unroll
        for (int i = 0; i < NX; ++i) gs.m[i][lane] = s.m[i];
#pragma unroll
        for (int i = 0; i < NP; ++i) gs.P[i][lane] = s.P[i];
        gs.ll[lane] = ll;
        gs.sprod[lane] = sprod;
        gs.esum[lane] = esum;
        gs.flags[lane] = (sbad ? 1 : 0) | (status << 8);
      } else if (live) {
        T llf = ll;
        if (lean) {
          // sum_k log S_k = esum log 2 + log(sprod); the -log(2 pi)/2 of every step
          // (explicit fma / single operations: the sliced and the plain instantiation must round identically)
          const T lsum = fma(T(esum), T(0.69314718055994530942), log(sprod));
          llf = llf - fma(T(0.5), lsum, T(K) * half_log_2pi<T>());
          if (sbad) llf = T(NAN);
        }
        if (a.out[CDK_OUT_LL]) static_cast<T*>(a.out[CDK_OUT_LL])[traj] = llf;
        if (a.out[CDK_OUT_STATUS]) static_cast<int*>(a.out[CDK_OUT_STATUS])[traj] = final_status(status, isfinite(llf));
      }
    }
    if (SLICED) __syncthreads();
  }
  if (use_tma && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  if (trace && lane == 0) {
    unsigned smid, wid;
    asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
    asm volatile("mov.u32 %0, %warpid;" : "=r"(wid));
    unsigned long long* r = trace + 4 * (traj0 >> 5);
    r[0] = t_entry;
    r[1] = globaltimer();
    r[2] = smid;
    r[3] = wid;
  }
}

// ======================================================================================================================
// EKS backward pass for the register-sized drifts (extended_kalman_smoother, inference_ekf.py:450-539 with _smooth
// :363-448): for k = K-2 .. 0, with the Jacobian and the drift frozen at the filtered mean m_f,
//   aux = psd_solve(P_f, L Qc L^T)^T,  G = J(m_f) + aux,
//   d/ds (m_s, P_s) = -( f(m_f) + G (m_s - m_f),  G P_s + P_s G^T - L Qc L^T ),  s in [0, t_{k+1} - t_k]  (reverse_rhs,
//   diffrax_utils.py:13-25), integrated with the caller's fixed-step solver from the smoothed moments of step k + 1.
// Same mapping as ekf_small_lw: one warp = 32 trajectories for the whole kernel, smoothed state, G and the frozen terms in
// registers, gaps run to the warp-wide maximum substep count, warps never synchronise with each other.  The filtered
// moments are read back from HBM through a private 3-deep cp.async ring (12 + 1 values per lane and step, issued two
// steps ahead); the smoothed rows leave through the same two-step staging blocks and TMA tensor stores as the filter's.
// ======================================================================================================================
constexpr int EK_RING = 3;

template <typename T, int NX>
struct alignas(128) EKSmem {
  T sm[32][2][NX];
  alignas(128) T sp[32][2][NX * NX];
  T inM[EK_RING][NX][32];
  T inP[EK_RING][NX * NX][32];
  T inT[EK_RING][32];
};

// generic explicit RK step y <- y + dt * sum_i b_i rhs(y_i) (same accumulation scheme as rk_step)
template <typename T, int NX, int SOLVER, class RHS>
__device__ __forceinline__ void rk_step_fn(St<T, NX>& y, T dt, RHS rhs) {
  using TB = Tab<SOLVER>;
  constexpr int NP = St<T, NX>::NP;
  constexpr int I0 = TB::b(0) != 0.0 ? 0 : (TB::S > 1 && TB::b(1) != 0.0 ? 1 : (TB::S > 2 && TB::b(2) != 0.0 ? 2 : 3));
  St<T, NX> k[TB::S];
  St<T, NX> ksum;
#pragma unroll
  for (int i = 0; i < TB::S; ++i) {
    St<T, NX> yi = y;
#pragma unroll
    for (int j = 0; j < i; ++j) {
      if (TB::a(i, j) != 0.0) {
        const T c = T(TB::a(i, j)) * dt;
#pragma unroll
        for (int e = 0; e < NX; ++e) yi.m[e] = fma(c, k[j].m[e], yi.m[e]);
#pragma unroll
        for (int e = 0; e < NP; ++e) yi.P[e] = fma(c, k[j].P[e], yi.P[e]);
      }
    }
    rhs(yi, k[i]);
    if (i == I0) {
      ksum = k[i];
    } else if (TB::b(i) != 0.0) {
      const T c = T(TB::b(i) / TB::b(I0));
      if (TB::b(i) == TB::b(I0)) {
#pragma unroll
        for (int e = 0; e < NX; ++e) ksum.m[e] += k[i].m[e];
#pragma unroll
        for (int e = 0; e < NP; ++e) ksum.P[e] += k[i].P[e];
      } else {
#pragma unroll
        for (int e = 0; e < NX; ++e) ksum.m[e] = fma(c, k[i].m[e], ksum.m[e]);
#pragma unroll
        for (int e = 0; e < NP; ++e) ksum.P[e] = fma(c, k[i].P[e], ksum.P[e]);
      }
    }
  }
  const T w = T(TB::b(I0)) * dt;
#pragma unroll
  for (int e = 0; e < NX; ++e) y.m[e] = fma(w, ksum.m[e], y.m[e]);
#pragma unroll
  for (int e = 0; e < NP; ++e) y.P[e] = fma(w, ksum.P[e], y.P[e]);
}

template <typename T, class Drift, int SOLVER>
__global__ void __launch_bounds__(32 * 14, 1) eks_small_lw(const KArgs<T> a, const __grid_constant__ V5Maps maps) {
  constexpr int NX = Drift::NX;
  constexpr int NP = St<T, NX>::NP;
  constexpr int NTH = Drift::NTHETA;
  using S = EKSmem<T, NX>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  S& sm = *reinterpret_cast<S*>(smem_raw + (size_t)warp * sizeof(S));
  const long long N = a.d.N;
  const int K = a.d.K;
  const long long traj0 = (long long)blockIdx.x * blockDim.x + warp * 32;  // 1..14 warps per CTA (launch_eks_one)
  if (traj0 >= N) return;
  const long long traj = traj0 + lane;
  const bool live = traj < N;
  const int nlive = (int)((N - traj0) < 32 ? (N - traj0) : 32);
  const bool use_tma = sizeof(T) == 8 && maps.use_tma != 0;
  const long long tl = live ? traj : 0;

  // model constants, per lane (a leading N on any parameter is simply this lane's block)
  T th[NTH], lql[NP];
  {
    const T* thg = a.in[CDK_IN_F] + tl * a.in_stride[CDK_IN_F];
    const T* Lm = a.in[CDK_IN_L] + tl * a.in_stride[CDK_IN_L];
    const T* Qc = a.in[CDK_IN_QC] + tl * a.in_stride[CDK_IN_QC];
#pragma unroll
    for (int i = 0; i < NTH; ++i) th[i] = thg[i];
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int j = i; j < NX; ++j) {
        T acc = T(0);
        for (int p = 0; p < NX; ++p) {
          T lq = T(0);
          for (int q = 0; q < NX; ++q) lq += Lm[i * NX + q] * Qc[q * NX + p];
          acc += lq * Lm[j * NX + p];
        }
        lql[pidx<NX>(i, j)] = acc;
      }
  }
  const T* __restrict__ FMg = a.in[CDK_IN_FM] + tl * a.in_stride[CDK_IN_FM];
  const T* __restrict__ FPg = a.in[CDK_IN_FP] + tl * a.in_stride[CDK_IN_FP];
  const T* __restrict__ Tg = a.in[CDK_IN_T] + tl * a.in_stride[CDK_IN_T];
  T* const SMg = static_cast<T*>(a.out[CDK_OUT_SM]);
  T* const SPg = static_cast<T*>(a.out[CDK_OUT_SP]);
  auto prefetch = [&](int kk) {  // filtered moments and time stamp of step kk -> ring slot kk % EK_RING
    if (live && kk >= 0) {
      const int r = kk % EK_RING;
#pragma unroll
      for (int i = 0; i < NX; ++i) cp_async_elem(&sm.inM[r][i][lane], FMg + (long long)kk * NX + i);
#pragma unroll
      for (int i = 0; i < NX * NX; ++i) cp_async_elem(&sm.inP[r][i][lane], FPg + (long long)kk * NX * NX + i);
      cp_async_elem(&sm.inT[r][lane], Tg + kk);
    }
    cp_async_commit();
  };
  prefetch(K - 1);
  prefetch(K - 2);
  prefetch(K - 3);
  const T dt0 = T(a.d.dt0);
  const int max_steps = a.d.max_steps;
  int status = 0;

  auto tma_store = [&](int k0) {  // lane 0: store the two-step block starting at the (even) step k0
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tma_store_2d(&maps.m[0], &sm.sm[0][0][0], k0 * NX, (int)traj0);
    tma_store_2d(&maps.m[1], &sm.sp[0][0][0], k0 * NX * NX, (int)traj0);
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  };
  auto flush_generic = [&](int k0, int nrow) {  // fp32 / odd K / unaligned outputs: cooperative copy of rows [k0, k0 + nrow)
#pragma unroll
    for (int arr = 0; arr < 2; ++arr) {
      T* __restrict__ G = arr == 0 ? SMg : SPg;
      const int len = arr ? NX * NX : NX;
      const T* src = arr ? &sm.sp[0][0][0] : &sm.sm[0][0][0];
      const int per = nrow * len, off = (k0 & 1) * len;
      for (int u = lane; u < nlive * per; u += 32) {
        const int slot = u / per, e = u - slot * per;
        G[((traj0 + slot) * (long long)K + k0) * len + e] = src[slot * 2 * len + off + e];
      }
    }
    __syncwarp();
  };
  auto stage = [&](int row, const St<T, NX>& v) {
    T full[NX * NX];
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int j = 0; j < NX; ++j) full[i * NX + j] = v.P[pidx<NX>(i, j)];
    if (row == 0) {
      stage_row<0, NX>(&sm.sm[lane][0][0], v.m);
      stage_row<0, NX * NX>(&sm.sp[lane][0][0], full);
    } else {
      stage_row<1, NX>(&sm.sm[lane][0][0], v.m);
      stage_row<1, NX * NX>(&sm.sp[lane][0][0], full);
    }
  };

  // step K-1: smoothed = filtered (:466-470 / :813-814 in the linear twin)
  St<T, NX> s;
  T t1 = T(0);
  asm volatile("cp.async.wait_group 2;" ::: "memory");
  __syncwarp();
  if (live) {
    const int r = (K - 1) % EK_RING;
#pragma unroll
    for (int i = 0; i < NX; ++i) s.m[i] = sm.inM[r][i][lane];
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int j = i; j < NX; ++j) s.P[pidx<NX>(i, j)] = sm.inP[r][i * NX + j][lane];
    t1 = sm.inT[r][lane];
    // the reference copies the filtered covariance verbatim: keep its lower triangle too
    T full[NX * NX];
#pragma unroll
    for (int i = 0; i < NX * NX; ++i) full[i] = sm.inP[r][i][lane];
    if (((K - 1) & 1) == 0) {
      stage_row<0, NX>(&sm.sm[lane][0][0], s.m);
      stage_row<0, NX * NX>(&sm.sp[lane][0][0], full);
    } else {
      stage_row<1, NX>(&sm.sm[lane][0][0], s.m);
      stage_row<1, NX * NX>(&sm.sp[lane][0][0], full);
    }
  } else {
#pragma unroll
    for (int i = 0; i < NX; ++i) s.m[i] = T(0);
#pragma unroll
    for (int i = 0; i < NP; ++i) s.P[i] = T(0);
  }
  __syncwarp();
  if (((K - 1) & 1) == 0) {  // odd K: the last row is a block of its own (never the TMA path)
    flush_generic(K - 1, 1);
  }

  for (int k = K - 2; k >= 0; --k) {
    const int row = k & 1;
    prefetch(k - 2);
    asm volatile("cp.async.wait_group 2;" ::: "memory");  // own loads of step k have landed
    __syncwarp();
    if (live) {
      const int r = k % EK_RING;
      T mf[NX], Pf[NX][NX];
#pragma unroll
      for (int i = 0; i < NX; ++i) mf[i] = sm.inM[r][i][lane];
#pragma unroll
      for (int i = 0; i < NX; ++i)
#pragma unroll
        for (int j = 0; j < NX; ++j) Pf[i][j] = sm.inP[r][i * NX + j][lane];
      const T t0 = sm.inT[r][lane];
      // psd_solve(P_f, L Qc L^T): Cholesky of sym(P_f) + 1e-9 I (utils.py:202-207), three right-hand sides
      T Lc[NX][NX], inv[NX];
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        T sjj = T(0.5) * (Pf[j][j] + Pf[j][j]) + T(1e-9);
#pragma unroll
        for (int q = 0; q < j; ++q) sjj -= Lc[j][q] * Lc[j][q];
        const T dj = sqrt(sjj);
        Lc[j][j] = dj;
        inv[j] = T(1) / dj;
#pragma unroll
        for (int i = j + 1; i < NX; ++i) {
          T v = T(0.5) * (Pf[i][j] + Pf[j][i]);
#pragma unroll
          for (int q = 0; q < j; ++q) v -= Lc[i][q] * Lc[j][q];
          Lc[i][j] = v * inv[j];
        }
      }
      T G[NX][NX];
      Drift::jac(th, mf, G);
#pragma unroll
      for (int c = 0; c < NX; ++c) {  // column c of X = (P_f + eps I)^-1 L Qc L^T;  aux = X^T
        T w[NX], x[NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) {
          T v = lql[pidx<NX>(i, c)];
#pragma unroll
          for (int q = 0; q < i; ++q) v -= Lc[i][q] * w[q];
          w[i] = v * inv[i];
        }
#pragma unroll
        for (int i = NX - 1; i >= 0; --i) {
          T v = w[i];
#pragma unroll
          for (int q = i + 1; q < NX; ++q) v -= Lc[q][i] * x[q];
          x[i] = v * inv[i];
        }
#pragma unroll
        for (int i = 0; i < NX; ++i) G[c][i] += x[i];
      }
      T c0[NX];
      Drift::f(th, mf, c0);
      auto rhs = [&](const St<T, NX>& y, St<T, NX>& kk) {
        T GP[NX][NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) {
          T acc = c0[i];
#pragma unroll
          for (int q = 0; q < NX; ++q) acc = fma(G[i][q], y.m[q] - mf[q], acc);
          kk.m[i] = -acc;
#pragma unroll
          for (int j = 0; j < NX; ++j) {
            T g = T(0);
#pragma unroll
            for (int q = 0; q < NX; ++q) g = fma(G[i][q], y.P[pidx<NX>(q, j)], g);
            GP[i][j] = g;
          }
        }
#pragma unroll
        for (int i = 0; i < NX; ++i)
#pragma unroll
          for (int j = i; j < NX; ++j) kk.P[pidx<NX>(i, j)] = lql[pidx<NX>(i, j)] - (GP[i][j] + GP[j][i]);
      };
      const T span = t1 - t0;  // integrate s from 0 to t_{k+1} - t_k
      StepClock<T> clk(T(0), span, dt0);
      while (clk.running() && clk.n < max_steps) {
        rk_step_fn<T, NX, SOLVER>(s, clk.dt(), rhs);
        clk.advance();
      }
      if (clk.running()) {  // diffrax max_steps exceeded: NaN, as in the reference
        status = 2;
#pragma unroll
        for (int i = 0; i < NX; ++i) s.m[i] = T(NAN);
#pragma unroll
        for (int i = 0; i < NP; ++i) s.P[i] = T(NAN);
      }
      t1 = t0;
    }
    if (use_tma && row == 1) {  // the block (k-1, k) is about to be rewritten: its predecessor (k+1, k+2) must have been read
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      __syncwarp();
    }
    if (live) stage(row, s);
    __syncwarp();
    if (use_tma) {
      if (row == 0 && lane == 0) tma_store(k);
    } else if (row == 0 || k == 0) {
      const int nrow = (k + 1 < K && row == 0) ? 2 : 1;
      flush_generic(k, nrow);
    }
  }
  if (use_tma && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  cp_async_wait_all();
  if (live && a.out[CDK_OUT_STATUS]) {
    bool bad = false;
#pragma unroll
    for (int i = 0; i < NX; ++i) bad |= !isfinite(s.m[i]);
    merge_smoother_status(static_cast<int*>(a.out[CDK_OUT_STATUS]), traj, status, !bad);
  }
}

// ======================================================================================================================
// d log-likelihood / d theta for the register CD-EKF (SURVEY section 8f rank 1: what jax.value_and_grad of
// marginal_log_prob gives the reference's fit_sgd, src/utils/optimize_utils.py:102) -- FORWARD mode, drift parameters.
// Tangent of the moment ODE (inference_ekf.py:76-123) w.r.t. theta_p:  m' and P' obey
//   dm'/dt = J m' + df/dtheta_p,   dP'/dt = J' P + J P' + (J' P + J P')^T,   J' = (dJ/dm)[m'] + dJ/dtheta_p,
// and an explicit RK step of the augmented system (m, P, m', P') IS the derivative of the RK step of (m, P) (the step
// sizes do not depend on theta), so the result is the exact derivative of the discrete filter the forward kernels run.
// Tangent of the scalar-emission update (:153-199, :285-289) with S = H P H^T + R, r = y - H m - d, K = P H^T / (S + 1e-9):
//   l' = -r r'/S + (r^2/S^2 - 1/S) S'/2,   K' = (P' H^T) / (S + eps) - K S' / (S + eps),
//   m+' = m' + K' r + K r',   P+' = P' - (K' S K^T + K S' K^T + K S K'^T).
// One lane per trajectory, one launch per parameter (the base filter is recomputed: 18 doubles of state instead of 36).
// ======================================================================================================================
template <typename T, int NE, int SOLVER, class RHS>
__device__ __forceinline__ void rk_step_flat(T (&y)[NE], T dt, RHS rhs) {
  using TB = Tab<SOLVER>;
  constexpr int I0 = TB::b(0) != 0.0 ? 0 : (TB::S > 1 && TB::b(1) != 0.0 ? 1 : (TB::S > 2 && TB::b(2) != 0.0 ? 2 : 3));
  T k[TB::S][NE], ksum[NE];
#pragma unroll
  for (int i = 0; i < TB::S; ++i) {
    T yi[NE];
#pragma unroll
    for (int e = 0; e < NE; ++e) yi[e] = y[e];
#pragma unroll
    for (int j = 0; j < i; ++j) {
      if (TB::a(i, j) != 0.0) {
        const T c = T(TB::a(i, j)) * dt;
#pragma unroll
        for (int e = 0; e < NE; ++e) yi[e] = fma(c, k[j][e], yi[e]);
      }
    }
    rhs(yi, k[i]);
    if (i == I0) {
#pragma unroll
      for (int e = 0; e < NE; ++e) ksum[e] = k[i][e];
    } else if (TB::b(i) != 0.0) {
      const T c = T(TB::b(i) / TB::b(I0));
#pragma unroll
      for (int e = 0; e < NE; ++e) ksum[e] = fma(c, k[i][e], ksum[e]);
    }
  }
  const T w = T(TB::b(I0)) * dt;
#pragma unroll
  for (int e = 0; e < NE; ++e) y[e] = fma(w, ksum[e], y[e]);
}

// Direction of differentiation = (kind, idx): CDK_GRAD_THETA idx 0..2 (sigma, rho, beta); CDK_GRAD_LQL / CDK_GRAD_P0
// idx = packed upper-triangle index of the SYMMETRIC matrix L Qc L^T / P0 (an off-diagonal direction moves both mirror
// entries); CDK_GRAD_R, CDK_GRAD_D (scalar emission); CDK_GRAD_H, CDK_GRAD_M0 idx 0..2.  Column `col` of grad.
enum { CDK_GRAD_THETA = 0, CDK_GRAD_LQL, CDK_GRAD_R, CDK_GRAD_D, CDK_GRAD_H, CDK_GRAD_M0, CDK_GRAD_P0 };

template <int SOLVER>
__global__ void __launch_bounds__(128) ekf_l63_grad_kernel(const KArgs<double> a, const int kind, const int idx,
                                                             double* __restrict__ grad, const int grad_stride, const int col) {
  using T = double;
  constexpr int NX = 3, NP = 6, NE = 2 * (NX + NP);
  const long long N = a.d.N;
  const int K = a.d.K;
  const long long traj = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (traj >= N) return;
  T th[3], lql[NP], H[NX];
  {
    const T* thg = a.in[CDK_IN_F] + traj * a.in_stride[CDK_IN_F];
    const T* Lm = a.in[CDK_IN_L] + traj * a.in_stride[CDK_IN_L];
    const T* Qc = a.in[CDK_IN_QC] + traj * a.in_stride[CDK_IN_QC];
    const T* Hg = a.in[CDK_IN_H] + traj * a.in_stride[CDK_IN_H];
#pragma unroll
    for (int i = 0; i < 3; ++i) th[i] = thg[i];
#pragma unroll
    for (int i = 0; i < NX; ++i) H[i] = Hg[i];
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int j = i; j < NX; ++j) {
        T acc = T(0);
#pragma unroll
        for (int q = 0; q < NX; ++q) {
          T lq = T(0);
#pragma unroll
          for (int r = 0; r < NX; ++r) lq += Lm[i * NX + r] * Qc[r * NX + q];
          acc += lq * Lm[j * NX + q];
        }
        lql[pidx<NX>(i, j)] = acc;
      }
  }
  const T dv = (a.in[CDK_IN_D] + traj * a.in_stride[CDK_IN_D])[0];
  const T R = (a.in[CDK_IN_R] + traj * a.in_stride[CDK_IN_R])[0];
  const T* __restrict__ Y = a.in[CDK_IN_Y] + traj * a.in_stride[CDK_IN_Y];
  const T* __restrict__ Tm = a.in[CDK_IN_T] + traj * a.in_stride[CDK_IN_T];
  // y = [m (3) | P (6) | m' (3) | P' (6)]
  T y[NE];
  {
    const T* m0 = a.in[CDK_IN_M0] + traj * a.in_stride[CDK_IN_M0];
    const T* P0 = a.in[CDK_IN_P0] + traj * a.in_stride[CDK_IN_P0];
#pragma unroll
    for (int i = 0; i < NX; ++i) y[i] = m0[i];
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int j = i; j < NX; ++j) y[NX + pidx<NX>(i, j)] = P0[i * NX + j];
#pragma unroll
    for (int e = NX + NP; e < NE; ++e) y[e] = T(0);
#pragma unroll
    for (int e = 0; e < NX; ++e)
      if (kind == CDK_GRAD_M0 && idx == e) y[NX + NP + e] = T(1);
#pragma unroll
    for (int e = 0; e < NP; ++e)
      if (kind == CDK_GRAD_P0 && idx == e) y[NX + NP + NX + e] = T(1);
  }
  const bool wrt_theta = kind == CDK_GRAD_THETA;
  const T ds = wrt_theta && idx == 0 ? T(1) : T(0), dr = wrt_theta && idx == 1 ? T(1) : T(0),
          db = wrt_theta && idx == 2 ? T(1) : T(0);
  const T dR = kind == CDK_GRAD_R ? T(1) : T(0), dd = kind == CDK_GRAD_D ? T(1) : T(0);
  T dH[NX], dlql[NP];
#pragma unroll
  for (int i = 0; i < NX; ++i) dH[i] = (kind == CDK_GRAD_H && idx == i) ? T(1) : T(0);
#pragma unroll
  for (int i = 0; i < NP; ++i) dlql[i] = (kind == CDK_GRAD_LQL && idx == i) ? T(1) : T(0);
  auto rhs = [&](const T (&u)[NE], T (&k)[NE]) {
    T m[NX] = {u[0], u[1], u[2]}, mt[NX] = {u[9], u[10], u[11]};
    T P[NP], Pt[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      P[i] = u[NX + i];
      Pt[i] = u[NX + NP + NX + i];
    }
    T f[NX], G[NX][NX], G2[NX][NX];
    DriftL63::f(th, m, f);
    DriftL63::jp(th, m, P, G);    // J P
    DriftL63::jp(th, m, Pt, G2);  // J P'
    // f' = J m' + df/dtheta_p
    const T ft0 = th[0] * (mt[1] - mt[0]) + ds * (m[1] - m[0]);
    const T ft1 = (th[1] - m[2]) * mt[0] - mt[1] - m[0] * mt[2] + dr * m[0];
    const T ft2 = m[1] * mt[0] + m[0] * mt[1] - th[2] * mt[2] - db * m[2];
    // J' P,  J' = [[-ds, ds, 0], [dr - z', 0, -x'], [y', x', -db]]
#pragma unroll
    for (int j = 0; j < NX; ++j) {
      const T p0 = P[pidx<NX>(0, j)], p1 = P[pidx<NX>(1, j)], p2 = P[pidx<NX>(2, j)];
      G2[0][j] += ds * (p1 - p0);
      G2[1][j] += (dr - mt[2]) * p0 - mt[0] * p2;
      G2[2][j] += mt[1] * p0 + mt[0] * p1 - db * p2;
    }
    k[0] = f[0]; k[1] = f[1]; k[2] = f[2];
    k[9] = ft0; k[10] = ft1; k[11] = ft2;
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
      for (int j = i; j < NX; ++j) {
        k[NX + pidx<NX>(i, j)] = (G[i][j] + G[j][i]) + lql[pidx<NX>(i, j)];
        k[NX + NP + NX + pidx<NX>(i, j)] = (G2[i][j] + G2[j][i]) + dlql[pidx<NX>(i, j)];
      }
  };
  const T dt0 = T(a.d.dt0), dtf = T(a.d.dt_final);
  const int max_steps = a.d.max_steps;
  T ll = T(0), llt = T(0);
  T t0 = Tm[0];
  for (int k = 0; k < K; ++k) {
    // ---- measurement update and its tangent (H' = dH, R' = dR, d' = dd are the parameter seeds) ----
    T HP[NX], HPt[NX];
#pragma unroll
    for (int j = 0; j < NX; ++j) {
      T acc = T(0), acct = T(0);
#pragma unroll
      for (int q = 0; q < NX; ++q) {
        acc += H[q] * y[NX + pidx<NX>(q, j)];
        acct += H[q] * y[NX + NP + NX + pidx<NX>(q, j)] + dH[q] * y[NX + pidx<NX>(q, j)];
      }
      HP[j] = acc;
      HPt[j] = acct;  // (H P)' = H P' + H' P
    }
    T S = R, St = dR, hm = dv, hmt = dd;
#pragma unroll
    for (int q = 0; q < NX; ++q) {
      S += HP[q] * H[q];
      St += HPt[q] * H[q] + HP[q] * dH[q];  // S' = (H P)' H^T + H P H'^T + R'
      hm += H[q] * y[q];
      hmt += H[q] * y[NX + NP + q] + dH[q] * y[q];
    }
    const T r = Y[k] - hm, rt = -hmt;
    const T iS = T(1) / S;
    ll += T(-0.5) * (r * r * iS) - T(0.5) * log(S) - half_log_2pi<T>();
    llt += -(r * rt * iS) + T(0.5) * (r * r * iS * iS - iS) * St;
    const T rb = T(1) / (S + T(1e-9));
    T Kg[NX], Kt[NX];
#pragma unroll
    for (int j = 0; j < NX; ++j) {
      Kg[j] = HP[j] * rb;
      Kt[j] = HPt[j] * rb - Kg[j] * St * rb;
    }
#pragma unroll
    for (int i = 0; i < NX; ++i) {
#pragma unroll
      for (int j = i; j < NX; ++j) {
        y[NX + NP + NX + pidx<NX>(i, j)] -= Kt[i] * S * Kg[j] + Kg[i] * St * Kg[j] + Kg[i] * S * Kt[j];
        y[NX + pidx<NX>(i, j)] -= Kg[i] * S * Kg[j];
      }
      y[NX + NP + i] += Kt[i] * r + Kg[i] * rt;
      y[i] += Kg[i] * r;
    }
    // ---- predict across the gap (diffrax stepping rule) ----
    const T t1 = k + 1 < K ? Tm[k + 1] : t0 + dtf;
    StepClock<T> clk(t0, t1, dt0);
    while (clk.running() && clk.n < max_steps) {
      rk_step_flat<T, NE, SOLVER>(y, clk.dt(), rhs);
      clk.advance();
    }
    if (clk.running()) {
#pragma unroll
      for (int e = 0; e < NE; ++e) y[e] = T(NAN);
    }
    t0 = t1;
  }
  if (a.out[CDK_OUT_LL]) static_cast<T*>(a.out[CDK_OUT_LL])[traj] = ll;
  grad[traj * grad_stride + col] = llt;
}

// ======================================================================================================================
// REVERSE mode: every column of d log-likelihood / d parameters in ONE backward launch (SURVEY section 8f rank 1; what
// jax.value_and_grad(marginal_log_prob) hands fit_sgd, src/utils/optimize_utils.py:102).  The forward filter
// (ekf_small_lw) has written the filtered and predicted moments of every step to HBM; this kernel walks k = K-1 .. 0 with
// the adjoint (am, AP) of the state:
//   gap k (k < K-1; the last predict does not enter the likelihood): re-integrate from (m_f, P_f)_k keeping the start state
//     of every substep (up to GR_CKPT of them in thread-local memory, otherwise recomputed from the gap start), then step
//     backwards through the substeps; each RK step is differentiated stage by stage,
//       cot(k_i) = b_i dt lam+ + dt sum_{j>i} a_ji lam(y_j),   lam(y_i) = VJP_rhs(y_i)[cot(k_i)],   lam = lam+ + sum_i lam(y_i),
//     with the closed-form VJP of the moment right-hand side (f(m), J P + P J^T + L Qc L^T) below;
//   update k: the scalar-emission update differentiated by hand (see the comments in the code).
// Adjoint covariances are FULL-matrix entry-wise gradients kept symmetric (packed upper triangle); the output columns use
// the convention of the forward-mode kernel: an off-diagonal column of a symmetric parameter moves both mirror entries,
// i.e. it is twice the packed entry.  One lane per trajectory; cost ~4 filter passes for all 23 columns (forward mode: one
// launch of ~2.2 filter passes per column).
// ======================================================================================================================
constexpr int GR_CKPT = 8;

struct GradAcc {
  double th[3], lql[6], R, d, H[3];
};

// VJP of the moment rhs at (m, P) with cotangent (cm, C): adds to (vm, V) and to the parameter accumulators.
__device__ __forceinline__ void l63_rhs_vjp(const double* th, const double (&m)[3], const double (&P)[6], const double (&cm)[3],
                                            const double (&C)[6], double (&vm)[3], double (&V)[6], GradAcc& g) {
  const double s = th[0], rz = th[1] - m[2], b = th[2], x = m[0], y = m[1], z = m[2];
  // J = [[-s, s, 0], [rz, -1, -x], [y, x, -b]];  full symmetric views of C and P
  const double C00 = C[0], C01 = C[1], C02 = C[2], C11 = C[3], C12 = C[4], C22 = C[5];
  const double P00 = P[0], P01 = P[1], P02 = P[2], P11 = P[3], P12 = P[4], P22 = P[5];
  // W = J^T C:  W_ab = sum_i J_ia C_ib;  dL/dP = W + W^T
  const double W00 = -s * C00 + rz * C01 + y * C02, W01 = -s * C01 + rz * C11 + y * C12, W02 = -s * C02 + rz * C12 + y * C22;
  const double W10 = s * C00 - C01 + x * C02, W11 = s * C01 - C11 + x * C12, W12 = s * C02 - C12 + x * C22;
  const double W20 = -x * C01 - b * C02, W21 = -x * C11 - b * C12, W22 = -x * C12 - b * C22;
  V[0] += 2.0 * W00;
  V[1] += W01 + W10;
  V[2] += W02 + W20;
  V[3] += 2.0 * W11;
  V[4] += W12 + W21;
  V[5] += 2.0 * W22;
  // M = C P (only the entries the sparse dJ/dm, dJ/dtheta touch):  dL/dJ = 2 M
  const double M00 = C00 * P00 + C01 * P01 + C02 * P02, M01 = C00 * P01 + C01 * P11 + C02 * P12;
  const double M10 = C01 * P00 + C11 * P01 + C12 * P02, M12 = C01 * P02 + C11 * P12 + C12 * P22;
  const double M20 = C02 * P00 + C12 * P01 + C22 * P02, M21 = C02 * P01 + C12 * P11 + C22 * P12, M22 = C02 * P02 + C12 * P12 + C22 * P22;
  // mean: Jf^T cm + <dJ/dm, 2 M>   (J10 = rho - z, J12 = -x, J20 = y, J21 = x)
  vm[0] += -s * cm[0] + rz * cm[1] + y * cm[2] + 2.0 * (M21 - M12);
  vm[1] += s * cm[0] - cm[1] + x * cm[2] + 2.0 * M20;
  vm[2] += -x * cm[1] - b * cm[2] - 2.0 * M10;
  // parameters: df/dtheta^T cm + <dJ/dtheta, 2 M>;  d(L Qc L^T) enters dP entry-wise
  g.th[0] += (y - x) * cm[0] + 2.0 * (M01 - M00);
  g.th[1] += x * cm[1] + 2.0 * M10;
  g.th[2] += -z * cm[2] - 2.0 * M22;
#pragma unroll
  for (int e = 0; e < 6; ++e) g.lql[e] += C[e];
}

template <int SOLVER>
__device__ __forceinline__ void l63_rk_step_vjp(const double* th, const double* lql, const St<double, 3>& y, const double dt,
                                                St<double, 3>& lam, GradAcc& g) {
  using TB = Tab<SOLVER>;
  constexpr int S = TB::S;
  St<double, 3> yi[S], k[S];
  // forward: stage inputs and increments (rhs WITHOUT dt, as rk_step)
#pragma unroll
  for (int i = 0; i < S; ++i) {
    yi[i] = y;
#pragma unroll
    for (int j = 0; j < i; ++j)
      if (TB::a(i, j) != 0.0) {
        const double c = TB::a(i, j) * dt;
#pragma unroll
        for (int e = 0; e < 3; ++e) yi[i].m[e] = fma(c, k[j].m[e], yi[i].m[e]);
#pragma unroll
        for (int e = 0; e < 6; ++e) yi[i].P[e] = fma(c, k[j].P[e], yi[i].P[e]);
      }
    ekf_rhs<double, DriftL63>(th, lql, yi[i], k[i]);
  }
  // backward
  St<double, 3> ly[S];
  St<double, 3> out = lam;
#pragma unroll
  for (int i = S - 1; i >= 0; --i) {
    double cm[3], C[6];
#pragma unroll
    for (int e = 0; e < 3; ++e) cm[e] = TB::b(i) * dt * lam.m[e];
#pragma unroll
    for (int e = 0; e < 6; ++e) C[e] = TB::b(i) * dt * lam.P[e];
#pragma unroll
    for (int j = i + 1; j < S; ++j)
      if (TB::a(j, i) != 0.0) {
        const double c = TB::a(j, i) * dt;
#pragma unroll
        for (int e = 0; e < 3; ++e) cm[e] = fma(c, ly[j].m[e], cm[e]);
#pragma unroll
        for (int e = 0; e < 6; ++e) C[e] = fma(c, ly[j].P[e], C[e]);
      }
#pragma unroll
    for (int e = 0; e < 3; ++e) ly[i].m[e] = 0.0;
#pragma unroll
    for (int e = 0; e < 6; ++e) ly[i].P[e] = 0.0;
    l63_rhs_vjp(th, yi[i].m, yi[i].P, cm, C, ly[i].m, ly[i].P, g);
#pragma unroll
    for (int e = 0; e < 3; ++e) out.m[e] += ly[i].m[e];
#pragma unroll
    for (int e = 0; e < 6; ++e) out.P[e] += ly[i].P[e];
  }
  lam = out;
}

template <int SOLVER>
__global__ void __launch_bounds__(128) ekf_l63_grad_rev_kernel(const KArgs<double> a, const double* __restrict__ FMg,
                                                                 const double* __restrict__ FPg, const double* __restrict__ PMg,
                                                                 const double* __restrict__ PPg, double* __restrict__ grad) {
  constexpr int NX = 3;
  const long long N = a.d.N;
  const int K = a.d.K;
  const long long traj = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (traj >= N) return;
  double th[3], lql[6], H[3];
  {
    const double* thg = a.in[CDK_IN_F] + traj * a.in_stride[CDK_IN_F];
    const double* Lm = a.in[CDK_IN_L] + traj * a.in_stride[CDK_IN_L];
    const double* Qc = a.in[CDK_IN_QC] + traj * a.in_stride[CDK_IN_QC];
    const double* Hg = a.in[CDK_IN_H] + traj * a.in_stride[CDK_IN_H];
    for (int i = 0; i < 3; ++i) th[i] = thg[i];
    for (int i = 0; i < 3; ++i) H[i] = Hg[i];
    for (int i = 0; i < NX; ++i)
      for (int j = i; j < NX; ++j) {
        double acc = 0.0;
        for (int q = 0; q < NX; ++q) {
          double lq = 0.0;
          for (int r = 0; r < NX; ++r) lq += Lm[i * NX + r] * Qc[r * NX + q];
          acc += lq * Lm[j * NX + q];
        }
        lql[pidx<NX>(i, j)] = acc;
      }
  }
  const double dv = (a.in[CDK_IN_D] + traj * a.in_stride[CDK_IN_D])[0];
  const double R = (a.in[CDK_IN_R] + traj * a.in_stride[CDK_IN_R])[0];
  const double* __restrict__ Y = a.in[CDK_IN_Y] + traj * a.in_stride[CDK_IN_Y];
  const double* __restrict__ Tm = a.in[CDK_IN_T] + traj * a.in_stride[CDK_IN_T];
  const double* fm = FMg + traj * (long long)K * 3;
  const double* fp = FPg + traj * (long long)K * 9;
  const double* pm = PMg + traj * (long long)K * 3;
  const double* pp = PPg + traj * (long long)K * 9;
  const double dt0 = a.d.dt0;
  const int max_steps = a.d.max_steps;
  GradAcc g;
  for (int i = 0; i < 3; ++i) g.th[i] = g.H[i] = 0.0;
  for (int i = 0; i < 6; ++i) g.lql[i] = 0.0;
  g.R = g.d = 0.0;
  St<double, 3> lam;  // adjoint of the PREDICTED state entering update k+1 (zero beyond the last observation)
  for (int i = 0; i < 3; ++i) lam.m[i] = 0.0;
  for (int i = 0; i < 6; ++i) lam.P[i] = 0.0;
  auto load_state = [&](const double* mrow, const double* prow, St<double, 3>& s) {
    for (int i = 0; i < 3; ++i) s.m[i] = mrow[i];
    for (int i = 0; i < 3; ++i)
      for (int j = i; j < 3; ++j) s.P[pidx<3>(i, j)] = prow[i * 3 + j];
  };
  for (int k = K - 1; k >= 0; --k) {
    if (k < K - 1) {
      // ---- predict over [t_k, t_{k+1}], backwards ----
      St<double, 3> y0;
      load_state(fm + (long long)k * 3, fp + (long long)k * 9, y0);
      const double t0 = Tm[k], t1 = Tm[k + 1];
      // number of substeps; the time grid does not depend on the state
      StepClock<double> count(t0, t1, dt0);
      while (count.running() && count.n < max_steps) count.advance();
      const int q = count.n;
      // start state of substep i for i % stride == 0 (i / stride < GR_CKPT) is kept; the others are re-integrated
      const int stride = (q + GR_CKPT - 1) / GR_CKPT > 0 ? (q + GR_CKPT - 1) / GR_CKPT : 1;
      St<double, 3> ck[GR_CKPT];
      {
        St<double, 3> s = y0;
        StepClock<double> clk(t0, t1, dt0);
        for (int i = 0; i < q; ++i) {
          if (i % stride == 0) ck[i / stride] = s;
          rk_step<double, DriftL63, SOLVER>(th, lql, s, clk.dt());
          clk.advance();
        }
      }
      for (int i = q - 1; i >= 0; --i) {
        // (tprev, tnext) and the start state of substep i
        const int base = (i / stride) * stride;
        StepClock<double> clk(t0, t1, dt0);
        for (int u = 0; u < base; ++u) clk.advance();
        St<double, 3> s = ck[i / stride];
        for (int u = base; u < i; ++u) {
          rk_step<double, DriftL63, SOLVER>(th, lql, s, clk.dt());
          clk.advance();
        }
        l63_rk_step_vjp<SOLVER>(th, lql, s, clk.dt(), lam, g);
      }
    }
    // ---- update k, backwards.  Forward (ekf_update, scalar emission):  HP = H P, S = HP.H + R, r = y - H.m - d,
    //      ll = -r^2 / (2 S) - log(S) / 2 - c,  rb = 1 / (S + 1e-9),  K = HP rb,  P_f = P - S K K^T,  m_f = m + K r ----
    St<double, 3> sp;  // the predicted state that entered the update
    if (k == 0) {
      const double* m0 = a.in[CDK_IN_M0] + traj * a.in_stride[CDK_IN_M0];
      const double* P0 = a.in[CDK_IN_P0] + traj * a.in_stride[CDK_IN_P0];
      load_state(m0, P0, sp);
    } else {
      load_state(pm + (long long)(k - 1) * 3, pp + (long long)(k - 1) * 9, sp);
    }
    double Pf[3][3];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) Pf[i][j] = sp.P[pidx<3>(i, j)];
    double HP[3], S = R, hm = dv;
    for (int j = 0; j < 3; ++j) HP[j] = H[0] * Pf[0][j] + H[1] * Pf[1][j] + H[2] * Pf[2][j];
    for (int q2 = 0; q2 < 3; ++q2) {
      S += HP[q2] * H[q2];
      hm += H[q2] * sp.m[q2];
    }
    const double r = Y[k] - hm, iS = 1.0 / S, rb = 1.0 / (S + 1e-9);
    double Kg[3];
    for (int j = 0; j < 3; ++j) Kg[j] = HP[j] * rb;
    // adjoints in: lam.m = dL/dm_f, lam.P = dL/dP_f (full-matrix, symmetric)
    double A[3][3];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) A[i][j] = lam.P[pidx<3>(i, j)];
    double AK[3];  // A K
    for (int i = 0; i < 3; ++i) AK[i] = A[i][0] * Kg[0] + A[i][1] * Kg[1] + A[i][2] * Kg[2];
    double aK[3], a_r = 0.0, a_S = 0.0;
    // m_f = m + K r
    for (int i = 0; i < 3; ++i) {
      aK[i] = lam.m[i] * r;
      a_r += Kg[i] * lam.m[i];
    }
    // P_f = P - S K K^T
    a_S -= Kg[0] * AK[0] + Kg[1] * AK[1] + Kg[2] * AK[2];
    for (int i = 0; i < 3; ++i) aK[i] -= 2.0 * S * AK[i];
    // K = HP rb
    double aHP[3], a_rb = 0.0;
    for (int j = 0; j < 3; ++j) {
      aHP[j] = aK[j] * rb;
      a_rb += HP[j] * aK[j];
    }
    a_S -= rb * rb * a_rb;  // rb = 1 / (S + eps)
    // ll_k
    a_r += -r * iS;
    a_S += 0.5 * r * r * iS * iS - 0.5 * iS;
    // r = y - hm, hm = H.m + d
    const double a_hm = -a_r;
    g.d += a_hm;
    // S = HP.H + R
    g.R += a_S;
    for (int j = 0; j < 3; ++j) {
      aHP[j] += a_S * H[j];
      g.H[j] += a_S * HP[j] + a_hm * sp.m[j];
    }
    // HP_j = sum_i H_i P_ij
    for (int i = 0; i < 3; ++i) g.H[i] += Pf[i][0] * aHP[0] + Pf[i][1] * aHP[1] + Pf[i][2] * aHP[2];
    // adjoint of the predicted state: dL/dm = lam.m + H a_hm;  dL/dP = A + sym(H aHP^T)
    for (int i = 0; i < 3; ++i) lam.m[i] += H[i] * a_hm;
    for (int i = 0; i < 3; ++i)
      for (int j = i; j < 3; ++j) lam.P[pidx<3>(i, j)] += 0.5 * (H[i] * aHP[j] + H[j] * aHP[i]);
  }
  // ---- columns: theta 3 | LQL packed 6 | R | d | H 3 | m0 3 | P0 packed 6 (off-diagonals of symmetric parameters: both
  //      mirror entries move, i.e. twice the symmetric entry-wise gradient) ----
  double* out = grad + traj * CDK_GRAD_COLS_L63;
  for (int i = 0; i < 3; ++i) out[i] = g.th[i];
  const bool offd[6] = {false, true, true, false, true, false};
  for (int e = 0; e < 6; ++e) out[3 + e] = offd[e] ? 2.0 * g.lql[e] : g.lql[e];
  out[9] = g.R;
  out[10] = g.d;
  for (int i = 0; i < 3; ++i) out[11 + i] = g.H[i];
  for (int i = 0; i < 3; ++i) out[14 + i] = lam.m[i];
  for (int e = 0; e < 6; ++e) out[17 + e] = offd[e] ? 2.0 * lam.P[e] : lam.P[e];
}

typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

encode_tiled_fn get_encode_tiled() {
  static encode_tiled_fn fn = []() -> encode_tiled_fn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<encode_tiled_fn>(p);
  }();
  return fn;
}

// Warps per CTA for a batch of N trajectories: the smallest count that still fits the batch into one wave of
// `ctas_per_sm` CTAs per SM (so the warps spread over every SM and sub-partition), at most `max_warps`.
// CDK_LW_WARPS=k forces k (experiments).
int lw_num_sms() {
  static const int num_sms = []() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1)
      n = 148;
    return n;
  }();
  return num_sms;
}

int lw_warps_per_cta(long long N, int max_warps, int ctas_per_sm) {
  static const int forced = []() {
    const char* e = getenv("CDK_LW_WARPS");
    return e ? atoi(e) : 0;
  }();
  if (forced >= 1) return forced < max_warps ? forced : max_warps;
  const long long nwarps = (N + 31) / 32, slots = (long long)lw_num_sms() * ctas_per_sm;
  const long long w = (nwarps + slots - 1) / slots;
  return (int)(w < 1 ? 1 : (w > max_warps ? max_warps : w));
}

// Build the four output tensor maps.  Returns false when the TMA path does not apply (fp32, odd K, unaligned pointers,
// CDK_EKF_TMA=0): the kernel then uses the cooperative-copy flush.
template <typename T>
bool make_maps(const KArgs<T>& a, int NX, int box_rows, V5Maps& maps, const int* slot_list = nullptr) {
  memset(&maps, 0, sizeof(maps));
  static const bool disabled = []() {
    const char* e = getenv("CDK_EKF_TMA");
    return e && e[0] == '0';
  }();
  if (disabled || sizeof(T) != 8 || (a.d.K & 1) || a.d.N > 0x7fffffffLL) return false;
  encode_tiled_fn enc = get_encode_tiled();
  if (!enc) return false;
  const int default_slots[4] = {CDK_OUT_FM, CDK_OUT_FP, CDK_OUT_PM, CDK_OUT_PP};
  const int* slots = slot_list ? slot_list : default_slots;  // even entries: [N][K][NX] arrays, odd: [N][K][NX*NX]
  for (int i = 0; i < 4; ++i) {
    if (slots[i] < 0) continue;
    void* ptr = a.out[slots[i]];
    if (!ptr) continue;
    if (reinterpret_cast<uintptr_t>(ptr) & 15) return false;
    const cuuint64_t len = (i & 1) ? NX * NX : NX;
    const cuuint64_t gdim[2] = {len * (cuuint64_t)a.d.K, (cuuint64_t)a.d.N};
    const cuuint64_t gstr[1] = {len * (cuuint64_t)a.d.K * sizeof(T)};
    const cuuint32_t box[2] = {(cuuint32_t)(2 * len), (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(&maps.m[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return false;
  }
  maps.use_tma = 1;
  return true;
}

template <typename T, class Drift, int NY, int SOLVER>
int launch_one(const KArgs<T>& a, cudaStream_t s) {
  constexpr int NX = Drift::NX;
  constexpr int NPAR = Drift::NTHETA + NX * (NX + 1) / 2 + NY * NX + NY + NY * NY;
  using SW = LWSmem<T, NX, NY>;
  const uint32_t par_mask = (1u << CDK_IN_F) | (1u << CDK_IN_L) | (1u << CDK_IN_QC) | (1u << CDK_IN_H) |
                            (1u << CDK_IN_D) | (1u << CDK_IN_R);
  const bool par_batched = (a.d.batched_mask & par_mask) != 0;
  if (a.d.N == 0) return CDK_OK;
  // Kernel variant: 14 = ONE CTA per SM of up to 14 warps (drift parameters in registers), or -- CDK_LW_WPC=7, and always
  // when every lane carries its own parameter block in shared memory -- two CTAs per SM of up to 7 warps.
  static const int wpc_env = []() {
    const char* e = getenv("CDK_LW_WPC");
    return e && atoi(e) == 7 ? 7 : 14;
  }();
  const int warp_bytes = (int)((sizeof(SW) + sizeof(T) * NPAR * (par_batched ? 32 : 1) + 127) & ~size_t(127));
  const int wpc = (size_t)warp_bytes * wpc_env > 227 * 1024 ? 7 : wpc_env;
  // Occupancy-aware geometry: a trajectory is a serial chain of K steps, so what matters for a batch smaller than one
  // full wave (148 SMs x 14 warps x 32 = 66,304 trajectories) is that its ceil(N / 32) warps spread over ALL SMs and all
  // four sub-partitions of each -- N / 8 = 8,192 trajectories (the 8-GPU shard of BASELINE config 3) are 256 warps, i.e.
  // 128 CTAs of 2 warps instead of 19 CTAs of 14.  Warps never synchronise with each other, so the kernel is the same.
  int warps = lw_warps_per_cta(a.d.N, wpc, wpc == 7 ? 2 : 1);
  int nout = 0;
  for (int slot : {CDK_OUT_FM, CDK_OUT_FP, CDK_OUT_PM, CDK_OUT_PP}) nout += a.out[slot] != nullptr;
  static const bool forced = getenv("CDK_LW_WARPS") != nullptr;
  const long long nwarps = (a.d.N + 31) / 32;
  // Time slicing (see the kernel): when the batch is more than one BALANCED wave -- 12 resident warps per SM, three per
  // sub-partition, or 8 when all four moment arrays are written (the scattered 48 / 144-byte output rows of more warps cap
  // the pass at ~1.8 TB/s of DRAM writes; measured balanced rates in profiles/r02_c3_outputs_probe.jsonl: 12.0 / 9.5
  // trajectories per us with 12 warps, 11.3 / 10.6 with 8, log-likelihood only / all outputs) -- every SM gets
  // G = ceil(groups / SMs) groups of 32 trajectories and works through them in K-segments of 50 steps.  CDK_LW_SLICE=0
  // disables, CDK_LW_SLICE=w forces w resident warps.
  // (read at every launch, not cached: the tests switch them; CDK_LW_SLICE_SMS pretends a smaller GPU so that a small batch
  // takes the sliced path)
  const char* slice_e = getenv("CDK_LW_SLICE");
  const int slice_env = slice_e ? atoi(slice_e) : -1;
  const char* sms_e = getenv("CDK_LW_SLICE_SMS");
  const char* segk_e = getenv("CDK_LW_SEGK");  // segment length (even); default: chosen below
  const int segk_env = segk_e && atoi(segk_e) >= 2 ? (atoi(segk_e) & ~1) : 50;
  int G = warps, segk = a.d.K > 0 ? a.d.K : 1;
  size_t smw = (size_t)warp_bytes * warps;
  long long wblocks = (a.d.N + 32 * warps - 1) / (32 * warps);
  const bool ponly_l = (a.d.reserved[2] & CDK_FLAG_PREDICT_ONLY) != 0;
  bool sliced = false;
  if (!forced && slice_env != 0 && wpc == 14 && !par_batched && !ponly_l && a.d.K >= 200 && (a.d.K & 1) == 0) {
    const int sms = sms_e && atoi(sms_e) > 0 ? atoi(sms_e) : lw_num_sms();
    for (int wres : {slice_env > 0 ? slice_env : (nout >= 3 ? 8 : 12), 8}) {
      if (wres < 1 || wres > 12 || nwarps <= (long long)sms * wres) continue;
      const long long Gs = (nwarps + sms - 1) / sms;
      const size_t need = (size_t)warp_bytes * wres + (size_t)Gs * sizeof(LWGroup<T, NX>);
      if (Gs < wres || need > 227 * 1024) continue;
      warps = wres;
      G = (int)Gs;
      // segment length: the pass costs ceil(G nseg / W) rounds of segk steps; fewest total steps, then fewest segments
      // (every item pays a barrier and a refill of its input ring: 250-step segments measured 3 % faster than 50-step ones)
      segk = segk_env;
      if (!segk_e) {
        long long best = -1;
        for (int ns = 2; ns <= 24; ++ns) {
          const int sk = (((a.d.K + ns - 1) / ns) + 1) & ~1;
          const int nsr = (a.d.K + sk - 1) / sk;  // segments this length really gives
          const long long cost = ((Gs * nsr + wres - 1) / wres) * sk;
          if (best < 0 || cost < best) {
            best = cost;
            segk = sk;
          }
        }
      }
      smw = need;
      wblocks = (nwarps + Gs - 1) / Gs;
      sliced = true;
      break;
    }
  }
  if (!sliced) {
    // CTAs of 8 warps instead of 14 when all four moment arrays are written and the batch is about one full wave (only
    // reached when slicing is off): 6.93 ms against 7.30 ms at N = 65,536.  Two such CTAs share an SM, so 108 SMs carry
    // 16 warps -- four per sub-partition, balanced -- and 40 carry 8, where 14 warps per SM put (4, 4, 3, 3) warps on the
    // sub-partitions of every SM.
    if (!forced && wpc == 14 && warps > 8 && nout >= 3 && nwarps > 1761 && nwarps <= 2368) warps = 8;
    G = warps;
    smw = (size_t)warp_bytes * warps;
    wblocks = (a.d.N + 32 * warps - 1) / (32 * warps);
  }
  if (wblocks > 2147483647LL) return CDK_E_SIZE;
  V5Maps maps;
  make_maps<T>(a, NX, 32, maps);
  auto kw = wpc == 7 ? ekf_small_lw<T, Drift, NY, SOLVER, 7>
                     : (sliced ? ekf_small_lw<T, Drift, NY, SOLVER, 14, true> : ekf_small_lw<T, Drift, NY, SOLVER, 14>);
  {
    const size_t cap = (size_t)warp_bytes * wpc > smw ? (size_t)warp_bytes * wpc : smw;
    if (cap > 48 * 1024 && cudaFuncSetAttribute(kw, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(ekf_small_lw)");
  }
  static const int token_env = []() {  // experiment, default off (see the kernel)
    const char* e = getenv("CDK_LW_TOKEN");
    return e ? atoi(e) : 0;
  }();
  const int use_token = wpc == 14 ? token_env : 0;  // with two CTAs per SM the lock would have to span CTAs
  kw<<<(unsigned)wblocks, 32 * warps, smw, s>>>(a, maps, warp_bytes, use_token, G, segk);
  note_launch();
  return check_launch("ekf_small_lw");
}

template <typename T, class Drift, int NY>
int launch_solver(const KArgs<T>& a, cudaStream_t s) {
  switch (a.d.solver) {
    case CDK_RK4: return launch_one<T, Drift, NY, CDK_RK4>(a, s);
    case CDK_DOPRI5: return launch_one<T, Drift, NY, CDK_DOPRI5>(a, s);
    case CDK_EULER: return launch_one<T, Drift, NY, CDK_EULER>(a, s);
    case CDK_HEUN: return launch_one<T, Drift, NY, CDK_HEUN>(a, s);
  }
  return CDK_E_UNSUPPORTED;
}

template <typename T, class Drift>
int launch_ny(const KArgs<T>& a, cudaStream_t s) {
  switch (a.d.m) {
    case 1: return launch_solver<T, Drift, 1>(a, s);
    case 2: return launch_solver<T, Drift, 2>(a, s);
    case 3: return launch_solver<T, Drift, 3>(a, s);
  }
  return CDK_E_UNSUPPORTED;
}

template <typename T, class Drift, int SOLVER>
int launch_eks_one(const KArgs<T>& a, cudaStream_t s) {
  constexpr int NX = Drift::NX;
  using S = EKSmem<T, NX>;
  if (a.d.N == 0) return CDK_OK;
  const int warps = lw_warps_per_cta(a.d.N, 14, 1);  // same occupancy-aware geometry as the filter
  const long long blocks = (a.d.N + 32 * warps - 1) / (32 * warps);
  if (blocks > 2147483647LL) return CDK_E_SIZE;
  V5Maps maps;
  const int slots[4] = {CDK_OUT_SM, CDK_OUT_SP, -1, -1};
  make_maps<T>(a, NX, 32, maps, slots);
  const size_t smem = sizeof(S) * warps;
  auto kern = eks_small_lw<T, Drift, SOLVER>;
  if (sizeof(S) * 14 > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(S) * 14)) != cudaSuccess)
    return check_launch("cudaFuncSetAttribute(eks_small_lw)");
  kern<<<(unsigned)blocks, 32 * warps, smem, s>>>(a, maps);
  note_launch();
  return check_launch("eks_small_lw");
}

}  // namespace

// Fast path coverage: EKF filter, state_order first/second, Lorenz-63 (n = 3), m <= 3, solvers rk4/dopri5/euler/heun.
template <typename T>
int launch_ekf_small(const KArgs<T>& a, cudaStream_t s) {
  const cdk_desc& d = a.d;
  // the fast path is written for h(x) = H x + d; any other emission runs in the generic kernel
  if (d.state_order == CDK_ORDER_ZEROTH || d.emission_id != CDK_EMISSION_LINEAR) return CDK_E_UNSUPPORTED;
  if (d.drift_id == CDK_DRIFT_LORENZ63 && d.n == 3) return launch_ny<T, DriftL63>(a, s);
  return CDK_E_UNSUPPORTED;
}

int set_lw_trace(void* devbuf) {
  unsigned long long* p = static_cast<unsigned long long*>(devbuf);
  return cudaMemcpyToSymbol(g_lw_trace, &p, sizeof(p)) == cudaSuccess ? CDK_OK : CDK_E_CUDA;
}

// Gradient of the Lorenz-63 CD-EKF log-likelihood (scalar emission, num_iter 1, state_order first / second):
// grad [N, 23], columns = theta (3) | L Qc L^T packed (6) | R | d | H (3) | m0 (3) | P0 packed (6); `groups` (bit g = group g
// in that order, 0 = theta only) selects which columns are computed (the others are left untouched).
int launch_ekf_l63_grad(const KArgs<double>& a, double* grad, cudaStream_t s) {
  const cdk_desc& d = a.d;
  if (d.drift_id != CDK_DRIFT_LORENZ63 || d.n != 3 || d.m != 1 || d.num_iter != 1 || d.state_order == CDK_ORDER_ZEROTH)
    return CDK_E_UNSUPPORTED;
  if (d.N == 0) return CDK_OK;
  const long long blocks = (d.N + 127) / 128;
  if (blocks > 2147483647LL) return CDK_E_SIZE;
  if (a.out[CDK_OUT_SCRATCH] && (d.reserved[3] & CDK_GRAD_REVERSE)) {
    // reverse mode: forward filter into the scratch block (FM | FP | PM | PP, N*K*24 doubles), then ONE backward launch
    double* sc = static_cast<double*>(a.out[CDK_OUT_SCRATCH]);
    const long long NK = d.N * (long long)d.K;
    KArgs<double> f = a;
    f.d.reserved[3] = 0;
    f.out[CDK_OUT_FM] = sc;
    f.out[CDK_OUT_FP] = sc + NK * 3;
    f.out[CDK_OUT_PM] = sc + NK * 12;
    f.out[CDK_OUT_PP] = sc + NK * 15;
    f.out[CDK_OUT_LLCUM] = nullptr;
    f.out[CDK_OUT_GRAD] = nullptr;
    f.out[CDK_OUT_SCRATCH] = nullptr;
    int rc = launch_ekf_small<double>(f, s);
    if (rc != CDK_OK) return rc;
    const double *FM = sc, *FP = sc + NK * 3, *PM = sc + NK * 12, *PP = sc + NK * 15;
    switch (d.solver) {
      case CDK_RK4: ekf_l63_grad_rev_kernel<CDK_RK4><<<(unsigned)blocks, 128, 0, s>>>(a, FM, FP, PM, PP, grad); break;
      case CDK_DOPRI5: ekf_l63_grad_rev_kernel<CDK_DOPRI5><<<(unsigned)blocks, 128, 0, s>>>(a, FM, FP, PM, PP, grad); break;
      case CDK_EULER: ekf_l63_grad_rev_kernel<CDK_EULER><<<(unsigned)blocks, 128, 0, s>>>(a, FM, FP, PM, PP, grad); break;
      case CDK_HEUN: ekf_l63_grad_rev_kernel<CDK_HEUN><<<(unsigned)blocks, 128, 0, s>>>(a, FM, FP, PM, PP, grad); break;
      default: return CDK_E_UNSUPPORTED;
    }
    note_launch();
    return check_launch("ekf_l63_grad_rev_kernel");
  }
  const int groups = (d.reserved[3] & 127) ? (d.reserved[3] & 127) : 1;
  static const int kinds[7] = {CDK_GRAD_THETA, CDK_GRAD_LQL, CDK_GRAD_R, CDK_GRAD_D, CDK_GRAD_H, CDK_GRAD_M0, CDK_GRAD_P0};
  static const int count[7] = {3, 6, 1, 1, 3, 3, 6};
  int col = 0;
  for (int g = 0; g < 7; ++g) {
    for (int idx = 0; idx < count[g]; ++idx, ++col) {
      if (!((groups >> g) & 1)) continue;
      switch (d.solver) {
        case CDK_RK4: ekf_l63_grad_kernel<CDK_RK4><<<(unsigned)blocks, 128, 0, s>>>(a, kinds[g], idx, grad, CDK_GRAD_COLS_L63, col); break;
        case CDK_DOPRI5: ekf_l63_grad_kernel<CDK_DOPRI5><<<(unsigned)blocks, 128, 0, s>>>(a, kinds[g], idx, grad, CDK_GRAD_COLS_L63, col); break;
        case CDK_EULER: ekf_l63_grad_kernel<CDK_EULER><<<(unsigned)blocks, 128, 0, s>>>(a, kinds[g], idx, grad, CDK_GRAD_COLS_L63, col); break;
        case CDK_HEUN: ekf_l63_grad_kernel<CDK_HEUN><<<(unsigned)blocks, 128, 0, s>>>(a, kinds[g], idx, grad, CDK_GRAD_COLS_L63, col); break;
        default: return CDK_E_UNSUPPORTED;
      }
      note_launch();
    }
  }
  return check_launch("ekf_l63_grad_kernel");
}

// EKS backward pass fast path: Lorenz-63, solvers rk4 / dopri5 / euler / heun (anything else: generic_smooth_kernel).
template <typename T>
int launch_eks_small(const KArgs<T>& a, cudaStream_t s) {
  const cdk_desc& d = a.d;
  static const bool disabled = []() {
    const char* e = getenv("CDK_EKS_FAST");
    return e && e[0] == '0';
  }();
  if (disabled || d.drift_id != CDK_DRIFT_LORENZ63 || d.n != 3 || d.emission_id != CDK_EMISSION_LINEAR) return CDK_E_UNSUPPORTED;
  switch (d.solver) {
    case CDK_RK4: return launch_eks_one<T, DriftL63, CDK_RK4>(a, s);
    case CDK_DOPRI5: return launch_eks_one<T, DriftL63, CDK_DOPRI5>(a, s);
    case CDK_EULER: return launch_eks_one<T, DriftL63, CDK_EULER>(a, s);
    case CDK_HEUN: return launch_eks_one<T, DriftL63, CDK_HEUN>(a, s);
  }
  return CDK_E_UNSUPPORTED;
}

template int launch_eks_small<double>(const KArgs<double>&, cudaStream_t);
template int launch_eks_small<float>(const KArgs<float>&, cudaStream_t);
template int launch_ekf_small<double>(const KArgs<double>&, cudaStream_t);
template int launch_ekf_small<float>(const KArgs<float>&, cudaStream_t);

}  // namespace cdk
