// cdk_generic.cu -- shared-memory kernels for arbitrary (runtime) state / emission dimensions: ONE CTA PER TRAJECTORY.
//
// Covers, for n <= CDK_MAX_N, m <= CDK_MAX_M and every solver in the registry:
//   ALGO_KF_FILTER   cdlgssm_filter            cd_linear/inference.py:555-632 (+ compute_pushforward :105-144,
//                                               _predict :185-206, _condition_on :209-259)
//   ALGO_KF_SMOOTH   cdlgssm_smoother scan     cd_linear/inference.py:746-794 (+ _smooth :636-690)
//   ALGO_EKF_FILTER  extended_kalman_filter    cd_nonlinear/inference_ekf.py:202-326 (all three state orders)
//   ALGO_EKF_SMOOTH  extended_kalman_smoother  cd_nonlinear/inference_ekf.py:450-539 (+ _smooth :363-448)
//   ALGO_UKF_FILTER  unscented_kalman_filter   cd_nonlinear/inference_ukf.py:206-308
// The whole per-trajectory state (moments, RK stage vectors, Jacobian, Cholesky factors) lives in shared memory
// (up to ~200 KB of the 227 KB a B200 CTA may use); the threads of the CTA split every small matrix product by
// output element.  Matrices are stored with an odd leading dimension so that row-strided accesses (Cholesky,
// triangular solves, A B^T products) are bank-conflict free for 64-bit words.
#include <stdlib.h>

#include "cdk_dense.cuh"

namespace cdk {
namespace {

enum { ODE_PUSH = 0, ODE_EKF = 1, ODE_MEAN = 2, ODE_BACK = 3, ODE_UKF = 4, ODE_UKFC = 5 };

// Drifts whose Jacobian is a fixed sparse stencil evaluated on the fly (no n x n Jacobian buffer, no dense J P product)
__host__ __device__ inline bool stencil_drift(int id) { return id == CDK_DRIFT_LORENZ63 || id == CDK_DRIFT_LORENZ96; }
// The UKF runs in closed form (see ode_rhs, ODE_UKFC) unless the caller asks for literal sigma points
// (and always for a user-defined drift, which need not be a polynomial of degree <= 2)
__host__ __device__ inline bool ukf_closed(const cdk_desc& d) {
  return !(d.reserved[2] & CDK_FLAG_UKF_SIGMA_POINTS) && d.drift_id != CDK_DRIFT_USER;
}

// shared-memory layout, computed identically on host (size) and device (offsets); units = elements of T
struct Lay {
  int n, m, du, ldn, ldm, nn, S, nth, mpoff;
  int TH, LQL, H, R, DV, BV, BU, DU, YV, UV, MU, P, ODEY, YS, ACC, KS, J, W1, W2, W3, SM, SL, RV, MF, PF, C0, PHI, YP, total;
  Lay() = default;
  // reg_ode: the launcher has chosen the register-resident stencil ODE (ode_solve_stencil), so the shared-memory RHS and its
  // Jacobian buffer are never used by this launch
  __host__ __device__ Lay(const cdk_desc& d, int algo, int nslots, bool reg_ode = false) {
    n = d.n; m = d.m; du = d.d_u; ldn = ldp(n); ldm = ldp(m); nn = n * ldn;
    const bool lin = algo == ALGO_KF_FILTER || algo == ALGO_KF_SMOOTH;
    const bool smooth = algo == ALGO_KF_SMOOTH || algo == ALGO_EKF_SMOOTH;
    const bool ukf = algo == ALGO_UKF_FILTER;
    const bool ukfc = ukf && ukf_closed(d);
    const bool ekf_reg = algo == ALGO_EKF_FILTER && reg_ode;
    nth = lin ? nn : ((ukf || ekf_reg) ? d.n_theta : (d.n_theta > nn ? d.n_theta : nn));
    const int mx = n > m ? n : m;
    const int wsz = mx * ldp(mx);
    mpoff = (n + 1) & ~1;           // offset of P behind MU inside the (m, P) ODE state
    const int S_mp = mpoff + nn;
    S = lin ? (2 * nn > S_mp ? 2 * nn : S_mp) : S_mp;  // kf smoother type 2 integrates (m, P) as well
    int o = 0;
    auto take = [&](int cnt) { int r = o; o += (cnt + 1) & ~1; return r; };
    TH = take(nth); LQL = take(nn); H = take(m * ldn); R = take(m * ldm); DV = take(m); BV = take(n);
    BU = take(n * du); DU = take(m * du); YV = take(m); UV = take(du);
    MU = take(n); P = take(nn);  // contiguous: [MU | P] is the (m, P) ODE state (n is padded to even by take())
    ODEY = take(lin ? 2 * nn : 0);
    YS = take(S); ACC = take(S); KS = take(nslots * S);
    if ((ukfc || ekf_reg) && nslots == 1 && m <= n && stencil_drift(d.drift_id)) {
      // closed-form UKF (or the EKF on the register-resident stencil ODE), stencil Jacobian, chain tableau: the RHS needs
      // no scratch at all (J P is formed in the output block and symmetrised in place) and the update's three [m x n]
      // scratch matrices are only live while the ODE stage buffers are not -- 84 KB for n = 40, m = 20: two CTAs per SM.
      J = KS; W1 = YS; W2 = KS; W3 = ACC;
    } else if (ukf && !ukfc && nslots == 1 && m <= n) {
      // sigma-point UKF with a chain tableau: 110 KB instead of 164 KB for n = 40, m = 20, so that TWO trajectories share
      // an SM.  J (the factor of P inside the update) and W3 (update / model-load scratch) are only live while the ODE
      // stage buffers are not, so they alias KS and ACC; the RHS needs neither (see ode_rhs).
      J = KS; W1 = take(wsz); W2 = take(wsz); W3 = ACC;
    } else {
      J = take(nn); W1 = take(wsz); W2 = take(wsz); W3 = take(wsz);
    }
    SM = take(m * ldm); SL = take(m * ldm); RV = take(2 * m);
    MF = take(smooth ? n : 0); PF = take(smooth ? nn : 0); C0 = take(n);
    // user emission: its parameters phi, and (UKF) the 2n + 1 sigma points pushed through h, [2n + 1] x ldm
    PHI = take(emission_params(d)); YP = take(ukf && user_emission(d) ? (2 * n + 1) * ldm : 0);
    total = o;
  }
};

template <typename T>
struct GArgs {
  KArgs<T> k;
  RtTab tab;
  int nslots;  // RK stage buffers kept in shared memory (1 for "chain" tableaux, S otherwise)
  int algo;
  int reg_ode;  // allow the register-resident Lorenz-96 moment ODE (ode_solve_stencil)
  Lay lay;      // computed once on the host: the offsets are then constant-bank operands, not ~40 integer instructions
                // the compiler re-derives from (n, m) wherever a register is short
};

template <typename T>
struct Ctx {
  const GArgs<T>& g;
  const Lay& L;
  T* sh;
  __device__ Ctx(const GArgs<T>& g_, T* sh_) : g(g_), L(g_.lay), sh(sh_) {}
  __device__ T* p(int off) const { return sh + off; }
};

// (J(x) P)[r][c] for the stencil drifts, straight from x and P (4 / 3 terms per entry instead of a length-n dot product)
template <typename T>
__device__ __forceinline__ T stencil_jp(int id, const T* th, int n, int r, int c, const T* x, const T* P, int ld) {
  if (id == CDK_DRIFT_LORENZ96) {
    const int ip = r + 1 == n ? 0 : r + 1, im1 = r == 0 ? n - 1 : r - 1, im2 = im1 == 0 ? n - 1 : im1 - 1;
    return x[im1] * (P[ip * ld + c] - P[im2 * ld + c]) + (x[ip] - x[im2]) * P[im1 * ld + c] - P[r * ld + c];
  }
  const T p0 = P[c], p1 = P[ld + c], p2 = P[2 * ld + c];  // Lorenz-63: J = [[-s, s, 0], [r - z, -1, -x], [y, x, -b]]
  if (r == 0) return th[0] * (p1 - p0);
  if (r == 1) return (th[1] - x[2]) * p0 - p1 - x[0] * p2;
  return x[1] * p0 + x[0] * p1 - th[2] * p2;
}

// k = dt * rhs(kind, ys).  All arrays in shared memory.  Ends with a barrier.
template <typename T>
__device__ void ode_rhs(const Ctx<T>& c, int kind, const T* ys, T* k, T dt) {
  const Lay& L = c.L;
  const int n = L.n, ld = L.ldn;
  const cdk_desc& d = c.g.k.d;
  const T* lql = c.p(L.LQL);
  if (kind == ODE_PUSH) {
    // dA = F A ; dQ = F Q + Q F^T + L Qc L^T   (cd_linear/inference.py:114-131)
    const T* F = c.p(L.TH);
    const T* A = ys;
    const T* Q = ys + L.nn;
    T* FQ = c.p(L.W1);
    mm_dmma<T, false, false>(F, ld, A, ld, n, n, n, [&](int i, int j, double v) { k[i * ld + j] = dt * (T)v; });
    mm_dmma<T, false, false>(F, ld, Q, ld, n, n, n, [&](int i, int j, double v) { FQ[i * ld + j] = (T)v; });
    __syncthreads();
    FOR_T(e, n * n) {  // Q F^T = (F Q)^T for the symmetric Q
      const int i = e / n, j = e - i * n;
      k[L.nn + i * ld + j] = dt * ((FQ[i * ld + j] + FQ[j * ld + i]) + lql[i * ld + j]);
    }
    __syncthreads();
    return;
  }
  if (kind == ODE_MEAN) {
    const T* th = c.p(L.TH);
    FOR_T(i, n) k[i] = dt * drift_f<T>(d.drift_id, th, n, i, [&](int j) { return ys[j]; });
    __syncthreads();
    return;
  }
  const T* mm = ys;
  const T* P = ys + L.P - L.MU;  // same relative offset as [MU | P]
  T* km = k;
  T* kP = k + (L.P - L.MU);
  if (kind == ODE_EKF) {
    // inference_ekf.py:76-123
    const T* th = c.p(L.TH);
    T* J = c.p(L.J);
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      J[i * ld + j] = drift_jac<T>(d.drift_id, th, n, i, j, mm);
    }
    __syncthreads();
    const bool second = d.state_order == CDK_ORDER_SECOND && (d.drift_id == CDK_DRIFT_QUADRATIC || d.drift_id == CDK_DRIFT_USER);
    FOR_T(i, n) {
      T f = drift_f<T>(d.drift_id, th, n, i, [&](int j) { return mm[j]; });
      if (second) {
        T s = T(0);
#if CDK_HAS_USER_DRIFT
        if (d.drift_id == CDK_DRIFT_USER) {
          for (int q = 0; q < n; ++q) s += cdk_user::graddiv<T>(th, n, q, mm) * P[q * ld + i];
        } else
#endif
        for (int q = 0; q < n; ++q) s += drift_graddiv<T>(d.drift_id, th, n, q) * P[q * ld + i];
        f += T(0.5) * s;
      }
      km[i] = dt * f;
    }
    T* JP = c.p(L.W1);
    mm_dmma<T, false, false>(J, ld, P, ld, n, n, n, [&](int i, int j, double v) { JP[i * ld + j] = (T)v; });
    __syncthreads();
    FOR_T(e, n * n) {  // P J^T = (J P)^T for the symmetric P
      const int i = e / n, j = e - i * n;
      kP[i * ld + j] = dt * ((JP[i * ld + j] + JP[j * ld + i]) + lql[i * ld + j]);
    }
    __syncthreads();
    return;
  }
  if (kind == ODE_UKFC) {
    // The sigma-point moment ODE (Sarkka eq. 3.183, inference_ukf.py:130-152) in CLOSED FORM.  Every drift of the registry
    // is a polynomial of degree <= 2, f(m + d) = f(m) + J d + B(d, d) exactly, and the sigma set is symmetric
    // (X_i^+- = m +- c L_i, L L^T = P, w = 1 / (2 (n + lambda)), c^2 = n + lambda), so
    //   sum_k w_m[k] f(X_k)                      = f(m) + sum_i B(L_i, L_i) = f(m) + 0.5 tr(Hess f . P)
    //   sum_k w_c[k] (f(X_k) - fbar)(X_k - m)^T  = w c sum_i (2 c J L_i) L_i^T = J P
    // hold in exact arithmetic: the unscented predict of these models is dm = f(m) + 0.5 tr(Hess P),
    // dP = J P + P J^T + L Qc L^T -- no Cholesky factorisation of P at every RK stage (18 per observation-step of BASELINE
    // config 4) and no 2n + 1 drift evaluations.  The literal sigma-point evaluation below (ODE_UKF) stays available
    // (CDK_FLAG_UKF_SIGMA_POINTS) and both are checked against the oracle, which evaluates sigma points as the reference
    // does; they differ by the rounding of the reference's own f(X^+) - f(X^-) cancellation (~1e-13).
    const T* th = c.p(L.TH);
    FOR_T(i, n) {
      km[i] = dt * (drift_f<T>(d.drift_id, th, n, i, [&](int j) { return mm[j]; }) + drift_half_trhp<T>(d.drift_id, th, n, i, P, ld));
    }
    T* JP = kP;  // formed in the output block, symmetrised in place
    if (stencil_drift(d.drift_id)) {
      FOR_T(e, n * n) {
        const int i = e / n, j = e - i * n;
        JP[i * ld + j] = stencil_jp<T>(d.drift_id, th, n, i, j, mm, P, ld);
      }
    } else {
      T* J = c.p(L.J);
      FOR_T(e, n * n) {
        const int i = e / n, j = e - i * n;
        J[i * ld + j] = drift_jac<T>(d.drift_id, th, n, i, j, mm);
      }
      __syncthreads();
      mm_dmma<T, false, false>(J, ld, P, ld, n, n, n, [&](int i, int j, double v) { JP[i * ld + j] = (T)v; });
    }
    __syncthreads();
    FOR_T(e, n * n) {
      const int a = e / n, b = e - a * n;
      if (a <= b) {  // one thread owns the pair (a, b), (b, a)
        const T sab = JP[a * ld + b] + JP[b * ld + a];
        kP[a * ld + b] = dt * (sab + lql[a * ld + b]);
        if (a != b) kP[b * ld + a] = dt * (sab + lql[b * ld + a]);
      }
    }
    __syncthreads();
    return;
  }
  if (kind == ODE_BACK) {
    // reverse-time smoothing ODE (cd_linear/inference.py:664-684, inference_ekf.py:399-441; reverse_rhs
    // diffrax_utils.py:13-25): d/ds (m_s, P_s) = -( c0 + G (m_s - m_f),  G P_s + P_s G^T - L Qc L^T )
    const T* G = c.p(L.J);
    const T* mf = c.p(L.MF);
    const T* c0 = c.p(L.C0);
    FOR_T(i, n) {
      T s = c0[i];
      for (int q = 0; q < n; ++q) s += G[i * ld + q] * (mm[q] - mf[q]);
      km[i] = -dt * s;
    }
    T* GP = c.p(L.W1);
    mm_dmma<T, false, false>(G, ld, P, ld, n, n, n, [&](int i, int j, double v) { GP[i * ld + j] = (T)v; });
    __syncthreads();
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      kP[i * ld + j] = -dt * ((GP[i * ld + j] + GP[j * ld + i]) - lql[i * ld + j]);
    }
    __syncthreads();
    return;
  }
  // ODE_UKF: the literal sigma points (cdk_dense.cuh, ukf_sigma_rhs; the gradient's re-integration calls it too)
  ukf_sigma_rhs<T>(d, c.p(L.TH), n, ld, mm, P, lql, c.p(L.W1), c.p(L.W2), km, kP, dt);
}

// Integrate y (length S, shared memory, in place) from t0 to t1 with the fixed-step explicit RK in g.tab.
// Restates diffrax diffeqsolve + ConstantStepSize (diffrax_utils.py:150-163).  Returns true when max_steps was hit.
template <typename T>
__device__ bool ode_solve(const Ctx<T>& c, int kind, T* y, int S, T t0, T t1, T dt0, int max_steps) {
  const RtTab& tab = c.g.tab;
  const int nslots = c.g.nslots;
  T* ys = c.p(c.L.YS);
  T* acc = c.p(c.L.ACC);
  T* ks = c.p(c.L.KS);
  StepClock<T> clk(t0, t1, dt0);
  while (clk.running()) {
    if (clk.n >= max_steps) {
      FOR_T(e, S) y[e] = T(NAN);
      __syncthreads();
      return true;
    }
    const T dt = clk.dt();
    for (int i = 0; i < tab.S; ++i) {
      const int nz = tab.nnz[i];
      FOR_T(e, S) {
        T v = y[e];
        // chain tableaux (nslots == 1) only ever reference the previous stage, which sits in slot 0
        for (int q = 0; q < nz; ++q) v += T(tab.val[i][q]) * ks[(nslots == 1 ? 0 : tab.col[i][q] * S) + e];
        ys[e] = v;
        if (i == 0) acc[e] = v;
      }
      __syncthreads();
      T* ki = ks + (nslots == 1 ? 0 : i * S);
      ode_rhs<T>(c, kind, ys, ki, dt);
      const T bi = T(tab.b[i]);
      if (bi != T(0)) {
        FOR_T(e, S) acc[e] += bi * ki[e];
      }
      __syncthreads();
    }
    FOR_T(e, S) y[e] = acc[e];
    __syncthreads();
    clk.advance();
  }
  return false;
}

// Moment ODE of the Lorenz-96 drift (EKF first / second order -- identical for this drift, SURVEY F8 -- and the closed-form
// unscented predict) for chain tableaux, with the RK state in REGISTERS.  Thread t owns a SEGMENT of one covariance row:
// row r = t % n, columns [c0, c0 + SEG), c0 = min(SEG * (t / n), n - SEG) (the last segment of a row overlaps its neighbour
// instead of being short: both owners compute and store identical values, and no entry needs a bounds predicate), and, for
// the first segment of a row, mean entry r.  It keeps y, the running combination and the previous stage increment of its
// entries.  Only the STAGE INPUT lives in shared memory (two buffers, YS and KS, alternating: ONE barrier per stage),
// because an entry's derivative reads its neighbours:
//   d/dt P_rc = (J P)_rc + (J P)_cr + (L Qc L^T)_rc,   (J P)_rc = x_{r-1} (P_{r+1,c} - P_{r-2,c}) + (x_{r+1} - x_{r-2}) P_{r-1,c} - P_rc,
// and with P_{c',r} read as P_{r,c'} the transposed term needs only a window of row r: the thread's own stage inputs
// (already in registers) plus three halo entries.  Per stage and thread: 3 + 10 window loads, 3 row coefficients, 3 column
// loads per entry (contiguous: immediate offsets from three row pointers) -- ~37 loads and ~150 instructions for 7
// entries, against ~500 with one entry per (thread, slot) and ~1,200 (index arithmetic of the run-time-n loops, four
// barriers) for ode_solve + ode_rhs on the same ODE.
constexpr int STENCIL_SEG = 7;  // 6 segments x 40 rows = 240 threads for n = 40 (BASELINE config 4)

__host__ __device__ inline bool stencil_fits(int n, int threads) {
  return n >= STENCIL_SEG && n * ((n + STENCIL_SEG - 1) / STENCIL_SEG) <= threads;
}

template <typename T>
struct StencilRegs {
  int act;                       // owns a segment
  int own_m;                     // ... and mean entry r
  int o_x, o_row;                // element offsets inside a stage buffer: x_{c0}, P_{r,c0}
  int o_colT;                    // P_{c0,r} (the transposed entries follow with stride ld)
  int o_up, o_d1, o_d2;          // P_{r+1,c0}, P_{r-1,c0}, P_{r-2,c0}
  int o_xl0, o_xl1, o_xh;        // x_{c0-2}, x_{c0-1}, x_{c0+SEG} (cyclic)
  int o_pl0, o_pl1, o_ph;        // P_{r,c0-2}, P_{r,c0-1}, P_{r,c0+SEG} (cyclic)
  int o_xr, o_xrp, o_xrm1, o_xrm2;  // x_r, x_{r+1}, x_{r-1}, x_{r-2}
  int o_u0, o_u1, o_u2, o_u3;    // P_{r+1,r-1}, P_{r-1,r+1}, P_{r-2,r-1}, P_{r-1,r-2} (unscented mean term)
  T lql[STENCIL_SEG];
};

template <typename T>
__device__ __forceinline__ void stencil_init(const Ctx<T>& c, StencilRegs<T>& R) {
  constexpr int SEG = STENCIL_SEG;
  const int n = c.L.n, ld = c.L.ldn, poff = c.L.P - c.L.MU;
  const T* lql = c.p(c.L.LQL);
  const int t = threadIdx.x;
  const int r = t % n, seg = t / n;
  int c0 = SEG * seg;
  R.act = c0 < n;
  if (!R.act) c0 = 0;
  if (c0 > n - SEG) c0 = n - SEG;
  R.own_m = R.act && seg == 0;
  auto wrap = [&](int q) { return q < 0 ? q + n : (q >= n ? q - n : q); };
  const int rp = wrap(r + 1), rm1 = wrap(r - 1), rm2 = wrap(r - 2);
  R.o_x = c0;
  R.o_row = poff + r * ld + c0;
  R.o_colT = poff + c0 * ld + r;
  R.o_up = poff + rp * ld + c0;
  R.o_d1 = poff + rm1 * ld + c0;
  R.o_d2 = poff + rm2 * ld + c0;
  R.o_xl0 = wrap(c0 - 2); R.o_xl1 = wrap(c0 - 1); R.o_xh = wrap(c0 + SEG);
  R.o_pl0 = poff + r * ld + R.o_xl0; R.o_pl1 = poff + r * ld + R.o_xl1; R.o_ph = poff + r * ld + R.o_xh;
  R.o_xr = r; R.o_xrp = rp; R.o_xrm1 = rm1; R.o_xrm2 = rm2;
  R.o_u0 = poff + rp * ld + rm1; R.o_u1 = poff + rm1 * ld + rp; R.o_u2 = poff + rm2 * ld + rm1; R.o_u3 = poff + rm1 * ld + rm2;
#pragma unroll
  for (int j = 0; j < SEG; ++j) R.lql[j] = lql[r * ld + c0 + j];
}

// The row-segment right-hand side reads P_{c',r} as P_{r,c'}: it integrates dP = J P + P J^T, whose ANTISYMMETRIC part obeys the
// same (chaotic, unstable) dynamics as the symmetric one.  The EKF symmetrises P in every update, so its covariance enters a
// gap exactly symmetric; the UKF never does (inference_ukf.py:202), and the rounding-level asymmetry of its update then
// doubles every few steps (1e-16 -> O(1) in ~240 steps of BASELINE config 4, found by the full-size test).  The reference's
// unscented right-hand side factors chol of the SYMMETRISED covariance (jnp.linalg.cholesky) and returns a symmetric
// derivative: the symmetric part evolves from sym(P) and the antisymmetric part is carried along unchanged.  UKFC does exactly
// that: integrate S = sym(P), then add the old antisymmetric part back.
// (The EKF's covariance is exactly symmetric after an update, but not between the gaps of a FORECAST -- no updates --, where the
// rounding asymmetry of one gap would be amplified by the next: it integrates sym(P) as well; the reference's own
// F P + P F^T keeps an exactly symmetric P exactly symmetric, so there is no antisymmetric part to carry.)
template <typename T, bool UKFC>
__device__ __forceinline__ T stencil_load_entry(const T* y, const StencilRegs<T>& R, int j, int ld) {
  return T(0.5) * (y[R.o_row + j] + y[R.o_colT + j * ld]);
}
template <typename T, bool UKFC>
__device__ __forceinline__ T stencil_antisym(const T* y, const StencilRegs<T>& R, int j, int ld) {
  if (!UKFC) return T(0);
  const T prc = y[R.o_row + j];
  return prc - T(0.5) * (prc + y[R.o_colT + j * ld]);
}

// Integrate (m, P) (shared memory, [MU | P] layout of `y`) from t0 to t1.  UKFC adds the unscented second-order mean term.
template <typename T, bool UKFC>
__device__ bool ode_solve_stencil(const Ctx<T>& c, const StencilRegs<T>& R, T* y, T t0, T t1, T dt0, int max_steps) {
  constexpr int SEG = STENCIL_SEG;
  const Lay& L = c.L;
  const RtTab& tab = c.g.tab;
  const T F = c.p(L.TH)[0];
  const bool act = R.act, own_m = R.own_m;
  // aP is the running combination y + sum_s b_s k_s: it equals y at the start of every step, so y itself needs no copy
  T aP[SEG], kP[SEG], yP[SEG];
  T am = T(0), km = T(0), ym = T(0);
#pragma unroll
  for (int j = 0; j < SEG; ++j) {
    aP[j] = stencil_load_entry<T, UKFC>(y, R, j, c.L.ldn);
    kP[j] = T(0);
  }
  if (own_m) am = y[R.o_xr];
  StepClock<T> clk(t0, t1, dt0);
  bool hit = false;
  const int boff0 = L.YS, boff1 = L.KS;
  int flip = 0;
  while (clk.running()) {
    if (clk.n >= max_steps) {
      hit = true;
#pragma unroll
      for (int j = 0; j < SEG; ++j) aP[j] = T(NAN);
      am = T(NAN);
      break;
    }
    const T dt = clk.dt();
#pragma unroll
    for (int j = 0; j < SEG; ++j) yP[j] = aP[j];
    ym = am;
    for (int st = 0; st < tab.S; ++st) {
      // chain tableau: only the previous stage; a = 0 at stage 0, where k still holds the previous step's (finite) value
      const T a = (st > 0 && tab.nnz[st]) ? T(tab.val[st][0]) : T(0);
      // the two stage buffers alternate over ALL stages of the solve (not per step: with an odd stage count -- euler, bosh3 --
      // the last stage of a step and the first of the next would otherwise share a buffer with no barrier between the reads of
      // the one and the writes of the other); an integer select keeps the pointer in the shared window (LDS / STS)
      T* B = c.sh + (flip ? boff1 : boff0);
      flip ^= 1;
      // stage input y + a k_{st-1}: kept in registers (it is this thread's part of the row window) and published
      T sP[SEG];
#pragma unroll
      for (int j = 0; j < SEG; ++j) sP[j] = fma(a, kP[j], yP[j]);
      const T sm = fma(a, km, ym);
      if (act) {
        T* row = B + R.o_row;
#pragma unroll
        for (int j = 0; j < SEG; ++j) row[j] = sP[j];
        if (own_m) B[R.o_xr] = sm;
      }
      __syncthreads();
      if (act) {
        const T b = T(tab.b[st]);
        // windows: index q <-> column c0 - 2 + q
        T xw[SEG + 3], pr[SEG + 3];
        xw[0] = B[R.o_xl0]; xw[1] = B[R.o_xl1]; xw[SEG + 2] = B[R.o_xh];
        pr[0] = B[R.o_pl0]; pr[1] = B[R.o_pl1]; pr[SEG + 2] = B[R.o_ph];
        const T* xs = B + R.o_x;
#pragma unroll
        for (int j = 0; j < SEG; ++j) {
          xw[j + 2] = xs[j];
          pr[j + 2] = sP[j];
        }
        const T ar = B[R.o_xrm1], br = B[R.o_xrp] - B[R.o_xrm2];
        const T* Pu = B + R.o_up;
        const T* Pd1 = B + R.o_d1;
        const T* Pd2 = B + R.o_d2;
#pragma unroll
        for (int j = 0; j < SEG; ++j) {
          const int q = j + 2;
          // (J P)_rc + (J P)_cr + LQL_rc as one fma chain: 3 differences, 5 fma
          T v = fma(T(-2), pr[q], R.lql[j]);
          v = fma(ar, Pu[j] - Pd2[j], v);
          v = fma(br, Pd1[j], v);
          v = fma(xw[q - 1], pr[q + 1] - pr[q - 2], v);
          v = fma(xw[q + 1] - xw[q - 2], pr[q - 1], v);
          kP[j] = dt * v;
          aP[j] = fma(b, kP[j], aP[j]);
        }
        if (own_m) {
          T f = fma(br, ar, F - sm);
          if (UKFC)  // 0.5 tr(Hess f_r P) = sym(P)_{r+1,r-1} - sym(P)_{r-2,r-1}
            f += T(0.5) * ((B[R.o_u0] + B[R.o_u1]) - (B[R.o_u2] + B[R.o_u3]));
          km = dt * f;
          am = fma(b, km, am);
        }
      }
    }
    clk.advance();
  }
  T a0[SEG];
#pragma unroll
  for (int j = 0; j < SEG; ++j) a0[j] = stencil_antisym<T, UKFC>(y, R, j, c.L.ldn);
  __syncthreads();  // the last stage's readers and the readers of the old state are done before the state block is rewritten
  if (act) {
#pragma unroll
    for (int j = 0; j < SEG; ++j) y[R.o_row + j] = UKFC ? aP[j] + a0[j] : aP[j];
    if (own_m) y[R.o_xr] = am;
  }
  __syncthreads();
  return hit;
}

// The same register-resident moment ODE for the reference's DEFAULT solver, Dormand-Prince 5 with a constant step
// (diffrax_utils.py:121-127): six stages with a full tableau, so the increments k_1 .. k_5 of the thread's entries stay in
// registers as well (5 x 7 doubles; ~170 registers: one CTA per SM, its own kernel instantiation) and the stage loop is
// unrolled over the compile-time tableau.  (Through the shared-memory solver with six stage buffers the default solver ran
// at a quarter of the RK4 rate on BASELINE config 4's model.)
template <typename T, bool UKFC>
__device__ bool ode_solve_stencil_dopri5(const Ctx<T>& c, const StencilRegs<T>& R, T* y, T t0, T t1, T dt0, int max_steps) {
  constexpr int SEG = STENCIL_SEG;
  using TB = Tab<CDK_DOPRI5>;
  constexpr int S = TB::S;
  const Lay& L = c.L;
  const T F = c.p(L.TH)[0];
  const bool act = R.act, own_m = R.own_m;
  T yP[SEG], kk[S - 1][SEG];
  T ym = T(0), kkm[S - 1];
#pragma unroll
  for (int j = 0; j < SEG; ++j) yP[j] = stencil_load_entry<T, UKFC>(y, R, j, c.L.ldn);
  if (own_m) ym = y[R.o_xr];
#pragma unroll
  for (int q = 0; q < S - 1; ++q) {
    kkm[q] = T(0);
#pragma unroll
    for (int j = 0; j < SEG; ++j) kk[q][j] = T(0);
  }
  StepClock<T> clk(t0, t1, dt0);
  bool hit = false;
  const int boff0 = L.YS, boff1 = L.KS;
  while (clk.running()) {
    if (clk.n >= max_steps) {
      hit = true;
#pragma unroll
      for (int j = 0; j < SEG; ++j) yP[j] = T(NAN);
      ym = T(NAN);
      break;
    }
    const T dt = clk.dt();
    T aP[SEG], am = ym;
#pragma unroll
    for (int j = 0; j < SEG; ++j) aP[j] = yP[j];
#pragma unroll
    for (int st = 0; st < S; ++st) {
      T* B = c.sh + ((st & 1) ? boff1 : boff0);
      T sP[SEG], sm = ym;
#pragma unroll
      for (int j = 0; j < SEG; ++j) sP[j] = yP[j];
#pragma unroll
      for (int q = 0; q < st; ++q) {
        if (TB::a(st, q) != 0.0) {
          const T aq = T(TB::a(st, q));
#pragma unroll
          for (int j = 0; j < SEG; ++j) sP[j] = fma(aq, kk[q][j], sP[j]);
          sm = fma(aq, kkm[q], sm);
        }
      }
      if (act) {
        T* row = B + R.o_row;
#pragma unroll
        for (int j = 0; j < SEG; ++j) row[j] = sP[j];
        if (own_m) B[R.o_xr] = sm;
      }
      __syncthreads();
      if (act) {
        T xw[SEG + 3], pr[SEG + 3];
        xw[0] = B[R.o_xl0]; xw[1] = B[R.o_xl1]; xw[SEG + 2] = B[R.o_xh];
        pr[0] = B[R.o_pl0]; pr[1] = B[R.o_pl1]; pr[SEG + 2] = B[R.o_ph];
        const T* xs = B + R.o_x;
#pragma unroll
        for (int j = 0; j < SEG; ++j) {
          xw[j + 2] = xs[j];
          pr[j + 2] = sP[j];
        }
        const T ar = B[R.o_xrm1], br = B[R.o_xrp] - B[R.o_xrm2];
        const T* Pu = B + R.o_up;
        const T* Pd1 = B + R.o_d1;
        const T* Pd2 = B + R.o_d2;
        const T b = T(TB::b(st));
#pragma unroll
        for (int j = 0; j < SEG; ++j) {
          const int q = j + 2;
          T v = fma(T(-2), pr[q], R.lql[j]);
          v = fma(ar, Pu[j] - Pd2[j], v);
          v = fma(br, Pd1[j], v);
          v = fma(xw[q - 1], pr[q + 1] - pr[q - 2], v);
          v = fma(xw[q + 1] - xw[q - 2], pr[q - 1], v);
          const T kv = dt * v;
          if (st < S - 1) kk[st < S - 1 ? st : 0][j] = kv;
          if (TB::b(st) != 0.0) aP[j] = fma(b, kv, aP[j]);
        }
        if (own_m) {
          T f = fma(br, ar, F - sm);
          if (UKFC) f += T(0.5) * ((B[R.o_u0] + B[R.o_u1]) - (B[R.o_u2] + B[R.o_u3]));
          const T kv = dt * f;
          if (st < S - 1) kkm[st < S - 1 ? st : 0] = kv;
          if (TB::b(st) != 0.0) am = fma(b, kv, am);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < SEG; ++j) yP[j] = aP[j];
    ym = am;
    clk.advance();
  }
  T a0[SEG];
#pragma unroll
  for (int j = 0; j < SEG; ++j) a0[j] = stencil_antisym<T, UKFC>(y, R, j, c.L.ldn);
  __syncthreads();
  if (act) {
#pragma unroll
    for (int j = 0; j < SEG; ++j) y[R.o_row + j] = UKFC ? yP[j] + a0[j] : yP[j];
    if (own_m) y[R.o_xr] = ym;
  }
  __syncthreads();
  return hit;
}

// load a [r x c] row-major global matrix into shared memory with leading dimension ld
template <typename T>
__device__ void load_mat(T* dst, const T* src, int r, int c, int ld) {
  FOR_T(e, r * c) {
    const int i = e / c, j = e - i * c;
    dst[i * ld + j] = src[e];
  }
}
template <typename T>
__device__ void store_mat(T* dst, const T* src, int r, int c, int ld) {
  FOR_T(e, r * c) {
    const int i = e / c, j = e - i * c;
    dst[e] = src[i * ld + j];
  }
}

template <typename T>
__device__ void load_model(const Ctx<T>& c, long long traj, bool linear) {
  const Lay& L = c.L;
  const KArgs<T>& a = c.g.k;
  const int n = L.n, m = L.m, du = L.du;
  auto src = [&](int slot) { return a.in[slot] + traj * a.in_stride[slot]; };
  if (linear) {
    load_mat<T>(c.p(L.TH), src(CDK_IN_F), n, n, L.ldn);
    FOR_T(i, n) c.p(L.BV)[i] = src(CDK_IN_B)[i];
    if (du > 0) {
      FOR_T(i, n * du) c.p(L.BU)[i] = src(CDK_IN_BU)[i];
      FOR_T(i, m * du) c.p(L.DU)[i] = src(CDK_IN_DU)[i];
    }
  } else {
    FOR_T(i, a.d.n_theta) c.p(L.TH)[i] = src(CDK_IN_F)[i];
  }
  if (!linear && user_emission(a.d)) {
    FOR_T(i, emission_params(a.d)) c.p(L.PHI)[i] = src(CDK_IN_H)[i];  // phi; L.H then holds J = d h / dx at the mean
  } else {
    load_mat<T>(c.p(L.H), src(CDK_IN_H), m, n, L.ldn);
    FOR_T(i, m) c.p(L.DV)[i] = src(CDK_IN_D)[i];
  }
  if (a.d.reserved[2] & CDK_FLAG_DIAG_R) {
    FOR_T(i, m) c.p(L.R)[i] = src(CDK_IN_R)[i];  // 1-D emissions.cov: the diagonal (linear model only, validated)
  } else {
    load_mat<T>(c.p(L.R), src(CDK_IN_R), m, m, L.ldm);
  }
  // L Qc L^T via W1 = L, W2 = Qc, W3 = L Qc
  T* Lm = c.p(L.W1);
  T* Qc = c.p(L.W2);
  T* LQ = c.p(L.W3);
  load_mat<T>(Lm, src(CDK_IN_L), n, n, L.ldn);
  load_mat<T>(Qc, src(CDK_IN_QC), n, n, L.ldn);
  __syncthreads();
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    T s = T(0);
    for (int q = 0; q < n; ++q) s += Lm[i * L.ldn + q] * Qc[q * L.ldn + j];
    LQ[i * L.ldn + j] = s;
  }
  __syncthreads();
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    T s = T(0);
    for (int q = 0; q < n; ++q) s += LQ[i * L.ldn + q] * Lm[j * L.ldn + q];
    c.p(L.LQL)[i * L.ldn + j] = s;
  }
  __syncthreads();
}

// Linear-model measurement update for a 1-D (diagonal) emission covariance: the reference's Woodbury branch
// (cd_linear/inference.py:240-254) and its log-likelihood (:613), restated literally:
//   U = H chol(sym P),  X = U / R[:, None],  S_inv = diag(1/R) - X psd_solve(I + U^T X, X^T),  K = P H^T S_inv,
//   S = diag(R) + H P H^T,  P <- sym(P - K S K^T),  m <- m + K (y - D u - d - H m);
//   ll = log N(y; H m + D u + d, chol(H P H^T + (R_i + R_j) / 2)) -- the reference adds the VECTOR R to H P H^T by
//   broadcasting (entry (i, j) gets R[j]) and TFP's Cholesky factors the symmetrised matrix; for a constant vector this is
//   diag(R)-free of error only on the diagonal, and it is reproduced as is (parity is with the reference, not the textbook).
// Scratch: J, the pushforward buffers ODEY (2 n x n, idle during the update), W1..W3, SM, SL.
template <typename T>
__device__ T condition_on_diag_r(const Ctx<T>& c) {
  const Lay& L = c.L;
  const int n = L.n, m = L.m, ldn = L.ldn, ldm = L.ldm;
  T* mu = c.p(L.MU);
  T* P = c.p(L.P);
  const T* H = c.p(L.H);
  const T* R = c.p(L.R);  // [m]
  const T* dv = c.p(L.DV);
  const T* yv = c.p(L.YV);
  T* Lp = c.p(L.J);        // chol(sym P)
  T* Ma = c.p(L.ODEY);     // sym(P), then M = I + U^T X
  T* Lm = Ma + L.nn;       // chol(sym(M) + 1e-9 I)
  T* W1 = c.p(L.W1);       // H P [m x n]; then Z = psd_solve(M, X^T) as [n x ldm]; then (P H^T)^T [m x n]
  T* U = c.p(L.W2);        // [m x n], later Kt
  T* X = c.p(L.W3);        // [m x n], later S Kt
  T* Sm = c.p(L.SM);
  T* Sl = c.p(L.SL);
  T* rv = c.p(L.RV);
  T* zv = rv + m;
  __shared__ T ll_sh;
  FOR_T(e, m * n) {
    const int a = e / n, j = e - a * n;
    T s = T(0);
    for (int q = 0; q < n; ++q) s += H[a * ldn + q] * P[q * ldn + j];
    W1[a * ldn + j] = s;
  }
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    Ma[i * ldn + j] = T(0.5) * (P[i * ldn + j] + P[j * ldn + i]);
  }
  FOR_T(a, m) {
    T s = dv[a];
    for (int q = 0; q < n; ++q) s += H[a * ldn + q] * mu[q];
    rv[a] = yv[a] - s;
  }
  __syncthreads();
  FOR_T(e, m * m) {  // H P H^T (plain) in Sm; the log-likelihood's matrix in X (scratch)
    const int a = e / m, b = e - a * m;
    T s = T(0);
    for (int q = 0; q < n; ++q) s += W1[a * ldn + q] * H[b * ldn + q];
    Sm[a * ldm + b] = s;
  }
  __syncthreads();
  FOR_T(e, m * m) {
    const int a = e / m, b = e - a * m;
    // sym(H P H^T + R[None, :]) = (hph_ab + hph_ba) / 2 + (R_a + R_b) / 2
    X[a * ldm + b] = T(0.5) * ((Sm[a * ldm + b] + R[b]) + (Sm[b * ldm + a] + R[a]));
  }
  __syncthreads();
  chol<T>(X, Sl, m, ldm, T(0));
  mvn_ll_warp<T>(Sl, ldm, rv, m, &ll_sh);
  chol<T>(Ma, Lp, n, ldn, T(0));  // jnp.linalg.cholesky(P) symmetrises its input
  FOR_T(e, m * n) {  // U = H Lp (Lp lower), X = U / R[:, None]
    const int a = e / n, j = e - a * n;
    T s = T(0);
    for (int q = j; q < n; ++q) s += H[a * ldn + q] * Lp[q * ldn + j];
    U[a * ldn + j] = s;
    X[a * ldn + j] = s / R[a];
  }
  __syncthreads();
  FOR_T(e, n * n) {  // M = I + U^T X
    const int i = e / n, j = e - i * n;
    T s = i == j ? T(1) : T(0);
    for (int a = 0; a < m; ++a) s += U[a * ldn + i] * X[a * ldn + j];
    Ma[i * ldn + j] = s;
  }
  __syncthreads();
  T* Ms = U;  // sym(M) (U is no longer needed; n x ldn fits the max(n, m)-sized scratch)
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    Ms[i * ldn + j] = T(0.5) * (Ma[i * ldn + j] + Ma[j * ldn + i]);
  }
  T* Z = W1;  // [n x ldm] <- X^T, then psd_solve(M, X^T)  (H P is no longer needed; max(n, m)-sized scratch)
  __syncthreads();
  FOR_T(e, n * m) {
    const int i = e / m, a = e - i * m;
    Z[i * ldm + a] = X[a * ldn + i];
  }
  chol<T>(Ms, Lm, n, ldn, T(1e-9));
  chol_solve<T>(Lm, n, ldn, Z, m, ldm);
  T* Si = Sl;  // S_inv = diag(1 / R) - X Z
  FOR_T(e, m * m) {
    const int a = e / m, b = e - a * m;
    T s = a == b ? T(1) / R[a] : T(0);
    for (int q = 0; q < n; ++q) s -= X[a * ldn + q] * Z[q * ldm + b];
    Si[a * ldm + b] = s;
  }
  __syncthreads();
  FOR_T(e, m * n) {  // (P H^T)^T, row a = P H[a, :]^T
    const int a = e / n, i = e - a * n;
    T s = T(0);
    for (int q = 0; q < n; ++q) s += P[i * ldn + q] * H[a * ldn + q];
    W1[a * ldn + i] = s;
  }
  __syncthreads();
  T* Kt = U;  // Kt[a][i] = K[i][a] = sum_b (P H^T)[i][b] S_inv[b][a]
  FOR_T(e, m * n) {
    const int a = e / n, i = e - a * n;
    T s = T(0);
    for (int b = 0; b < m; ++b) s += W1[b * ldn + i] * Si[b * ldm + a];
    Kt[a * ldn + i] = s;
  }
  FOR_T(a, m) Sm[a * ldm + a] += R[a];  // S = diag(R) + H P H^T
  __syncthreads();
  T* SK = X;
  FOR_T(e, m * n) {
    const int a = e / n, j = e - a * n;
    T s = T(0);
    for (int b = 0; b < m; ++b) s += Sm[a * ldm + b] * Kt[b * ldn + j];
    SK[a * ldn + j] = s;
  }
  __syncthreads();
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    T s = T(0);
    for (int a = 0; a < m; ++a) s += Kt[a * ldn + i] * SK[a * ldn + j];
    P[i * ldn + j] -= s;
  }
  FOR_T(i, n) {
    T s = T(0);
    for (int a = 0; a < m; ++a) s += Kt[a * ldn + i] * rv[a];
    mu[i] += s;
  }
  __syncthreads();
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    if (i < j) {
      const T v = T(0.5) * (P[i * ldn + j] + P[j * ldn + i]);
      P[i * ldn + j] = v;
      P[j * ldn + i] = v;
    }
  }
  __syncthreads();
  return ll_sh;
}

// The moments of the UKF update with a user emission, restating inference_ukf.py:162-203 literally (as tests/user_emission_oracle.py does):
// sigma points X_p = m, m +- c L_i (L L^T = P, c^2 = n + lambda), Y_p = h(X_p), yhat = sum_p w_m[p] Y_p,
// S = sum_p w_c[p] dY_p dY_p^T + R, C = sum_p w_c[p] dX_p dY_p^T -- the centre point's w_c[0], which carries
// 1 - alpha^2 + beta, included.  One (point, component) evaluation of h per thread.  Out: Sm = S, Ct = C^T [m x n],
// rv = y - yhat.  Scratch: J (the factor of P), YP (the points through h, then their deviations), rv + m (yhat).
template <typename T>
__device__ void ukf_user_moments(const Ctx<T>& c, T* Sm, T* Ct, T* rv) {
  const Lay& L = c.L;
  const cdk_desc& d = c.g.k.d;
  const int n = L.n, m = L.m, ldn = L.ldn, ldm = L.ldm, np = 2 * n + 1;
  const T* mu = c.p(L.MU);
  const T* R = c.p(L.R);
  const T* phi = c.p(L.PHI);
  const T* yv = c.p(L.YV);
  T* Lc = c.p(L.J);
  T* Y = c.p(L.YP);
  T* yhat = rv + m;
  chol<T>(c.p(L.P), Lc, n, ldn, T(0));  // ends with a barrier
  const double lam = d.alpha * d.alpha * (d.n + d.kappa) - d.n;  // ukf_weights (inference_ukf.py:42, :63-89)
  const T w0m = T(lam / (d.n + lam)), wi = T(1.0 / (2.0 * (d.n + lam)));
  const T w0c = T(lam / (d.n + lam) + (1.0 - d.alpha * d.alpha + d.beta));
  const T cs = sqrt(T(d.n + lam));
  auto xp = [&](int p, int j) -> T {  // component j of sigma point p
    if (p == 0) return mu[j];
    const T v = cs * Lc[j * ldn + (p <= n ? p - 1 : p - 1 - n)];
    return p <= n ? mu[j] + v : mu[j] - v;
  };
  FOR_T(e, np * m) {
    const int p = e / m, a = e - p * m;
    Y[p * ldm + a] = user_h<T>(phi, n, m, a, [&](int j) { return xp(p, j); });
  }
  __syncthreads();
  FOR_T(a, m) {
    T s = T(0);
    for (int p = 0; p < np; ++p) s += (p == 0 ? w0m : wi) * Y[p * ldm + a];
    yhat[a] = s;
    rv[a] = yv[a] - s;
  }
  __syncthreads();
  FOR_T(e, np * m) {
    const int p = e / m, a = e - p * m;
    Y[p * ldm + a] -= yhat[a];
  }
  __syncthreads();
  FOR_T(e, m * m) {
    const int a = e / m, b = e - a * m;
    T s = T(0);
    for (int p = 0; p < np; ++p) s += (p == 0 ? w0c : wi) * Y[p * ldm + a] * Y[p * ldm + b];
    Sm[a * ldm + b] = s + R[a * ldm + b];
  }
  FOR_T(e, m * n) {
    const int a = e / n, j = e - a * n;
    T s = T(0);  // dX_0 = 0
    for (int p = 1; p < np; ++p) s += wi * (xp(p, j) - mu[j]) * Y[p * ldm + a];
    Ct[a * ldn + j] = s;
  }
}

// Measurement update shared by KF / EKF / UKF.  On entry MU, P hold the prediction; on exit the filtered moments.
// Returns the log-likelihood increment (same value in every thread).
template <typename T>
__device__ T condition_on(const Ctx<T>& c, int algo, int num_iter) {
  const Lay& L = c.L;
  const cdk_desc& d = c.g.k.d;
  const int n = L.n, m = L.m, ldn = L.ldn, ldm = L.ldm;
  T* mu = c.p(L.MU);
  T* P = c.p(L.P);
  T* H = c.p(L.H);  // user emission: J = d h / dx at the running mean, re-evaluated in every iteration
  const T* phi = c.p(L.PHI);
  const T* R = c.p(L.R);
  const T* dv = c.p(L.DV);
  const T* yv = c.p(L.YV);
  T* HP = c.p(L.W1);  // [m x n]
  T* Kt = c.p(L.W2);  // [m x n]  (S + boost)^-1 H P
  T* SK = c.p(L.W3);  // [m x n]  S Kt
  T* Sm = c.p(L.SM);
  T* Sl = c.p(L.SL);
  T* rv = c.p(L.RV);
  T* zv = rv + m;
  __shared__ T ll_sh;
  // ukf: literal sigma points through chol(P).  The closed-form UKF (linear emission: S = H P H^T + R and the cross term
  // P H^T exactly) takes the H P products of the KF / EKF branch, but -- like the reference's UKF -- never symmetrises.
  // A user emission (cdk.h, CDK_EMISSION_USER): the EKF linearises h at the running mean of every iteration (the iterated
  // update of inference_ekf.py:153-199 with H = jacfwd(h), re-using the running covariance); the UKF takes the literal
  // sigma-point update (ukf_user_moments) whether its predict runs in closed form or not.
  const bool ue = algo != ALGO_KF_FILTER && user_emission(d);
  const bool ukf_user = algo == ALGO_UKF_FILTER && ue;
  const bool ukf = algo == ALGO_UKF_FILTER && !ukf_closed(d) && !ue;
  const bool no_sym = algo == ALGO_UKF_FILTER;
  for (int it = 0; it < num_iter; ++it) {
    if (ue && !ukf_user) {
      FOR_T(e, m * n) {
        const int a = e / n, j = e - a * n;
        H[a * ldn + j] = user_h_jac<T>(phi, n, m, a, j, mu);
      }
      __syncthreads();
    }
    if (ukf_user) {
      ukf_user_moments<T>(c, Sm, HP, rv);
    } else if (!ukf) {
      mm_dmma<T, false, false>(H, ldn, P, ldn, m, n, n, [&](int a, int j, double v) { HP[a * ldn + j] = (T)v; });
      __syncthreads();
      mm_dmma<T, false, true>(HP, ldn, H, ldn, m, m, n, [&](int a, int b, double v) { Sm[a * ldm + b] = R[a * ldm + b] + (T)v; });
    } else {
      // inference_ukf.py:162-203 with h(x) = H x + d:  Y_i^+- - yhat = +-c H L_i, X_i^+- - m = +-c L_i
      //   S = 2 w c^2 (H Lc)(H Lc)^T + R,  cross^T = 2 w c^2 (H Lc) Lc^T
      T* Lc = c.p(L.J);
      chol<T>(P, Lc, n, ldn, T(0));
      T* HL = SK;
      FOR_T(e, m * n) {
        const int a = e / n, j = e - a * n;
        T s = T(0);
        for (int q = j; q < n; ++q) s += H[a * ldn + q] * Lc[q * ldn + j];
        HL[a * ldn + j] = s;
      }
      __syncthreads();
      const T lam = T(d.alpha * d.alpha * (d.n + d.kappa) - d.n);
      const T c2 = T(2) * (T(1) / (T(2) * (T(d.n) + lam))) * (T(d.n) + lam);
      FOR_T(e, m * m) {
        const int a = e / m, b = e - a * m;
        T s = T(0);
        for (int q = 0; q < n; ++q) s += HL[a * ldn + q] * HL[b * ldn + q];
        Sm[a * ldm + b] = c2 * s + R[a * ldm + b];
      }
      FOR_T(e, m * n) {
        const int a = e / n, j = e - a * n;
        T s = T(0);
        for (int q = 0; q <= j; ++q) s += HL[a * ldn + q] * Lc[j * ldn + q];
        HP[a * ldn + j] = c2 * s;  // cross^T
      }
    }
    if (!ukf_user) {
      FOR_T(a, m) {
        T s;
        if (ue) {
          s = user_h<T>(phi, n, m, a, [&](int j) { return mu[j]; });
        } else {
          s = dv[a];
          for (int q = 0; q < n; ++q) s += H[a * ldn + q] * mu[q];
        }
        rv[a] = yv[a] - s;  // yv already has D u subtracted (linear model)
      }
    }
    __syncthreads();
    // MVN(.).log_prob(y) factors S un-boosted (TFP); psd_solve(S, .) factors sym(S) + 1e-9 I: two independent m x m
    // factorisations, one warp each, side by side.  The un-boosted factor is parked in SK (free until S Kt below).
    const int w1 = blockDim.x > 32 ? 1 : 0;
    if (it == 0) chol_prep<T, false>(Sm, SK, m, ldm, T(0));
    chol_prep<T, true>(Sm, Sl, m, ldm, T(1e-9));
    __syncthreads();
    if (it == 0) chol_warp<T>(0, SK, m, ldm);
    chol_warp<T>(w1, Sl, m, ldm);
    __syncthreads();
    if (it == 0) mvn_ll_warp<T>(SK, ldm, rv, m, &ll_sh);  // warp 0 only; the others start on the solve
    chol_solve<T>(Sl, m, ldm, HP, Kt, n, ldn);           // Kt = (sym(S) + 1e-9 I)^-1 H P; ends with a barrier
    mm_dmma<T, false, false>(Sm, ldm, Kt, ldn, m, n, m, [&](int a, int j, double v) { SK[a * ldn + j] = (T)v; });
    __syncthreads();
    mm_dmma<T, true, false>(Kt, ldn, SK, ldn, n, n, m, [&](int i, int j, double v) { P[i * ldn + j] -= (T)v; });
    FOR_T(i, n) {
      T s = T(0);
      for (int a = 0; a < m; ++a) s += Kt[a * ldn + i] * rv[a];
      mu[i] += s;
    }
    __syncthreads();
  }
  if (!no_sym) {
    // symmetrize (cd_linear/inference.py:259, inference_ekf.py:199); the UKF does not (inference_ukf.py:202)
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      if (i < j) {
        const T v = T(0.5) * (P[i * ldn + j] + P[j * ldn + i]);
        P[i * ldn + j] = v;
        P[j * ldn + i] = v;
      }
    }
    __syncthreads();
  }
  return ll_sh;
}

// REGODE: the launcher has established that the predict step is the Lorenz-96 moment ODE with a chain tableau
// (ode_solve_stencil, RK state in registers); that instantiation contains no other ODE code, so its register allocation is
// not burdened by the shared-memory solver and vice versa.
template <typename T, int REGODE>
__global__ void __launch_bounds__(256, REGODE == 2 ? 1 : 2) generic_filter_kernel(const GArgs<T> g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Ctx<T> c(g, reinterpret_cast<T*>(smem_raw));
  const Lay& L = c.L;
  const KArgs<T>& a = g.k;
  const cdk_desc& d = a.d;
  const int n = L.n, m = L.m, du = L.du, ldn = L.ldn, K = d.K;
  const int algo = g.algo;
  const bool linear = algo == ALGO_KF_FILTER;
  const long long traj = blockIdx.x;
  FOR_T(e, L.total) c.sh[e] = T(0);
  __syncthreads();
  load_model<T>(c, traj, linear);
  T* mu = c.p(L.MU);
  T* P = c.p(L.P);
  FOR_T(i, n) mu[i] = (a.in[CDK_IN_M0] + traj * a.in_stride[CDK_IN_M0])[i];
  load_mat<T>(P, a.in[CDK_IN_P0] + traj * a.in_stride[CDK_IN_P0], n, n, ldn);
  __syncthreads();
  const T* Y = a.in[CDK_IN_Y] + traj * a.in_stride[CDK_IN_Y];
  const T* Tm = a.in[CDK_IN_T] + traj * a.in_stride[CDK_IN_T];
  const T* U = du > 0 ? a.in[CDK_IN_U] + traj * a.in_stride[CDK_IN_U] : nullptr;
  T* FM = static_cast<T*>(a.out[CDK_OUT_FM]);
  T* FP = static_cast<T*>(a.out[CDK_OUT_FP]);
  T* PM = static_cast<T*>(a.out[CDK_OUT_PM]);
  T* PP = static_cast<T*>(a.out[CDK_OUT_PP]);
  T* LLC = static_cast<T*>(a.out[CDK_OUT_LLCUM]);
  const long long row0 = traj * (long long)K;
  const T dt0 = T(d.dt0);
  T ll = T(0);
  int status = 0;
  T* yv = c.p(L.YV);
  T* uv = c.p(L.UV);
  // forecast (CDK_FLAG_PREDICT_ONLY): no updates; Tm holds K + 1 stamps, t_init first
  const bool ponly = (d.reserved[2] & CDK_FLAG_PREDICT_ONLY) != 0;
  StencilRegs<T> sreg;
  if constexpr (REGODE != 0) stencil_init<T>(c, sreg);
  for (int k = 0; k < K; ++k) {
    FOR_T(i, du) uv[i] = U[(long long)k * du + i];
    __syncthreads();
    if (!ponly) {
      FOR_T(i, m) {
        T v = Y[(long long)k * m + i];
        if (du > 0) {  // y - D u (cd_linear/inference.py:258, :613)
          const T* DU = c.p(L.DU);
          for (int q = 0; q < du; ++q) v -= DU[i * du + q] * uv[q];
        }
        yv[i] = v;
      }
      __syncthreads();
      if (linear && (d.reserved[2] & CDK_FLAG_DIAG_R)) {
        ll += condition_on_diag_r<T>(c);
      } else {
        ll += condition_on<T>(c, algo, algo == ALGO_EKF_FILTER ? d.num_iter : 1);
      }
      if (FM) FOR_T(i, n) FM[(row0 + k) * n + i] = mu[i];
      if (FP) store_mat<T>(FP + (row0 + k) * n * n, P, n, n, ldn);
      if (LLC && threadIdx.x == 0) LLC[row0 + k] = ll;
    }
    const T t0 = Tm[k];
    const T t1 = (ponly || k + 1 < K) ? Tm[k + 1] : t0 + T(d.dt_final);
    bool hit = false;
    if constexpr (REGODE == 1) {
      if (algo == ALGO_UKF_FILTER) {
        hit = ode_solve_stencil<T, true>(c, sreg, mu, t0, t1, dt0, d.max_steps);
      } else {
        hit = ode_solve_stencil<T, false>(c, sreg, mu, t0, t1, dt0, d.max_steps);
      }
    } else if constexpr (REGODE == 2) {
      if (algo == ALGO_UKF_FILTER) {
        hit = ode_solve_stencil_dopri5<T, true>(c, sreg, mu, t0, t1, dt0, d.max_steps);
      } else {
        hit = ode_solve_stencil_dopri5<T, false>(c, sreg, mu, t0, t1, dt0, d.max_steps);
      }
    } else if (linear) {
      // pushforward from (I, 0), then m = A m + B u + b, P = A P A^T + Q (cd_linear/inference.py:619-620)
      T* A = c.p(L.ODEY);
      T* Q = A + L.nn;
      FOR_T(e, n * ldn) {
        const int i = e / ldn, j = e - i * ldn;
        A[e] = i == j ? T(1) : T(0);
        Q[e] = T(0);
      }
      __syncthreads();
      hit = ode_solve<T>(c, ODE_PUSH, A, 2 * L.nn, t0, t1, dt0, d.max_steps);
      T* AP = c.p(L.W1);
      T* mnew = c.p(L.C0);
      mm_dmma<T, false, false>(A, ldn, P, ldn, n, n, n, [&](int i, int j, double v) { AP[i * ldn + j] = (T)v; });
      FOR_T(i, n) {
        T s = T(0);
        for (int q = 0; q < n; ++q) s += A[i * ldn + q] * mu[q];
        if (du > 0) {
          const T* BU = c.p(L.BU);
          for (int q = 0; q < du; ++q) s += BU[i * du + q] * uv[q];
        }
        mnew[i] = s + c.p(L.BV)[i];
      }
      __syncthreads();
      mm_dmma<T, false, true>(AP, ldn, A, ldn, n, n, n, [&](int i, int j, double v) { P[i * ldn + j] = (T)v + Q[i * ldn + j]; });
      FOR_T(i, n) mu[i] = mnew[i];
      __syncthreads();
    } else if (algo == ALGO_EKF_FILTER && d.state_order == CDK_ORDER_ZEROTH) {
      // inference_ekf.py:126-138: only the mean is integrated; P += sqrt(dt) (c L) Qc (c L)^T
      hit = ode_solve<T>(c, ODE_MEAN, mu, n, t0, t1, dt0, d.max_steps);
      const T sc = sqrt(t1 - t0) * T(d.cov_rescaling) * T(d.cov_rescaling);
      const T* lql = c.p(L.LQL);
      FOR_T(e, n * n) {
        const int i = e / n, j = e - i * n;
        P[i * ldn + j] += sc * lql[i * ldn + j];
      }
      __syncthreads();
    } else {
      const int kind = algo == ALGO_UKF_FILTER ? (ukf_closed(d) ? ODE_UKFC : ODE_UKF) : ODE_EKF;
      hit = ode_solve<T>(c, kind, mu, L.mpoff + L.nn, t0, t1, dt0, d.max_steps);
    }
    if (hit) status = 2;
    if (PM) FOR_T(i, n) PM[(row0 + k) * n + i] = mu[i];
    if (PP) store_mat<T>(PP + (row0 + k) * n * n, P, n, n, ldn);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (a.out[CDK_OUT_LL]) static_cast<T*>(a.out[CDK_OUT_LL])[traj] = ll;
    if (a.out[CDK_OUT_STATUS]) static_cast<int*>(a.out[CDK_OUT_STATUS])[traj] = final_status(status, isfinite(ll));
  }
}

// Backward pass of the smoothers.  Reads the filtered moments from HBM (CDK_IN_FM / CDK_IN_FP).
template <typename T>
__global__ void generic_smooth_kernel(const GArgs<T> g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Ctx<T> c(g, reinterpret_cast<T*>(smem_raw));
  const Lay& L = c.L;
  const KArgs<T>& a = g.k;
  const cdk_desc& d = a.d;
  const int n = L.n, du = L.du, ldn = L.ldn, K = d.K;
  const bool linear = g.algo == ALGO_KF_SMOOTH;
  const int stype = linear ? d.smoother_type : 2;
  const long long traj = blockIdx.x;
  FOR_T(e, L.total) c.sh[e] = T(0);
  __syncthreads();
  load_model<T>(c, traj, linear);
  const T* Tm = a.in[CDK_IN_T] + traj * a.in_stride[CDK_IN_T];
  const T* U = du > 0 ? a.in[CDK_IN_U] + traj * a.in_stride[CDK_IN_U] : nullptr;
  const T* FMg = a.in[CDK_IN_FM] + traj * a.in_stride[CDK_IN_FM];
  const T* FPg = a.in[CDK_IN_FP] + traj * a.in_stride[CDK_IN_FP];
  T* SMg = static_cast<T*>(a.out[CDK_OUT_SM]) + traj * (long long)K * n;
  T* SPg = static_cast<T*>(a.out[CDK_OUT_SP]) + traj * (long long)K * n * n;
  T* SCg = a.out[CDK_OUT_SCROSS] ? static_cast<T*>(a.out[CDK_OUT_SCROSS]) + traj * (long long)(K - 1) * n * n : nullptr;
  T* ms = c.p(L.MU);
  T* Ps = c.p(L.P);
  T* mf = c.p(L.MF);
  T* Pf = c.p(L.PF);
  FOR_T(i, n) ms[i] = FMg[(long long)(K - 1) * n + i];
  load_mat<T>(Ps, FPg + (long long)(K - 1) * n * n, n, n, ldn);
  __syncthreads();
  FOR_T(i, n) SMg[(long long)(K - 1) * n + i] = ms[i];
  store_mat<T>(SPg + (long long)(K - 1) * n * n, Ps, n, n, ldn);
  int status = 0;
  const T* lql = c.p(L.LQL);
  for (int k = K - 2; k >= 0; --k) {
    FOR_T(i, n) mf[i] = FMg[(long long)k * n + i];
    load_mat<T>(Pf, FPg + (long long)k * n * n, n, n, ldn);
    __syncthreads();
    const T t0 = Tm[k], t1 = Tm[k + 1];
    if (stype == 1) {
      // Sarkka Alg 3.17 (cd_linear/inference.py:746-773): the pushforward is re-integrated here (:753)
      T* A = c.p(L.ODEY);
      T* Q = A + L.nn;
      FOR_T(e, n * ldn) {
        const int i = e / ldn, j = e - i * ldn;
        A[e] = i == j ? T(1) : T(0);
        Q[e] = T(0);
      }
      __syncthreads();
      if (ode_solve<T>(c, ODE_PUSH, A, 2 * L.nn, t0, t1, T(d.dt0), d.max_steps)) status = 2;
      T* APf = c.p(L.W1);  // A Pf, then Ct = (Pp + boost)^-1 A Pf  (C = Ct^T)
      T* Pp = c.p(L.W2);   // A Pf A^T + Q
      T* Lp = c.p(L.W3);
      T* Dm = c.p(L.J);    // Ps - Pp, then scratch
      T* rv = c.p(L.C0);
      mm_dmma<T, false, false>(A, ldn, Pf, ldn, n, n, n, [&](int i, int j, double v) { APf[i * ldn + j] = (T)v; });
      __syncthreads();
      mm_dmma<T, false, true>(APf, ldn, A, ldn, n, n, n, [&](int i, int j, double v) { Pp[i * ldn + j] = Q[i * ldn + j] + (T)v; });
      FOR_T(i, n) {
        // m_s^+ - A m_f - B u - b   (:763-766)
        T s = T(0);
        for (int q = 0; q < n; ++q) s += A[i * ldn + q] * mf[q];
        if (du > 0) {
          const T* BU = c.p(L.BU);
          for (int q = 0; q < du; ++q) s += BU[i * du + q] * U[(long long)k * du + q];
        }
        rv[i] = ms[i] - s - c.p(L.BV)[i];
      }
      __syncthreads();
      FOR_T(e, n * n) {
        const int i = e / n, j = e - i * n;
        Dm[i * ldn + j] = Ps[i * ldn + j] - Pp[i * ldn + j];
        Q[i * ldn + j] = T(0.5) * (Pp[i * ldn + j] + Pp[j * ldn + i]);  // sym(Pp) (Q no longer needed)
      }
      __syncthreads();
      chol<T>(Q, Lp, n, ldn, T(1e-9));
      chol_solve<T>(Lp, n, ldn, APf, n, ldn);  // APf <- Ct
      const T* Ct = APf;
      T* CD = Pp;  // C (Ps - Pp)
      mm_dmma<T, true, false>(Ct, ldn, Dm, ldn, n, n, n, [&](int i, int j, double v) { CD[i * ldn + j] = (T)v; });
      mm_dmma<T, true, false>(Ct, ldn, Ps, ldn, n, n, n, [&](int i, int j, double v) { Q[i * ldn + j] = (T)v; });  // C P_s^+
      T* msn = c.p(L.YS);
      FOR_T(i, n) {
        T s = T(0);
        for (int q = 0; q < n; ++q) s += Ct[q * ldn + i] * rv[q];
        msn[i] = mf[i] + s;
      }
      __syncthreads();
      if (SCg) {
        // cross = C P_s^+ + m_s m_s^{+T}   (:771)
        FOR_T(e, n * n) {
          const int i = e / n, j = e - i * n;
          SCg[(long long)k * n * n + e] = Q[i * ldn + j] + msn[i] * ms[j];
        }
      }
      __syncthreads();
      mm_dmma<T, false, false>(CD, ldn, Ct, ldn, n, n, n, [&](int i, int j, double v) { Ps[i * ldn + j] = Pf[i * ldn + j] + (T)v; });
      FOR_T(i, n) ms[i] = msn[i];
      __syncthreads();
    } else {
      // backward ODE: aux = psd_solve(P_f, L Qc L^T)^T; G = F_or_J(m_f) + aux; c0 = F m_f or f(m_f)
      T* Lp = c.p(L.W3);
      T* X = c.p(L.W1);
      T* G = c.p(L.J);
      T* Psym = c.p(L.W2);
      T* c0 = c.p(L.C0);
      FOR_T(e, n * n) {
        const int i = e / n, j = e - i * n;
        Psym[i * ldn + j] = T(0.5) * (Pf[i * ldn + j] + Pf[j * ldn + i]);
        X[i * ldn + j] = lql[i * ldn + j];
      }
      __syncthreads();
      chol<T>(Psym, Lp, n, ldn, T(1e-9));
      chol_solve<T>(Lp, n, ldn, X, n, ldn);
      const T* th = c.p(L.TH);
      FOR_T(e, n * n) {
        const int i = e / n, j = e - i * n;
        const T fj = linear ? th[i * ldn + j] : drift_jac<T>(d.drift_id, th, n, i, j, mf);
        G[i * ldn + j] = fj + X[j * ldn + i];
      }
      FOR_T(i, n) {
        if (linear) {
          T s = T(0);
          for (int q = 0; q < n; ++q) s += th[i * ldn + q] * mf[q];
          c0[i] = s;
        } else {
          c0[i] = drift_f<T>(d.drift_id, th, n, i, [&](int q) { return mf[q]; });
        }
      }
      __syncthreads();
      // cd_linear type 2 ignores the user's settings (cd_linear/inference.py:688): host passes defaults in g.tab/d
      if (ode_solve<T>(c, ODE_BACK, ms, L.mpoff + L.nn, T(0), t1 - t0, T(d.dt0), d.max_steps)) status = 2;
      if (SCg) FOR_T(e, n * n) SCg[(long long)k * n * n + e] = T(NAN);  // :792
    }
    FOR_T(i, n) SMg[(long long)k * n + i] = ms[i];
    store_mat<T>(SPg + (long long)k * n * n, Ps, n, n, ldn);
    __syncthreads();
  }
  if (threadIdx.x == 0 && a.out[CDK_OUT_STATUS]) {
    bool bad = false;
    for (int i = 0; i < n; ++i) bad |= !isfinite(ms[i]);
    merge_smoother_status(static_cast<int*>(a.out[CDK_OUT_STATUS]), traj, status, !bad);
  }
}

}  // namespace

template <typename T>
int launch_generic(int algo, const KArgs<T>& a, cudaStream_t s) {
  GArgs<T> g;
  g.k = a;
  g.algo = algo;
  if (algo == ALGO_KF_SMOOTH && a.d.smoother_type == 2) {
    // _smooth passes no diffeqsolve settings: always Dopri5 / dt0 = 0.01 / max_steps = 1e5 (cd_linear/inference.py:688)
    g.k.d.solver = CDK_DOPRI5;
    g.k.d.dt0 = 0.01;
    g.k.d.max_steps = 100000;
  }
  if (!fill_rt_tab(g.k.d.solver, g.tab)) return CDK_E_ENUM;
  g.nslots = g.k.d.solver == CDK_DOPRI5 ? g.tab.S : 1;
  static const int reg_ode_env = []() {
    const char* e = getenv("CDK_GENERIC_REG_ODE");
    return e && e[0] == '0' ? 0 : 1;
  }();
  g.reg_ode = reg_ode_env;
  const int nmax = a.d.n > a.d.m ? a.d.n : a.d.m;
  const int threads = nmax <= 4 ? 32 : (nmax <= 8 ? 64 : (nmax <= 16 ? 128 : 256));
  const bool smooth = algo == ALGO_KF_SMOOTH || algo == ALGO_EKF_SMOOTH;
  // Lorenz-96 moment ODE with a chain tableau: RK state in registers (ode_solve_stencil); CDK_GENERIC_REG_ODE=0 disables
  const cdk_desc& dd = g.k.d;
  const bool dopri = dd.solver == CDK_DOPRI5;
  const bool reg_ode = g.reg_ode && !smooth && dd.drift_id == CDK_DRIFT_LORENZ96 && (g.nslots == 1 || dopri) &&
                       stencil_fits(dd.n, threads) &&
                       ((algo == ALGO_EKF_FILTER && dd.state_order != CDK_ORDER_ZEROTH) || (algo == ALGO_UKF_FILTER && ukf_closed(dd)));
  // on the register path Dopri5 keeps its stage increments in registers: the shared-memory layout is the one-slot one
  if (reg_ode && dopri) g.nslots = 1;
  g.lay = Lay(g.k.d, algo, g.nslots, reg_ode);
  const Lay& L = g.lay;
  const size_t smem = (size_t)L.total * sizeof(T);
  int dev = 0, max_optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (smem > (size_t)max_optin) return CDK_E_SIZE;
  auto kern = smooth ? generic_smooth_kernel<T>
                     : (reg_ode ? (dopri ? generic_filter_kernel<T, 2> : generic_filter_kernel<T, 1>) : generic_filter_kernel<T, 0>);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return check_launch("cudaFuncSetAttribute(generic)");
  }
  if (a.d.N > 2147483647LL) return CDK_E_SIZE;
  kern<<<(unsigned)a.d.N, threads, smem, s>>>(g);
  note_launch();
  return check_launch(smooth ? "generic_smooth_kernel" : "generic_filter_kernel");
}

bool has_user_drift() { return CDK_HAS_USER_DRIFT != 0; }
bool has_user_emission() { return CDK_HAS_USER_EMISSION != 0; }
int user_emission_params(int n, int m) {
#if CDK_HAS_USER_EMISSION
  return cdk_user_emission::num_params(n, m);
#else
  return -1;
#endif
}

template int launch_generic<double>(int, const KArgs<double>&, cudaStream_t);
template int launch_generic<float>(int, const KArgs<float>&, cudaStream_t);

}  // namespace cdk
