// cdk_ekfgrad.cu -- reverse-mode gradient of the CD-EKF and closed-form CD-UKF log-likelihoods for every registry drift
// and emission size (cdk_ekf_grad_dense_f64, cdk_ukf_grad_dense_f64): ONE CTA PER TRAJECTORY, like generic_filter_kernel.
//
// The forward pass is the filter launch cdk_ekf_filter_f64 (cdk_ukf_filter_f64) makes, with its filtered and predicted
// moments written to the scratch.  ekf_grad_dense_kernel then walks k = K-1 .. 0 with the cotangent (mu_bar, P_bar) of the moments entering
// update k+1:
//   update VJP      both Cholesky factors recomputed from the stored predicted moments (the un-boosted one of the
//                   log-density, sym(S) + 1e-9 I of the gain); accumulates H_bar, d_bar, R_bar;
//   moment-ODE VJP  the gap is re-integrated from the stored filtered moments (StepClock rule), the substep start states
//                   kept at two checkpoint levels of EG_CK slots, then stepped back substep by substep and stage by
//                   stage for any tableau: kbar_i = b_i ybar + sum_{j>i} a_ji Ybar_j.  Stage inputs, stage cotangents
//                   and checkpoints live in the trajectory's slice of the scratch (L2-resident); shared memory holds
//                   the model, the gradient accumulators and a few n x n working matrices.
// The right-hand side is dm = f(m) [+ 0.5 g^T P], dP = J P + (J P)^T + Sigma; its VJP for a cotangent (a, A) is
//   As = A + A^T,  P_bar = J^T As [+ 0.5 g a^T],  Jb = As P^T,  m_bar = J^T a + x-contraction(Jb),
//   theta_bar += theta-contraction(a, Jb),  Sigma_bar += A
// with the registry contractions of cdk_dense.cuh.  The gap after the last observation does not affect the
// log-likelihood and is not differentiated.  A user drift (CDK_DRIFT_USER, in a variant built with
// build_user_drift(code, grad=True)) replaces the registry contractions by dual-number evaluations of its own code
// (eg_user_vjp, cdk_dual.cuh, DESIGN 4.2f); all of that is compiled only under CDK_HAS_USER_DRIFT.
//
// UKF mode (EgArgs::ukf).  The closed-form unscented predict (cdk_generic.cu, ODE_UKFC) replaces the bracketed EKF term
// by the exact half-trace 0.5 tr(Hess f . sym P) (drift_half_trhp, for every drift whatever state_order says), whose VJP
// adds 0.5 sum_r a_r Hess f_r to P_bar and, for the quadratic drift, a_r sym(P) to C_bar_r.  The update VJP is the EKF's,
// symmetrisation of P_f_bar included, although the UKF update leaves P_f unsymmetrised: the parameters only ever move the
// covariances along symmetric directions (Sigma, R and P0 get symmetric parts), and on symmetric moments the UKF update
// is, in exact arithmetic, the EKF update -- P - Kt^T S Kt is then symmetric -- so the two updates have the same
// derivative along every direction the parameter gradient sees.  The forward's rounding-level antisymmetric part of P
// is carried unchanged across a gap by the symmetric right-hand side, here as in the filter.  The torch reference
// (oracle/cd_torch_ukf.py) differentiates the unsymmetrised update literally and pins the gradient.
#include "cdk_dense.cuh"
#if CDK_HAS_USER_DRIFT
#include "cdk_dual.cuh"
#endif

namespace cdk {
namespace {

constexpr int EG_CK = 32;  // checkpoint slots per level: a gap of up to EG_CK^2 substeps is re-integrated once
constexpr int EG_CLOCK = (int)((sizeof(StepClock<double>) + 7) / 8);

__host__ __device__ inline int eg_threads(int n, int m) {
  const int nmax = n > m ? n : m;
  return nmax <= 4 ? 32 : (nmax <= 8 ? 64 : (nmax <= 16 ? 128 : 256));
}

#if CDK_HAS_USER_DRIFT
// Directions seeded per dual evaluation of the user's drift (the W of cdk_dual::Dual; see DESIGN 4.2f for the choice).
constexpr int EG_DW = 8;
using EgDual = cdk_dual::Dual<EG_DW>;
#endif

// Shared-memory layout (doubles), computed on the host.  A moment state [mu | P] has st = mpoff + n * ldn entries, the
// layout of generic_filter_kernel.  With m <= n the update's [m x n] buffers alias ODE buffers that are idle then.
struct EgLay {
  int n, m, ldn, ldm, nn, mpoff, st, nth, S;
  int TH, THB, LQL, H, R, DV, SIGB, HB, RB, DB, YC, YS, KS, ACC, YB, J, W1, W2;
  int G, KT, U, GB, SM, L0, LB, SI, SB, RV, ZV, RBV, YV, CLK, total;
#if CDK_HAS_USER_DRIFT
  int DU, PART, WQ, GV;
#endif
  EgLay() = default;
  __host__ __device__ EgLay(const cdk_desc& d, int stages) {
    n = d.n; m = d.m; ldn = ldp(n); ldm = ldp(m); nn = n * ldn; nth = d.n_theta; S = stages;
    mpoff = (n + 1) & ~1;
    st = mpoff + nn;
    int o = 0;
    auto take = [&](int cnt) { int r = o; o += (cnt + 1) & ~1; return r; };
    TH = take(nth); THB = take(nth); LQL = take(nn); H = take(m * ldn); R = take(m * ldm); DV = take(m);
    SIGB = take(nn); HB = take(m * ldn); RB = take(m * ldm); DB = take(m);
    YC = take(st); YS = take(st); KS = take(st); ACC = take(st); YB = take(st);
    J = take(nn); W1 = take(nn); W2 = take(nn);
    if (m <= n) {
      G = YS; KT = KS; U = ACC; GB = J;
    } else {
      G = take(m * ldn); KT = take(m * ldn); U = take(m * ldn); GB = take(m * ldn);
    }
    SM = take(m * ldm); L0 = take(m * ldm); LB = take(m * ldm); SI = take(m * ldm); SB = take(m * ldm);
    RV = take(m); ZV = take(m); RBV = take(m); YV = take(m);
    CLK = take(2 * EG_CK * EG_CLOCK);
#if CDK_HAS_USER_DRIFT
    // user drift: one dual copy of [x | theta] for the CTA, one partial sum of EG_DW tangents per thread, w_q and g(x)
    DU = PART = WQ = GV = 0;
    if (d.drift_id == CDK_DRIFT_USER) {
      DU = take((n + nth) * (EG_DW + 1));
      PART = take(eg_threads(n, m) * EG_DW);
      WQ = take(n);
      GV = take(n);
    }
#endif
    total = o;
  }
  // per-trajectory backward scratch (doubles): checkpoints at two levels, stage inputs, stage cotangents
  __host__ __device__ long long bwd() const { return (long long)(2 * EG_CK + 2 * S) * st; }
};

struct EgArgs {
  KArgs<double> k;
  RtTab tab;
  double a[6][6];  // dense Butcher matrix
  EgLay lay;
  double* sc;      // scratch: FM | FP | PM | PP ([N][K][...] each), then N backward slices
  const int* status;
  double* grad;
  int cols;
  int ukf;         // the closed-form UKF's predict (half-trace mean term) instead of the EKF's
};

struct Eg {
  const EgArgs& g;
  const EgLay& L;
  double* sh;
  __device__ Eg(const EgArgs& g_, double* sh_) : g(g_), L(g_.lay), sh(sh_) {}
  __device__ double* p(int off) const { return sh + off; }
  __device__ bool second() const {
#if CDK_HAS_USER_DRIFT
    if (g.k.d.drift_id == CDK_DRIFT_USER) return !g.ukf && g.k.d.state_order == CDK_ORDER_SECOND;
#endif
    return !g.ukf && g.k.d.state_order == CDK_ORDER_SECOND && g.k.d.drift_id == CDK_DRIFT_QUADRATIC;
  }
};

// k = dt * rhs(y), y and k in shared memory.  Ends with a barrier.
__device__ void eg_rhs(const Eg& c, const double* y, double* k, double dt) {
  const EgLay& L = c.L;
  const int n = L.n, ld = L.ldn, id = c.g.k.d.drift_id;
  const double* th = c.p(L.TH);
  const double* lql = c.p(L.LQL);
  const double* P = y + L.mpoff;
  double* J = c.p(L.J);
  double* JP = c.p(L.W1);
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    J[i * ld + j] = drift_jac<double>(id, th, n, i, j, y);
  }
  __syncthreads();
  mm_dmma<double, false, false>(J, ld, P, ld, n, n, n, [&](int i, int j, double v) { JP[i * ld + j] = v; });
  const bool second = c.second();
  FOR_T(i, n) {
    double f = drift_f<double>(id, th, n, i, [&](int j) { return y[j]; });
    if (second) {
      double s = 0.0;
#if CDK_HAS_USER_DRIFT
      if (id == CDK_DRIFT_USER) {  // the x-dependent g(x) of the filter (cdk_generic.cu, ODE_EKF)
        for (int q = 0; q < n; ++q) s += cdk_user::graddiv<double>(th, n, q, y) * P[q * ld + i];
      } else
#endif
      for (int q = 0; q < n; ++q) s += drift_graddiv<double>(id, th, n, q) * P[q * ld + i];
      f += 0.5 * s;
    }
    if (c.g.ukf) f += drift_half_trhp<double>(id, th, n, i, P, ld);
    k[i] = dt * f;
  }
  __syncthreads();
  double* kP = k + L.mpoff;
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    kP[i * ld + j] = dt * ((JP[i * ld + j] + JP[j * ld + i]) + lql[i * ld + j]);
  }
  __syncthreads();
}

#if CDK_HAS_USER_DRIFT
// The mean and parameter cotangents of eg_rhs_vjp for the user drift, from dual evaluations of its own f / jac / graddiv
// at the stage input y (J, Jb and outP = J^T As are in place).  With w_q = 0.5 sum_i P_qi a_i ('second' order only):
//   m_bar_l      = (J^T a)_l + sum_ik Jb_ik dJ_ik/dx_l + sum_q w_q dg_q/dx_l
//   theta_bar_e += sum_i a_i df_i/dtheta_e + sum_ik Jb_ik dJ_ik/dtheta_e + sum_q w_q dg_q/dtheta_e
//   P_bar       += 0.5 g(x) a^T
// The n + n_theta directions (x, then theta) are seeded EG_DW at a time into the CTA's one dual copy of [x | theta];
// for each chunk the threads share out the evaluations (jac (i, k), f i, graddiv q), each sums its weighted tangents in
// registers, and one thread per direction adds the per-thread partial sums in thread order: the result is the same bits
// from run to run.  Ends with a barrier.
__device__ void eg_user_vjp(const Eg& c, const double* y, const double* ab, const double* Jb, double* out, double* outP,
                            bool second) {
  const EgLay& L = c.L;
  const int n = L.n, ld = L.ldn, nv = n + L.nth;
  const double* th = c.p(L.TH);
  const double* P = y + L.mpoff;
  const double* J = c.p(L.J);
  double* wq = c.p(L.WQ);
  double* gv = c.p(L.GV);
  double* part = c.p(L.PART);
  double* thb = c.p(L.THB);
  EgDual* xd = reinterpret_cast<EgDual*>(c.p(L.DU));
  EgDual* td = xd + n;
  FOR_T(l, n) {
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += J[i * ld + l] * ab[i];
    out[l] = s;
    if (second) {
      double w = 0.0;
      for (int i = 0; i < n; ++i) w += P[l * ld + i] * ab[i];
      wq[l] = 0.5 * w;
      gv[l] = cdk_user::graddiv<double>(th, n, l, y);
    }
  }
  FOR_T(v, nv) xd[v] = EgDual(v < n ? y[v] : th[v - n]);
  __syncthreads();
  if (second) {
    FOR_T(e, n * n) {
      const int q = e / n, l = e - q * n;
      outP[q * ld + l] += 0.5 * gv[q] * ab[l];
    }
  }
  const int nj = n * n, E = nj + n + (second ? n : 0);
  for (int c0 = 0; c0 < nv; c0 += EG_DW) {
    FOR_T(e, nv * EG_DW) {
      const int v = e / EG_DW, w = e - v * EG_DW;
      xd[v].d[w] = c0 + w == v ? 1.0 : 0.0;
    }
    __syncthreads();
    const bool fth = c0 + EG_DW > n;  // the chunk holds parameter directions: f's tangents enter (its x-tangents are J)
    double acc[EG_DW];
#pragma unroll
    for (int w = 0; w < EG_DW; ++w) acc[w] = 0.0;
    for (int e = threadIdx.x; e < E; e += blockDim.x) {
      if (e < nj) {
        const int i = e / n, k = e - i * n;
        const EgDual v = cdk_user::jac<EgDual>(td, n, i, k, xd);
        const double wt = Jb[i * ld + k];
#pragma unroll
        for (int w = 0; w < EG_DW; ++w) acc[w] += wt * v.d[w];
      } else if (e < nj + n) {
        if (!fth) continue;
        const int i = e - nj;
        const EgDual v = cdk_user::f<EgDual>(td, n, i, [&](int j) { return xd[j]; });
        const double wt = ab[i];
#pragma unroll
        for (int w = 0; w < EG_DW; ++w)
          if (c0 + w >= n) acc[w] += wt * v.d[w];
      } else {
        const int q = e - nj - n;
        const EgDual v = cdk_user::graddiv<EgDual>(td, n, q, xd);
        const double wt = wq[q];
#pragma unroll
        for (int w = 0; w < EG_DW; ++w) acc[w] += wt * v.d[w];
      }
    }
#pragma unroll
    for (int w = 0; w < EG_DW; ++w) part[threadIdx.x * EG_DW + w] = acc[w];
    __syncthreads();
    FOR_T(w, EG_DW) {
      const int v = c0 + w;
      if (v < nv) {
        double s = 0.0;
        for (int t = 0; t < (int)blockDim.x; ++t) s += part[t * EG_DW + w];
        if (v < n) out[v] += s; else thb[v - n] += s;
      }
    }
  }
  __syncthreads();
}
#endif

// VJP of the right-hand side at y (shared) for the cotangent kb (shared, already scaled by dt): writes the cotangent of y
// to `out` (the stage's slot in the scratch) and accumulates theta_bar and Sigma_bar.  Ends with a barrier.
__device__ void eg_rhs_vjp(const Eg& c, const double* y, const double* kb, double* out) {
  const EgLay& L = c.L;
  const int n = L.n, ld = L.ldn, id = c.g.k.d.drift_id;
  const double* th = c.p(L.TH);
  const double* P = y + L.mpoff;
  const double* ab = kb;
  const double* Ab = kb + L.mpoff;
  double* J = c.p(L.J);
  double* As = c.p(L.W1);
  double* Jb = c.p(L.W2);
  double* sigb = c.p(L.SIGB);
  double* outP = out + L.mpoff;
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    J[i * ld + j] = drift_jac<double>(id, th, n, i, j, y);
    As[i * ld + j] = Ab[i * ld + j] + Ab[j * ld + i];
    sigb[i * ld + j] += Ab[i * ld + j];
  }
  __syncthreads();
  mm_dmma<double, true, false>(J, ld, As, ld, n, n, n, [&](int i, int j, double v) { outP[i * ld + j] = v; });  // J^T As
  mm_dmma<double, false, true>(As, ld, P, ld, n, n, n, [&](int i, int j, double v) { Jb[i * ld + j] = v; });    // As P^T
  __syncthreads();
  const bool second = c.second();
#if CDK_HAS_USER_DRIFT
  if (id == CDK_DRIFT_USER) {
    eg_user_vjp(c, y, ab, Jb, out, outP, second);
    return;
  }
#endif
  FOR_T(l, n) {
    double s = drift_jac_vjp_x<double>(id, th, n, l, Jb, ld);
    for (int i = 0; i < n; ++i) s += J[i * ld + l] * ab[i];
    out[l] = s;
  }
  if (second) {
    FOR_T(e, n * n) {
      const int q = e / n, l = e - q * n;
      outP[q * ld + l] += 0.5 * drift_graddiv<double>(id, th, n, q) * ab[l];
    }
  }
  const bool ukf = c.g.ukf;
  if (ukf) {
    FOR_T(e, n * n) {
      const int q = e / n, l = e - q * n;
      outP[q * ld + l] += drift_half_trhp_vjp_p<double>(id, th, n, q, l, ab);
    }
  }
  double* thb = c.p(L.THB);
  FOR_T(e, L.nth) {
    thb[e] += drift_theta_vjp<double>(id, th, n, e, y, ab, Jb, ld, P, second);
    if (ukf) thb[e] += drift_half_trhp_vjp_theta<double>(id, n, e, ab, P, ld);
  }
  __syncthreads();
}

// One substep of the state YC (in place) through the stages of any tableau; the stage inputs are left in stg[s * st].
__device__ void eg_step(const Eg& c, double dt, double* __restrict__ stg) {
  const EgLay& L = c.L;
  const int st = L.st, S = L.S;
  double* y = c.p(L.YC);
  double* ys = c.p(L.YS);
  double* k = c.p(L.KS);
  double* acc = c.p(L.ACC);
  FOR_T(e, st) {
    acc[e] = y[e];
    for (int s = 0; s < S; ++s) stg[s * st + e] = y[e];
  }
  for (int s = 0; s < S; ++s) {
    FOR_T(e, st) ys[e] = stg[s * st + e];
    __syncthreads();
    eg_rhs(c, ys, k, dt);
    const double b = c.g.tab.b[s];
    FOR_T(e, st) {
      const double kv = k[e];
      if (b != 0.0) acc[e] += b * kv;
      for (int s2 = s + 1; s2 < S; ++s2) {
        const double a = c.g.a[s2][s];
        if (a != 0.0) stg[s2 * st + e] += a * kv;
      }
    }
    __syncthreads();
  }
  FOR_T(e, st) y[e] = acc[e];
  __syncthreads();
}

// VJP of the substep eg_step just took (stage inputs in stg): YB is the cotangent of its end state on entry and of its
// start state on exit.  stb[s * st] receives the stage-input cotangents.
__device__ void eg_step_vjp(const Eg& c, double dt, const double* __restrict__ stg, double* __restrict__ stb) {
  const EgLay& L = c.L;
  const int st = L.st, S = L.S;
  double* yb = c.p(L.YB);
  double* ys = c.p(L.YS);
  double* kb = c.p(L.KS);
  for (int s = S - 1; s >= 0; --s) {
    const double b = c.g.tab.b[s];
    FOR_T(e, st) {
      double v = b * yb[e];
      for (int s2 = s + 1; s2 < S; ++s2) {
        const double a = c.g.a[s2][s];
        if (a != 0.0) v += a * stb[s2 * st + e];
      }
      kb[e] = dt * v;
      ys[e] = stg[s * st + e];
    }
    __syncthreads();
    eg_rhs_vjp(c, ys, kb, stb + s * st);
  }
  FOR_T(e, st) {
    double v = yb[e];
    for (int s = 0; s < S; ++s) v += stb[s * st + e];
    yb[e] = v;
  }
  __syncthreads();
}

// VJP of the measurement update (condition_on, num_iter = 1, then the symmetrisation) at the predicted moments in YC for
// the emission in YV: YB holds the cotangent of the filtered moments on entry and of the predicted ones on exit, plus
// the log-density's own derivative.  Accumulates H_bar, d_bar, R_bar.
__device__ void eg_update_vjp(const Eg& c) {
  const EgLay& L = c.L;
  const int n = L.n, m = L.m, ldn = L.ldn, ldm = L.ldm;
  const double* mu = c.p(L.YC);
  const double* P = mu + L.mpoff;
  double* mub = c.p(L.YB);
  double* Pb = mub + L.mpoff;
  const double* H = c.p(L.H);
  const double* R = c.p(L.R);
  const double* dv = c.p(L.DV);
  const double* yv = c.p(L.YV);
  double* G = c.p(L.G);    // H P
  double* Kt = c.p(L.KT);  // (sym(S) + 1e-9 I)^-1 H P
  double* U = c.p(L.U);    // Kt P_f_bar, then S_bar H + G_bar
  double* Gb = c.p(L.GB);  // K_bar^T, then G_bar = (sym(S) + 1e-9 I)^-1 K_bar^T
  double* Sm = c.p(L.SM);
  double* L0 = c.p(L.L0);
  double* Lb = c.p(L.LB);
  double* Si = c.p(L.SI);
  double* Sb = c.p(L.SB);
  double* rv = c.p(L.RV);
  double* zv = c.p(L.ZV);
  double* rb = c.p(L.RBV);
  double* W1 = c.p(L.W1);
  FOR_T(e, n * n) {  // the filter symmetrises P_f
    const int i = e / n, j = e - i * n;
    if (i < j) {
      const double v = 0.5 * (Pb[i * ldn + j] + Pb[j * ldn + i]);
      Pb[i * ldn + j] = v;
      Pb[j * ldn + i] = v;
    }
  }
  mm_dmma<double, false, false>(H, ldn, P, ldn, m, n, n, [&](int a, int j, double v) { G[a * ldn + j] = v; });
  FOR_T(a, m) {
    double s = dv[a];
    for (int q = 0; q < n; ++q) s += H[a * ldn + q] * mu[q];
    rv[a] = yv[a] - s;
  }
  __syncthreads();
  mm_dmma<double, false, true>(G, ldn, H, ldn, m, m, n, [&](int a, int b, double v) { Sm[a * ldm + b] = R[a * ldm + b] + v; });
  __syncthreads();
  chol_prep<double, false>(Sm, L0, m, ldm, 0.0);
  chol_prep<double, true>(Sm, Lb, m, ldm, 1e-9);
  FOR_T(e, m * m) {
    const int a = e / m, b = e - a * m;
    Si[a * ldm + b] = a == b ? 1.0 : 0.0;
  }
  __syncthreads();
  chol_warp<double>(0, L0, m, ldm);
  chol_warp<double>(blockDim.x > 32 ? 1 : 0, Lb, m, ldm);
  __syncthreads();
  chol_solve<double>(L0, m, ldm, Si, m, ldm);     // S^-1
  chol_solve<double>(Lb, m, ldm, G, Kt, n, ldn);  // Kt
  FOR_T(a, m) {  // z = S^-1 r;  r_bar = Kt mu_f_bar - z
    double z = 0.0, kb = 0.0;
    for (int b = 0; b < m; ++b) z += Si[a * ldm + b] * rv[b];
    for (int q = 0; q < n; ++q) kb += Kt[a * ldn + q] * mub[q];
    zv[a] = z;
    rb[a] = kb - z;
  }
  mm_dmma<double, false, false>(Kt, ldn, Pb, ldn, m, n, n, [&](int a, int j, double v) { U[a * ldn + j] = v; });
  __syncthreads();
  // S_bar = 0.5 z z^T - 0.5 S^-1 - Kt P_f_bar Kt^T;  K_bar^T = r mu_f_bar^T - 2 S Kt P_f_bar
  mm_dmma<double, false, true>(U, ldn, Kt, ldn, m, m, n, [&](int a, int b, double v) {
    Sb[a * ldm + b] = 0.5 * zv[a] * zv[b] - 0.5 * Si[a * ldm + b] - v;
  });
  mm_dmma<double, false, false>(Sm, ldm, U, ldn, m, n, m, [&](int a, int j, double v) { Gb[a * ldn + j] = rv[a] * mub[j] - 2.0 * v; });
  __syncthreads();
  chol_solve<double>(Lb, m, ldm, Gb, n, ldn);  // G_bar
  mm_dmma<double, false, true>(Gb, ldn, Kt, ldn, m, m, n, [&](int a, int b, double v) { L0[a * ldm + b] = v; });  // G_bar Kt^T
  __syncthreads();
  double* RBg = c.p(L.RB);
  FOR_T(e, m * m) {  // S_bar -= sym(G_bar Kt^T)
    const int a = e / m, b = e - a * m;
    const double v = Sb[a * ldm + b] - 0.5 * (L0[a * ldm + b] + L0[b * ldm + a]);
    Sb[a * ldm + b] = v;
    RBg[a * ldm + b] += v;
  }
  __syncthreads();
  double* HBg = c.p(L.HB);
  mm_dmma<double, false, false>(Sb, ldm, G, ldn, m, n, m, [&](int a, int j, double v) { HBg[a * ldn + j] += 2.0 * v; });
  __syncthreads();
  mm_dmma<double, false, false>(Gb, ldn, P, ldn, m, n, n, [&](int a, int j, double v) {
    HBg[a * ldn + j] += v - rb[a] * mu[j];
  });
  mm_dmma<double, false, false>(Sb, ldm, H, ldn, m, n, m, [&](int a, int j, double v) { U[a * ldn + j] = v + Gb[a * ldn + j]; });
  double* DBg = c.p(L.DB);
  FOR_T(a, m) DBg[a] -= rb[a];
  FOR_T(l, n) {  // mu_bar = mu_f_bar - H^T r_bar
    double s = 0.0;
    for (int a = 0; a < m; ++a) s += H[a * ldn + l] * rb[a];
    mub[l] -= s;
  }
  __syncthreads();
  mm_dmma<double, true, false>(H, ldn, U, ldn, n, n, m, [&](int i, int j, double v) { W1[i * ldn + j] = v; });
  __syncthreads();
  FOR_T(e, n * n) {  // P_bar = P_f_bar + sym(H^T (S_bar H + G_bar))
    const int i = e / n, j = e - i * n;
    Pb[i * ldn + j] += 0.5 * (W1[i * ldn + j] + W1[j * ldn + i]);
  }
  __syncthreads();
}

__device__ void eg_load(double* dst, const double* __restrict__ src, int st) {
  FOR_T(e, st) dst[e] = src[e];
}
__device__ void eg_save(double* __restrict__ dst, const double* src, int st) {
  FOR_T(e, st) dst[e] = src[e];
}

__global__ void __launch_bounds__(256) ekf_grad_dense_kernel(const EgArgs g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Eg c(g, reinterpret_cast<double*>(smem_raw));
  const EgLay& L = c.L;
  const KArgs<double>& a = g.k;
  const cdk_desc& d = a.d;
  const int n = L.n, m = L.m, ldn = L.ldn, ldm = L.ldm, st = L.st, K = d.K;
  const long long traj = blockIdx.x;
  double* grow = g.grad + traj * (long long)g.cols;
  if (g.status[traj] != 0) {
    FOR_T(e, g.cols) grow[e] = NAN;
    return;
  }
  FOR_T(e, L.total) c.sh[e] = 0.0;
  __syncthreads();
  auto src = [&](int slot) { return a.in[slot] + traj * a.in_stride[slot]; };
  {  // model: theta, H, R, d and L Qc L^T (J, W1, W2 as scratch)
    FOR_T(i, L.nth) c.p(L.TH)[i] = src(CDK_IN_F)[i];
    FOR_T(e, m * n) c.p(L.H)[(e / n) * ldn + e % n] = src(CDK_IN_H)[e];
    FOR_T(e, m * m) c.p(L.R)[(e / m) * ldm + e % m] = src(CDK_IN_R)[e];
    FOR_T(i, m) c.p(L.DV)[i] = src(CDK_IN_D)[i];
    double* Lm = c.p(L.J);
    double* Qc = c.p(L.W1);
    double* LQ = c.p(L.W2);
    FOR_T(e, n * n) {
      Lm[(e / n) * ldn + e % n] = src(CDK_IN_L)[e];
      Qc[(e / n) * ldn + e % n] = src(CDK_IN_QC)[e];
    }
    __syncthreads();
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      double s = 0.0;
      for (int q = 0; q < n; ++q) s += Lm[i * ldn + q] * Qc[q * ldn + j];
      LQ[i * ldn + j] = s;
    }
    __syncthreads();
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      double s = 0.0;
      for (int q = 0; q < n; ++q) s += LQ[i * ldn + q] * Lm[j * ldn + q];
      c.p(L.LQL)[i * ldn + j] = s;
    }
    __syncthreads();
  }
  const long long NK = d.N * (long long)K;
  const double* FMg = g.sc + traj * (long long)K * n;
  const double* FPg = g.sc + NK * n + traj * (long long)K * n * n;
  const double* PMg = g.sc + NK * (n + n * n) + traj * (long long)K * n;
  const double* PPg = g.sc + NK * (2 * n + n * n) + traj * (long long)K * n * n;
  double* ck1 = g.sc + NK * (2 * n + 2 * n * n) + traj * L.bwd();
  double* ck2 = ck1 + EG_CK * st;
  double* stg = ck2 + EG_CK * st;
  double* stb = stg + L.S * st;
  StepClock<double>* ckc1 = reinterpret_cast<StepClock<double>*>(c.p(L.CLK));
  StepClock<double>* ckc2 = reinterpret_cast<StepClock<double>*>(c.p(L.CLK) + EG_CK * EG_CLOCK);
  FOR_T(e, L.S * st) stb[e] = 0.0;  // the padding entries are never written by the stage VJP
  const double* Y = a.in[CDK_IN_Y] + traj * a.in_stride[CDK_IN_Y];
  const double* Tm = a.in[CDK_IN_T] + traj * a.in_stride[CDK_IN_T];
  const double dt0 = d.dt0;
  double* yc = c.p(L.YC);
  auto load_moments = [&](const double* mg, const double* pg) {
    FOR_T(i, n) yc[i] = mg[i];
    FOR_T(e, n * n) yc[L.mpoff + (e / n) * ldn + e % n] = pg[e];
    __syncthreads();
  };
  for (int k = K - 1; k >= 0; --k) {
    if (k < K - 1) {
      // ---- gap [t_k, t_{k+1}]: forward from the filtered moments, substep starts at checkpoint level 1 ----
      const double t0 = Tm[k], t1 = Tm[k + 1];
      StepClock<double> cnt(t0, t1, dt0);
      while (cnt.running()) cnt.advance();  // status 0: the filter took these cnt.n <= max_steps substeps
      const int q = cnt.n;
      const int s1 = q > EG_CK ? (q + EG_CK - 1) / EG_CK : 1;
      if (q > 0) {
        load_moments(FMg + (long long)k * n, FPg + (long long)k * n * n);
        StepClock<double> clk(t0, t1, dt0);
        for (int i = 0; i < q; ++i) {
          if (i % s1 == 0) {
            eg_save(ck1 + (i / s1) * st, yc, st);
            if (threadIdx.x == 0) ckc1[i / s1] = clk;
          }
          eg_step(c, clk.dt(), stg);
          clk.advance();
        }
      }
      const int nseg = q > 0 ? (q + s1 - 1) / s1 : 0;
      for (int seg = nseg - 1; seg >= 0; --seg) {
        const int i0 = seg * s1, len = q - i0 < s1 ? q - i0 : s1;
        const int s2 = len > EG_CK ? (len + EG_CK - 1) / EG_CK : 1;
        if (len > 1) {  // level 2: the substep starts of this segment
          StepClock<double> clk = ckc1[seg];
          eg_load(yc, ck1 + seg * st, st);
          __syncthreads();
          for (int u = 0; u < len - 1; ++u) {
            if (u % s2 == 0) {
              eg_save(ck2 + (u / s2) * st, yc, st);
              if (threadIdx.x == 0) ckc2[u / s2] = clk;
            }
            eg_step(c, clk.dt(), stg);
            clk.advance();
          }
          if ((len - 1) % s2 == 0) {
            eg_save(ck2 + ((len - 1) / s2) * st, yc, st);
            if (threadIdx.x == 0) ckc2[(len - 1) / s2] = clk;
          }
          __syncthreads();
        }
        for (int u = len - 1; u >= 0; --u) {
          StepClock<double> clk = len > 1 ? ckc2[u / s2] : ckc1[seg];
          eg_load(yc, len > 1 ? ck2 + (u / s2) * st : ck1 + seg * st, st);
          __syncthreads();
          for (int v = (len > 1 ? (u / s2) * s2 : u); v < u; ++v) {
            eg_step(c, clk.dt(), stg);
            clk.advance();
          }
          eg_step(c, clk.dt(), stg);  // the stage inputs of substep i0 + u
          eg_step_vjp(c, clk.dt(), stg, stb);
        }
      }
    }
    // ---- update VJP at k, from the predicted moments entering it ----
    if (k == 0) {
      load_moments(src(CDK_IN_M0), src(CDK_IN_P0));
    } else {
      load_moments(PMg + (long long)(k - 1) * n, PPg + (long long)(k - 1) * n * n);
    }
    FOR_T(i, m) c.p(L.YV)[i] = Y[(long long)k * m + i];
    __syncthreads();
    eg_update_vjp(c);
  }
  // ---- gradient row: theta | Sigma (sym) | H | d | R (sym) | m0 | P0 (sym) ----
  const double* sigb = c.p(L.SIGB);
  const double* HB = c.p(L.HB);
  const double* RB = c.p(L.RB);
  const double* yb = c.p(L.YB);
  const int nth = L.nth;
  FOR_T(e, nth) grow[e] = c.p(L.THB)[e];
  double* gS = grow + nth;
  double* gH = gS + n * n;
  double* gd = gH + m * n;
  double* gR = gd + m;
  double* gm0 = gR + m * m;
  double* gP0 = gm0 + n;
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    gS[e] = 0.5 * (sigb[i * ldn + j] + sigb[j * ldn + i]);
    gP0[e] = 0.5 * (yb[L.mpoff + i * ldn + j] + yb[L.mpoff + j * ldn + i]);
  }
  FOR_T(e, m * n) gH[e] = HB[(e / n) * ldn + e % n];
  FOR_T(i, m) gd[i] = c.p(L.DB)[i];
  FOR_T(e, m * m) {
    const int i = e / m, j = e - i * m;
    gR[e] = 0.5 * (RB[i * ldm + j] + RB[j * ldm + i]);
  }
  FOR_T(i, n) gm0[i] = yb[i];
}

}  // namespace

// The layout of the scratch and shared memory of cdk_ekf_grad_dense_f64 and cdk_ukf_grad_dense_f64 for `d` (false: beyond
// the 227 KB of one CTA)
static bool eg_layout(const cdk_desc& d, EgLay& lay, RtTab& rt) {
  if (!fill_rt_tab(d.solver, rt)) return false;
  lay = EgLay(d, rt.S);
  return (size_t)lay.total * sizeof(double) <= 227u * 1024u;
}

bool ekf_grad_dense_fits(const cdk_desc& d) {
  EgLay lay;
  RtTab rt;
  return eg_layout(d, lay, rt);
}

bool ekf_grad_has_user_drift() { return CDK_HAS_USER_DRIFT != 0; }

long long ekf_grad_dense_scratch_doubles(const cdk_desc& d) {
  EgLay lay;
  RtTab rt;
  eg_layout(d, lay, rt);
  return d.N * ((long long)d.K * (2 * d.n + 2 * d.n * d.n) + lay.bwd() + 1);
}

// The backward launch behind a forward filter pass whose moments are in out[CDK_OUT_SCRATCH] and whose status is `status`;
// `ukf`: the forward pass was the closed-form UKF filter.
int launch_ekf_grad_dense(const KArgs<double>& a, const int* status, double* grad, bool ukf, cudaStream_t s) {
  EgArgs g;
  g.k = a;
  if (!eg_layout(a.d, g.lay, g.tab)) return CDK_E_SIZE;
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j < 6; ++j) g.a[i][j] = 0.0;
  for (int i = 0; i < g.tab.S; ++i)
    for (int q = 0; q < g.tab.nnz[i]; ++q) g.a[i][g.tab.col[i][q]] = g.tab.val[i][q];
  g.sc = static_cast<double*>(a.out[CDK_OUT_SCRATCH]);
  g.status = status;
  g.grad = grad;
  g.cols = CDK_GRAD_COLS_EKF(a.d.n, a.d.m, a.d.n_theta);
  g.ukf = ukf ? 1 : 0;
  const int threads = eg_threads(a.d.n, a.d.m);
  const size_t smem = (size_t)g.lay.total * sizeof(double);
  if (smem > 48 * 1024 && cudaFuncSetAttribute(ekf_grad_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("cudaFuncSetAttribute(ekf_grad_dense_kernel)");
  if (a.d.N > 2147483647LL) return CDK_E_SIZE;
  ekf_grad_dense_kernel<<<(unsigned)a.d.N, threads, smem, s>>>(g);
  note_launch();
  return check_launch("ekf_grad_dense_kernel");
}

}  // namespace cdk
