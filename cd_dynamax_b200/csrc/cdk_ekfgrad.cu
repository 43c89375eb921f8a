// cdk_ekfgrad.cu -- reverse-mode gradient of the CD-EKF, closed-form CD-UKF and sigma-point CD-UKF log-likelihoods for
// every registry drift and emission size (cdk_ekf_grad_dense_f64, cdk_ukf_grad_dense_f64, cdk_ukf_grad_sigma_f64; the
// last also for user drifts): ONE CTA PER TRAJECTORY, like generic_filter_kernel.  The sigma-point predict's right-hand
// side and its VJP are described at eg_sigma_rhs_vjp (ukf_sigma_grad_kernel, DESIGN 4.2g).
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
// (eg_user_vjp, cdk_dual.cuh, DESIGN 4.2f); all of that is compiled only under CDK_HAS_USER_DRIFT.  A user emission
// (CDK_EMISSION_USER, in a variant built with build_variant(..., emission_grad=True)) re-linearises h at every step's
// predicted mean and contracts the second derivatives of its own h / jac, again from dual numbers (eg_emission_vjp,
// DESIGN 4.2h); all of that is compiled only under CDK_HAS_USER_EMISSION.
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
#if CDK_HAS_USER_DRIFT || CDK_HAS_USER_EMISSION
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
#if CDK_HAS_USER_EMISSION
// Directions seeded per dual evaluation of the user's emission: 4 rather than 8, so that the dual copy of [x | phi] of
// the range emission to 20 beacons at n = 40 fits in the moment buffers it aliases (DESIGN 4.2h).
constexpr int EG_EW = 4;
using EgEDual = cdk_dual::Dual<EG_EW>;
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
#if CDK_HAS_USER_EMISSION
  int nph, PHI, PHB, ED;
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
#if CDK_HAS_USER_EMISSION
    // user emission: phi and its cotangent, and the emission's dual scratch ED = [per-thread partial sums | dual x |
    // dual phi].  ED is needed only after the update VJP, when the four moment buffers YC..ACC are idle until the next
    // gap reloads them: it aliases them when it fits there, else it is appended.  Aliased, the dual x lies behind the
    // partial sums (threads * EG_EW >= 128 >= n doubles), so copying mu out of YC into it overwrites nothing unread.
    nph = PHI = PHB = ED = 0;
    if (d.emission_id == CDK_EMISSION_USER) {
      nph = cdk_user_emission::num_params(n, m);
      PHI = take(nph);
      PHB = take(nph);
      const int need = eg_threads(n, m) * EG_EW + (n + nph) * (EG_EW + 1);
      ED = need <= YB - YC ? YC : take(need);
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

// k = dt * rhs(y), y and k in shared memory.  Ends with a barrier.  SIGMA: the literal sigma-point unscented predict of
// the filter (ukf_sigma_rhs), with Lc and D in W1 and W2 as there.
template <bool SIGMA>
__device__ void eg_rhs(const Eg& c, const double* y, double* k, double dt) {
  const EgLay& L = c.L;
  const int n = L.n, ld = L.ldn, id = c.g.k.d.drift_id;
  const double* th = c.p(L.TH);
  const double* lql = c.p(L.LQL);
  const double* P = y + L.mpoff;
  if (SIGMA) {
    ukf_sigma_rhs<double>(c.g.k.d, th, n, ld, y, P, lql, c.p(L.W1), c.p(L.W2), k, k + L.mpoff, dt);
    return;
  }
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

#if CDK_HAS_USER_DRIFT || CDK_HAS_USER_EMISSION
// The chunk loop of the dual-number contractions: the nv directions of the dual copies (dual(v), v < nv; the first nx
// of them the state's, then the parameters') are seeded W at a time; for each chunk the threads share out the E
// evaluations, eval(e, c0, fth, acc) adding evaluation e's weighted tangents of the chunk starting at direction c0 to the
// thread's acc[W] in registers (fth: the chunk holds parameter directions), and one thread per direction adds the
// per-thread partial sums (part, blockDim.x * W doubles) in thread order and hands the sum to sink(v, s): the result is
// the same bits from run to run.  The dual copies hold their values on entry.  Ends with a barrier.
template <int W, class DA, class EV, class SK>
__device__ __forceinline__ void eg_dual_chunks(DA dual, int nx, int nv, int E, double* part, EV eval, SK sink) {
  for (int c0 = 0; c0 < nv; c0 += W) {
    FOR_T(e, nv * W) {
      const int v = e / W, w = e - v * W;
      dual(v).d[w] = c0 + w == v ? 1.0 : 0.0;
    }
    __syncthreads();
    const bool fth = c0 + W > nx;
    double acc[W];
#pragma unroll
    for (int w = 0; w < W; ++w) acc[w] = 0.0;
    for (int e = threadIdx.x; e < E; e += blockDim.x) eval(e, c0, fth, acc);
#pragma unroll
    for (int w = 0; w < W; ++w) part[threadIdx.x * W + w] = acc[w];
    __syncthreads();
    FOR_T(w, W) {
      const int v = c0 + w;
      if (v < nv) {
        double s = 0.0;
        for (int t = 0; t < (int)blockDim.x; ++t) s += part[t * W + w];
        sink(v, s);
      }
    }
  }
  __syncthreads();
}
#endif

#if CDK_HAS_USER_DRIFT
// The mean and parameter cotangents of eg_rhs_vjp for the user drift, from dual evaluations of its own f / jac / graddiv
// at the stage input y (J, Jb and outP = J^T As are in place).  With w_q = 0.5 sum_i P_qi a_i ('second' order only):
//   m_bar_l      = (J^T a)_l + sum_ik Jb_ik dJ_ik/dx_l + sum_q w_q dg_q/dx_l
//   theta_bar_e += sum_i a_i df_i/dtheta_e + sum_ik Jb_ik dJ_ik/dtheta_e + sum_q w_q dg_q/dtheta_e
//   P_bar       += 0.5 g(x) a^T
// The n + n_theta directions (x, then theta) are seeded EG_DW at a time into the CTA's one dual copy of [x | theta]
// (eg_dual_chunks); the threads share out the evaluations jac (i, k), f i and graddiv q.  Ends with a barrier.
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
  eg_dual_chunks<EG_DW>(
      [&](int v) -> EgDual& { return xd[v]; }, n, nv, E, part,
      [&](int e, int c0, bool fth, double(&acc)[EG_DW]) {
        if (e < nj) {
          const int i = e / n, k = e - i * n;
          const EgDual v = cdk_user::jac<EgDual>(td, n, i, k, xd);
          const double wt = Jb[i * ld + k];
#pragma unroll
          for (int w = 0; w < EG_DW; ++w) acc[w] += wt * v.d[w];
        } else if (e < nj + n) {
          if (!fth) return;  // no parameter direction in the chunk: f's x-tangents are J
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
      },
      [&](int v, double s) {
        if (v < n) out[v] += s; else thb[v - n] += s;
      });
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

#if CDK_HAS_USER_DRIFT
// theta_bar_e += sum_p sum_j Fb[p][j] df_j/dtheta_e (X_p) over the np points X (rows of ldn; Fb likewise) for the user
// drift: dual evaluations of its f with only theta seeded, EG_DW directions at a time, into the CTA's one dual copy of
// theta (eg_dual_chunks); x enters as plain constants.  Ends with a barrier.
__device__ void eg_user_theta(const Eg& c, const double* X, const double* Fb, int np) {
  const EgLay& L = c.L;
  const int n = L.n, ld = L.ldn, nth = L.nth, E = np * n;
  const double* th = c.p(L.TH);
  double* thb = c.p(L.THB);
  EgDual* td = reinterpret_cast<EgDual*>(c.p(L.DU)) + n;
  FOR_T(v, nth) td[v] = EgDual(th[v]);
  __syncthreads();
  eg_dual_chunks<EG_DW>(
      [&](int v) -> EgDual& { return td[v]; }, 0, nth, E, c.p(L.PART),
      [&](int e, int, bool, double(&acc)[EG_DW]) {
        const int p = e / n, j = e - p * n;
        const double* x = X + p * ld;
        const EgDual v = cdk_user::f<EgDual>(td, n, j, [&](int q) { return EgDual(x[q]); });
        const double wt = Fb[p * ld + j];
#pragma unroll
        for (int w = 0; w < EG_DW; ++w) acc[w] += wt * v.d[w];
      },
      [&](int v, double s) { thb[v] += s; });
}
#endif

// theta_bar += sum over the np points X (rows) of sum_j Fb[p][j] df_j/dtheta (X_p): the registry's f-contraction, one thread
// per parameter and the points in order; the user drift's from dual numbers.  Ends with a barrier.
__device__ void eg_sigma_theta(const Eg& c, const double* X, const double* Fb, int np) {
  const EgLay& L = c.L;
  const int n = L.n, ld = L.ldn, id = c.g.k.d.drift_id;
#if CDK_HAS_USER_DRIFT
  if (id == CDK_DRIFT_USER) {
    eg_user_theta(c, X, Fb, np);
    return;
  }
#endif
  double* thb = c.p(L.THB);
  FOR_T(e, L.nth) {
    double s = 0.0;
    for (int p = 0; p < np; ++p) s += drift_theta_vjp_f<double>(id, n, e, X + p * ld, Fb + p * ld);
    thb[e] += s;
  }
  __syncthreads();
}

// VJP of the sigma-point right-hand side (ukf_sigma_rhs) at y = (m, P) for the cotangent kb = (a, A) (already scaled by dt):
// writes the cotangent of y to `out` (the stage's slot in the scratch) and accumulates theta_bar and Sigma_bar.  With
// Lc = chol(P), X_i^+- = m +- c Lc[:, i], D[:, i] = f(X_i^+) - f(X_i^-), wc = w c:
//   As = A + A^T,  Sigma_bar += A,  D_bar = wc As Lc,  Lc_bar = wc As D (direct part)
//   F_bar_i^+- = w a +- D_bar[:, i],  f0_bar = w0 a,  X_bar_i^+- = J(X_i^+-)^T F_bar_i^+-
//   m_bar = J(m)^T f0_bar + sum_i (X_bar_i^+ + X_bar_i^-),  Lc_bar[:, i] += c (X_bar_i^+ - X_bar_i^-)
//   theta_bar += sum over the 2n + 1 points of F_bar^T df/dtheta
//   P_bar = sym(Lc^-T Phi(Lc^T tril(Lc_bar)) Lc^-1),  Phi: the lower triangle with the diagonal halved
// (the symmetric Cholesky VJP, torch's linalg.cholesky backward).  The stage VJP leaves YC, ACC, J, W1 and W2 idle; they
// hold Lc, As (then F_bar), D (then X_bar), D_bar (then the transposed solve) and Lc_bar, and the sigma points of one sign
// (then Phi) sit behind the layout at XS = L.total.  Ends with a barrier.
__device__ void eg_sigma_rhs_vjp(const Eg& c, const double* y, const double* kb, double* out) {
  const EgLay& L = c.L;
  const cdk_desc& d = c.g.k.d;
  const int n = L.n, ld = L.ldn, id = d.drift_id;
  const double* th = c.p(L.TH);
  const double* mm = y;
  const double* P = y + L.mpoff;
  const double* ab = kb;
  const double* Ab = kb + L.mpoff;
  double* Lc = c.p(L.YC);
  double* As = c.p(L.ACC);
  double* Fb = As;
  double* D = c.p(L.J);
  double* Xb = D;
  double* Db = c.p(L.W1);
  double* Lb = c.p(L.W2);
  double* X = c.p(L.total);
  double* sigb = c.p(L.SIGB);
  double* outP = out + L.mpoff;
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    As[i * ld + j] = Ab[i * ld + j] + Ab[j * ld + i];
    sigb[i * ld + j] += Ab[i * ld + j];
  }
  // chol's first loop copies P into Lc (YC) before its first barrier; the loop above writes only As (ACC) and SIGB, which
  // that copy does not touch, so no barrier is needed here.  chol ends with a barrier.
  chol<double>(P, Lc, n, ld, 0.0);
  const UkfSigmaWeights<double> u(d);
  const double cs = u.cs, w = u.w, wc = u.w * u.cs;
  FOR_T(e, n * n) {
    const int j = e / n, i = e - j * n;
    const double fp = drift_f<double>(id, th, n, j, [&](int q) { return mm[q] + cs * Lc[q * ld + i]; });
    const double fm = drift_f<double>(id, th, n, j, [&](int q) { return mm[q] - cs * Lc[q * ld + i]; });
    D[j * ld + i] = fp - fm;
  }
  __syncthreads();
  mm_dmma<double, false, false>(As, ld, Lc, ld, n, n, n, [&](int i, int j, double v) { Db[i * ld + j] = wc * v; });
  mm_dmma<double, false, false>(As, ld, D, ld, n, n, n, [&](int i, int j, double v) { Lb[i * ld + j] = wc * v; });
  __syncthreads();
  for (int sg = 0; sg < 2; ++sg) {  // the points X_i^+ (rows of X), then X_i^-
    FOR_T(e, n * n) {
      const int i = e / n, q = e - i * n;
      const double v = cs * Lc[q * ld + i];
      X[i * ld + q] = sg == 0 ? mm[q] + v : mm[q] - v;
      Fb[i * ld + q] = sg == 0 ? w * ab[q] + Db[q * ld + i] : w * ab[q] - Db[q * ld + i];
    }
    __syncthreads();
    FOR_T(e, n * n) {
      const int i = e / n, l = e - i * n;
      const double* x = X + i * ld;
      double xb = 0.0;
      for (int j = 0; j < n; ++j) xb += drift_jac<double>(id, th, n, j, l, x) * Fb[i * ld + j];
      if (sg == 0) {
        Xb[i * ld + l] = xb;
        Lb[l * ld + i] += cs * xb;
      } else {
        Xb[i * ld + l] += xb;
        Lb[l * ld + i] -= cs * xb;
      }
    }
    eg_sigma_theta(c, X, Fb, n);
  }
  FOR_T(j, n) Fb[j] = u.w0 * ab[j];  // the centre point m
  __syncthreads();
  FOR_T(l, n) {
    double s = 0.0;
    for (int j = 0; j < n; ++j) s += drift_jac<double>(id, th, n, j, l, mm) * Fb[j];
    for (int i = 0; i < n; ++i) s += Xb[i * ld + l];
    out[l] = s;
  }
  FOR_T(e, n * n) {  // only the lower triangle of Lc_bar enters
    const int i = e / n, j = e - i * n;
    if (j > i) Lb[i * ld + j] = 0.0;
  }
  eg_sigma_theta(c, mm, Fb, 1);
  // ---- Cholesky VJP: Phi(Lc^T Lc_bar) into X, two solves with Lc^T, P_bar = sym ----
  mm_dmma<double, true, false>(Lc, ld, Lb, ld, n, n, n, [&](int i, int j, double v) {
    X[i * ld + j] = i > j ? v : (i == j ? 0.5 * v : 0.0);
  });
  __syncthreads();
  chol_solve_lt<double>(Lc, n, ld, X, n, ld);  // Y = Lc^-T Phi
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    Db[i * ld + j] = X[j * ld + i];
  }
  __syncthreads();
  chol_solve_lt<double>(Lc, n, ld, Db, n, ld);  // Z^T = Lc^-T Y^T,  Z = Lc^-T Phi Lc^-1
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    outP[i * ld + j] = 0.5 * (Db[i * ld + j] + Db[j * ld + i]);
  }
  __syncthreads();
}

// One substep of the state YC (in place) through the stages of any tableau; the stage inputs are left in stg[s * st].
template <bool SIGMA>
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
    eg_rhs<SIGMA>(c, ys, k, dt);
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
template <bool SIGMA>
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
    if (SIGMA) {
      eg_sigma_rhs_vjp(c, ys, kb, stb + s * st);
    } else {
      eg_rhs_vjp(c, ys, kb, stb + s * st);
    }
  }
  FOR_T(e, st) {
    double v = yb[e];
    for (int s = 0; s < S; ++s) v += stb[s * st + e];
    yb[e] = v;
  }
  __syncthreads();
}

#if CDK_HAS_USER_EMISSION
// The user emission's part of the update VJP at the predicted mean mu (YC), once the linear update VJP has run with
// H = J(mu) and r = y - h(mu): HB holds this step's cotangent Hb of J(mu), RBV the residual's r_bar.  Then
//   mu_bar_l  += sum_aj Hb_aj dJ_aj/dx_l                      (-sum_a r_bar_a J_al is the linear VJP's -H^T r_bar)
//   phi_bar_e += sum_aj Hb_aj dJ_aj/dphi_e - sum_a r_bar_a dh_a/dphi_e
// from dual evaluations of the user's jac (a, j) and h (a), the n + n_phi directions (x, then phi) seeded EG_EW at a time
// (eg_dual_chunks); h enters only chunks that hold phi directions, its x-tangents being J.  Ends with a barrier.
__device__ void eg_emission_vjp(const Eg& c) {
  const EgLay& L = c.L;
  const int n = L.n, m = L.m, ld = L.ldn, nph = L.nph, nj = m * n;
  const double* mu = c.p(L.YC);
  const double* phi = c.p(L.PHI);
  const double* Hb = c.p(L.HB);
  const double* rb = c.p(L.RBV);
  double* mub = c.p(L.YB);
  double* phb = c.p(L.PHB);
  double* part = c.p(L.ED);
  EgEDual* xd = reinterpret_cast<EgEDual*>(part + eg_threads(n, m) * EG_EW);
  EgEDual* pd = xd + n;
  FOR_T(v, n) xd[v] = EgEDual(mu[v]);  // before pd, which may overwrite YC
  __syncthreads();
  FOR_T(v, nph) pd[v] = EgEDual(phi[v]);
  __syncthreads();
  eg_dual_chunks<EG_EW>(
      [&](int v) -> EgEDual& { return v < n ? xd[v] : pd[v - n]; }, n, n + nph, nj + m, part,
      [&](int e, int c0, bool fth, double(&acc)[EG_EW]) {
        if (e < nj) {
          const int a = e / n, j = e - a * n;
          const EgEDual v = cdk_user_emission::jac<EgEDual>(pd, n, m, a, j, xd);
          const double wt = Hb[a * ld + j];
#pragma unroll
          for (int w = 0; w < EG_EW; ++w) acc[w] += wt * v.d[w];
        } else {
          if (!fth) return;  // no parameter direction in the chunk
          const int a = e - nj;
          const EgEDual v = cdk_user_emission::h<EgEDual>(pd, n, m, a, [&](int q) { return xd[q]; });
          const double wt = -rb[a];
#pragma unroll
          for (int w = 0; w < EG_EW; ++w)
            if (c0 + w >= n) acc[w] += wt * v.d[w];
        }
      },
      [&](int v, double s) {
        if (v < n) mub[v] += s; else phb[v - n] += s;
      });
}
#endif

// VJP of the measurement update (condition_on, num_iter = 1, then the symmetrisation) at the predicted moments in YC for
// the emission in YV: YB holds the cotangent of the filtered moments on entry and of the predicted ones on exit, plus
// the log-density's own derivative.  Accumulates H_bar, d_bar, R_bar.  A user emission (ue) runs the same VJP with
// H = J(mu) and r = y - h(mu), recomputed by the filter's code; its H_bar is this step's alone (J moves with mu), the
// terms of H mu + d are dropped, and eg_emission_vjp contracts H_bar and r_bar with the emission's derivatives.
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
  const bool ue = user_emission(c.g.k.d);
#if CDK_HAS_USER_EMISSION
  if (ue) {  // H = J(mu) as condition_on computes it; this step's H_bar starts from zero
    double* Hw = c.p(L.H);
    double* HBw = c.p(L.HB);
    const double* phi = c.p(L.PHI);
    FOR_T(e, m * n) {
      const int a = e / n, j = e - a * n;
      Hw[a * ldn + j] = user_h_jac<double>(phi, n, m, a, j, mu);
      HBw[a * ldn + j] = 0.0;
    }
    __syncthreads();
  }
#endif
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
    double s;
#if CDK_HAS_USER_EMISSION
    if (ue) {
      s = user_h<double>(c.p(L.PHI), n, m, a, [&](int j) { return mu[j]; });
    } else
#endif
    {
      s = dv[a];
      for (int q = 0; q < n; ++q) s += H[a * ldn + q] * mu[q];
    }
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
    HBg[a * ldn + j] += ue ? v : v - rb[a] * mu[j];
  });
  mm_dmma<double, false, false>(Sb, ldm, H, ldn, m, n, m, [&](int a, int j, double v) { U[a * ldn + j] = v + Gb[a * ldn + j]; });
  double* DBg = c.p(L.DB);
  if (!ue) FOR_T(a, m) DBg[a] -= rb[a];
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
#if CDK_HAS_USER_EMISSION
  if (ue) eg_emission_vjp(c);
#endif
}

__device__ void eg_load(double* dst, const double* __restrict__ src, int st) {
  FOR_T(e, st) dst[e] = src[e];
}
__device__ void eg_save(double* __restrict__ dst, const double* src, int st) {
  FOR_T(e, st) dst[e] = src[e];
}

// The backward walk of one trajectory (one CTA); SIGMA: the literal sigma-point unscented predict.
template <bool SIGMA>
__device__ __forceinline__ void eg_body(const EgArgs& g, double* smem) {
  Eg c(g, smem);
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
#if CDK_HAS_USER_EMISSION
    if (user_emission(d)) {  // phi from the H slot (n_phi per trajectory); d is not read
      FOR_T(i, L.nph) c.p(L.PHI)[i] = src(CDK_IN_H)[i];
    } else
#endif
    FOR_T(e, m * n) c.p(L.H)[(e / n) * ldn + e % n] = src(CDK_IN_H)[e];
    FOR_T(e, m * m) c.p(L.R)[(e / m) * ldm + e % m] = src(CDK_IN_R)[e];
#if CDK_HAS_USER_EMISSION
    if (!user_emission(d))
#endif
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
          eg_step<SIGMA>(c, clk.dt(), stg);
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
            eg_step<SIGMA>(c, clk.dt(), stg);
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
            eg_step<SIGMA>(c, clk.dt(), stg);
            clk.advance();
          }
          eg_step<SIGMA>(c, clk.dt(), stg);  // the stage inputs of substep i0 + u
          eg_step_vjp<SIGMA>(c, clk.dt(), stg, stb);
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
  // ---- gradient row: theta | Sigma (sym) | H | d | R (sym) | m0 | P0 (sym); a user emission: phi in place of H | d ----
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
#if CDK_HAS_USER_EMISSION
  if (user_emission(d)) gR = gH + L.nph;
#endif
  double* gm0 = gR + m * m;
  double* gP0 = gm0 + n;
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    gS[e] = 0.5 * (sigb[i * ldn + j] + sigb[j * ldn + i]);
    gP0[e] = 0.5 * (yb[L.mpoff + i * ldn + j] + yb[L.mpoff + j * ldn + i]);
  }
#if CDK_HAS_USER_EMISSION
  if (user_emission(d)) {
    FOR_T(e, L.nph) gH[e] = c.p(L.PHB)[e];
  } else
#endif
  {
    FOR_T(e, m * n) gH[e] = HB[(e / n) * ldn + e % n];
    FOR_T(i, m) gd[i] = c.p(L.DB)[i];
  }
  FOR_T(e, m * m) {
    const int i = e / m, j = e - i * m;
    gR[e] = 0.5 * (RB[i * ldm + j] + RB[j * ldm + i]);
  }
  FOR_T(i, n) gm0[i] = yb[i];
}

__global__ void __launch_bounds__(256) ekf_grad_dense_kernel(const EgArgs g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  eg_body<false>(g, reinterpret_cast<double*>(smem_raw));
}

// cdk_ukf_grad_sigma_f64: the same walk through the literal sigma-point predict (its own instantiation, so that the
// EKF and closed-form UKF kernel above keeps its code)
__global__ void __launch_bounds__(256) ukf_sigma_grad_kernel(const EgArgs g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  eg_body<true>(g, reinterpret_cast<double*>(smem_raw));
}

}  // namespace

// Shared memory of the backward kernel in doubles: the layout, and for the sigma-point predict one more n x ldn block (XS,
// behind the layout) for the sigma points of one sign
static long long eg_smem_doubles(const EgLay& lay, bool sigma) { return lay.total + (sigma ? (lay.nn + 1) / 2 * 2 : 0); }

// The layout of the scratch and shared memory of cdk_ekf_grad_dense_f64, cdk_ukf_grad_dense_f64 and (sigma)
// cdk_ukf_grad_sigma_f64 for `d` (false: beyond the 227 KB of one CTA)
static bool eg_layout(const cdk_desc& d, EgLay& lay, RtTab& rt, bool sigma = false) {
  if (!fill_rt_tab(d.solver, rt)) return false;
  lay = EgLay(d, rt.S);
  return (size_t)eg_smem_doubles(lay, sigma) * sizeof(double) <= 227u * 1024u;
}

bool ekf_grad_dense_fits(const cdk_desc& d, bool sigma) {
  EgLay lay;
  RtTab rt;
  return eg_layout(d, lay, rt, sigma);
}

bool ekf_grad_has_user_drift() { return CDK_HAS_USER_DRIFT != 0; }
bool ekf_grad_has_user_emission() { return CDK_HAS_USER_EMISSION != 0; }

long long ekf_grad_dense_scratch_doubles(const cdk_desc& d) {
  EgLay lay;
  RtTab rt;
  eg_layout(d, lay, rt);
  return d.N * ((long long)d.K * (2 * d.n + 2 * d.n * d.n) + lay.bwd() + 1);
}

// The backward launch behind a forward filter pass whose moments are in out[CDK_OUT_SCRATCH] and whose status is `status`;
// `ukf`: the forward pass was the closed-form UKF filter; `sigma`: the sigma-point UKF filter (ukf_sigma_grad_kernel).
int launch_ekf_grad_dense(const KArgs<double>& a, const int* status, double* grad, bool ukf, bool sigma, cudaStream_t s) {
  EgArgs g;
  g.k = a;
  if (!eg_layout(a.d, g.lay, g.tab, sigma)) return CDK_E_SIZE;
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j < 6; ++j) g.a[i][j] = 0.0;
  for (int i = 0; i < g.tab.S; ++i)
    for (int q = 0; q < g.tab.nnz[i]; ++q) g.a[i][g.tab.col[i][q]] = g.tab.val[i][q];
  g.sc = static_cast<double*>(a.out[CDK_OUT_SCRATCH]);
  g.status = status;
  g.grad = grad;
  g.cols = CDK_GRAD_COLS_EKF(a.d.n, a.d.m, a.d.n_theta);
#if CDK_HAS_USER_EMISSION
  if (user_emission(a.d)) g.cols = CDK_GRAD_COLS_EKF_UE(a.d.n, a.d.m, a.d.n_theta, g.lay.nph);
#endif
  g.ukf = ukf || sigma ? 1 : 0;
  const int threads = eg_threads(a.d.n, a.d.m);
  const size_t smem = (size_t)eg_smem_doubles(g.lay, sigma) * sizeof(double);
  if (a.d.N > 2147483647LL) return CDK_E_SIZE;
  if (sigma) {
    if (smem > 48 * 1024 && cudaFuncSetAttribute(ukf_sigma_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(ukf_sigma_grad_kernel)");
    ukf_sigma_grad_kernel<<<(unsigned)a.d.N, threads, smem, s>>>(g);
    note_launch();
    return check_launch("ukf_sigma_grad_kernel");
  }
  if (smem > 48 * 1024 && cudaFuncSetAttribute(ekf_grad_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("cudaFuncSetAttribute(ekf_grad_dense_kernel)");
  ekf_grad_dense_kernel<<<(unsigned)a.d.N, threads, smem, s>>>(g);
  note_launch();
  return check_launch("ekf_grad_dense_kernel");
}

}  // namespace cdk
