// cdk_kfwarp.cu -- continuous-discrete Kalman filter for n <= 16, m <= 8: ONE WARP PER TRAJECTORY on the FP64 tensor cores.
//
// Replaces cdlgssm_filter (src/continuous_discrete_linear_gaussian_ssm/inference.py:555-632) with compute_pushforward
// (:105-144: dA = F A, dQ = F Q + Q F^T + L Qc L^T from (I, 0) over every gap), _predict (:185-206) and _condition_on
// (:209-259) for BASELINE config 2 (n = 16, m = 4, N = 262,144, K = 500), fp64, chain tableaux (Euler .. RK4).
//
// B200 mapping:
//  * 94 % of the work is the pushforward: 2 n^3 FMAs per RK stage.  Every 16x16 matrix of the RK state (A, Q, the stage
//    increments, the running combination) lives in REGISTERS in the accumulator layout of mma.sync.m8n8k4.f64 (SASS DMMA):
//    8 doubles per lane per matrix.  A stage writes its input to the warp's private shared-memory slice once (as the B
//    operand), runs 2 x 16 DMMAs against F, forms F Q + (F Q)^T with one more shared-memory round trip, and does the
//    y + a dt k / acc + b dt k updates lane-locally on the fragments.  Leading dimension 20 (= 4 mod 16) makes the A/B
//    fragment loads bank-conflict free.
//  * the warps of a CTA never synchronise with each other (only __syncwarp): like ekf_small_lw they drift out of phase, so
//    the latency-bound measurement update of one warp hides behind the DMMA-bound pushforward of the others.
//  * one warp = one trajectory also makes every per-step output row (n + n^2 doubles) one contiguous, coalesced store.
//  * dimensions are padded to 16 x 16 / 8 x 16 with zeros (identity block for A), which leaves the arithmetic on the real
//    entries unchanged.
// Everything this fast path does not cover (inputs, fp32, n > 16, the type-2 smoother) stays on generic_filter_kernel.
#include <stdlib.h>

#include "cdk_common.cuh"

namespace cdk {
namespace {

constexpr int KW_LD = 20;   // leading dimension (doubles) of every shared-memory matrix
constexpr int KW_WPC = 4;   // warps (trajectories) per CTA
constexpr int KW_MAT = 16 * KW_LD, KW_MAT8 = 8 * KW_LD;
constexpr int KW_MODEL = 3 * KW_MAT + 2 * KW_MAT8 + 16 + 8;  // F, LQL, H, R, b, d, Rk (the RK map of one full step)
constexpr int KW_RK_OFF = 2 * KW_MAT + 2 * KW_MAT8 + 16 + 8;  // offset of Rk inside the model block

struct KwTab {
  int S;
  double a[6];  // chain tableau: stage i reads only stage i-1, with coefficient a[i]
  double b[6];
  // poly != 0 (any tableau that is not a chain, i.e. Dopri5 -- the reference's DEFAULT solver, diffrax_utils.py:121-124):
  // the pushforward ODEs are linear with constant coefficients, y' = Ly + g, and one explicit RK step of ANY tableau is
  // then y + h sum_{j>=1} c_j (h L)^{j-1} (L y + g) with c_j = b^T A^{j-1} 1 (its stability polynomial): the same
  // S applications of L as the S stages, evaluated by Horner's rule with THREE matrices in registers instead of the
  // S stage increments a non-chain tableau would have to keep (6 x 2 x 2 KB per warp for Dopri5).  Same result as
  // stepping through the stages up to rounding.
  int poly;
  double c[7];  // c[1..S]
};

struct F16 {
  double v[2][2][2];  // [row block][col block][r]: element (8 rb + gid, 8 cb + 2 tig + r)
};

__device__ __forceinline__ void dmma(double& d0, double& d1, double av, double bv) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(av), "d"(bv));
}

// D[RB x CB tiles] = opA * opB over KD (multiple of 4), operands in shared memory with leading dimension KW_LD.
template <bool TRANSA, bool TRANSB, int KD, int RB, int CB>
__device__ __forceinline__ void mm(double (&d)[RB][CB][2], const double* __restrict__ sA, const double* __restrict__ sB) {
  const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
#pragma unroll
  for (int rb = 0; rb < RB; ++rb)
#pragma unroll
    for (int cb = 0; cb < CB; ++cb) d[rb][cb][0] = d[rb][cb][1] = 0.0;
#pragma unroll
  for (int kk = 0; kk < KD / 4; ++kk) {
    double av[RB], bv[CB];
#pragma unroll
    for (int rb = 0; rb < RB; ++rb)
      av[rb] = TRANSA ? sA[(4 * kk + tig) * KW_LD + 8 * rb + gid] : sA[(8 * rb + gid) * KW_LD + 4 * kk + tig];
#pragma unroll
    for (int cb = 0; cb < CB; ++cb)
      bv[cb] = TRANSB ? sB[(8 * cb + gid) * KW_LD + 4 * kk + tig] : sB[(4 * kk + tig) * KW_LD + 8 * cb + gid];
#pragma unroll
    for (int rb = 0; rb < RB; ++rb)
#pragma unroll
      for (int cb = 0; cb < CB; ++cb) dmma(d[rb][cb][0], d[rb][cb][1], av[rb], bv[cb]);
  }
}

// D1 = A * B1 and D2 = A * B2 (all 16 x 16, row-major in shared memory, leading dimension KW_LD) in one sweep: the
// fragments of A are loaded once per k-step and the eight DMMAs of a k-step are mutually independent, so the dependent
// accumulation chain of every output tile is eight tensor instructions apart.
__device__ __forceinline__ void mm2_shared_a(double (&d1)[2][2][2], double (&d2)[2][2][2], const double* __restrict__ sA,
                                             const double* __restrict__ sB1, const double* __restrict__ sB2) {
  const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
#pragma unroll
  for (int rb = 0; rb < 2; ++rb)
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) d1[rb][cb][0] = d1[rb][cb][1] = d2[rb][cb][0] = d2[rb][cb][1] = 0.0;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    double av[2], b1[2], b2[2];
#pragma unroll
    for (int rb = 0; rb < 2; ++rb) av[rb] = sA[(8 * rb + gid) * KW_LD + 4 * kk + tig];
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) {
      b1[cb] = sB1[(4 * kk + tig) * KW_LD + 8 * cb + gid];
      b2[cb] = sB2[(4 * kk + tig) * KW_LD + 8 * cb + gid];
    }
#pragma unroll
    for (int rb = 0; rb < 2; ++rb)
#pragma unroll
      for (int cb = 0; cb < 2; ++cb) {
        dmma(d1[rb][cb][0], d1[rb][cb][1], av[rb], b1[cb]);
        dmma(d2[rb][cb][0], d2[rb][cb][1], av[rb], b2[cb]);
      }
  }
}

template <int RB, int CB>
__device__ __forceinline__ void store_c(const double (&d)[RB][CB][2], double* s) {
  const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
#pragma unroll
  for (int rb = 0; rb < RB; ++rb)
#pragma unroll
    for (int cb = 0; cb < CB; ++cb) {
      s[(8 * rb + gid) * KW_LD + 8 * cb + 2 * tig] = d[rb][cb][0];
      s[(8 * rb + gid) * KW_LD + 8 * cb + 2 * tig + 1] = d[rb][cb][1];
    }
}
template <int RB, int CB>
__device__ __forceinline__ void load_c(double (&d)[RB][CB][2], const double* s) {
  const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
#pragma unroll
  for (int rb = 0; rb < RB; ++rb)
#pragma unroll
    for (int cb = 0; cb < CB; ++cb) {
      d[rb][cb][0] = s[(8 * rb + gid) * KW_LD + 8 * cb + 2 * tig];
      d[rb][cb][1] = s[(8 * rb + gid) * KW_LD + 8 * cb + 2 * tig + 1];
    }
}
// d(r, c) = s(c, r)
__device__ __forceinline__ void load_ct(double (&d)[2][2][2], const double* s) {
  const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
#pragma unroll
  for (int rb = 0; rb < 2; ++rb)
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) {
      d[rb][cb][0] = s[(8 * cb + 2 * tig) * KW_LD + 8 * rb + gid];
      d[rb][cb][1] = s[(8 * cb + 2 * tig + 1) * KW_LD + 8 * rb + gid];
    }
}

// write a C-layout 16x16 fragment to a global row-major n x n matrix
__device__ __forceinline__ void store_global(const double (&d)[2][2][2], double* __restrict__ G, int n) {
  const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
#pragma unroll
  for (int rb = 0; rb < 2; ++rb)
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) {
      const int r = 8 * rb + gid, c = 8 * cb + 2 * tig;
      if (r < n) {
        if (c < n) G[r * n + c] = d[rb][cb][0];
        if (c + 1 < n) G[r * n + c + 1] = d[rb][cb][1];
      }
    }
}

// (A, Q) over [t0, t1] from (I, 0): dA = F A, dQ = F Q + Q F^T + L Qc L^T (cd_linear/inference.py:105-144) with the diffrax
// ConstantStepSize stepping rule.  Results stay in registers (C-fragment layout); sYA / sYQ / sT are the warp's stage
// buffers.  Returns true when max_steps was exceeded (results are NaN then, as in the reference).
template <bool POLY>
__device__ __forceinline__ bool pushforward(const KwTab& tab, const double dt0, const int max_steps,
                                            const double t0, const double t1, const double* sF, const double* sLQL,
                                            const double* sRk, double* sYA, double* sYQ, double* sT, F16& yA, F16& yQ,
                                            const bool direct_t = false) {
  const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
  bool hit = false;
#pragma unroll
  for (int rb = 0; rb < 2; ++rb)
#pragma unroll
    for (int cb = 0; cb < 2; ++cb)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        yA.v[rb][cb][r] = (8 * rb + gid == 8 * cb + 2 * tig + r) ? 1.0 : 0.0;
        yQ.v[rb][cb][r] = 0.0;
      }
  StepClock<double> clk(t0, t1, dt0);
  while (clk.running()) {
    if (clk.n >= max_steps) {
      hit = true;
#pragma unroll
      for (int i = 0; i < 8; ++i) (&yA.v[0][0][0])[i] = (&yQ.v[0][0][0])[i] = NAN;
      break;
    }
    const double dt = clk.dt();
    // dA = F A is linear with constant coefficients, so one explicit RK step of length dt0 maps A to Rk A with the SAME
    // matrix Rk for every full-length substep of every gap (Rk = the RK step applied to the identity, computed once per
    // model by rk_map): one product instead of one per stage.  Clipped substeps (and Q, whose step map is not a
    // similarity transform of the truncated polynomial) take the stages.  Same result as stepping A up to rounding.
    const bool fastA = clk.full() && sRk != nullptr;
    F16 accA = yA, accQ = yQ, kA, kQ;
    if (fastA) {
      store_c<2, 2>(yA.v, sYA);
      __syncwarp();
      mm<false, false, 16, 2, 2>(accA.v, sRk, sYA);
      __syncwarp();
      // a full substep ends at t + dt0 rounded, so its length differs from dt0 by up to half an ulp of t: 1.8e-12
      // at t = 1e4, i.e. 7e-10 of dt0 = 0.0025, and the reference steps with that length.  Rk(dt) = Rk(dt0) + (dt - dt0) F
      // Rk(dt0) + O(dt0^S (dt - dt0)): one more product restores it.  Below 2^-40 dt0 the term is under 2^-40 dt0 |F| of A
      // per step and the product is skipped, so grids at moderate t keep the one-product step.
      const double ddt = dt - dt0;
      if (fabs(ddt) > 0x1p-40 * dt0) {
        F16 fa;
        store_c<2, 2>(accA.v, sYA);
        __syncwarp();
        mm<false, false, 16, 2, 2>(fa.v, sF, sYA);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 8; ++i) (&accA.v[0][0][0])[i] = fma(ddt, (&fa.v[0][0][0])[i], (&accA.v[0][0][0])[i]);
      }
    }
    if constexpr (POLY) {
      // Horner evaluation of the step polynomial (see KwTab): v = L y + g, w = c_S v, w = c_j v + dt L w (j = S-1 .. 1),
      // y += dt w; for A: L = F . , g = 0; for Q: L = F . + (F .)^T, g = L Qc L^T.  kA / kQ hold v, iA / iQ hold w.
      F16 wA, wQ;
#pragma unroll 1
      for (int j = tab.S; j >= 1; --j) {
        const bool first = j == tab.S;
        // operand of this application of L: y for the first pass (-> v), w afterwards
        if (!fastA) store_c<2, 2>(first ? yA.v : wA.v, sYA);
        store_c<2, 2>(first ? yQ.v : wQ.v, sYQ);
        __syncwarp();
        F16 fa, fq, fqt;
        if (fastA) {
          mm<false, false, 16, 2, 2>(fq.v, sF, sYQ);
        } else {
          mm2_shared_a(fa.v, fq.v, sF, sYA, sYQ);
        }
        store_c<2, 2>(fq.v, sT);
        __syncwarp();
        load_ct(fqt.v, sT);
        if (first) {
          F16 lq;
          load_c<2, 2>(lq.v, sLQL);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            (&kQ.v[0][0][0])[i] = ((&fq.v[0][0][0])[i] + (&fqt.v[0][0][0])[i]) + (&lq.v[0][0][0])[i];
            (&wQ.v[0][0][0])[i] = tab.c[j] * (&kQ.v[0][0][0])[i];
            if (!fastA) {
              (&kA.v[0][0][0])[i] = (&fa.v[0][0][0])[i];
              (&wA.v[0][0][0])[i] = tab.c[j] * (&fa.v[0][0][0])[i];
            }
          }
        }
        if (!first) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            (&wQ.v[0][0][0])[i] = fma(dt, (&fq.v[0][0][0])[i] + (&fqt.v[0][0][0])[i], tab.c[j] * (&kQ.v[0][0][0])[i]);
            if (!fastA) (&wA.v[0][0][0])[i] = fma(dt, (&fa.v[0][0][0])[i], tab.c[j] * (&kA.v[0][0][0])[i]);
          }
        }
        __syncwarp();
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        (&accQ.v[0][0][0])[i] = fma(dt, (&wQ.v[0][0][0])[i], (&yQ.v[0][0][0])[i]);
        if (!fastA) (&accA.v[0][0][0])[i] = fma(dt, (&wA.v[0][0][0])[i], (&yA.v[0][0][0])[i]);
      }
    } else {
#pragma unroll 1
    for (int st = 0; st < tab.S; ++st) {
      // stage input y + a dt k_{st-1} -> shared memory (B operand)
      F16 iA = yA, iQ = yQ;
      if (st > 0) {
        const double c = tab.a[st] * dt;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (!fastA) (&iA.v[0][0][0])[i] = fma(c, (&kA.v[0][0][0])[i], (&iA.v[0][0][0])[i]);
          (&iQ.v[0][0][0])[i] = fma(c, (&kQ.v[0][0][0])[i], (&iQ.v[0][0][0])[i]);
        }
      }
      if (!fastA) store_c<2, 2>(iA.v, sYA);
      store_c<2, 2>(iQ.v, sYQ);
      __syncwarp();
      F16 fq;
      if (fastA) {
        mm<false, false, 16, 2, 2>(fq.v, sF, sYQ);  // F Q
      } else {
        mm2_shared_a(kA.v, fq.v, sF, sYA, sYQ);  // dA = F A and F Q
      }
      F16 fqt, lq;
      if (direct_t) {
        mm<false, true, 16, 2, 2>(fqt.v, sYQ, sF);  // Q F^T on the tensor cores: no shared-memory round trip
      } else {
        store_c<2, 2>(fq.v, sT);
        __syncwarp();
        load_ct(fqt.v, sT);  // Q F^T = (F Q)^T for the symmetric Q
      }
      load_c<2, 2>(lq.v, sLQL);
#pragma unroll
      for (int i = 0; i < 8; ++i) (&kQ.v[0][0][0])[i] = ((&fq.v[0][0][0])[i] + (&fqt.v[0][0][0])[i]) + (&lq.v[0][0][0])[i];
      const double w = tab.b[st] * dt;
      if (w != 0.0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (!fastA) (&accA.v[0][0][0])[i] = fma(w, (&kA.v[0][0][0])[i], (&accA.v[0][0][0])[i]);
          (&accQ.v[0][0][0])[i] = fma(w, (&kQ.v[0][0][0])[i], (&accQ.v[0][0][0])[i]);
        }
      }
      __syncwarp();
    }
    }
    yA = accA;
    yQ = accQ;
    clk.advance();
  }
  return hit;
}

// Rk = one explicit RK step of length dt0 of dA = F A applied to the identity (chain tableau), into sRk.
template <bool POLY>
__device__ __forceinline__ void rk_map(const KwTab& tab, const double dt0, const double* sF, double* sRk, double* sYA) {
  const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
  F16 eye, acc, kA;
#pragma unroll
  for (int rb = 0; rb < 2; ++rb)
#pragma unroll
    for (int cb = 0; cb < 2; ++cb)
#pragma unroll
      for (int r = 0; r < 2; ++r) eye.v[rb][cb][r] = (8 * rb + gid == 8 * cb + 2 * tig + r) ? 1.0 : 0.0;
  acc = eye;
  if constexpr (POLY) {  // Rk = I + h sum_j c_j (h F)^{j-1} F by Horner: v = F, w = c_S v, w = c_j v + h F w, Rk = I + h w
    F16 v, w;
#pragma unroll 1
    for (int j = tab.S; j >= 1; --j) {
      const bool first = j == tab.S;
      store_c<2, 2>(first ? eye.v : w.v, sYA);
      __syncwarp();
      mm<false, false, 16, 2, 2>(kA.v, sF, sYA);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (first) {
          (&v.v[0][0][0])[i] = (&kA.v[0][0][0])[i];
          (&w.v[0][0][0])[i] = tab.c[j] * (&kA.v[0][0][0])[i];
        } else {
          (&w.v[0][0][0])[i] = fma(dt0, (&kA.v[0][0][0])[i], tab.c[j] * (&v.v[0][0][0])[i]);
        }
      }
      __syncwarp();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) (&acc.v[0][0][0])[i] = fma(dt0, (&w.v[0][0][0])[i], (&eye.v[0][0][0])[i]);
    store_c<2, 2>(acc.v, sRk);
    __syncwarp();
    return;
  }
#pragma unroll 1
  for (int st = 0; st < tab.S; ++st) {
    F16 iA = eye;
    if (st > 0) {
      const double c = tab.a[st] * dt0;
#pragma unroll
      for (int i = 0; i < 8; ++i) (&iA.v[0][0][0])[i] = fma(c, (&kA.v[0][0][0])[i], (&iA.v[0][0][0])[i]);
    }
    store_c<2, 2>(iA.v, sYA);
    __syncwarp();
    mm<false, false, 16, 2, 2>(kA.v, sF, sYA);
    const double w = tab.b[st] * dt0;
#pragma unroll
    for (int i = 0; i < 8; ++i) (&acc.v[0][0][0])[i] = fma(w, (&kA.v[0][0][0])[i], (&acc.v[0][0][0])[i]);
    __syncwarp();
  }
  store_c<2, 2>(acc.v, sRk);
  __syncwarp();
}

// Model constants (padded with zeros) into the CTA's or the warp's model block; L Qc L^T hoisted
// (cd_linear/inference.py:121-131).  scr0..2 are three 16 x KW_LD scratch matrices of the calling warp.
__device__ __forceinline__ void load_model_kw(const KArgs<double>& a, const long long tj, double* model, double* scr0,
                                              double* scr1, double* scr2) {
  const int lane = threadIdx.x & 31;
  const int n = a.d.n, m = a.d.m;
  double* sF = model;
  double* sLQL = sF + KW_MAT;
  double* sH = sLQL + KW_MAT;
  double* sR = sH + KW_MAT8;
  double* sb = sR + KW_MAT8;
  double* sd = sb + 16;
  auto src = [&](int slot) { return a.in[slot] + tj * a.in_stride[slot]; };
  for (int e = lane; e < KW_MODEL; e += 32) model[e] = 0.0;
  __syncwarp();
  double* Lm = scr0;
  double* Qc = scr1;
  double* LQ = scr2;
  for (int e = lane; e < n * n; e += 32) {
    const int i = e / n, j = e - i * n;
    sF[i * KW_LD + j] = src(CDK_IN_F)[e];
    Lm[i * KW_LD + j] = src(CDK_IN_L)[e];
    Qc[i * KW_LD + j] = src(CDK_IN_QC)[e];
  }
  for (int e = lane; e < m * n; e += 32) sH[(e / n) * KW_LD + (e % n)] = src(CDK_IN_H)[e];
  for (int e = lane; e < m * m; e += 32) sR[(e / m) * KW_LD + (e % m)] = src(CDK_IN_R)[e];
  for (int e = lane; e < n; e += 32) sb[e] = src(CDK_IN_B)[e];
  for (int e = lane; e < m; e += 32) sd[e] = src(CDK_IN_D)[e];
  __syncwarp();
  for (int e = lane; e < n * n; e += 32) {
    const int i = e / n, j = e - i * n;
    double s = 0.0;
    for (int q = 0; q < n; ++q) s += Lm[i * KW_LD + q] * Qc[q * KW_LD + j];
    LQ[i * KW_LD + j] = s;
  }
  __syncwarp();
  for (int e = lane; e < n * n; e += 32) {
    const int i = e / n, j = e - i * n;
    double s = 0.0;
    for (int q = 0; q < n; ++q) s += LQ[i * KW_LD + q] * Lm[j * KW_LD + q];
    sLQL[i * KW_LD + j] = s;
  }
}

// read a C-layout 16x16 fragment from a global row-major n x n matrix (zero padding outside n x n)
__device__ __forceinline__ void load_global(double (&d)[2][2][2], const double* __restrict__ G, int n) {
  const int lane = threadIdx.x & 31, gid = lane >> 2, tig = lane & 3;
#pragma unroll
  for (int rb = 0; rb < 2; ++rb)
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) {
      const int r = 8 * rb + gid, c = 8 * cb + 2 * tig;
      d[rb][cb][0] = (r < n && c < n) ? G[r * n + c] : 0.0;
      d[rb][cb][1] = (r < n && c + 1 < n) ? G[r * n + c + 1] : 0.0;
    }
}

struct KwSmemCounts {
  // per-warp doubles / per-model doubles
  static constexpr int PER_WARP = 4 * KW_MAT + 3 * KW_MAT8 + 8 * 9 + 16 + 16 + 8 + 8 + 8 + 8;
  static constexpr int PER_MODEL = KW_MODEL;  // F, LQL, H, R, b, d, Rk
};

template <bool POLY>
__global__ void __launch_bounds__(32 * KW_WPC, 3) kf_warp_filter(const KArgs<double> a, const __grid_constant__ KwTab tab, const int model_per_warp, const int use_rk) {
  extern __shared__ __align__(16) double kw_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, gid = lane >> 2, tig = lane & 3;
  const cdk_desc& d = a.d;
  const int n = d.n, m = d.m, K = d.K;
  const long long traj = (long long)blockIdx.x * KW_WPC + warp;
  double* model = kw_smem + (model_per_warp ? warp * KwSmemCounts::PER_MODEL : 0);
  double* wbase = kw_smem + (model_per_warp ? KW_WPC : 1) * KwSmemCounts::PER_MODEL + warp * KwSmemCounts::PER_WARP;
  double* sF = model;
  double* sLQL = sF + KW_MAT;
  double* sH = sLQL + KW_MAT;
  double* sR = sH + KW_MAT8;
  double* sb = sR + KW_MAT8;
  double* sd = sb + 16;
  const double* sRk = (use_rk & 1) ? model + KW_RK_OFF : nullptr;
  double* sP = wbase;
  double* sYA = sP + KW_MAT;
  double* sYQ = sYA + KW_MAT;
  double* sT = sYQ + KW_MAT;
  double* sHP = sT + KW_MAT;  // H P, then K^T in place
  double* sSK = sHP + KW_MAT8;
  double* sS = sSK + KW_MAT8;
  double* sL = sS + KW_MAT8;  // [8][9] Cholesky factor
  double* smu = sL + 72;
  double* smn = smu + 16;
  double* sy = smn + 16;
  double* sr = sy + 8;
  double* sz = sr + 8;
  double* sllv = sz + 8;

  // ---- model constants (padded with zeros); L Qc L^T hoisted (cd_linear/inference.py:121-131) ----
  const bool loader = model_per_warp ? true : warp == 0;
  const long long tj = traj < d.N ? traj : d.N - 1;
  auto src = [&](int slot) { return a.in[slot] + tj * a.in_stride[slot]; };
  if (loader) {
    for (int e = lane; e < KwSmemCounts::PER_MODEL; e += 32) model[e] = 0.0;
    __syncwarp();
    double* Lm = sYA;  // scratch of this warp
    double* Qc = sYQ;
    double* LQ = sT;
    for (int e = lane; e < n * n; e += 32) {
      const int i = e / n, j = e - i * n;
      sF[i * KW_LD + j] = src(CDK_IN_F)[e];
      Lm[i * KW_LD + j] = src(CDK_IN_L)[e];
      Qc[i * KW_LD + j] = src(CDK_IN_QC)[e];
    }
    for (int e = lane; e < m * n; e += 32) sH[(e / n) * KW_LD + (e % n)] = src(CDK_IN_H)[e];
    for (int e = lane; e < m * m; e += 32) sR[(e / m) * KW_LD + (e % m)] = src(CDK_IN_R)[e];
    for (int e = lane; e < n; e += 32) sb[e] = src(CDK_IN_B)[e];
    for (int e = lane; e < m; e += 32) sd[e] = src(CDK_IN_D)[e];
    __syncwarp();
    for (int e = lane; e < n * n; e += 32) {
      const int i = e / n, j = e - i * n;
      double s = 0.0;
      for (int q = 0; q < n; ++q) s += Lm[i * KW_LD + q] * Qc[q * KW_LD + j];
      LQ[i * KW_LD + j] = s;
    }
    __syncwarp();
    for (int e = lane; e < n * n; e += 32) {
      const int i = e / n, j = e - i * n;
      double s = 0.0;
      for (int q = 0; q < n; ++q) s += LQ[i * KW_LD + q] * Lm[j * KW_LD + q];
      sLQL[i * KW_LD + j] = s;
    }
    __syncwarp();
    rk_map<POLY>(tab, d.dt0, sF, model + KW_RK_OFF, sYA);
  }
  __syncthreads();  // the only CTA-wide barrier: the shared model block is ready
  if (traj >= d.N) return;
  for (int e = lane; e < KwSmemCounts::PER_WARP; e += 32) wbase[e] = 0.0;
  __syncwarp();
  for (int e = lane; e < n * n; e += 32) sP[(e / n) * KW_LD + (e % n)] = src(CDK_IN_P0)[e];
  if (lane < n) smu[lane] = src(CDK_IN_M0)[lane];
  __syncwarp();

  const double* __restrict__ Y = a.in[CDK_IN_Y] + traj * a.in_stride[CDK_IN_Y];
  const double* __restrict__ Tm = a.in[CDK_IN_T] + traj * a.in_stride[CDK_IN_T];
  double* FM = static_cast<double*>(a.out[CDK_OUT_FM]);
  double* FP = static_cast<double*>(a.out[CDK_OUT_FP]);
  double* PM = static_cast<double*>(a.out[CDK_OUT_PM]);
  double* PP = static_cast<double*>(a.out[CDK_OUT_PP]);
  double* LLC = static_cast<double*>(a.out[CDK_OUT_LLCUM]);
  double* AQ = (d.reserved[2] & CDK_FLAG_KEEP_PUSHFORWARD) ? static_cast<double*>(a.out[CDK_OUT_SCRATCH]) : nullptr;
  const long long row0 = traj * (long long)K;
  const double dt0 = d.dt0;
  double ll = 0.0;
  int status = 0;
  double y_next = lane < m ? Y[lane] : 0.0;
  double t_cur = Tm[0];
  double t_nxt = K > 1 ? Tm[1] : t_cur + d.dt_final;

  for (int k = 0; k < K; ++k) {
    // ================= update (cd_linear/inference.py:613-616, _condition_on :209-259) =================
    if (lane < m) sy[lane] = y_next;
    if (k + 1 < K && lane < m) y_next = Y[(long long)(k + 1) * m + lane];
    const double t0 = t_cur, t1 = t_nxt;
    t_cur = t1;
    t_nxt = k + 2 < K ? Tm[k + 2] : t1 + d.dt_final;
    __syncwarp();
    {
      double hp[1][2][2];
      mm<false, false, 16, 1, 2>(hp, sH, sP);  // H P  [8 x 16]
      store_c<1, 2>(hp, sHP);
      if (lane < 8) {  // innovation r = y - d - H mu (rows >= m are zero)
        double s = 0.0;
        if (lane < m) {
          s = sy[lane] - sd[lane];
          for (int q = 0; q < n; ++q) s -= sH[lane * KW_LD + q] * smu[q];
        }
        sr[lane] = s;
      }
      __syncwarp();
      double sf[1][1][2];
      mm<false, true, 16, 1, 1>(sf, sHP, sH);  // H P H^T
      {
        const int r = gid, c = 2 * tig;
        sS[r * KW_LD + c] = sf[0][0][0] + sR[r * KW_LD + c];
        sS[r * KW_LD + c + 1] = sf[0][0][1] + sR[r * KW_LD + c + 1];
      }
      __syncwarp();
      // MVN(H mu + d, S).log_prob(y): un-boosted Cholesky (TFP); then psd_solve: chol(sym(S) + 1e-9 I)
      for (int pass = 0; pass < 2; ++pass) {
        for (int j = 0; j < m; ++j) {
          if (lane >= j && lane < m) {
            const double boost = pass ? 1e-9 : 0.0;
            double sjj = sS[j * KW_LD + j] + boost;
            for (int q = 0; q < j; ++q) sjj -= sL[j * 9 + q] * sL[j * 9 + q];
            const double dj = sqrt(sjj);
            if (lane == j) {
              sL[j * 9 + j] = dj;
            } else {
              double v = pass ? 0.5 * (sS[lane * KW_LD + j] + sS[j * KW_LD + lane]) : sS[lane * KW_LD + j];
              for (int q = 0; q < j; ++q) v -= sL[lane * 9 + q] * sL[j * 9 + q];
              sL[lane * 9 + j] = v / dj;
            }
          }
          __syncwarp();
        }
        if (pass == 0) {
          if (lane == 0) {
            double quad = 0.0, logdet = 0.0;
            for (int i = 0; i < m; ++i) {
              double v = sr[i];
              for (int q = 0; q < i; ++q) v -= sL[i * 9 + q] * sz[q];
              v /= sL[i * 9 + i];
              sz[i] = v;
              quad += v * v;
              logdet += log(sL[i * 9 + i]);
            }
            sllv[0] = -0.5 * quad - logdet - m * half_log_2pi<double>();
          }
          __syncwarp();
        }
      }
      ll += sllv[0];
      // K^T = (S + boost)^-1 H P, one column per lane, in place in sHP
      if (lane < n) {
        for (int i = 0; i < m; ++i) {
          double v = sHP[i * KW_LD + lane];
          for (int q = 0; q < i; ++q) v -= sL[i * 9 + q] * sHP[q * KW_LD + lane];
          sHP[i * KW_LD + lane] = v / sL[i * 9 + i];
        }
        for (int i = m - 1; i >= 0; --i) {
          double v = sHP[i * KW_LD + lane];
          for (int q = i + 1; q < m; ++q) v -= sL[q * 9 + i] * sHP[q * KW_LD + lane];
          sHP[i * KW_LD + lane] = v / sL[i * 9 + i];
        }
      }
      __syncwarp();
      const double* sKt = sHP;
      double sk[1][2][2];
      mm<false, false, 8, 1, 2>(sk, sS, sKt);  // S K^T  (un-boosted S, :257)
      store_c<1, 2>(sk, sSK);
      if (lane < n) {  // mu += K r
        double s = 0.0;
        for (int q = 0; q < m; ++q) s += sKt[q * KW_LD + lane] * sr[q];
        smu[lane] += s;
      }
      __syncwarp();
      F16 ksk, P;
      mm<true, false, 8, 2, 2>(ksk.v, sKt, sSK);  // K S K^T
      load_c<2, 2>(P.v, sP);
#pragma unroll
      for (int i = 0; i < 8; ++i) (&P.v[0][0][0])[i] -= (&ksk.v[0][0][0])[i];
      store_c<2, 2>(P.v, sT);
      __syncwarp();
      F16 Pt;
      load_ct(Pt.v, sT);  // symmetrize (:259)
#pragma unroll
      for (int i = 0; i < 8; ++i) (&P.v[0][0][0])[i] = 0.5 * ((&P.v[0][0][0])[i] + (&Pt.v[0][0][0])[i]);
      store_c<2, 2>(P.v, sP);
      if (FP) store_global(P.v, FP + (row0 + k) * n * n, n);
      if (FM && lane < n) FM[(row0 + k) * n + lane] = smu[lane];
      if (LLC && lane == 0) LLC[row0 + k] = ll;
      __syncwarp();
    }
    // ================= pushforward (A, Q) over [t0, t1] from (I, 0)  (:105-144; diffrax ConstantStepSize) =================
    F16 yA, yQ;
    if (pushforward<POLY>(tab, dt0, d.max_steps, t0, t1, sF, sLQL, sRk, sYA, sYQ, sT, yA, yQ, (use_rk & 2) != 0)) status = 2;
    if (AQ && k + 1 < K) {  // CDK_FLAG_KEEP_PUSHFORWARD: the type-1 smoother will read (A_k, Q_k) back
      double* dst = AQ + ((traj * (long long)(K - 1) + k) * 2) * n * n;
      store_global(yA.v, dst, n);
      store_global(yQ.v, dst + n * n, n);
    }
    // ================= discrete predict: mu = A mu + b, P = A P A^T + Q  (:204-205) =================
    store_c<2, 2>(yA.v, sYA);
    __syncwarp();
    {
      F16 ap;
      mm<false, false, 16, 2, 2>(ap.v, sYA, sP);
      store_c<2, 2>(ap.v, sT);
      if (lane < 16) {
        double s = 0.0;
        for (int q = 0; q < n; ++q) s += sYA[lane * KW_LD + q] * smu[q];
        smn[lane] = lane < n ? s + sb[lane] : 0.0;
      }
      __syncwarp();
      F16 pn;
      mm<false, true, 16, 2, 2>(pn.v, sT, sYA);
#pragma unroll
      for (int i = 0; i < 8; ++i) (&pn.v[0][0][0])[i] += (&yQ.v[0][0][0])[i];
      store_c<2, 2>(pn.v, sP);
      if (lane < 16) smu[lane] = smn[lane];
      if (PP) store_global(pn.v, PP + (row0 + k) * n * n, n);
      if (PM && lane < n) PM[(row0 + k) * n + lane] = smn[lane];
      __syncwarp();
    }
  }
  if (lane == 0) {
    if (a.out[CDK_OUT_LL]) static_cast<double*>(a.out[CDK_OUT_LL])[traj] = ll;
    if (a.out[CDK_OUT_STATUS]) static_cast<int*>(a.out[CDK_OUT_STATUS])[traj] = final_status(status, isfinite(ll));
  }
}


// ======================================================================================================================
// Backward pass of cdlgssm_smoother, smoother_type 'cd_smoother_1' (cd_linear/inference.py:746-773, Sarkka Alg. 3.17):
// for k = K-2 .. 0 re-integrate the pushforward (A, Q) over [t_k, t_{k+1}] (:753), then
//   C = psd_solve(A P_f A^T + Q, A P_f)^T,  m_s = m_f + C (m_s^+ - A m_f - b),  P_s = P_f + C (P_s^+ - A P_f A^T - Q) C^T,
//   cross = C P_s^+ + m_s m_s^{+T}.
// Same mapping as the filter: one warp per trajectory, every n x n product on the FP64 tensor cores, the 16 x 16 Cholesky
// and the two triangular solves warp-cooperative in shared memory (one lane per row / per right-hand-side column).
// ======================================================================================================================
constexpr int KS_WPC = 6;  // 6 warps x 16 KB + model: two CTAs (12 trajectories) per SM
struct KsSmemCounts {
  static constexpr int PER_WARP = 6 * KW_MAT + 5 * 16;
};

template <bool POLY>
__global__ void __launch_bounds__(32 * KS_WPC, 2) kf_warp_smooth(const KArgs<double> a, const __grid_constant__ KwTab tab, const int model_per_warp, const int use_rk) {
  extern __shared__ __align__(16) double kw_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const cdk_desc& d = a.d;
  const int n = d.n, K = d.K;
  const long long traj = (long long)blockIdx.x * KS_WPC + warp;
  double* model = kw_smem + (model_per_warp ? warp * KwSmemCounts::PER_MODEL : 0);
  double* wbase = kw_smem + (model_per_warp ? KS_WPC : 1) * KwSmemCounts::PER_MODEL + warp * KsSmemCounts::PER_WARP;
  double* sF = model;
  double* sLQL = sF + KW_MAT;
  double* sb = sLQL + KW_MAT + 2 * KW_MAT8;
  const double* sRk = (use_rk & 1) ? model + KW_RK_OFF : nullptr;
  double* sPs = wbase;        // smoothed covariance of step k+1
  double* sPf = sPs + KW_MAT;  // filtered covariance of step k
  double* sYA = sPf + KW_MAT;  // stage buffer, then A
  double* sYQ = sYA + KW_MAT;  // stage buffer, then sym(P_pred) -> its Cholesky factor -> C (P_s^+ - P_pred)
  double* sT = sYQ + KW_MAT;   // stage buffer, then A P_f -> C^T
  double* sDm = sT + KW_MAT;   // P_s^+ - P_pred
  double* sms = sDm + KW_MAT;
  double* smf = sms + 16;
  double* srv = smf + 16;
  double* smn = srv + 16;
  double* sinv = smn + 16;

  const long long tj = traj < d.N ? traj : d.N - 1;
  if (model_per_warp || warp == 0) {
    load_model_kw(a, tj, model, sYA, sYQ, sT);
    __syncwarp();
    rk_map<POLY>(tab, d.dt0, sF, model + KW_RK_OFF, sYA);
  }
  __syncthreads();  // the only CTA-wide barrier: the shared model block is ready
  if (traj >= d.N) return;
  for (int e = lane; e < KsSmemCounts::PER_WARP; e += 32) wbase[e] = 0.0;
  __syncwarp();

  const double* __restrict__ Tm = a.in[CDK_IN_T] + traj * a.in_stride[CDK_IN_T];
  const double* __restrict__ FMg = a.in[CDK_IN_FM] + traj * a.in_stride[CDK_IN_FM];
  const double* __restrict__ FPg = a.in[CDK_IN_FP] + traj * a.in_stride[CDK_IN_FP];
  double* __restrict__ SMg = static_cast<double*>(a.out[CDK_OUT_SM]) + traj * (long long)K * n;
  double* __restrict__ SPg = static_cast<double*>(a.out[CDK_OUT_SP]) + traj * (long long)K * n * n;
  double* __restrict__ SCg =
      a.out[CDK_OUT_SCROSS] ? static_cast<double*>(a.out[CDK_OUT_SCROSS]) + traj * (long long)(K - 1) * n * n : nullptr;
  const double dt0 = d.dt0;
  int status = 0;
  const double* AQ =
      (d.reserved[2] & CDK_FLAG_KEEP_PUSHFORWARD) ? static_cast<const double*>(a.out[CDK_OUT_SCRATCH]) : nullptr;

  // last step: smoothed = filtered (:813-814)
  for (int e = lane; e < n * n; e += 32) {
    const double v = FPg[(long long)(K - 1) * n * n + e];
    sPs[(e / n) * KW_LD + (e % n)] = v;
    SPg[(long long)(K - 1) * n * n + e] = v;
  }
  if (lane < n) {
    const double v = FMg[(long long)(K - 1) * n + lane];
    sms[lane] = v;
    SMg[(long long)(K - 1) * n + lane] = v;
  }
  __syncwarp();

  for (int k = K - 2; k >= 0; --k) {
    for (int e = lane; e < n * n; e += 32) sPf[(e / n) * KW_LD + (e % n)] = FPg[(long long)k * n * n + e];
    if (lane < n) smf[lane] = FMg[(long long)k * n + lane];
    const double t0 = Tm[k], t1 = Tm[k + 1];
    F16 yA, yQ;
    if (AQ) {  // the filter kept (A_k, Q_k) of this gap (bit-identical to re-integrating it)
      const double* src = AQ + ((traj * (long long)(K - 1) + k) * 2) * n * n;
      load_global(yA.v, src, n);
      load_global(yQ.v, src + n * n, n);  // (zero padding: the padded rows of P_f are zero, so A's identity pad is moot)
    } else if (pushforward<POLY>(tab, dt0, d.max_steps, t0, t1, sF, sLQL, sRk, sYA, sYQ, sT, yA, yQ, (use_rk & 2) != 0)) {
      status = 2;
    }
    store_c<2, 2>(yA.v, sYA);
    __syncwarp();
    {
      F16 ap;
      mm<false, false, 16, 2, 2>(ap.v, sYA, sPf);  // A P_f
      store_c<2, 2>(ap.v, sT);
      if (lane < 16) {  // rv = m_s^+ - A m_f - b   (:763-766)
        double s = 0.0;
        for (int q = 0; q < n; ++q) s += sYA[lane * KW_LD + q] * smf[q];
        srv[lane] = lane < n ? sms[lane] - s - sb[lane] : 0.0;
      }
      __syncwarp();
      F16 pp, ps, ppt;
      mm<false, true, 16, 2, 2>(pp.v, sT, sYA);  // A P_f A^T
      load_c<2, 2>(ps.v, sPs);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        (&pp.v[0][0][0])[i] += (&yQ.v[0][0][0])[i];                      // P_pred = A P_f A^T + Q
        (&ps.v[0][0][0])[i] -= (&pp.v[0][0][0])[i];                      // P_s^+ - P_pred
      }
      store_c<2, 2>(ps.v, sDm);
      store_c<2, 2>(pp.v, sYQ);
      __syncwarp();
      load_ct(ppt.v, sYQ);
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 8; ++i) (&pp.v[0][0][0])[i] = 0.5 * ((&pp.v[0][0][0])[i] + (&ppt.v[0][0][0])[i]);  // symmetrize
      store_c<2, 2>(pp.v, sYQ);
      __syncwarp();
    }
    // ---- psd_solve: Cholesky of sym(P_pred) + 1e-9 I, in place (lower triangle of sYQ), lane = row ----
    for (int j = 0; j < n; ++j) {
      if (lane >= j && lane < n) {
        double sjj = sYQ[j * KW_LD + j] + 1e-9;
        for (int q = 0; q < j; ++q) sjj -= sYQ[j * KW_LD + q] * sYQ[j * KW_LD + q];
        const double dj = sqrt(sjj);
        const double idj = 1.0 / dj;
        if (lane == j) {
          sinv[j] = idj;
        } else {
          double v = sYQ[lane * KW_LD + j];
          for (int q = 0; q < j; ++q) v -= sYQ[lane * KW_LD + q] * sYQ[j * KW_LD + q];
          sYQ[lane * KW_LD + j] = v * idj;
        }
      }
      __syncwarp();
    }
    // ---- C^T = (P_pred + boost)^-1 A P_f: one right-hand-side column per lane, in place in sT ----
    if (lane < n) {
      for (int i = 0; i < n; ++i) {
        double v = sT[i * KW_LD + lane];
        for (int q = 0; q < i; ++q) v -= sYQ[i * KW_LD + q] * sT[q * KW_LD + lane];
        sT[i * KW_LD + lane] = v * sinv[i];
      }
      for (int i = n - 1; i >= 0; --i) {
        double v = sT[i * KW_LD + lane];
        for (int q = i + 1; q < n; ++q) v -= sYQ[q * KW_LD + i] * sT[q * KW_LD + lane];
        sT[i * KW_LD + lane] = v * sinv[i];
      }
    }
    __syncwarp();
    {
      const double* sCt = sT;
      F16 cd, cps;
      mm<true, false, 16, 2, 2>(cd.v, sCt, sDm);   // C (P_s^+ - P_pred)
      mm<true, false, 16, 2, 2>(cps.v, sCt, sPs);  // C P_s^+
      if (lane < 16) {  // m_s = m_f + C rv
        double s = 0.0;
        for (int q = 0; q < n; ++q) s += sCt[q * KW_LD + lane] * srv[q];
        smn[lane] = lane < n ? smf[lane] + s : 0.0;
      }
      __syncwarp();
      store_c<2, 2>(cd.v, sYQ);  // the Cholesky factor is no longer needed
      if (SCg) {                 // cross = C P_s^+ + m_s m_s^{+T}   (:771)
        const int gid = lane >> 2, tig = lane & 3;
#pragma unroll
        for (int rb = 0; rb < 2; ++rb)
#pragma unroll
          for (int cb = 0; cb < 2; ++cb)
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              const int i = 8 * rb + gid, j = 8 * cb + 2 * tig + r;
              cps.v[rb][cb][r] += smn[i] * sms[j];
            }
        store_global(cps.v, SCg + (long long)k * n * n, n);
      }
      __syncwarp();
      F16 pn, pf;
      mm<false, false, 16, 2, 2>(pn.v, sYQ, sCt);  // C (P_s^+ - P_pred) C^T
      load_c<2, 2>(pf.v, sPf);
#pragma unroll
      for (int i = 0; i < 8; ++i) (&pn.v[0][0][0])[i] += (&pf.v[0][0][0])[i];
      __syncwarp();
      store_c<2, 2>(pn.v, sPs);
      store_global(pn.v, SPg + (long long)k * n * n, n);
      if (lane < 16) sms[lane] = smn[lane];
      if (lane < n) SMg[(long long)k * n + lane] = smn[lane];
      __syncwarp();
    }
  }
  if (lane == 0 && a.out[CDK_OUT_STATUS]) {
    bool bad = false;
    for (int i = 0; i < n; ++i) bad |= !isfinite(sms[i]);
    merge_smoother_status(static_cast<int*>(a.out[CDK_OUT_STATUS]), traj, status, !bad);
  }
}

// ======================================================================================================================
// Reverse-mode gradient of the filter's log-likelihood (cdk_kf_grad_f64).  kf_warp_filter runs first and writes the
// filtered and predicted moments to scratch; kf_warp_grad then walks k = K-1 .. 0 with the adjoint (mu_bar, P_bar) of the
// predicted moments that enter update k+1, one warp per trajectory, every n x n product on the FP64 tensor cores:
//   update VJP      (m <= 8, warp-cooperative in shared memory like the forward update),
//   predict VJP     mu' = A mu_f + b, P' = A P_f A^T + Q,
//   pushforward VJP the gap is re-integrated from (I, 0) stage by stage (any tableau, Dopri5 included) with the substep
//                   start states kept at two checkpoint levels of KG_CK slots in the trajectory's scratch, then stepped
//                   back substep by substep: the stage inputs of the substep are rebuilt in shared memory and the stage
//                   cotangents (Ca, Cq) give A_i_bar = F^T Ca, Q_i_bar = F^T Cq + Cq F, F_bar += Ca A_i^T + 2 Cq Q_i,
//                   Sigma_bar += Cq (Cq stays symmetric).
// Adjoints of symmetric matrices (P, Q, S) are kept symmetric: every perturbation of the parameters that keeps Sigma, R and
// P0 symmetric keeps them symmetric, so this gives the exact derivative along those directions.
// ======================================================================================================================
constexpr int KG_CK = 32;           // checkpoint slots per level; a gap of up to KG_CK^2 substeps is re-integrated once
constexpr int KG_STATE = 16 * 32;   // one (A, Q) state in fragment layout: 16 doubles per lane
constexpr int KG_WPC_MAX = 8;

struct KgTab {
  int S;
  double a[6][6];  // dense Butcher matrix (a[i][j], j < i)
  double b[6];
};

// fragment-layout state <-> global scratch (coalesced: element i of every lane is contiguous)
__device__ __forceinline__ void kg_save(double* __restrict__ dst, const F16& A, const F16& Q) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    dst[i * 32 + lane] = (&A.v[0][0][0])[i];
    dst[(8 + i) * 32 + lane] = (&Q.v[0][0][0])[i];
  }
}
__device__ __forceinline__ void kg_load(const double* __restrict__ src, F16& A, F16& Q) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    (&A.v[0][0][0])[i] = src[i * 32 + lane];
    (&Q.v[0][0][0])[i] = src[(8 + i) * 32 + lane];
  }
}

// One explicit RK substep of (A, Q) through the stages of any tableau.  The stage inputs are accumulated in place in
// sStg[2 st] (A) / sStg[2 st + 1] (Q), which hold them afterwards for kg_step_vjp; y is advanced in place.
__device__ __forceinline__ void kg_step(const KgTab& tab, const double dt, const double* sF, const double* sLQL, double* sStg,
                                        double* sT, F16& yA, F16& yQ) {
  F16 accA = yA, accQ = yQ;
#pragma unroll 1
  for (int st = 0; st < tab.S; ++st) {
    store_c<2, 2>(yA.v, sStg + (2 * st) * KW_MAT);
    store_c<2, 2>(yQ.v, sStg + (2 * st + 1) * KW_MAT);
  }
  __syncwarp();
#pragma unroll 1
  for (int st = 0; st < tab.S; ++st) {
    F16 kA, fq, fqt, lq;
    mm2_shared_a(kA.v, fq.v, sF, sStg + (2 * st) * KW_MAT, sStg + (2 * st + 1) * KW_MAT);  // F A_i, F Q_i
    store_c<2, 2>(fq.v, sT);
    __syncwarp();
    load_ct(fqt.v, sT);
    load_c<2, 2>(lq.v, sLQL);
#pragma unroll
    for (int i = 0; i < 8; ++i) (&fq.v[0][0][0])[i] = ((&fq.v[0][0][0])[i] + (&fqt.v[0][0][0])[i]) + (&lq.v[0][0][0])[i];
    const double w = tab.b[st] * dt;
    if (w != 0.0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        (&accA.v[0][0][0])[i] = fma(w, (&kA.v[0][0][0])[i], (&accA.v[0][0][0])[i]);
        (&accQ.v[0][0][0])[i] = fma(w, (&fq.v[0][0][0])[i], (&accQ.v[0][0][0])[i]);
      }
    }
#pragma unroll 1
    for (int s2 = st + 1; s2 < tab.S; ++s2) {  // lane-local: every lane updates its own fragment entries
      const double c = tab.a[s2][st] * dt;
      if (c == 0.0) continue;
      F16 iA, iQ;
      load_c<2, 2>(iA.v, sStg + (2 * s2) * KW_MAT);
      load_c<2, 2>(iQ.v, sStg + (2 * s2 + 1) * KW_MAT);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        (&iA.v[0][0][0])[i] = fma(c, (&kA.v[0][0][0])[i], (&iA.v[0][0][0])[i]);
        (&iQ.v[0][0][0])[i] = fma(c, (&fq.v[0][0][0])[i], (&iQ.v[0][0][0])[i]);
      }
      store_c<2, 2>(iA.v, sStg + (2 * s2) * KW_MAT);
      store_c<2, 2>(iQ.v, sStg + (2 * s2 + 1) * KW_MAT);
    }
    __syncwarp();
  }
  yA = accA;
  yQ = accQ;
}

// VJP of the substep kg_step just took (its stage inputs in sStg): (lamA, lamQ) is the cotangent of the substep's end
// state on entry and of its start state on exit; gF / gS accumulate F_bar / Sigma_bar.  The stage buffers are overwritten
// with the stage-input cotangents.
__device__ __forceinline__ void kg_step_vjp(const KgTab& tab, const double dt, const double* sFt, double* sStg, double* sCa,
                                            double* sCq, double* sT, F16& lamA, F16& lamQ, F16& gF, F16& gS) {
#pragma unroll 1
  for (int st = tab.S - 1; st >= 0; --st) {
    F16 ca, cq;
    const double w = tab.b[st] * dt;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      (&ca.v[0][0][0])[i] = w * (&lamA.v[0][0][0])[i];
      (&cq.v[0][0][0])[i] = w * (&lamQ.v[0][0][0])[i];
    }
#pragma unroll 1
    for (int s2 = st + 1; s2 < tab.S; ++s2) {
      const double c = tab.a[s2][st] * dt;
      if (c == 0.0) continue;
      F16 bA, bQ;
      load_c<2, 2>(bA.v, sStg + (2 * s2) * KW_MAT);
      load_c<2, 2>(bQ.v, sStg + (2 * s2 + 1) * KW_MAT);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        (&ca.v[0][0][0])[i] = fma(c, (&bA.v[0][0][0])[i], (&ca.v[0][0][0])[i]);
        (&cq.v[0][0][0])[i] = fma(c, (&bQ.v[0][0][0])[i], (&cq.v[0][0][0])[i]);
      }
    }
    store_c<2, 2>(ca.v, sCa);
    store_c<2, 2>(cq.v, sCq);
    __syncwarp();
    F16 x, y;
    mm<false, true, 16, 2, 2>(x.v, sCa, sStg + (2 * st) * KW_MAT);       // Ca A_i^T
    mm<false, false, 16, 2, 2>(y.v, sCq, sStg + (2 * st + 1) * KW_MAT);  // Cq Q_i
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      (&gF.v[0][0][0])[i] += (&x.v[0][0][0])[i] + 2.0 * (&y.v[0][0][0])[i];
      (&gS.v[0][0][0])[i] += (&cq.v[0][0][0])[i];
    }
    mm2_shared_a(x.v, y.v, sFt, sCa, sCq);  // F^T Ca, F^T Cq
    store_c<2, 2>(y.v, sT);
    __syncwarp();
    F16 yt;
    load_ct(yt.v, sT);
#pragma unroll
    for (int i = 0; i < 8; ++i) (&y.v[0][0][0])[i] += (&yt.v[0][0][0])[i];
    store_c<2, 2>(x.v, sStg + (2 * st) * KW_MAT);
    store_c<2, 2>(y.v, sStg + (2 * st + 1) * KW_MAT);
    __syncwarp();
  }
#pragma unroll 1
  for (int st = 0; st < tab.S; ++st) {  // the start state feeds every stage input with coefficient 1
    F16 bA, bQ;
    load_c<2, 2>(bA.v, sStg + (2 * st) * KW_MAT);
    load_c<2, 2>(bQ.v, sStg + (2 * st + 1) * KW_MAT);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      (&lamA.v[0][0][0])[i] += (&bA.v[0][0][0])[i];
      (&lamQ.v[0][0][0])[i] += (&bQ.v[0][0][0])[i];
    }
  }
  __syncwarp();
}

struct KgLayout {
  // per-warp shared memory (doubles): P_bar, the work slots, small vectors, Cholesky factors, checkpoint clocks
  static constexpr int VEC = 16 * 4 + 8 * 4 + 72 * 2;
  static constexpr int CLOCK = (int)((sizeof(StepClock<double>) + 7) / 8);
  static __host__ __device__ int slots(int S) { return 2 * S + 3 > 7 ? 2 * S + 3 : 7; }
  static __host__ __device__ int per_warp(int S) { return (1 + slots(S)) * KW_MAT + VEC + 2 * KG_CK * CLOCK; }
  // per-trajectory scratch (doubles): FM, FP, PM, PP of the forward pass ([N][K][...] each), the checkpoints, the status
  static __host__ __device__ long long moments(int K, int n) { return (long long)K * (2 * n + 2 * n * n); }
  static __host__ __device__ long long per_traj(int K, int n) { return moments(K, n) + 2 * KG_CK * KG_STATE + 1; }
};

__global__ void __launch_bounds__(32 * KG_WPC_MAX, 1) kf_warp_grad(const KArgs<double> a, const __grid_constant__ KgTab tab,
                                                                  const int model_per_warp, const int per_warp,
                                                                  const double* __restrict__ sc, double* __restrict__ ckpt,
                                                                  const int* __restrict__ status, double* __restrict__ grad) {
  extern __shared__ __align__(16) double kw_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, gid = lane >> 2, tig = lane & 3;
  const int wpc = blockDim.x >> 5;
  const cdk_desc& d = a.d;
  const int n = d.n, m = d.m, K = d.K;
  const long long N = d.N;
  const long long traj = (long long)blockIdx.x * wpc + warp;
  double* model = kw_smem + (model_per_warp ? warp * KwSmemCounts::PER_MODEL : 0);
  double* wbase = kw_smem + (model_per_warp ? wpc : 1) * KwSmemCounts::PER_MODEL + warp * per_warp;
  double* sF = model;
  double* sLQL = sF + KW_MAT;
  double* sH = sLQL + KW_MAT;
  double* sR = sH + KW_MAT8;
  double* sb = sR + KW_MAT8;
  double* sd = sb + 16;
  double* sFt = model + KW_RK_OFF;  // F^T in the slot of the filter's RK map
  double* sPb = wbase;
  double* W = sPb + KW_MAT;
  const int nslots = KgLayout::slots(tab.S);
  double* smu = W + nslots * KW_MAT;  // predicted mean entering the update
  double* smub = smu + 16;            // adjoint of the mean
  double* smf = smub + 16;            // filtered mean
  double* sv = smf + 16;
  double* sr = sv + 16;
  double* sz = sr + 8;
  double* srb = sz + 8;
  double* sy = srb + 8;
  double* sL0 = sy + 8;   // [8][9] Cholesky factor of S (log-likelihood)
  double* sLb = sL0 + 72;  // [8][9] Cholesky factor of sym(S) + 1e-9 I (gain)
  StepClock<double>* ckc1 = reinterpret_cast<StepClock<double>*>(sLb + 72);
  StepClock<double>* ckc2 = reinterpret_cast<StepClock<double>*>(sLb + 72 + KG_CK * KgLayout::CLOCK);

  const long long tj = traj < N ? traj : N - 1;
  if (model_per_warp || warp == 0) {
    load_model_kw(a, tj, model, W, W + KW_MAT, W + 2 * KW_MAT);
    __syncwarp();
    for (int e = lane; e < KW_MAT; e += 32) {
      const int i = e / KW_LD, j = e - i * KW_LD;
      sFt[e] = j < 16 ? sF[j * KW_LD + i] : 0.0;
    }
  }
  __syncthreads();  // the only CTA-wide barrier: the shared model block is ready
  if (traj >= N) return;
  const int cols = 3 * n * n + m * n + m * m + 2 * n + m;
  double* grow = grad + traj * (long long)cols;
  if (status[traj] != 0) {
    for (int e = lane; e < cols; e += 32) grow[e] = NAN;
    return;
  }
  for (int e = lane; e < per_warp; e += 32) wbase[e] = 0.0;
  __syncwarp();

  const long long NK = N * (long long)K;
  const double* FMg = sc + traj * (long long)K * n;
  const double* FPg = sc + NK * n + traj * (long long)K * n * n;
  const double* PMg = sc + NK * (n + n * n) + traj * (long long)K * n;
  const double* PPg = sc + NK * (2 * n + n * n) + traj * (long long)K * n * n;
  double* ck1 = ckpt + traj * (long long)(2 * KG_CK * KG_STATE);
  double* ck2 = ck1 + KG_CK * KG_STATE;
  const double* __restrict__ Y = a.in[CDK_IN_Y] + traj * a.in_stride[CDK_IN_Y];
  const double* __restrict__ Tm = a.in[CDK_IN_T] + traj * a.in_stride[CDK_IN_T];
  const double dt0 = d.dt0;

  F16 gF, gS;
#pragma unroll
  for (int i = 0; i < 8; ++i) (&gF.v[0][0][0])[i] = (&gS.v[0][0][0])[i] = 0.0;
  double gH[1][2][2] = {{{0.0, 0.0}, {0.0, 0.0}}}, gR[1][1][2] = {{{0.0, 0.0}}};
  double gb = 0.0, gd = 0.0;

  for (int k = K - 1; k >= 0; --k) {
    if (k < K - 1) {
      // ================= gap [t_k, t_{k+1}]: forward from (I, 0), substep starts at checkpoint level 1 =================
      const double t0 = Tm[k], t1 = Tm[k + 1];
      StepClock<double> cnt(t0, t1, dt0);
      while (cnt.running()) cnt.advance();  // status 0: the filter took these cnt.n <= max_steps substeps
      const int q = cnt.n;
      const int s1 = q > KG_CK ? (q + KG_CK - 1) / KG_CK : 1;
      F16 yA, yQ;
#pragma unroll
      for (int rb = 0; rb < 2; ++rb)
#pragma unroll
        for (int cb = 0; cb < 2; ++cb)
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            yA.v[rb][cb][r] = (8 * rb + gid == 8 * cb + 2 * tig + r) ? 1.0 : 0.0;
            yQ.v[rb][cb][r] = 0.0;
          }
      {
        StepClock<double> clk(t0, t1, dt0);
        for (int i = 0; i < q; ++i) {
          if (i % s1 == 0) {
            kg_save(ck1 + (i / s1) * KG_STATE, yA, yQ);
            if (lane == 0) ckc1[i / s1] = clk;
          }
          kg_step(tab, clk.dt(), sF, sLQL, W + 3 * KW_MAT, W + 2 * KW_MAT, yA, yQ);
          clk.advance();
        }
      }
      // ================= predict VJP: mu' = A mu_f + b, P' = A P_f A^T + Q  (cotangents smub, sPb) =================
      double* sA = W + 3 * KW_MAT;
      double* sPf = W + 4 * KW_MAT;
      double* sT1 = W + 5 * KW_MAT;
      F16 lamA, lamQ;
      {
        __syncwarp();
        store_c<2, 2>(yA.v, sA);
        F16 pf;
        load_global(pf.v, FPg + (long long)k * n * n, n);
        store_c<2, 2>(pf.v, sPf);
        if (lane < 16) smf[lane] = lane < n ? FMg[(long long)k * n + lane] : 0.0;
        if (lane < n) gb += smub[lane];
        __syncwarp();
        F16 t1m, t2m;
        mm<false, false, 16, 2, 2>(t1m.v, sPb, sA);  // P'_bar A
        store_c<2, 2>(t1m.v, sT1);
        __syncwarp();
        mm<false, false, 16, 2, 2>(t2m.v, sT1, sPf);  // P'_bar A P_f
        load_c<2, 2>(lamQ.v, sPb);
#pragma unroll
        for (int rb = 0; rb < 2; ++rb)
#pragma unroll
          for (int cb = 0; cb < 2; ++cb)
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              const int i = 8 * rb + gid, j = 8 * cb + 2 * tig + r;
              lamA.v[rb][cb][r] = 2.0 * t2m.v[rb][cb][r] + smub[i] * smf[j];
            }
        if (lane < 16) {
          double s = 0.0;
          for (int qq = 0; qq < n; ++qq) s += sA[qq * KW_LD + lane] * smub[qq];
          sv[lane] = lane < n ? s : 0.0;
        }
        F16 pb, pbt;
        mm<true, false, 16, 2, 2>(pb.v, sA, sT1);  // A^T P'_bar A
        __syncwarp();
        if (lane < 16) smub[lane] = sv[lane];
        store_c<2, 2>(pb.v, sT1);
        __syncwarp();
        load_ct(pbt.v, sT1);
#pragma unroll
        for (int i = 0; i < 8; ++i) (&pb.v[0][0][0])[i] = 0.5 * ((&pb.v[0][0][0])[i] + (&pbt.v[0][0][0])[i]);
        store_c<2, 2>(pb.v, sPb);
        __syncwarp();
      }
      // ================= pushforward VJP, substep by substep from the last =================
      double* sCa = W;
      double* sCq = W + KW_MAT;
      double* sT = W + 2 * KW_MAT;
      double* sStg = W + 3 * KW_MAT;
      const int nseg = q > 0 ? (q + s1 - 1) / s1 : 0;
      for (int seg = nseg - 1; seg >= 0; --seg) {
        const int i0 = seg * s1, len = (q - i0 < s1 ? q - i0 : s1);
        const int s2 = len > KG_CK ? (len + KG_CK - 1) / KG_CK : 1;
        if (len > 1) {  // level 2: the substep starts of this segment
          StepClock<double> clk = ckc1[seg];
          kg_load(ck1 + seg * KG_STATE, yA, yQ);
          for (int u = 0; u < len - 1; ++u) {
            if (u % s2 == 0) {
              kg_save(ck2 + (u / s2) * KG_STATE, yA, yQ);
              if (lane == 0) ckc2[u / s2] = clk;
            }
            kg_step(tab, clk.dt(), sF, sLQL, sStg, sT, yA, yQ);
            clk.advance();
          }
          if ((len - 1) % s2 == 0) {
            kg_save(ck2 + ((len - 1) / s2) * KG_STATE, yA, yQ);
            if (lane == 0) ckc2[(len - 1) / s2] = clk;
          }
          __syncwarp();
        }
        for (int u = len - 1; u >= 0; --u) {
          StepClock<double> clk = len > 1 ? ckc2[u / s2] : ckc1[seg];
          kg_load(len > 1 ? ck2 + (u / s2) * KG_STATE : ck1 + seg * KG_STATE, yA, yQ);
          for (int v = (len > 1 ? (u / s2) * s2 : u); v < u; ++v) {
            kg_step(tab, clk.dt(), sF, sLQL, sStg, sT, yA, yQ);
            clk.advance();
          }
          kg_step(tab, clk.dt(), sF, sLQL, sStg, sT, yA, yQ);  // rebuilds the stage inputs of substep i0 + u
          kg_step_vjp(tab, clk.dt(), sFt, sStg, sCa, sCq, sT, lamA, lamQ, gF, gS);
        }
      }
    }
    // ================= update VJP at k (cotangents of the filtered moments in smub / sPb) =================
    {
      double* sP = W;
      double* sT = W + KW_MAT;
      double* sG = W + 2 * KW_MAT;
      double* sS = sG + KW_MAT8;
      double* sKt = W + 3 * KW_MAT;
      double* sKtPb = sKt + KW_MAT8;
      double* sGb = W + 4 * KW_MAT;
      double* sSb = sGb + KW_MAT8;
      double* sWm = W + 5 * KW_MAT;
      double* sX8 = sWm + KW_MAT8;
      double* sSi = W + 6 * KW_MAT;
      {
        F16 p;
        if (k == 0) {
          load_global(p.v, a.in[CDK_IN_P0] + traj * a.in_stride[CDK_IN_P0], n);
          if (lane < 16) smu[lane] = lane < n ? (a.in[CDK_IN_M0] + traj * a.in_stride[CDK_IN_M0])[lane] : 0.0;
        } else {
          load_global(p.v, PPg + (long long)(k - 1) * n * n, n);
          if (lane < 16) smu[lane] = lane < n ? PMg[(long long)(k - 1) * n + lane] : 0.0;
        }
        store_c<2, 2>(p.v, sP);
        if (lane < 8) sy[lane] = lane < m ? Y[(long long)k * m + lane] : 0.0;
      }
      __syncwarp();
      double hp[1][2][2];
      mm<false, false, 16, 1, 2>(hp, sH, sP);  // G = H P
      store_c<1, 2>(hp, sG);
      store_c<1, 2>(hp, sKt);
      if (lane < 8) {
        double s = 0.0;
        if (lane < m) {
          s = sy[lane] - sd[lane];
          for (int qq = 0; qq < n; ++qq) s -= sH[lane * KW_LD + qq] * smu[qq];
        }
        sr[lane] = s;
      }
      __syncwarp();
      {
        double sf[1][1][2];
        mm<false, true, 16, 1, 1>(sf, sG, sH);  // S = H P H^T + R
        sS[gid * KW_LD + 2 * tig] = sf[0][0][0] + sR[gid * KW_LD + 2 * tig];
        sS[gid * KW_LD + 2 * tig + 1] = sf[0][0][1] + sR[gid * KW_LD + 2 * tig + 1];
      }
      __syncwarp();
      for (int pass = 0; pass < 2; ++pass) {  // chol(S) and chol(sym(S) + 1e-9 I), as the filter
        double* Lf = pass ? sLb : sL0;
        for (int j = 0; j < m; ++j) {
          if (lane >= j && lane < m) {
            double sjj = sS[j * KW_LD + j] + (pass ? 1e-9 : 0.0);
            for (int qq = 0; qq < j; ++qq) sjj -= Lf[j * 9 + qq] * Lf[j * 9 + qq];
            const double dj = sqrt(sjj);
            if (lane == j) {
              Lf[j * 9 + j] = dj;
            } else {
              double v = pass ? 0.5 * (sS[lane * KW_LD + j] + sS[j * KW_LD + lane]) : sS[lane * KW_LD + j];
              for (int qq = 0; qq < j; ++qq) v -= Lf[lane * 9 + qq] * Lf[j * 9 + qq];
              Lf[lane * 9 + j] = v / dj;
            }
          }
          __syncwarp();
        }
      }
      if (lane < m) {  // column `lane` of S^-1 (un-boosted factor), in place in sSi
        for (int i = 0; i < m; ++i) {
          double v = i == lane ? 1.0 : 0.0;
          for (int qq = 0; qq < i; ++qq) v -= sL0[i * 9 + qq] * sSi[qq * KW_LD + lane];
          sSi[i * KW_LD + lane] = v / sL0[i * 9 + i];
        }
        for (int i = m - 1; i >= 0; --i) {
          double v = sSi[i * KW_LD + lane];
          for (int qq = i + 1; qq < m; ++qq) v -= sL0[qq * 9 + i] * sSi[qq * KW_LD + lane];
          sSi[i * KW_LD + lane] = v / sL0[i * 9 + i];
        }
      } else if (lane >= 16 && lane < 16 + n) {  // K^T = (sym(S) + 1e-9 I)^-1 G, column lane - 16, in place in sKt
        const int c = lane - 16;
        for (int i = 0; i < m; ++i) {
          double v = sKt[i * KW_LD + c];
          for (int qq = 0; qq < i; ++qq) v -= sLb[i * 9 + qq] * sKt[qq * KW_LD + c];
          sKt[i * KW_LD + c] = v / sLb[i * 9 + i];
        }
        for (int i = m - 1; i >= 0; --i) {
          double v = sKt[i * KW_LD + c];
          for (int qq = i + 1; qq < m; ++qq) v -= sLb[qq * 9 + i] * sKt[qq * KW_LD + c];
          sKt[i * KW_LD + c] = v / sLb[i * 9 + i];
        }
      }
      __syncwarp();
      if (lane < 8) {  // z = S^-1 r;  r_bar = K^T mu_f_bar - z
        double z = 0.0, kb = 0.0;
        if (lane < m) {
          for (int qq = 0; qq < m; ++qq) z += sSi[lane * KW_LD + qq] * sr[qq];
          for (int qq = 0; qq < n; ++qq) kb += sKt[lane * KW_LD + qq] * smub[qq];
        }
        sz[lane] = z;
        srb[lane] = lane < m ? kb - z : 0.0;
      }
      {
        double x[1][2][2];
        mm<false, false, 16, 1, 2>(x, sKt, sPb);  // K^T P_f_bar
        store_c<1, 2>(x, sKtPb);
      }
      __syncwarp();
      double sbar[1][1][2];
      {
        double kpk[1][1][2], u[1][2][2];
        mm<false, true, 16, 1, 1>(kpk, sKtPb, sKt);  // K^T P_f_bar K
        mm<false, false, 8, 1, 2>(u, sS, sKtPb);     // S K^T P_f_bar
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const int i = gid, j = 2 * tig + r;
          sbar[0][0][r] = (i < m && j < m) ? 0.5 * sz[i] * sz[j] - 0.5 * sSi[i * KW_LD + j] - kpk[0][0][r] : 0.0;
        }
#pragma unroll
        for (int cb = 0; cb < 2; ++cb)
#pragma unroll
          for (int r = 0; r < 2; ++r) {  // K_bar^T = r mu_f_bar^T - 2 S K^T P_f_bar
            const int i = gid, j = 8 * cb + 2 * tig + r;
            u[0][cb][r] = i < m ? sr[i] * smub[j] - 2.0 * u[0][cb][r] : 0.0;
          }
        store_c<1, 2>(u, sGb);
      }
      __syncwarp();
      if (lane < n) {  // G_bar = (sym(S) + 1e-9 I)^-1 K_bar^T, column `lane`, in place in sGb
        for (int i = 0; i < m; ++i) {
          double v = sGb[i * KW_LD + lane];
          for (int qq = 0; qq < i; ++qq) v -= sLb[i * 9 + qq] * sGb[qq * KW_LD + lane];
          sGb[i * KW_LD + lane] = v / sLb[i * 9 + i];
        }
        for (int i = m - 1; i >= 0; --i) {
          double v = sGb[i * KW_LD + lane];
          for (int qq = i + 1; qq < m; ++qq) v -= sLb[qq * 9 + i] * sGb[qq * KW_LD + lane];
          sGb[i * KW_LD + lane] = v / sLb[i * 9 + i];
        }
      }
      __syncwarp();
      {
        double gk[1][1][2];
        mm<false, true, 16, 1, 1>(gk, sGb, sKt);  // G_bar K
        store_c<1, 1>(gk, sX8);
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 2; ++r) {  // S_bar -= sym(G_bar K)
          const int i = gid, j = 2 * tig + r;
          sbar[0][0][r] -= 0.5 * (gk[0][0][r] + sX8[j * KW_LD + i]);
          gR[0][0][r] += sbar[0][0][r];
        }
        store_c<1, 1>(sbar, sSb);
      }
      __syncwarp();
      {
        double p1[1][2][2], p2[1][2][2], p3[1][2][2], gbv[1][2][2];
        mm<false, false, 8, 1, 2>(p1, sSb, sG);   // S_bar G
        mm<false, false, 16, 1, 2>(p2, sGb, sP);  // G_bar P
        mm<false, false, 8, 1, 2>(p3, sSb, sH);   // S_bar H
        load_c<1, 2>(gbv, sGb);
#pragma unroll
        for (int cb = 0; cb < 2; ++cb)
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            const int i = gid, j = 8 * cb + 2 * tig + r;
            gH[0][cb][r] += 2.0 * p1[0][cb][r] + p2[0][cb][r] - srb[i] * smu[j];
            p3[0][cb][r] += gbv[0][cb][r];  // W = S_bar H + G_bar
          }
        store_c<1, 2>(p3, sWm);
      }
      if (lane < m) gd -= srb[lane];
      if (lane < n) {  // mu_bar = mu_f_bar - H^T r_bar
        double s = 0.0;
        for (int i = 0; i < m; ++i) s += sH[i * KW_LD + lane] * srb[i];
        smub[lane] -= s;
      }
      __syncwarp();
      {
        F16 X, Xt, pb;
        mm<true, false, 8, 2, 2>(X.v, sH, sWm);  // H^T W
        store_c<2, 2>(X.v, sT);
        __syncwarp();
        load_ct(Xt.v, sT);
        load_c<2, 2>(pb.v, sPb);
#pragma unroll
        for (int i = 0; i < 8; ++i)
          (&pb.v[0][0][0])[i] += 0.5 * ((&X.v[0][0][0])[i] + (&Xt.v[0][0][0])[i]);  // P_bar = P_f_bar + H^T S_bar H + sym(H^T G_bar)
        __syncwarp();
        store_c<2, 2>(pb.v, sPb);
        __syncwarp();
      }
    }
  }
  // ================= gradient row: F | b | Sigma (sym) | H | d | R (sym) | m0 | P0 (sym) =================
  double* sT = W;
  store_global(gF.v, grow, n);
  if (lane < n) grow[n * n + lane] = gb;
  store_c<2, 2>(gS.v, sT);
  __syncwarp();
  {
    F16 t;
    load_ct(t.v, sT);
#pragma unroll
    for (int i = 0; i < 8; ++i) (&gS.v[0][0][0])[i] = 0.5 * ((&gS.v[0][0][0])[i] + (&t.v[0][0][0])[i]);
  }
  store_global(gS.v, grow + n * n + n, n);
  double* gHrow = grow + 2 * n * n + n;
#pragma unroll
  for (int cb = 0; cb < 2; ++cb)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int i = gid, j = 8 * cb + 2 * tig + r;
      if (i < m && j < n) gHrow[i * n + j] = gH[0][cb][r];
    }
  if (lane < m) gHrow[m * n + lane] = gd;
  double* sX8 = W + KW_MAT;
  __syncwarp();
  store_c<1, 1>(gR, sX8);
  __syncwarp();
  double* gRrow = gHrow + m * n + m;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int i = gid, j = 2 * tig + r;
    if (i < m && j < m) gRrow[i * m + j] = 0.5 * (gR[0][0][r] + sX8[j * KW_LD + i]);
  }
  if (lane < n) gRrow[m * m + lane] = smub[lane];
  F16 p0;
  load_c<2, 2>(p0.v, sPb);
  store_global(p0.v, gRrow + m * m + n, n);
}

}  // namespace

// Fast path coverage: KF filter and type-1 smoother, fp64, n <= 16, m <= 8, no inputs, every solver of the registry (chain
// tableaux through their stages, Dopri5 -- the reference default -- through its step polynomial).
template <typename T>
int launch_kf_warp(int algo, const KArgs<T>& a, cudaStream_t s) {
  return CDK_E_UNSUPPORTED;
}

bool kf_warp_eligible(const cdk_desc& d, bool smooth) {
  static const bool disabled = []() {
    const char* e = getenv("CDK_KF_WARP");
    return e && e[0] == '0';
  }();
  if (disabled || d.n > 16 || d.m > 8 || d.d_u != 0) return false;
  if (!smooth && (d.reserved[2] & CDK_FLAG_DIAG_R)) return false;  // the Woodbury update lives in the generic kernel
  if (d.reserved[2] & CDK_FLAG_PREDICT_ONLY) return false;          // forecasts (no updates): generic kernel
  if (smooth && d.smoother_type != 1) return false;  // type 2 (backward ODE) stays on the generic kernel
  RtTab rt;
  return fill_rt_tab(d.solver, rt);  // chain tableaux step through the stages, the others (Dopri5) through the polynomial
}

template <>
int launch_kf_warp<double>(int algo, const KArgs<double>& a, cudaStream_t s) {
  const cdk_desc& d = a.d;
  const bool smooth = algo == ALGO_KF_SMOOTH;
  if (!kf_warp_eligible(d, smooth)) return CDK_E_UNSUPPORTED;
  RtTab rt;
  if (!fill_rt_tab(d.solver, rt)) return CDK_E_ENUM;
  KwTab tab;
  tab.S = rt.S;
  tab.poly = 0;
  for (int i = 0; i < 6; ++i) {
    if (rt.nnz[i] > 1 || (rt.nnz[i] == 1 && rt.col[i][0] != i - 1)) tab.poly = 1;  // not a chain tableau
    tab.a[i] = rt.nnz[i] ? rt.val[i][0] : 0.0;
    tab.b[i] = rt.b[i];
  }
  {
    // c_j = b^T A^{j-1} 1, j = 1 .. S (the coefficients of the step polynomial; c_1 = sum b = 1 for a consistent method)
    double Adense[6][6] = {};
    for (int i = 0; i < rt.S; ++i)
      for (int q = 0; q < rt.nnz[i]; ++q) Adense[i][rt.col[i][q]] = rt.val[i][q];
    double vec[6];
    for (int i = 0; i < 6; ++i) vec[i] = i < rt.S ? 1.0 : 0.0;
    for (int j = 0; j < 7; ++j) tab.c[j] = 0.0;
    for (int j = 1; j <= rt.S; ++j) {
      double cj = 0.0;
      for (int i = 0; i < rt.S; ++i) cj += rt.b[i] * vec[i];
      tab.c[j] = cj;
      double nv[6] = {};
      for (int i = 0; i < rt.S; ++i)
        for (int q = 0; q < rt.S; ++q) nv[i] += Adense[i][q] * vec[q];
      for (int i = 0; i < 6; ++i) vec[i] = nv[i];
    }
  }
  const uint32_t model_mask = (1u << CDK_IN_F) | (1u << CDK_IN_L) | (1u << CDK_IN_QC) | (1u << CDK_IN_H) | (1u << CDK_IN_R) |
                              (1u << CDK_IN_B) | (1u << CDK_IN_D);
  const int model_per_warp = (d.batched_mask & model_mask) != 0;
  static const int use_rk = []() {  // CDK_KF_RKMAP=0: step A through the RK stages like Q (A/B testing)
    const char* e = getenv("CDK_KF_RKMAP");
    return e ? atoi(e) : 1;  // bit 0: RK map for A; bit 1: Q F^T as a second tensor-core product
  }();
  if (smooth) {
    const size_t smem = sizeof(double) * ((model_per_warp ? KS_WPC : 1) * KwSmemCounts::PER_MODEL + KS_WPC * KsSmemCounts::PER_WARP);
    const long long blocks = (d.N + KS_WPC - 1) / KS_WPC;
    if (blocks > 2147483647LL) return CDK_E_SIZE;
    auto ks = tab.poly ? kf_warp_smooth<true> : kf_warp_smooth<false>;
    if (cudaFuncSetAttribute(ks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return check_launch("cudaFuncSetAttribute(kf_warp_smooth)");
    ks<<<(unsigned)blocks, 32 * KS_WPC, smem, s>>>(a, tab, model_per_warp, use_rk);
    note_launch();
    return check_launch("kf_warp_smooth");
  }
  const size_t smem = sizeof(double) * ((model_per_warp ? KW_WPC : 1) * KwSmemCounts::PER_MODEL + KW_WPC * KwSmemCounts::PER_WARP);
  const long long blocks = (d.N + KW_WPC - 1) / KW_WPC;
  if (blocks > 2147483647LL) return CDK_E_SIZE;
  auto kf = tab.poly ? kf_warp_filter<true> : kf_warp_filter<false>;
  if (cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("cudaFuncSetAttribute(kf_warp_filter)");
  kf<<<(unsigned)blocks, 32 * KW_WPC, smem, s>>>(a, tab, model_per_warp, use_rk);
  note_launch();
  return check_launch("kf_warp_filter");
}

long long kf_grad_scratch_doubles(const cdk_desc& d) { return d.N * KgLayout::per_traj(d.K, d.n); }

// Gradient of the log-likelihood of kf_warp_filter (cdk_kf_grad_f64): the forward filter into scratch, then kf_warp_grad.
int launch_kf_grad(const KArgs<double>& a, double* grad, cudaStream_t s) {
  const cdk_desc& d = a.d;
  double* sc = static_cast<double*>(a.out[CDK_OUT_SCRATCH]);
  const long long NK = d.N * (long long)d.K;
  const int n = d.n;
  int* status = a.out[CDK_OUT_STATUS] ? static_cast<int*>(a.out[CDK_OUT_STATUS])
                                      : reinterpret_cast<int*>(sc + d.N * KgLayout::per_traj(d.K, n) - d.N);
  KArgs<double> f = a;
  f.d.reserved[2] &= ~CDK_FLAG_KEEP_PUSHFORWARD;
  f.out[CDK_OUT_FM] = sc;
  f.out[CDK_OUT_FP] = sc + NK * n;
  f.out[CDK_OUT_PM] = sc + NK * (n + n * n);
  f.out[CDK_OUT_PP] = sc + NK * (2 * n + n * n);
  f.out[CDK_OUT_LLCUM] = nullptr;
  f.out[CDK_OUT_STATUS] = status;
  f.out[CDK_OUT_SCRATCH] = nullptr;
  f.out[CDK_OUT_GRAD] = nullptr;
  int rc = launch_kf_warp<double>(ALGO_KF_FILTER, f, s);
  if (rc != CDK_OK) return rc;
  RtTab rt;
  if (!fill_rt_tab(d.solver, rt)) return CDK_E_ENUM;
  KgTab tab;
  tab.S = rt.S;
  for (int i = 0; i < 6; ++i) {
    tab.b[i] = rt.b[i];
    for (int j = 0; j < 6; ++j) tab.a[i][j] = 0.0;
    for (int q = 0; q < rt.nnz[i]; ++q) tab.a[i][rt.col[i][q]] = rt.val[i][q];
  }
  const uint32_t model_mask = (1u << CDK_IN_F) | (1u << CDK_IN_L) | (1u << CDK_IN_QC) | (1u << CDK_IN_H) | (1u << CDK_IN_R) |
                              (1u << CDK_IN_B) | (1u << CDK_IN_D);
  const int model_per_warp = (d.batched_mask & model_mask) != 0;
  // as many warps as the 227 KB of one CTA hold (the stage buffers of Dopri5 are the largest case)
  const int per_warp = KgLayout::per_warp(tab.S);
  const size_t budget = 227 * 1024 / sizeof(double) - (model_per_warp ? 0 : KwSmemCounts::PER_MODEL);
  int wpc = (int)(budget / (per_warp + (model_per_warp ? KwSmemCounts::PER_MODEL : 0)));
  wpc = wpc > KG_WPC_MAX ? KG_WPC_MAX : wpc;
  const size_t smem = sizeof(double) * ((model_per_warp ? wpc : 1) * KwSmemCounts::PER_MODEL + (size_t)wpc * per_warp);
  const long long blocks = (d.N + wpc - 1) / wpc;
  if (blocks > 2147483647LL) return CDK_E_SIZE;
  if (cudaFuncSetAttribute(kf_warp_grad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("cudaFuncSetAttribute(kf_warp_grad)");
  kf_warp_grad<<<(unsigned)blocks, 32 * wpc, smem, s>>>(a, tab, model_per_warp, per_warp, sc, sc + NK * (2 * n + 2 * n * n),
                                                          status, grad);
  note_launch();
  return check_launch("kf_warp_grad");
}

template int launch_kf_warp<float>(int, const KArgs<float>&, cudaStream_t);

}  // namespace cdk
