// cdk_enkf.cu -- continuous-discrete ensemble Kalman filter: ONE THREAD-BLOCK CLUSTER PER TRAJECTORY.
//
// Replaces ensemble_kalman_filter (src/continuous_discrete_nonlinear_gaussian_ssm/inference_enkf.py:151-276) with its
// _predict (:47-89, per-member SDE solve) and _condition_on (:92-148, stochastic perturbed-observation update).
// The reference draws from jax.random (threefry) and a diffrax VirtualBrownianTree, neither reproducible outside JAX;
// this kernel and the CPU oracle share a counter-based Philox4x32-10 stream instead (oracle/cd_oracle.py enkf_normals),
// so parity against the oracle is to rounding and parity against the reference is distributional (as in its own test,
// src/test_scripts/cdnlgssm_test_filter_linear_TRegular.py:434-470).
//
// B200 mapping (BASELINE config 5: n = 40, m = 20, E = 1,024 members, N = 1,024 trajectories, K = 500):
//  * the ensemble X[n][E] (320 KB in fp64) does not fit one SM's shared memory, so a trajectory is owned by a CLUSTER of
//    C CTAs (C = 4 here), each keeping E/C members resident in shared memory for the whole kernel (dimension-major, so
//    member-per-thread accesses are conflict-free).  Nothing but the per-step moments ever goes to HBM.
//  * per-member work (Philox + Box-Muller noise, drift, Euler-Maruyama / Heun step, gain application) is one thread per
//    member with the member's state in registers;
//  * the E-contractions -- the ensemble covariance X'X'^T that every step needs twice (filtered and predicted moments;
//    the predicted one also yields C_xy = C_xx H^T and C_yy = H C_xx H^T of the next update because h is linear) -- run
//    on the FP64 TENSOR CORES (mma.sync m8n8k4 f64, SASS DMMA): each warp owns whole 8x8 output tiles and sweeps the
//    members, anomalies are formed on the fly in the fragment loads.  tcgen05 has no FP64 kind; DMMA is the FP64 tensor
//    path on sm_100a (measured 37.1 TFLOP/s = the FMA-pipe peak, but at 1/16 of the instruction count);
//  * CTA partial sums / partial covariances are combined through distributed shared memory (cluster.map_shared_rank),
//    every CTA summing the partials in rank order so that all CTAs of the cluster hold bit-identical moments and can run
//    the small (m x m) gain algebra redundantly without another exchange.
#include <cooperative_groups.h>

#include <stdlib.h>

#include "cdk_dense.cuh"
#include "cdk_rng.cuh"

namespace cg = cooperative_groups;

namespace cdk {
namespace {

constexpr int ENKF_TPB = 256;

// ---- shared-memory layout (identical on host and device) -----------------------------------------------------------
struct ELay {
  int n, m, ldn, ldm, ldE, nth;
  // byte offsets
  size_t X, PSUM, CPART, CXX, MEAN, H, R, CHR, DV, G, HP, S, SL, KT, SK, YV, RV, TH, MISC, DB, PHI, YSUM, YPART, total;
  // dg: room for the [m x ldE] innovation block of the tensor-core gain application (EArgs::dg)
  // ue: a user emission (cdk.h CDK_EMISSION_USER) with nphi parameters: the [m x ldE] block then holds the members'
  //     h(x_e); YSUM / YPART receive this CTA's partial sums of the emission moments (sum_e h(x_e); [m + n] x ldm partial
  //     sums of dY dY^T and dX dY^T), and there is no H / d
  __host__ __device__ ELay(int n_, int m_, int nth_, int Eloc, size_t ts, int dg, bool ue = false, int nphi = 0) {
    n = n_; m = m_; nth = nth_;
    ldn = ldp(n); ldm = ldp(m);
    ldE = ((Eloc + 31) / 32) * 32 + 4;  // = 4 (mod 32): DMMA fragment loads X[i0 + gid][e0 + tig] are conflict-free
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 15) & ~size_t(15); return r; };
    X = take(ts * n * ldE);
    PSUM = take(8 * n);
    CPART = take(8 * n * ldn);
    CXX = take(ts * n * ldn);
    MEAN = take(ts * n);
    H = take(ue ? 0 : ts * m * ldn);
    R = take(ts * m * ldm);
    CHR = take(ts * m * ldm);
    DV = take(ts * m);
    G = take(ts * n * ldn);
    HP = take(ts * m * ldn);
    S = take(ts * m * ldm);
    SL = take(ts * m * ldm);
    KT = take(ts * m * ldn);
    SK = take(ts * (m > n ? m : n) * ldp(m > n ? m : n));
    YV = take(ts * m);
    RV = take(ts * 2 * m);
    TH = take(ts * (nth > 0 ? nth : 1));
    MISC = take(64);
    DB = take(dg || ue ? ts * m * ldE : 0);
    PHI = take(ue ? ts * (nphi > 0 ? nphi : 1) : 0);
    YSUM = take(ue ? 8 * m : 0);
    YPART = take(ue ? 8 * (size_t)(m + n) * ldm : 0);
    total = o;
  }
};

template <typename T>
struct EArgs {
  KArgs<T> k;
  int C;     // cluster size (CTAs per trajectory)
  int dg;    // 1: gain application X += K (Y~ - H X - d) as two tensor-core products over the CTA's members (needs ELay::DB)
  int Eloc;  // members per CTA (the last CTA may own fewer)
  int ue;    // user emission (then dg = 0: the tensor-core gain application forms H X, which needs a linear h)
};

// ---- FP64 tensor-core partial covariance ----------------------------------------------------------------------------
// Cp[i][j] = sum over this CTA's members e of (X[i][e] - mu[i]) (X[j][e] - mu[j]), i, j < n (full symmetric matrix written).
// mma.sync.m8n8k4.f64: A (8x4, row) lane -> (row gid = lane/4, col tig = lane%4); B (4x8, col) lane -> (row tig, col gid);
// C/D (8x8) lane -> (row gid, cols 2*tig, 2*tig+1).  With A = X'[i-block][members], B = X'[members][j-block] both
// fragments are the SAME load pattern X[blk*8 + gid][e0 + tig].
template <typename T>
__device__ void cov_partial_dmma(const T* __restrict__ X, int ldE, int nmem, const T* __restrict__ mu, int n,
                                 double* __restrict__ Cp, int ldc) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int gid = lane >> 2, tig = lane & 3;
  const int nb = (n + 7) >> 3;
  const int ntile = nb * (nb + 1) / 2;
  const int nk = (nmem + 3) & ~3;
  for (int t = warp; t < ntile; t += nwarp) {
    // upper-triangular tile index t -> (bi <= bj)
    int bi = 0, rem = t;
    while (rem >= nb - bi) {
      rem -= nb - bi;
      ++bi;
    }
    const int bj = bi + rem;
    const int ia = bi * 8 + gid, jb = bj * 8 + gid;
    const bool va = ia < n, vb = jb < n;
    const T* xa = X + (size_t)(va ? ia : 0) * ldE;
    const T* xb = X + (size_t)(vb ? jb : 0) * ldE;
    const double ma = va ? (double)mu[ia] : 0.0, mb = vb ? (double)mu[jb] : 0.0;
    double d[4][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};  // 4 independent accumulator sets (k-steps interleaved)
    for (int e0 = 0; e0 < nk; e0 += 16) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + 4 * u + tig;
        const bool ve = e < nmem;
        const double av = (va && ve) ? (double)xa[e] - ma : 0.0;
        const double bv = (vb && ve) ? (double)xb[e] - mb : 0.0;
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                     : "+d"(d[u][0]), "+d"(d[u][1])
                     : "d"(av), "d"(bv));
      }
    }
    const double c0 = (d[0][0] + d[1][0]) + (d[2][0] + d[3][0]);
    const double c1 = (d[0][1] + d[1][1]) + (d[2][1] + d[3][1]);
    const int ri = bi * 8 + gid, cj = bj * 8 + 2 * tig;
    if (ri < n) {
      if (cj < n) {
        Cp[ri * ldc + cj] = c0;
        Cp[cj * ldc + ri] = c0;
      }
      if (cj + 1 < n) {
        Cp[ri * ldc + cj + 1] = c1;
        Cp[(cj + 1) * ldc + ri] = c1;
      }
    }
  }
}

// Ensemble mean and covariance (divided by E - 1) of the whole cluster's members; result in sh MEAN / CXX of EVERY CTA.
template <typename T>
__device__ void moments(cg::cluster_group& cluster, const ELay& L, unsigned char* sh, int nmem, int E, int C) {
  const int n = L.n, ldn = L.ldn;
  T* X = reinterpret_cast<T*>(sh + L.X);
  double* psum = reinterpret_cast<double*>(sh + L.PSUM);
  double* Cp = reinterpret_cast<double*>(sh + L.CPART);
  T* Cxx = reinterpret_cast<T*>(sh + L.CXX);
  T* mean = reinterpret_cast<T*>(sh + L.MEAN);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  for (int i = warp; i < n; i += nwarp) {
    double s = 0.0;
    for (int e = lane; e < nmem; e += 32) s += (double)X[(size_t)i * L.ldE + e];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) psum[i] = s;
  }
  cluster.sync();
  FOR_T(i, n) {
    double s = 0.0;
    for (int r = 0; r < C; ++r) s += cluster.map_shared_rank(psum, r)[i];
    mean[i] = (T)(s / (double)E);
  }
  __syncthreads();
  cov_partial_dmma<T>(X, L.ldE, nmem, mean, n, Cp, ldn);
  cluster.sync();
  const double inv = 1.0 / (double)(E - 1);
  FOR_T(idx, n * n) {
    const int i = idx / n, j = idx - i * n;
    if (i <= j) {
      double s = 0.0;
      for (int r = 0; r < C; ++r) s += cluster.map_shared_rank(Cp, r)[i * ldn + j];
      const T v = (T)(s * inv);
      Cxx[i * ldn + j] = v;
      Cxx[j * ldn + i] = v;
    }
  }
  cluster.sync();  // nobody may overwrite psum / Cp (next moments call) or read a stale Cxx before everyone is done
}

// The emission moments of the stochastic update with a user emission (inference_enkf.py:92-148, which maps every member
// through h): Y_e = h(x_e) per member (one thread each, into the DB block), then over the whole cluster
//   ybar = mean_e Y_e,  C_yy = sum_e dY_e dY_e^T / (E - 1),  C_xy = sum_e dX_e dY_e^T / (E - 1)
// with dX about the ensemble mean already in MEAN (the moments of this same ensemble).  Partial sums are combined in rank
// order as in moments(), so every CTA holds bit-identical values.  Out (every CTA): HP = C_xy^T [m x n], S = C_yy + R,
// rv = y - ybar.  (A linear h gives C_xy = C_xx H^T and C_yy = H C_xx H^T straight from the predicted moments; a nonlinear
// one does not.)
template <typename T>
__device__ void user_emission_moments(cg::cluster_group& cluster, const ELay& L, unsigned char* sh, int nmem, int E, int C,
                                      const T* phi, const T* yv) {
  const int n = L.n, m = L.m, ldn = L.ldn, ldm = L.ldm, ldE = L.ldE;
  const T* X = reinterpret_cast<const T*>(sh + L.X);
  const T* mean = reinterpret_cast<const T*>(sh + L.MEAN);
  const T* R = reinterpret_cast<const T*>(sh + L.R);
  T* Yb = reinterpret_cast<T*>(sh + L.DB);
  double* ysum = reinterpret_cast<double*>(sh + L.YSUM);
  double* part = reinterpret_cast<double*>(sh + L.YPART);  // rows a < m: dY_a dY^T; rows m + j: dX_j dY^T
  T* HP = reinterpret_cast<T*>(sh + L.HP);
  T* Sm = reinterpret_cast<T*>(sh + L.S);
  T* rv = reinterpret_cast<T*>(sh + L.RV);
  T* ybar = rv + m;
  for (int el = threadIdx.x; el < nmem; el += blockDim.x)
    for (int a = 0; a < m; ++a) Yb[(size_t)a * ldE + el] = user_h<T>(phi, n, m, a, [&](int j) { return X[(size_t)j * ldE + el]; });
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  for (int a = warp; a < m; a += nwarp) {
    double s = 0.0;
    for (int e = lane; e < nmem; e += 32) s += (double)Yb[(size_t)a * ldE + e];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) ysum[a] = s;
  }
  cluster.sync();
  FOR_T(a, m) {
    double s = 0.0;
    for (int r = 0; r < C; ++r) s += cluster.map_shared_rank(ysum, r)[a];
    ybar[a] = (T)(s / (double)E);
  }
  __syncthreads();
  FOR_T(e, (m + n) * m) {
    const int r = e / m, b = e - r * m;
    const T* u = r < m ? Yb + (size_t)r * ldE : X + (size_t)(r - m) * ldE;
    const double uc = (double)(r < m ? ybar[r] : mean[r - m]);
    const T* v = Yb + (size_t)b * ldE;
    const double vc = (double)ybar[b];
    double s = 0.0;
    for (int el = 0; el < nmem; ++el) s += ((double)u[el] - uc) * ((double)v[el] - vc);
    part[r * ldm + b] = s;
  }
  cluster.sync();
  const double inv = 1.0 / (double)(E - 1);
  FOR_T(e, (m + n) * m) {
    const int r = e / m, b = e - r * m;
    double s = 0.0;
    for (int q = 0; q < C; ++q) s += cluster.map_shared_rank(part, q)[r * ldm + b];
    const T v = (T)(s * inv);
    if (r < m) {
      Sm[r * ldm + b] = v + R[r * ldm + b];
    } else {
      HP[b * ldn + (r - m)] = v;
    }
  }
  FOR_T(a, m) rv[a] = yv[a] - ybar[a];
  cluster.sync();  // nobody may overwrite ysum / part (next update) before every CTA has read them
}

// Lorenz-96 drift entry and Euler-Maruyama update with the oracle's operation order and NO fused multiply-adds
// (((x_{i+1} - x_{i-2}) x_{i-1} - x_i) + F;  (x + dt f) + noise): both member mappings and the NumPy oracle then agree bit for
// bit given the same deviates (the compiler is otherwise free to contract differently in differently shaped code).
__device__ __forceinline__ double l96_entry(double xp, double xm2, double xm1, double xi, double F) {
  return __dadd_rn(__dsub_rn(__dmul_rn(__dsub_rn(xp, xm2), xm1), xi), F);
}
__device__ __forceinline__ float l96_entry(float xp, float xm2, float xm1, float xi, float F) {
  return __fadd_rn(__fsub_rn(__fmul_rn(__fsub_rn(xp, xm2), xm1), xi), F);
}
__device__ __forceinline__ double em_update(double x, double dt, double f, double noise) {
  return __dadd_rn(__dadd_rn(x, __dmul_rn(dt, f)), noise);
}
__device__ __forceinline__ float em_update(float x, float dt, float f, float noise) {
  return __fadd_rn(__fadd_rn(x, __fmul_rn(dt, f)), noise);
}

// ---- per-member drift on a thread-private state ---------------------------------------------------------------------
// NX > 0 fixes the drift at compile time (NX = 40: Lorenz-96, NX = 3: Lorenz-63) so that fully unrolled code stays small.
template <typename T, int NX>
__device__ __forceinline__ T member_f(int drift_id, const T* th, int n, int i, const T* x) {
  if (NX == 3) {
    if (i == 0) return th[0] * (x[1] - x[0]);
    if (i == 1) return x[0] * (th[1] - x[2]) - x[1];
    return x[0] * x[1] - th[2] * x[2];
  }
  if (NX > 3) {
    const int ip = i + 1 == n ? 0 : i + 1, im1 = i == 0 ? n - 1 : i - 1, im2 = im1 == 0 ? n - 1 : im1 - 1;
    return l96_entry(x[ip], x[im2], x[im1], x[i], th[0]);
  }
  return drift_f<T>(drift_id, th, n, i, [&](int j) { return x[j]; });
}

// NX > 0: compile-time state dimension (member state in registers, loops unrolled); NX == 0: runtime n <= CDK_MAX_N
// (thread-private arrays in local memory).
//
// LIGHT (Lorenz-96 n = 40, Euler-Maruyama, diagonal diffusion -- BASELINE config 5): 512 threads per CTA, <= 128 registers.
// The per-member state of the legacy mapping (x and x_e in registers: 160 of 255 registers, 8 warps per SM, every phase of
// the kernel latency-bound at two warps per scheduler) is replaced by the ensemble's own shared-memory columns: lanes l and
// l + 16 of a warp share member 16 warp + l and sweep dimensions [0, 20) and [20, 40) IN PLACE with a three-value rolling
// window of old entries in registers (the stencil reads x_{i-2}, x_{i-1}, x_{i+1}); the three old values a sweep needs from the
// partner's half are read before anyone writes (one __syncwarp).  Same counters, same operation order: bit-identical to the
// legacy mapping.  Sixteen warps then also share the cooperative phases (moments, gain products, update algebra).
template <typename T, int NX, bool LIGHT>
__global__ void __launch_bounds__(LIGHT ? 2 * ENKF_TPB : ENKF_TPB, 1) enkf_kernel(const EArgs<T> g) {
  constexpr int NXA = NX > 0 ? NX : CDK_MAX_N;
  constexpr int UF = NX > 0 ? NX : 1;             // unroll factor of loops over the state dimension
  constexpr int UFP = NX > 0 ? (NX + 3) / 4 : 1;  // ... over normal quads (four normals per Philox call)
  extern __shared__ __align__(16) unsigned char sh[];
  cg::cluster_group cluster = cg::this_cluster();
  const KArgs<T>& a = g.k;
  const cdk_desc& d = a.d;
  const int n = NX > 0 ? NX : d.n, m = d.m, K = d.K, E = d.E, C = g.C;
  const int rank = (int)cluster.block_rank();
  const long long traj = blockIdx.x / C;
  const ELay L(n, m, d.n_theta, g.Eloc, sizeof(T), g.dg, g.ue, emission_params(d));
  const bool ue = user_emission(d) && g.ue;
  const int ldn = L.ldn, ldm = L.ldm, ldE = L.ldE;
  const int e_base = rank * g.Eloc;
  const int nmem = max(0, min(g.Eloc, E - e_base));
  T* X = reinterpret_cast<T*>(sh + L.X);
  T* Cxx = reinterpret_cast<T*>(sh + L.CXX);
  T* mean = reinterpret_cast<T*>(sh + L.MEAN);
  T* H = reinterpret_cast<T*>(sh + L.H);
  T* R = reinterpret_cast<T*>(sh + L.R);
  T* chR = reinterpret_cast<T*>(sh + L.CHR);
  T* dv = reinterpret_cast<T*>(sh + L.DV);
  T* G = reinterpret_cast<T*>(sh + L.G);
  T* HP = reinterpret_cast<T*>(sh + L.HP);
  T* Sm = reinterpret_cast<T*>(sh + L.S);
  T* Sl = reinterpret_cast<T*>(sh + L.SL);
  T* Kt = reinterpret_cast<T*>(sh + L.KT);
  T* SK = reinterpret_cast<T*>(sh + L.SK);
  T* yv = reinterpret_cast<T*>(sh + L.YV);
  T* rv = reinterpret_cast<T*>(sh + L.RV);
  T* zv = rv + m;
  T* th = reinterpret_cast<T*>(sh + L.TH);
  T* phi = reinterpret_cast<T*>(sh + L.PHI);
  int* misc = reinterpret_cast<int*>(sh + L.MISC);
  T* llsh = reinterpret_cast<T*>(sh + L.MISC + 16);

  auto src = [&](int slot) { return a.in[slot] + traj * a.in_stride[slot]; };
  const uint32_t ctr_traj = (uint32_t)(((unsigned long long)traj + d.rng_offset) & 0xffffffffull);
  const uint64_t seed = d.rng_seed;

  // ---- model constants: G = L chol(Qc) (inference_enkf.py:74-80), chol(R) for the perturbed observations (:135) ----
  FOR_T(e, (int)(L.total / sizeof(T)) - (int)(L.CXX / sizeof(T))) reinterpret_cast<T*>(sh + L.CXX)[e] = T(0);
  __syncthreads();
  FOR_T(i, d.n_theta) th[i] = src(CDK_IN_F)[i];
  {
    T* Lm = SK;   // [n x ldn] scratch
    T* Qc = Cxx;  // scratch until the first moments(); receives the product L chol(Qc) after the factorisation
    T* Lq = G;    // chol(Qc)
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      Lm[i * ldn + j] = src(CDK_IN_L)[e];
      Qc[i * ldn + j] = src(CDK_IN_QC)[e];
    }
    if (ue) {
      FOR_T(i, emission_params(d)) phi[i] = src(CDK_IN_H)[i];
    } else {
      FOR_T(e, m * n) {
        const int i = e / n, j = e - i * n;
        H[i * ldn + j] = src(CDK_IN_H)[e];
      }
      FOR_T(i, m) dv[i] = src(CDK_IN_D)[i];
    }
    FOR_T(e, m * m) {
      const int i = e / m, j = e - i * m;
      R[i * ldm + j] = src(CDK_IN_R)[e];
    }
    __syncthreads();
    chol<T>(Qc, Lq, n, ldn, T(0));  // Lq = chol(Qc) in G
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      T s = T(0);
      for (int q = j; q < n; ++q) s += Lm[i * ldn + q] * Lq[q * ldn + j];
      Qc[i * ldn + j] = s;  // Qc no longer needed after the factorisation
    }
    __syncthreads();
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      G[i * ldn + j] = Qc[i * ldn + j];
    }
    chol<T>(R, chR, m, ldm, T(0));
    __syncthreads();
  }
  // diagonal diffusion? (then the noise is G_ii dW_i: no n x n product per member and substep)
  int offdiag = 0;
  FOR_T(e, n * n) {
    const int i = e / n, j = e - i * n;
    if (i != j && G[i * ldn + j] != T(0)) offdiag = 1;
  }
  const bool diagG = __syncthreads_or(offdiag) == 0;
  offdiag = 0;
  FOR_T(e, m * m) {
    const int i = e / m, j = e - i * m;
    if (i != j && chR[i * ldm + j] != T(0)) offdiag = 1;
  }
  const bool diagR = __syncthreads_or(offdiag) == 0;  // diagonal chol(R): the measurement noise is chR_pp z_p

  // ---- initial ensemble: m0 + chol(P0) z (inference_enkf.py:260-262) ----
  {
    T* P0 = Cxx;
    T* Lp = SK;
    FOR_T(e, n * n) {
      const int i = e / n, j = e - i * n;
      P0[i * ldn + j] = src(CDK_IN_P0)[e];
    }
    FOR_T(i, n) mean[i] = src(CDK_IN_M0)[i];
    __syncthreads();
    chol<T>(P0, Lp, n, ldn, T(0));
    for (int el = threadIdx.x; el < nmem; el += blockDim.x) {
      T z[NXA];
#pragma unroll UFP
      for (int j = 0; j < NXA; j += 4) {
        if (j < n) {
          double z4[4];
          normal_quad((uint32_t)(e_base + el), ctr_traj, 0u, rng_c3(RNG_INIT, 0, j >> 2), seed, z4);
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (j + u < NXA) z[j + u] = (T)z4[u];
        }
      }
#pragma unroll UF
      for (int i = 0; i < NXA; ++i) {
        if (i < n) {
          T s = T(0);
#pragma unroll UF
          for (int j = 0; j < NXA; ++j)
            if (j <= i) s += Lp[i * ldn + j] * z[j];
          X[(size_t)i * ldE + el] = mean[i] + s;
        }
      }
    }
    __syncthreads();
  }
  moments<T>(cluster, L, sh, nmem, E, C);

  const T* Y = a.in[CDK_IN_Y] ? src(CDK_IN_Y) : nullptr;
  const T* Tm = src(CDK_IN_T);
  T* FM = static_cast<T*>(a.out[CDK_OUT_FM]);
  T* FP = static_cast<T*>(a.out[CDK_OUT_FP]);
  T* PM = static_cast<T*>(a.out[CDK_OUT_PM]);
  T* PP = static_cast<T*>(a.out[CDK_OUT_PP]);
  T* LLC = static_cast<T*>(a.out[CDK_OUT_LLCUM]);
  const long long row0 = traj * (long long)K;
  const T dt0 = T(d.dt0);
  T ll = T(0);
  int status = 0;

  auto write_moments = [&](T* Mo, T* Co, long long row) {
    if (rank != 0) return;
    if (Mo) FOR_T(i, n) Mo[row * n + i] = mean[i];
    if (Co) FOR_T(e, n * n) {
        const int i = e / n, j = e - i * n;
        Co[row * n * n + e] = Cxx[i * ldn + j];
      }
  };

  // forecast (CDK_FLAG_PREDICT_ONLY, forecast_ensemble_kalman_filter): no updates; Tm holds K + 1 stamps, t_init first
  const bool ponly = (d.reserved[2] & CDK_FLAG_PREDICT_ONLY) != 0;
  for (int k = 0; k < K; ++k) {
    if (!ponly) {
    // ================= update (inference_enkf.py:92-148), every CTA of the cluster redundantly =================
    FOR_T(i, m) yv[i] = Y[(long long)k * m + i];
    if (ue) {
      user_emission_moments<T>(cluster, L, sh, nmem, E, C, phi, yv);  // HP = C_xy^T, S = C_yy + R, rv = y - ybar
    } else {
    // HP = H Cxx (= C_xy^T because h is linear), S = H Cxx H^T + R: FP64 tensor cores
    mm_dmma<T, false, false>(H, ldn, Cxx, ldn, m, n, n, [&](int p, int j, double v) { HP[p * ldn + j] = (T)v; });
    __syncthreads();
    mm_dmma<T, false, true>(HP, ldn, H, ldn, m, m, n, [&](int p, int q2, double v) { Sm[p * ldm + q2] = (T)v + R[p * ldm + q2]; });
    FOR_T(p, m) {  // innovation of the ensemble mean
      T s = dv[p];
      for (int q = 0; q < n; ++q) s += H[p * ldn + q] * mean[q];
      rv[p] = yv[p] - s;
    }
    }
    __syncthreads();
    // MVN(ybar, S).log_prob(y) factors S un-boosted (:129); K^T = psd_solve(S, C_xy^T) factors sym(S) + 1e-9 I (:141-143):
    // one warp each, side by side (chol_warp); the un-boosted factor is parked in SK
    chol_prep<T, false>(Sm, SK, m, ldm, T(0));
    chol_prep<T, true>(Sm, Sl, m, ldm, T(1e-9));
    __syncthreads();
    chol_warp<T>(0, SK, m, ldm);
    chol_warp<T>(blockDim.x > 32 ? 1 : 0, Sl, m, ldm);
    __syncthreads();
    mvn_ll_warp<T>(SK, ldm, rv, m, llsh);          // warp 0; the others start on the solve
    chol_solve<T>(Sl, m, ldm, HP, Kt, n, ldn);     // ends with a barrier
    ll += *llsh;
    // per member: x += K ((y + chol(R) z) - (H x + d))   (:135-146)
    if (g.dg) {
      // Over the CTA's members at once: D = (y - d) 1^T + chol(R) Z - H X  [m x nmem],  X += K D, the two products on the FP64
      // tensor cores (per member this is 2 m n FMAs with one shared-memory operand load each: 11 % of the instruction stream).
      T* Db = reinterpret_cast<T*>(sh + L.DB);
      const bool pair_fill = (int)blockDim.x >= 2 * g.Eloc && diagR && d.perturb_measurements;
      if (pair_fill) {
        // twice as many threads as members (LIGHT): lanes l and l + 16 share a member and take alternate quads of the
        // observation noise, so all sixteen warps generate deviates instead of eight waiting at the barrier below
        const int lane = threadIdx.x & 31, half = lane >> 4;
        const int el = (threadIdx.x >> 5) * 16 + (lane & 15);
        if (el < nmem) {
          for (int p = 4 * half; p < m; p += 8) {
            double z4[4];
            normal_quad((uint32_t)(e_base + el), ctr_traj, (uint32_t)k, rng_c3(RNG_OBS, 0, p >> 2), seed, z4);
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (p + u < m) Db[(size_t)(p + u) * ldE + el] = (yv[p + u] + chR[(p + u) * ldm + p + u] * (T)z4[u]) - dv[p + u];
          }
        }
      } else
      for (int el = threadIdx.x; el < nmem; el += blockDim.x) {
        if (d.perturb_measurements) {
          T r[CDK_MAX_M];
          for (int p = 0; p < m; p += 4) {
            double z4[4];
            normal_quad((uint32_t)(e_base + el), ctr_traj, (uint32_t)k, rng_c3(RNG_OBS, 0, p >> 2), seed, z4);
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (p + u < m) r[p + u] = (T)z4[u];
          }
          if (diagR) {
            for (int p = 0; p < m; ++p) Db[(size_t)p * ldE + el] = (yv[p] + chR[p * ldm + p] * r[p]) - dv[p];
          } else {
            for (int p = m - 1; p >= 0; --p) {  // chol(R) z from the bottom row up
              T s = T(0);
              for (int q = 0; q <= p; ++q) s += chR[p * ldm + q] * r[q];
              Db[(size_t)p * ldE + el] = (yv[p] + s) - dv[p];
            }
          }
        } else {
          for (int p = 0; p < m; ++p) Db[(size_t)p * ldE + el] = yv[p] - dv[p];
        }
      }
      __syncthreads();
      mm_dmma_strip<T, false>(H, ldn, X, ldE, m, nmem, n, [&](int p, int e, double v) { Db[(size_t)p * ldE + e] -= (T)v; });
      __syncthreads();
      mm_dmma_strip<T, true>(Kt, ldn, Db, ldE, n, nmem, m, [&](int i, int e, double v) { X[(size_t)i * ldE + e] += (T)v; });
    } else
    for (int el = threadIdx.x; el < nmem; el += blockDim.x) {
      T x[NXA];
#pragma unroll UF
      for (int i = 0; i < NXA; ++i)
        if (i < n) x[i] = X[(size_t)i * ldE + el];
      T r[CDK_MAX_M];
      if (d.perturb_measurements) {
        for (int p = 0; p < m; p += 4) {
          double z4[4];
          normal_quad((uint32_t)(e_base + el), ctr_traj, (uint32_t)k, rng_c3(RNG_OBS, 0, p >> 2), seed, z4);
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (p + u < m) r[p + u] = (T)z4[u];
        }
        for (int p = m - 1; p >= 0; --p) {  // r <- chol(R) z, in place from the bottom row up
          T s = T(0);
          for (int q = 0; q <= p; ++q) s += chR[p * ldm + q] * r[q];
          r[p] = s;
        }
      } else {
        for (int p = 0; p < m; ++p) r[p] = T(0);
      }
      const T* Ye = reinterpret_cast<const T*>(sh + L.DB) + el;  // user emission: h(x_e), column el
      for (int p = 0; p < m; ++p) {
        T hx;
        if (ue) {
          hx = Ye[(size_t)p * ldE];
        } else {
          hx = dv[p];
#pragma unroll UF
          for (int i = 0; i < NXA; ++i)
            if (i < n) hx += H[p * ldn + i] * x[i];
        }
        r[p] = (yv[p] + r[p]) - hx;
      }
      for (int p = 0; p < m; ++p) {
        const T rp = r[p];
#pragma unroll UF
        for (int i = 0; i < NXA; ++i)
          if (i < n) x[i] += Kt[p * ldn + i] * rp;
      }
#pragma unroll UF
      for (int i = 0; i < NXA; ++i)
        if (i < n) X[(size_t)i * ldE + el] = x[i];
    }
    __syncthreads();
    if (FM || FP) {  // filtered moments (:225-228): an output only -- the next update reads the PREDICTED moments
      moments<T>(cluster, L, sh, nmem, E, C);
      write_moments(FM, FP, row0 + k);
    }
    if (LLC && rank == 0 && threadIdx.x == 0) LLC[row0 + k] = ll;
    }

    // ================= predict (inference_enkf.py:47-89): per-member SDE solve over the gap =================
    const T t0 = Tm[k];
    const T t1 = (ponly || k + 1 < K) ? Tm[k + 1] : t0 + T(d.dt_final);
    StepClock<T> clk(t0, t1, dt0);
    while (clk.running()) {
      if (clk.n >= d.max_steps) {  // diffrax max_steps exceeded: poison the ensemble, abandon the gap
        status = 2;
        for (int el = threadIdx.x; el < nmem; el += blockDim.x)
          for (int i = 0; i < n; ++i) X[(size_t)i * ldE + el] = T(NAN);
        break;
      }
      const T dt = clk.dt();
      const T sqdt = sqrt(dt);
      bool light_done = false;
      if constexpr (LIGHT && NX == 40) {
        if (diagG && d.solver == CDK_EULER) {
          light_done = true;
          constexpr int HN = NX / 2;
          const int lane = threadIdx.x & 31, half = lane >> 4;
          const int el = (threadIdx.x >> 5) * 16 + (lane & 15);
          const bool act = el < nmem;
          const int i0 = half * HN;
          T* xc = X + el;
          const T th0 = th[0];
          T xm2 = T(0), xm1 = T(0), cur = T(0), halo = T(0);
          if (act) {
            xm2 = xc[(size_t)(i0 == 0 ? NX - 2 : i0 - 2) * ldE];
            xm1 = xc[(size_t)(i0 == 0 ? NX - 1 : i0 - 1) * ldE];
            halo = xc[(size_t)(i0 + HN == NX ? 0 : i0 + HN) * ldE];
            cur = xc[(size_t)i0 * ldE];
          }
          __syncwarp();  // both halves hold their old halo values before either writes
          if (act) {
#pragma unroll
            for (int q0 = 0; q0 < HN; q0 += 8) {
              double z8[8];
              if (q0 + 4 < HN) {
                normal_oct((uint32_t)(e_base + el), ctr_traj, (uint32_t)k, rng_c3(RNG_DYN, clk.n, (i0 + q0) >> 2),
                           rng_c3(RNG_DYN, clk.n, ((i0 + q0) >> 2) + 1), seed, z8);
              } else {
                double z4[4];
                normal_quad((uint32_t)(e_base + el), ctr_traj, (uint32_t)k, rng_c3(RNG_DYN, clk.n, (i0 + q0) >> 2), seed, z4);
#pragma unroll
                for (int u = 0; u < 4; ++u) z8[u] = z4[u];
              }
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                if (q0 + u < HN) {
                  const int i = i0 + q0 + u;
                  const T nxt = (q0 + u + 1 < HN) ? xc[(size_t)(i + 1) * ldE] : halo;
                  const T noise = G[i * ldn + i] * (sqdt * (T)z8[u]);
                  xc[(size_t)i * ldE] = em_update(cur, dt, l96_entry(nxt, xm2, xm1, cur, th0), noise);
                  xm2 = xm1;
                  xm1 = cur;
                  cur = nxt;
                }
              }
            }
          }
          __syncwarp();  // the partner's new entries are this half's halo of the next substep
        }
      }
      if (!light_done)
      for (int el = threadIdx.x; el < nmem; el += blockDim.x) {
        T x[NXA], xe[NXA];  // xe first holds the noise G dW, then the Euler-Maruyama state
#pragma unroll UF
        for (int i = 0; i < NXA; ++i)
          if (i < n) x[i] = X[(size_t)i * ldE + el];
        if (diagG) {
#pragma unroll UFP
          for (int j = 0; j < NXA; j += 8) {
            if (j + 4 < n) {  // two quads at once (normal_oct: same values, interleaved chains)
              double z8[8];
              normal_oct((uint32_t)(e_base + el), ctr_traj, (uint32_t)k, rng_c3(RNG_DYN, clk.n, j >> 2),
                         rng_c3(RNG_DYN, clk.n, (j >> 2) + 1), seed, z8);
#pragma unroll
              for (int u = 0; u < 8; ++u)
                if (j + u < NXA && j + u < n) xe[j + u] = G[(j + u) * ldn + j + u] * (sqdt * (T)z8[u]);
            } else if (j < n) {
              double z4[4];
              normal_quad((uint32_t)(e_base + el), ctr_traj, (uint32_t)k, rng_c3(RNG_DYN, clk.n, j >> 2), seed, z4);
#pragma unroll
              for (int u = 0; u < 4; ++u)
                if (j + u < NXA && j + u < n) xe[j + u] = G[(j + u) * ldn + j + u] * (sqdt * (T)z4[u]);
            }
          }
        } else {
#pragma unroll UF
          for (int i = 0; i < NXA; ++i) xe[i] = T(0);
          for (int j = 0; j < n; j += 4) {  // quads stay a runtime loop: the rank-4 update below is the unrolled part
            double z4[4];
            normal_quad((uint32_t)(e_base + el), ctr_traj, (uint32_t)k, rng_c3(RNG_DYN, clk.n, j >> 2), seed, z4);
            for (int u = 0; u < 4 && j + u < n; ++u) {
              const T dw = sqdt * (T)z4[u];
#pragma unroll UF
              for (int i = 0; i < NXA; ++i)
                if (i < n) xe[i] += G[i * ldn + j + u] * dw;
            }
          }
        }
#pragma unroll UF
        for (int i = 0; i < NXA; ++i)
          if (i < n) xe[i] = em_update(x[i], dt, member_f<T, NX>(d.drift_id, th, n, i, x), xe[i]);
        if (d.solver == CDK_HEUN) {
          // x + dt/2 (f(x) + f(xe)) + noise, written as xe + dt/2 (f(xe) - f(x)) so the noise is not kept (oracle: same form)
          const T hdt = T(0.5) * dt;
#pragma unroll UF
          for (int i = 0; i < NXA; ++i)
            if (i < n)
              X[(size_t)i * ldE + el] =
                  xe[i] + hdt * (member_f<T, NX>(d.drift_id, th, n, i, xe) - member_f<T, NX>(d.drift_id, th, n, i, x));
        } else {
#pragma unroll UF
          for (int i = 0; i < NXA; ++i)
            if (i < n) X[(size_t)i * ldE + el] = xe[i];
        }
      }
      clk.advance();
    }
    __syncthreads();
    moments<T>(cluster, L, sh, nmem, E, C);  // predicted moments (:234-238); they also feed the next update
    write_moments(PM, PP, row0 + k);
  }
  if (rank == 0 && threadIdx.x == 0) {
    if (a.out[CDK_OUT_LL]) static_cast<T*>(a.out[CDK_OUT_LL])[traj] = ll;
    if (a.out[CDK_OUT_STATUS]) static_cast<int*>(a.out[CDK_OUT_STATUS])[traj] = final_status(status, isfinite(ll));
  }
  (void)misc;
}

template <typename T, int NX, bool LIGHT = false>
int launch_nx(const EArgs<T>& g, size_t smem, cudaStream_t s) {
  auto kern = enkf_kernel<T, NX, LIGHT>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("cudaFuncSetAttribute(enkf_kernel)");
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(g.k.d.N * g.C), 1, 1);
  cfg.blockDim = dim3(LIGHT ? 2 * ENKF_TPB : ENKF_TPB, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)g.C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, g);
  note_launch();
  (void)e;  // a failed launch is also recorded as the last error
  return check_launch("enkf_kernel");
}

}  // namespace

template <typename T>
int launch_enkf(const KArgs<T>& a, cudaStream_t s) {
  const cdk_desc& d = a.d;
  if (d.N * 8 > 2147483647LL) return CDK_E_SIZE;
  int dev = 0, max_optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  int forced = 0;
  if (const char* e = getenv("CDK_ENKF_CLUSTER")) forced = atoi(e);
  static const int dmma_gain_env = []() {
    const char* e = getenv("CDK_ENKF_DMMA_GAIN");
    return e && e[0] == '0' ? 0 : 1;
  }();
  EArgs<T> g;
  g.k = a;
  g.C = 0;
  g.dg = 0;
  g.ue = user_emission(d) ? 1 : 0;
  size_t smem = 0;
  for (int C = 1; C <= 8; C *= 2) {
    if (forced && C != forced) continue;
    const int Eloc = (((d.E + C - 1) / C) + 3) & ~3;
    if (!(forced || Eloc <= 2 * ENKF_TPB || C == 8)) continue;
    for (int dg = g.ue ? 0 : dmma_gain_env; dg >= 0 && g.C == 0; --dg) {  // prefer the tensor-core gain application if its block fits
      const ELay L(d.n, d.m, d.n_theta, Eloc, sizeof(T), dg, g.ue, emission_params(d));
      if (L.total <= (size_t)max_optin) {
        g.C = C;
        g.Eloc = Eloc;
        g.dg = dg;
        smem = L.total;
      }
    }
    if (g.C) break;
  }
  if (g.C == 0) return CDK_E_SIZE;  // ensemble too large for 8 CTAs x 227 KB
  if (d.n == 40 && d.drift_id == CDK_DRIFT_LORENZ96) {
    // two threads per member, state swept in shared memory (see the kernel); CDK_ENKF_LIGHT=0: the register mapping
    const char* le = getenv("CDK_ENKF_LIGHT");
    const bool light = !(le && le[0] == '0') && d.solver == CDK_EULER && g.dg && g.Eloc <= ENKF_TPB;
    return light ? launch_nx<T, 40, true>(g, smem, s) : launch_nx<T, 40>(g, smem, s);
  }
  if (d.n == 3 && d.drift_id == CDK_DRIFT_LORENZ63) return launch_nx<T, 3>(g, smem, s);
  return launch_nx<T, 0>(g, smem, s);
}

template int launch_enkf<double>(const KArgs<double>&, cudaStream_t);
template int launch_enkf<float>(const KArgs<float>&, cudaStream_t);

}  // namespace cdk
