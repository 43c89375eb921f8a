// cdk_common.cuh -- shared device/host helpers for the cdk kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "cdk.h"

namespace cdk {

// Kernel argument block, passed by value (lives in the constant bank).
template <typename T>
struct KArgs {
  cdk_desc d;
  const T* in[CDK_NUM_IN];
  void* out[CDK_NUM_OUT];
  long long in_stride[CDK_NUM_IN];  // elements per trajectory when the slot is batched, else 0
};

template <typename T>
__host__ __device__ inline T clip_tol() {
  // diffrax `_clip_to_end`: 1e-10 for float64 times, 1e-6 for float32 (restated; SURVEY App. C)
  return sizeof(T) == 8 ? T(1e-10) : T(1e-6);
}

// The substeps of one gap [t0, t1] under diffrax ConstantStepSize, in the element type T of the times (fp32 kernels step
// fp32 times with tol = 1e-6).  Every kernel steps its gaps with this rule:
//
//   StepClock<T> c(t0, t1, dt0);
//   while (c.running() && c.n < max_steps) { step(c.dt()); c.advance(); }
//   if (c.running()) ... max_steps exceeded (status 2) ...
//
// The first substep ends at min(t0 + dt0, t1); every later one at cand = tprev + dt0, or at t1 if cand > t1 - tol.  A gap
// that is already complete keeps tprev == tnext == t1 (a substep of length 0).  The members are the loop's registers.
template <typename T>
struct StepClock {
  T tprev, tnext, t1, dt0;
  int n;         // substeps taken
  bool clipped;  // the current substep ends at t1: the first if t0 + dt0 >= t1, a later one if tprev + dt0 > t1 - tol

  __host__ __device__ __forceinline__ StepClock(T t0, T t1_, T dt0_)
      : tprev(t0), tnext(fmin(t0 + dt0_, t1_)), t1(t1_), dt0(dt0_), n(0), clipped(!(t0 + dt0_ < t1_)) {}
  __host__ __device__ __forceinline__ bool running() const { return tprev < t1; }
  __host__ __device__ __forceinline__ T dt() const { return tnext - tprev; }
  // the current substep has the nominal length dt0 (up to the rounding of tprev + dt0)
  __host__ __device__ __forceinline__ bool full() const { return !clipped; }
  __host__ __device__ __forceinline__ void advance() {
    ++n;
    tprev = tnext;
    const T cand = tprev + dt0;
    clipped = cand > t1 - clip_tol<T>();
    tnext = clipped ? t1 : cand;
  }
};

// Per-trajectory status (CDK_OUT_STATUS): 0 ok, 1 non-finite result, 2 max_steps exceeded.  A max_steps failure outranks
// the NaN it causes.
//
// A filter's or sampler's final status, from the status of its steps and whether its result is finite.
__host__ __device__ __forceinline__ int final_status(int status, bool finite) {
  return status != 0 ? status : finite ? 0 : 1;
}
// A smoother's status, merged into st[i], which its filter wrote: non-finite smoothed moments after a filter that failed
// are that failure, not a new one, so the filter's status stays unless the filter was clean or the backward pass itself
// exceeded max_steps.
__host__ __device__ __forceinline__ void merge_smoother_status(int* st, long long i, int status, bool finite) {
  if (status == 0 && !finite && st[i] == 0) status = 1;
  if (status != 0) st[i] = status;
}

template <typename T>
__device__ __forceinline__ T half_log_2pi() {
  return T(0.91893853320467274178);
}

// ---- explicit Runge-Kutta tableaux (compile-time) ------------------------------------------------------------------
template <int SOLVER>
struct Tab;
// a(i,j) / b(i) are constexpr FUNCTIONS (not arrays) so that fully unrolled device code folds them to immediates.
template <>
struct Tab<CDK_EULER> {
  static constexpr int S = 1;
  __host__ __device__ static constexpr double a(int i, int j) {
    return 0.0;
  }
  __host__ __device__ static constexpr double b(int i) {
    return i == 0 ? 1.0 : 0.0;
  }
};
template <>
struct Tab<CDK_HEUN> {
  static constexpr int S = 2;
  __host__ __device__ static constexpr double a(int i, int j) {
    return (i == 1 && j == 0) ? 1.0 : 0.0;
  }
  __host__ __device__ static constexpr double b(int i) {
    return i == 0 ? 0.5 : i == 1 ? 0.5 : 0.0;
  }
};
template <>
struct Tab<CDK_MIDPOINT> {
  static constexpr int S = 2;
  __host__ __device__ static constexpr double a(int i, int j) {
    return (i == 1 && j == 0) ? 0.5 : 0.0;
  }
  __host__ __device__ static constexpr double b(int i) {
    return i == 0 ? 0.0 : i == 1 ? 1.0 : 0.0;
  }
};
template <>
struct Tab<CDK_RALSTON> {
  static constexpr int S = 2;
  __host__ __device__ static constexpr double a(int i, int j) {
    return (i == 1 && j == 0) ? 0.75 : 0.0;
  }
  __host__ __device__ static constexpr double b(int i) {
    return i == 0 ? 1.0 / 3.0 : i == 1 ? 2.0 / 3.0 : 0.0;
  }
};
template <>
struct Tab<CDK_BOSH3> {
  static constexpr int S = 3;
  __host__ __device__ static constexpr double a(int i, int j) {
    return (i == 1 && j == 0) ? 0.5 : 
           (i == 2 && j == 1) ? 0.75 : 0.0;
  }
  __host__ __device__ static constexpr double b(int i) {
    return i == 0 ? 2.0 / 9.0 : i == 1 ? 1.0 / 3.0 : i == 2 ? 4.0 / 9.0 : 0.0;
  }
};
template <>
struct Tab<CDK_RK4> {
  static constexpr int S = 4;
  __host__ __device__ static constexpr double a(int i, int j) {
    return (i == 1 && j == 0) ? 0.5 : 
           (i == 2 && j == 1) ? 0.5 : 
           (i == 3 && j == 2) ? 1.0 : 0.0;
  }
  __host__ __device__ static constexpr double b(int i) {
    return i == 0 ? 1.0 / 6.0 : i == 1 ? 1.0 / 3.0 : i == 2 ? 1.0 / 3.0 : i == 3 ? 1.0 / 6.0 : 0.0;
  }
};
template <>
struct Tab<CDK_DOPRI5> {
  static constexpr int S = 6;
  __host__ __device__ static constexpr double a(int i, int j) {
    return (i == 1 && j == 0) ? 1.0 / 5.0 : 
           (i == 2 && j == 0) ? 3.0 / 40.0 : 
           (i == 2 && j == 1) ? 9.0 / 40.0 : 
           (i == 3 && j == 0) ? 44.0 / 45.0 : 
           (i == 3 && j == 1) ? -56.0 / 15.0 : 
           (i == 3 && j == 2) ? 32.0 / 9.0 : 
           (i == 4 && j == 0) ? 19372.0 / 6561.0 : 
           (i == 4 && j == 1) ? -25360.0 / 2187.0 : 
           (i == 4 && j == 2) ? 64448.0 / 6561.0 : 
           (i == 4 && j == 3) ? -212.0 / 729.0 : 
           (i == 5 && j == 0) ? 9017.0 / 3168.0 : 
           (i == 5 && j == 1) ? -355.0 / 33.0 : 
           (i == 5 && j == 2) ? 46732.0 / 5247.0 : 
           (i == 5 && j == 3) ? 49.0 / 176.0 : 
           (i == 5 && j == 4) ? -5103.0 / 18656.0 : 0.0;
  }
  __host__ __device__ static constexpr double b(int i) {
    return i == 0 ? 35.0 / 384.0 : i == 1 ? 0.0 : i == 2 ? 500.0 / 1113.0 : i == 3 ? 125.0 / 192.0 : i == 4 ? -2187.0 / 6784.0 : i == 5 ? 11.0 / 84.0 : 0.0;
  }
};

// Runtime tableau (for the shared-memory kernels): up to 6 stages, stored SPARSE per stage (nnz / column / value) so the
// stage assembly is a short uniform loop instead of a scan over a dense row with floating-point compares.
struct RtTab {
  int S;
  int nnz[6];
  int col[6][5];
  double val[6][5];
  double b[6];
};

inline bool fill_rt_tab(int solver, RtTab& t) {
  auto copy = [&](auto tab) {
    using TT = decltype(tab);
    t.S = TT::S;
    for (int i = 0; i < 6; ++i) {
      t.nnz[i] = 0;
      for (int j = 0; j < 5; ++j) {
        t.col[i][j] = 0;
        t.val[i][j] = 0.0;
      }
      for (int j = 0; j < i && i < TT::S; ++j)
        if (TT::a(i, j) != 0.0) {
          t.col[i][t.nnz[i]] = j;
          t.val[i][t.nnz[i]] = TT::a(i, j);
          ++t.nnz[i];
        }
      t.b[i] = i < TT::S ? TT::b(i) : 0.0;
    }
  };
  switch (solver) {
    case CDK_EULER: copy(Tab<CDK_EULER>{}); return true;
    case CDK_HEUN: copy(Tab<CDK_HEUN>{}); return true;
    case CDK_MIDPOINT: copy(Tab<CDK_MIDPOINT>{}); return true;
    case CDK_RALSTON: copy(Tab<CDK_RALSTON>{}); return true;
    case CDK_BOSH3: copy(Tab<CDK_BOSH3>{}); return true;
    case CDK_RK4: copy(Tab<CDK_RK4>{}); return true;
    case CDK_DOPRI5: copy(Tab<CDK_DOPRI5>{}); return true;
  }
  return false;
}

bool has_user_drift();  // cdk_generic.cu: was this library compiled with CDK_USER_DRIFT_HEADER?
// cdk_ekfgrad.cu: was its dense gradient compiled with CDK_USER_DRIFT_HEADER (build_user_drift(code, grad=True))?
bool ekf_grad_has_user_drift();
// cdk_ekfgrad.cu: ... with CDK_USER_EMISSION_HEADER (build_variant(..., emission_grad=True))?
bool ekf_grad_has_user_emission();
bool has_user_emission();             // cdk_generic.cu: ... with CDK_USER_EMISSION_HEADER?
int user_emission_params(int n, int m);  // cdk_generic.cu: its num_params(n, m), or -1 without a user emission

// host-side launch bookkeeping (cdk_api.cu)
void note_launch();
int check_launch(const char* what);

// entry points implemented per translation unit; return CDK_E_UNSUPPORTED when the fast path does not cover `d`
template <typename T>
int launch_ekf_small(const KArgs<T>& a, cudaStream_t s);
template <typename T>
int launch_eks_small(const KArgs<T>& a, cudaStream_t s);
int launch_ekf_l63_grad(const KArgs<double>& a, double* grad, cudaStream_t s);
int launch_kf_grad(const KArgs<double>& a, double* grad, cudaStream_t s);  // cdk_kfwarp.cu
long long kf_grad_scratch_doubles(const cdk_desc& d);                      // its out[CDK_OUT_SCRATCH], in doubles
bool kf_warp_eligible(const cdk_desc& d, bool smooth);  // fp64 requests served by kf_warp_filter / kf_warp_smooth
// cdk_ekfgrad.cu: the backward launch of cdk_ekf_grad_dense_f64 (ukf: of cdk_ukf_grad_dense_f64; sigma: of
// cdk_ukf_grad_sigma_f64), its scratch (doubles) and its shared-memory budget
int launch_ekf_grad_dense(const KArgs<double>& a, const int* status, double* grad, bool ukf, bool sigma, cudaStream_t s);
long long ekf_grad_dense_scratch_doubles(const cdk_desc& d);
bool ekf_grad_dense_fits(const cdk_desc& d, bool sigma);
int set_lw_trace(void* devbuf);
template <typename T>
int launch_generic(int algo, const KArgs<T>& a, cudaStream_t s);
template <typename T>
int launch_enkf(const KArgs<T>& a, cudaStream_t s);
template <typename T>
int launch_kf_warp(int algo, const KArgs<T>& a, cudaStream_t s);

template <typename T>
int launch_sample_path(const KArgs<T>& a, cudaStream_t s);
template <typename T>
int launch_emission_moments(const KArgs<T>& a, cudaStream_t s);

enum { ALGO_KF_FILTER = 0, ALGO_KF_SMOOTH, ALGO_EKF_FILTER, ALGO_EKF_SMOOTH, ALGO_UKF_FILTER, ALGO_ENKF_FILTER, ALGO_SAMPLE,
       ALGO_EMISSIONS };

}  // namespace cdk
