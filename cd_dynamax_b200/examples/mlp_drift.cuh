// Example differentiable user-defined drift (LearnableUserDrift(..., differentiable=True) / build_user_drift(code,
// grad=True)): the neural drift of the reference's tutorials, a one-hidden-layer tanh network on n = 2 states,
//   f(x) = W2 tanh(W1 x + b1) + b2,   theta = W1 (16 x 2, row-major) | b1 (16) | W2 (2 x 16, row-major) | b2 (2),
// n_theta = 82.  It stays within the dual-number contract of csrc/cdk_dual.cuh (T arithmetic and unqualified tanh), so
// the gradient takes its parameter and second derivatives from these same functions.  Used by
// tests/test_gpu_user_drift_grad.py and scripts/user_drift_grad_bench.py.
namespace cdk_user {
constexpr int MLP_H = 16;
// t_h = tanh(W1 x + b1)_h
template <typename T> __device__ __forceinline__ T mlp_hidden(const T* th, int h, const T& x0, const T& x1) {
  return tanh(th[2 * h] * x0 + th[2 * h + 1] * x1 + th[2 * MLP_H + h]);
}
template <typename T, class XF> __device__ __forceinline__ T f(const T* th, int n, int i, XF x) {
  const T x0 = x(0), x1 = x(1);
  const T* W2 = th + 3 * MLP_H;
  T s = th[5 * MLP_H + i];
  for (int h = 0; h < MLP_H; ++h) s += W2[i * MLP_H + h] * mlp_hidden(th, h, x0, x1);
  return s;
}
// J_ij = sum_h W2_ih (1 - t_h^2) W1_hj
template <typename T> __device__ __forceinline__ T jac(const T* th, int n, int i, int j, const T* x) {
  const T* W2 = th + 3 * MLP_H;
  T s = T(0);
  for (int h = 0; h < MLP_H; ++h) {
    const T t = mlp_hidden(th, h, x[0], x[1]);
    s += W2[i * MLP_H + h] * (T(1) - t * t) * th[2 * h + j];
  }
  return s;
}
// g_k = sum_i d2 f_i / dx_i dx_k = sum_h (sum_i W2_ih W1_hi) (-2 t_h (1 - t_h^2)) W1_hk
template <typename T> __device__ __forceinline__ T graddiv(const T* th, int n, int k, const T* x) {
  const T* W2 = th + 3 * MLP_H;
  T s = T(0);
  for (int h = 0; h < MLP_H; ++h) {
    const T t = mlp_hidden(th, h, x[0], x[1]);
    const T c = W2[h] * th[2 * h] + W2[MLP_H + h] * th[2 * h + 1];
    s += c * (T(-2) * t * (T(1) - t * t)) * th[2 * h + k];
  }
  return s;
}
}
