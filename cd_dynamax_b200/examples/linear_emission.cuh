// Example user-defined emission: the linear emission h(x) = H x + d written as user code, phi = H ([m * n], row-major)
// followed by d ([m]).  It computes what LearnableLinear computes through the user-emission update paths, which is how
// tests/test_gpu_user_emission.py pins those paths against the stock ones.
namespace cdk_user_emission {
__host__ __device__ inline int num_params(int n, int m) { return m * n + m; }
template <typename T, class XF> __device__ __forceinline__ T h(const T* phi, int n, int m, int a, XF x) {
  T s = phi[m * n + a];
  for (int j = 0; j < n; ++j) s += phi[a * n + j] * x(j);
  return s;
}
template <typename T> __device__ __forceinline__ T jac(const T* phi, int n, int m, int a, int j, const T* x) {
  return phi[a * n + j];
}
}
