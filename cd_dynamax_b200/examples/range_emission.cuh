// Example user-defined emission (cd_dynamax_b200.LearnableUserEmission / build.build_variant): the range from the state
// to each of m beacons, h_a(x) = sqrt(sum_j (x_j - b_aj)^2 + eps), for any n and m.  phi = the beacon coordinates b
// ([m * n], row a = beacon a) followed by eps (> 0 keeps h smooth when the state sits on a beacon).  Used by
// tests/test_gpu_user_emission.py; __graft_entry__.build() pre-builds its variant libraries.
namespace cdk_user_emission {
__host__ __device__ inline int num_params(int n, int m) { return m * n + 1; }
template <typename T, class XF> __device__ __forceinline__ T h(const T* phi, int n, int m, int a, XF x) {
  T s = phi[m * n];
  for (int j = 0; j < n; ++j) {
    const T r = x(j) - phi[a * n + j];
    s += r * r;
  }
  return sqrt(s);
}
template <typename T> __device__ __forceinline__ T jac(const T* phi, int n, int m, int a, int j, const T* x) {
  return (x[j] - phi[a * n + j]) / h<T>(phi, n, m, a, [&](int q) { return x[q]; });
}
}
