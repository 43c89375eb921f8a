// cdk_dual.cuh -- vector-mode forward-mode dual numbers for device (and host) code: one fp64 value and W fp64 tangents.
//
// The reverse-mode CD-EKF gradient of a user-defined drift (cdk_ekfgrad.cu, CDK_DRIFT_USER) instantiates the user's
// templates f / jac / graddiv with T = cdk_dual::Dual<W> and seeds W directions (state components, then parameters) at
// a time, so that every partial derivative the stage VJP needs comes from the user's own code.  The operations below ARE
// the contract a differentiable user drift must stay within:
//   + - * / and unary -, with a Dual on either side and mixed with int / double constants; += -= *= /=;
//   comparisons (value only, so branches work); construction T(c) from a constant;
//   the unqualified functions sqrt exp log sin cos tan tanh sinh cosh atan fabs pow(T, double).
// They are declared in namespace cdk_dual, so argument-dependent lookup finds them from `namespace cdk_user`.  Qualified
// calls (::sin, std::exp) and intrinsics (__expf) bypass the overloads and do not compile with T = Dual.
#pragma once

namespace cdk_dual {

template <int W>
struct Dual {
  double v;
  double d[W];
  __host__ __device__ __forceinline__ Dual() : v(0.0) {
#pragma unroll
    for (int w = 0; w < W; ++w) d[w] = 0.0;
  }
  __host__ __device__ __forceinline__ Dual(double c) : v(c) {
#pragma unroll
    for (int w = 0; w < W; ++w) d[w] = 0.0;
  }
  __host__ __device__ __forceinline__ Dual& operator+=(const Dual& b) {
    v += b.v;
#pragma unroll
    for (int w = 0; w < W; ++w) d[w] += b.d[w];
    return *this;
  }
  __host__ __device__ __forceinline__ Dual& operator-=(const Dual& b) {
    v -= b.v;
#pragma unroll
    for (int w = 0; w < W; ++w) d[w] -= b.d[w];
    return *this;
  }
  __host__ __device__ __forceinline__ Dual& operator*=(const Dual& b) {
#pragma unroll
    for (int w = 0; w < W; ++w) d[w] = d[w] * b.v + v * b.d[w];
    v *= b.v;
    return *this;
  }
  __host__ __device__ __forceinline__ Dual& operator/=(const Dual& b) {
    const double q = v / b.v;
#pragma unroll
    for (int w = 0; w < W; ++w) d[w] = (d[w] - q * b.d[w]) / b.v;
    v = q;
    return *this;
  }
  __host__ __device__ __forceinline__ Dual& operator+=(double b) { v += b; return *this; }
  __host__ __device__ __forceinline__ Dual& operator-=(double b) { v -= b; return *this; }
  __host__ __device__ __forceinline__ Dual& operator*=(double b) {
    v *= b;
#pragma unroll
    for (int w = 0; w < W; ++w) d[w] *= b;
    return *this;
  }
  __host__ __device__ __forceinline__ Dual& operator/=(double b) {
    v /= b;
#pragma unroll
    for (int w = 0; w < W; ++w) d[w] /= b;
    return *this;
  }
};

// The value of every operation is the double operation on the values, bit for bit, so that a dual evaluation of the
// user's code has the value of its double evaluation.
// f(a) with f(a.v) = fv and f'(a.v) = fd
template <int W>
__host__ __device__ __forceinline__ Dual<W> chain(const Dual<W>& a, double fv, double fd) {
  Dual<W> r(fv);
#pragma unroll
  for (int w = 0; w < W; ++w) r.d[w] = fd * a.d[w];
  return r;
}

template <int W> __host__ __device__ __forceinline__ Dual<W> operator+(const Dual<W>& a) { return a; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator-(const Dual<W>& a) { return chain(a, -a.v, -1.0); }

template <int W> __host__ __device__ __forceinline__ Dual<W> operator+(Dual<W> a, const Dual<W>& b) { return a += b; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator-(Dual<W> a, const Dual<W>& b) { return a -= b; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator*(Dual<W> a, const Dual<W>& b) { return a *= b; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator/(Dual<W> a, const Dual<W>& b) { return a /= b; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator+(Dual<W> a, double b) { return a += b; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator-(Dual<W> a, double b) { return a -= b; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator*(Dual<W> a, double b) { return a *= b; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator/(Dual<W> a, double b) { return a /= b; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator+(double a, Dual<W> b) { return b += a; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator-(double a, const Dual<W>& b) { return chain(b, a - b.v, -1.0); }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator*(double a, Dual<W> b) { return b *= a; }
template <int W> __host__ __device__ __forceinline__ Dual<W> operator/(double a, const Dual<W>& b) {
  const double q = a / b.v;
  return chain(b, q, -q / b.v);
}

#define CDK_DUAL_CMP(op)                                                                                                   \
  template <int W> __host__ __device__ __forceinline__ bool operator op(const Dual<W>& a, const Dual<W>& b) { return a.v op b.v; } \
  template <int W> __host__ __device__ __forceinline__ bool operator op(const Dual<W>& a, double b) { return a.v op b; }           \
  template <int W> __host__ __device__ __forceinline__ bool operator op(double a, const Dual<W>& b) { return a op b.v; }
CDK_DUAL_CMP(<)
CDK_DUAL_CMP(<=)
CDK_DUAL_CMP(>)
CDK_DUAL_CMP(>=)
CDK_DUAL_CMP(==)
CDK_DUAL_CMP(!=)
#undef CDK_DUAL_CMP

template <int W> __host__ __device__ __forceinline__ Dual<W> sqrt(const Dual<W>& a) {
  const double s = ::sqrt(a.v);
  return chain(a, s, 0.5 / s);
}
template <int W> __host__ __device__ __forceinline__ Dual<W> exp(const Dual<W>& a) {
  const double e = ::exp(a.v);
  return chain(a, e, e);
}
template <int W> __host__ __device__ __forceinline__ Dual<W> log(const Dual<W>& a) { return chain(a, ::log(a.v), 1.0 / a.v); }
template <int W> __host__ __device__ __forceinline__ Dual<W> sin(const Dual<W>& a) { return chain(a, ::sin(a.v), ::cos(a.v)); }
template <int W> __host__ __device__ __forceinline__ Dual<W> cos(const Dual<W>& a) { return chain(a, ::cos(a.v), -::sin(a.v)); }
template <int W> __host__ __device__ __forceinline__ Dual<W> tan(const Dual<W>& a) {
  const double t = ::tan(a.v);
  return chain(a, t, 1.0 + t * t);
}
template <int W> __host__ __device__ __forceinline__ Dual<W> tanh(const Dual<W>& a) {
  const double t = ::tanh(a.v);
  return chain(a, t, 1.0 - t * t);
}
template <int W> __host__ __device__ __forceinline__ Dual<W> sinh(const Dual<W>& a) { return chain(a, ::sinh(a.v), ::cosh(a.v)); }
template <int W> __host__ __device__ __forceinline__ Dual<W> cosh(const Dual<W>& a) { return chain(a, ::cosh(a.v), ::sinh(a.v)); }
template <int W> __host__ __device__ __forceinline__ Dual<W> atan(const Dual<W>& a) { return chain(a, ::atan(a.v), 1.0 / (1.0 + a.v * a.v)); }
template <int W> __host__ __device__ __forceinline__ Dual<W> fabs(const Dual<W>& a) {
  return chain(a, ::fabs(a.v), a.v < 0.0 ? -1.0 : 1.0);
}
template <int W> __host__ __device__ __forceinline__ Dual<W> pow(const Dual<W>& a, double p) {
  const double v = ::pow(a.v, p);
  return chain(a, v, p == 0.0 ? 0.0 : p * ::pow(a.v, p - 1.0));
}

}  // namespace cdk_dual
