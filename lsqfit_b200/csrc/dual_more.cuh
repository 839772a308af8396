// More Dual<N> math for user models (run-time plug-ins, lsqfit_b200/user_functor.py): the functions a model body
// commonly needs beyond dual.cuh.  Only plug-ins include this header; the built-in functors do not use it.
//
// As in dual.cuh, every .v is computed exactly as the plain-double overload below computes it, so that
// Body::eval<double> and Body::eval<Dual<N>>().v agree bit for bit.
#pragma once
#include "dual.cuh"

namespace b200lm {

template <int N> __device__ __forceinline__ Dual<N> tanh(const Dual<N>& a) {
    const double t = ::tanh(a.v); return chain(a, t, 1.0 - t * t);
}
template <int N> __device__ __forceinline__ Dual<N> sinh(const Dual<N>& a) {
    return chain(a, ::sinh(a.v), ::cosh(a.v));
}
template <int N> __device__ __forceinline__ Dual<N> cosh(const Dual<N>& a) {
    return chain(a, ::cosh(a.v), ::sinh(a.v));
}
template <int N> __device__ __forceinline__ Dual<N> expm1(const Dual<N>& a) {
    return chain(a, ::expm1(a.v), ::exp(a.v));
}
template <int N> __device__ __forceinline__ Dual<N> log1p(const Dual<N>& a) {
    return chain(a, ::log1p(a.v), 1.0 / (1.0 + a.v));
}
template <int N> __device__ __forceinline__ Dual<N> erf(const Dual<N>& a) {
    return chain(a, ::erf(a.v), 1.1283791670955125739 * ::exp(-(a.v * a.v)));      // 2 / sqrt(pi)
}
// atan2(y, x): d = (x dy - y dx) / (x^2 + y^2)
template <int N> __device__ __forceinline__ Dual<N> atan2(const Dual<N>& y, const Dual<N>& x) {
    const double ir = 1.0 / (x.v * x.v + y.v * y.v);
    Dual<N> r; r.v = ::atan2(y.v, x.v);
#pragma unroll
    for (int i = 0; i < N; ++i) r.d[i] = fma(x.v, y.d[i], -(y.v * x.d[i])) * ir;
    return r;
}
template <int N> __device__ __forceinline__ Dual<N> atan2(const Dual<N>& y, double x) {
    return chain(y, ::atan2(y.v, x), x / (x * x + y.v * y.v));
}
template <int N> __device__ __forceinline__ Dual<N> atan2(double y, const Dual<N>& x) {
    return chain(x, ::atan2(y, x.v), -y / (x.v * x.v + y * y));
}
// |a|, derivative sign(a) (+1 at a = 0); the value is fabs(a.v), which keeps the sign bit of -0.0 cleared
template <int N> __device__ __forceinline__ Dual<N> abs(const Dual<N>& a) {
    Dual<N> r = a.v < 0.0 ? -a : a;
    r.v = ::fabs(a.v);
    return r;
}

// plain-double overloads (the templates above hide the global functions inside this namespace)
__device__ __forceinline__ double tanh(double a) { return ::tanh(a); }
__device__ __forceinline__ double sinh(double a) { return ::sinh(a); }
__device__ __forceinline__ double cosh(double a) { return ::cosh(a); }
__device__ __forceinline__ double expm1(double a) { return ::expm1(a); }
__device__ __forceinline__ double log1p(double a) { return ::log1p(a); }
__device__ __forceinline__ double erf(double a) { return ::erf(a); }
__device__ __forceinline__ double atan2(double y, double x) { return ::atan2(y, x); }
__device__ __forceinline__ double abs(double a) { return ::fabs(a); }

}  // namespace b200lm
