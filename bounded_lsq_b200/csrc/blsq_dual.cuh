// Forward-mode dual numbers for compiled residual models (blsq_user_model.cuh).
//
// A model whose residual is a template on its scalar type,
//
//   template <class T>
//   __device__ T residual(const T (&x)[N], int64_t pid, int r, const blsq_model_ctx& c) const;
//
// is evaluated once with T = blsq_dual::Dual<N> and x[k].d = e_k: the value
// v of the result is the residual and d[k] its derivative with respect to
// x_k, the exact Jacobian row up to rounding.  Everything is __host__
// __device__, so the rules can be checked on the host.
//
// VALUE CHANNEL.  The value of every operation is the single IEEE operation
// or the math function the double code calls on the values: a.v * b.v,
// ::exp(a.v), ...; nothing derivative-related feeds it.  Compiled with
// -fmad=false (the library's flags), the value of a dual evaluation is then
// bit-identical to the double instantiation of the same template, so f from
// the dual and f from residual<double> are the same bits.
//
// SUPPORTED.  Dual o Dual, Dual o double and double o Dual for + - * /
// (a double argument takes ints and literals), unary -, += -= *= /=, the
// comparisons == != < <= > >= on the values (so user branches compile), and
// these functions, found by argument-dependent lookup on an unqualified call:
//   exp expm1 log log1p sqrt cbrt pow(Dual, double) pow(Dual, Dual)
//   pow(double, Dual) sin cos tan atan atan2 sinh cosh tanh erf fabs fmin
//   fmax hypot
// (atan2, fmin, fmax and hypot in every Dual / double mix).  Any other
// function of a Dual is a compile error in the model's source.
//
// NON-DIFFERENTIABLE POINTS.  Where the derivative is infinite or undefined,
// it is taken as 0:
//   fabs(0)                    derivative 0
//   sqrt(0), cbrt(0)           derivative 0
//   pow(0, p) for p < 1        derivative with respect to the base 0
//   pow(a, b) with a <= 0      derivative with respect to the exponent 0
//   hypot(0, 0), atan2(0, 0)   derivative 0
// and at a tie of fmin / fmax (equal values) the derivative is the mean of
// the two arguments' derivatives.  Otherwise fmin / fmax take the derivative
// of the argument whose value they return (the other one when one is NaN).
// Where one partial derivative of an operation overflows, the others may be
// NaN (inf * 0 in the chain rule).
#pragma once
#include <float.h>
#include <math.h>

#ifdef __CUDACC__
#define BLSQ_HD __host__ __device__ __forceinline__
#else
#define BLSQ_HD inline
#endif

namespace blsq_dual {

template <int N>
struct Dual {
    double v;      // value
    double d[N];   // gradient
    BLSQ_HD Dual(double c = 0.0) : v(c) {
#pragma unroll
        for (int k = 0; k < N; k++) d[k] = 0.0;
    }
    BLSQ_HD Dual& operator+=(const Dual& b) { return *this = *this + b; }
    BLSQ_HD Dual& operator-=(const Dual& b) { return *this = *this - b; }
    BLSQ_HD Dual& operator*=(const Dual& b) { return *this = *this * b; }
    BLSQ_HD Dual& operator/=(const Dual& b) { return *this = *this / b; }
    BLSQ_HD Dual& operator+=(double b) { return *this = *this + b; }
    BLSQ_HD Dual& operator-=(double b) { return *this = *this - b; }
    BLSQ_HD Dual& operator*=(double b) { return *this = *this * b; }
    BLSQ_HD Dual& operator/=(double b) { return *this = *this / b; }
};

// value v, gradient s * a.d
template <int N>
BLSQ_HD Dual<N> chain(double v, double s, const Dual<N>& a) {
    Dual<N> o;
    o.v = v;
#pragma unroll
    for (int k = 0; k < N; k++) o.d[k] = s * a.d[k];
    return o;
}

// value v, gradient sa * a.d + sb * b.d
template <int N>
BLSQ_HD Dual<N> chain2(double v, double sa, const Dual<N>& a, double sb, const Dual<N>& b) {
    Dual<N> o;
    o.v = v;
#pragma unroll
    for (int k = 0; k < N; k++) o.d[k] = sa * a.d[k] + sb * b.d[k];
    return o;
}

// ---- arithmetic ----

template <int N>
BLSQ_HD Dual<N> operator+(const Dual<N>& a) { return a; }
template <int N>
BLSQ_HD Dual<N> operator-(const Dual<N>& a) {
    Dual<N> o;
    o.v = -a.v;
#pragma unroll
    for (int k = 0; k < N; k++) o.d[k] = -a.d[k];
    return o;
}

template <int N>
BLSQ_HD Dual<N> operator+(const Dual<N>& a, const Dual<N>& b) {
    Dual<N> o;
    o.v = a.v + b.v;
#pragma unroll
    for (int k = 0; k < N; k++) o.d[k] = a.d[k] + b.d[k];
    return o;
}
template <int N>
BLSQ_HD Dual<N> operator+(const Dual<N>& a, double b) {
    Dual<N> o = a;
    o.v = a.v + b;
    return o;
}
template <int N>
BLSQ_HD Dual<N> operator+(double a, const Dual<N>& b) {
    Dual<N> o = b;
    o.v = a + b.v;
    return o;
}

template <int N>
BLSQ_HD Dual<N> operator-(const Dual<N>& a, const Dual<N>& b) {
    Dual<N> o;
    o.v = a.v - b.v;
#pragma unroll
    for (int k = 0; k < N; k++) o.d[k] = a.d[k] - b.d[k];
    return o;
}
template <int N>
BLSQ_HD Dual<N> operator-(const Dual<N>& a, double b) {
    Dual<N> o = a;
    o.v = a.v - b;
    return o;
}
template <int N>
BLSQ_HD Dual<N> operator-(double a, const Dual<N>& b) {
    Dual<N> o = -b;
    o.v = a - b.v;
    return o;
}

template <int N>
BLSQ_HD Dual<N> operator*(const Dual<N>& a, const Dual<N>& b) {
    return chain2(a.v * b.v, b.v, a, a.v, b);
}
template <int N>
BLSQ_HD Dual<N> operator*(const Dual<N>& a, double b) { return chain(a.v * b, b, a); }
template <int N>
BLSQ_HD Dual<N> operator*(double a, const Dual<N>& b) { return chain(a * b.v, a, b); }

// d(a / b) = (a.d - q b.d) / b.v, with one reciprocal per row (q b.d first:
// an overflowing partial with respect to b leaves the one to a finite)
template <int N>
BLSQ_HD Dual<N> operator/(const Dual<N>& a, const Dual<N>& b) {
    Dual<N> o;
    o.v = a.v / b.v;
    const double rb = 1.0 / b.v;
#pragma unroll
    for (int k = 0; k < N; k++) o.d[k] = (a.d[k] - o.v * b.d[k]) * rb;
    return o;
}
template <int N>
BLSQ_HD Dual<N> operator/(const Dual<N>& a, double b) { return chain(a.v / b, 1.0 / b, a); }
template <int N>
BLSQ_HD Dual<N> operator/(double a, const Dual<N>& b) {
    const double q = a / b.v;
    return chain(q, -q / b.v, b);
}

// ---- comparisons, on the values ----

#define BLSQ_DUAL_CMP(OP)                                                                    \
    template <int N>                                                                         \
    BLSQ_HD bool operator OP(const Dual<N>& a, const Dual<N>& b) { return a.v OP b.v; }      \
    template <int N>                                                                         \
    BLSQ_HD bool operator OP(const Dual<N>& a, double b) { return a.v OP b; }                \
    template <int N>                                                                         \
    BLSQ_HD bool operator OP(double a, const Dual<N>& b) { return a OP b.v; }
BLSQ_DUAL_CMP(==)
BLSQ_DUAL_CMP(!=)
BLSQ_DUAL_CMP(<)
BLSQ_DUAL_CMP(<=)
BLSQ_DUAL_CMP(>)
BLSQ_DUAL_CMP(>=)
#undef BLSQ_DUAL_CMP

// ---- functions ----

template <int N>
BLSQ_HD Dual<N> exp(const Dual<N>& a) {
    const double e = ::exp(a.v);
    return chain(e, e, a);
}
template <int N>
BLSQ_HD Dual<N> expm1(const Dual<N>& a) { return chain(::expm1(a.v), ::exp(a.v), a); }
template <int N>
BLSQ_HD Dual<N> log(const Dual<N>& a) { return chain(::log(a.v), 1.0 / a.v, a); }
template <int N>
BLSQ_HD Dual<N> log1p(const Dual<N>& a) { return chain(::log1p(a.v), 1.0 / (1.0 + a.v), a); }
template <int N>
BLSQ_HD Dual<N> sqrt(const Dual<N>& a) {
    const double s = ::sqrt(a.v);
    return chain(s, s == 0.0 ? 0.0 : 0.5 / s, a);
}
template <int N>
BLSQ_HD Dual<N> cbrt(const Dual<N>& a) {
    const double c = ::cbrt(a.v);
    return chain(c, c == 0.0 ? 0.0 : 1.0 / (3.0 * c * c), a);
}

// p * x^(p-1) as p * (x^p / x) while x^p is a normal number (no rounding of
// p - 1), else from pow(x, p - 1); 0 at x = 0 for p < 1 (p = 0 included)
BLSQ_HD double dpow(double x, double p, double xp) {
    if (p == 0.0 || (x == 0.0 && p < 1.0)) return 0.0;
    if (::fabs(xp) >= DBL_MIN && ::fabs(xp) <= DBL_MAX) return p * (xp / x);
    return p * ::pow(x, p - 1.0);
}
// log(a) * a^b: the derivative of a^b with respect to b; 0 for a <= 0
BLSQ_HD double dpow_exp(double a, double ab) { return a > 0.0 ? ab * ::log(a) : 0.0; }

template <int N>
BLSQ_HD Dual<N> pow(const Dual<N>& a, double p) {
    const double v = ::pow(a.v, p);
    return chain(v, dpow(a.v, p, v), a);
}
template <int N>
BLSQ_HD Dual<N> pow(const Dual<N>& a, const Dual<N>& b) {
    const double v = ::pow(a.v, b.v);
    return chain2(v, dpow(a.v, b.v, v), a, dpow_exp(a.v, v), b);
}
template <int N>
BLSQ_HD Dual<N> pow(double a, const Dual<N>& b) {
    const double v = ::pow(a, b.v);
    return chain(v, dpow_exp(a, v), b);
}

template <int N>
BLSQ_HD Dual<N> sin(const Dual<N>& a) { return chain(::sin(a.v), ::cos(a.v), a); }
template <int N>
BLSQ_HD Dual<N> cos(const Dual<N>& a) { return chain(::cos(a.v), -::sin(a.v), a); }
template <int N>
BLSQ_HD Dual<N> tan(const Dual<N>& a) {
    const double t = ::tan(a.v);
    return chain(t, 1.0 + t * t, a);
}
template <int N>
BLSQ_HD Dual<N> atan(const Dual<N>& a) { return chain(::atan(a.v), 1.0 / (1.0 + a.v * a.v), a); }
template <int N>
BLSQ_HD Dual<N> sinh(const Dual<N>& a) { return chain(::sinh(a.v), ::cosh(a.v), a); }
template <int N>
BLSQ_HD Dual<N> cosh(const Dual<N>& a) { return chain(::cosh(a.v), ::sinh(a.v), a); }
template <int N>
BLSQ_HD Dual<N> tanh(const Dual<N>& a) {
    const double c = ::cosh(a.v);
    return chain(::tanh(a.v), 1.0 / (c * c), a);
}
template <int N>
BLSQ_HD Dual<N> erf(const Dual<N>& a) {
    return chain(::erf(a.v), 1.1283791670955126 * ::exp(-(a.v * a.v)), a);   // 2 / sqrt(pi)
}
template <int N>
BLSQ_HD Dual<N> fabs(const Dual<N>& a) {
    return chain(::fabs(a.v), a.v > 0.0 ? 1.0 : (a.v < 0.0 ? -1.0 : 0.0), a);
}

// atan2(y, x): d = (x dy - y dx) / h^2, h = hypot(x, y), scaled by h first
template <int N>
BLSQ_HD Dual<N> atan2(const Dual<N>& y, const Dual<N>& x) {
    const double h = ::hypot(x.v, y.v);
    const double sy = h == 0.0 ? 0.0 : (x.v / h) / h, sx = h == 0.0 ? 0.0 : -(y.v / h) / h;
    return chain2(::atan2(y.v, x.v), sy, y, sx, x);
}
template <int N>
BLSQ_HD Dual<N> hypot(const Dual<N>& a, const Dual<N>& b) {
    const double h = ::hypot(a.v, b.v);
    return chain2(h, h == 0.0 ? 0.0 : a.v / h, a, h == 0.0 ? 0.0 : b.v / h, b);
}
template <int N>
BLSQ_HD Dual<N> fmin(const Dual<N>& a, const Dual<N>& b) {
    const double v = ::fmin(a.v, b.v);
    if (a.v == b.v) return chain2(v, 0.5, a, 0.5, b);
    return chain(v, 1.0, v == a.v ? a : b);
}
template <int N>
BLSQ_HD Dual<N> fmax(const Dual<N>& a, const Dual<N>& b) {
    const double v = ::fmax(a.v, b.v);
    if (a.v == b.v) return chain2(v, 0.5, a, 0.5, b);
    return chain(v, 1.0, v == a.v ? a : b);
}

// the two-argument functions with one double argument: the double is a
// constant (zero gradient), the value is the same call on the values
#define BLSQ_DUAL_MIXED(F)                                                                   \
    template <int N>                                                                         \
    BLSQ_HD Dual<N> F(const Dual<N>& a, double b) { return F(a, Dual<N>(b)); }              \
    template <int N>                                                                         \
    BLSQ_HD Dual<N> F(double a, const Dual<N>& b) { return F(Dual<N>(a), b); }
BLSQ_DUAL_MIXED(atan2)
BLSQ_DUAL_MIXED(hypot)
BLSQ_DUAL_MIXED(fmin)
BLSQ_DUAL_MIXED(fmax)
#undef BLSQ_DUAL_MIXED

}  // namespace blsq_dual

#undef BLSQ_HD
