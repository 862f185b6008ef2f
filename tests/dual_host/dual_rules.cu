// Host check of the dual-number rules of blsq_dual.cuh (tests/test_autodiff_models.py).
//
// Reads lines "op form a b" (a, b as hex floats) and prints, per line, the
// value of the expression evaluated on Dual<2> operands, the value of the same
// expression on doubles, and the derivatives with respect to a and b, all as
// hex floats.  form: "DD" (both dual: a seeded with e_0, b with e_1), "Dd"
// (b a double constant), "dD" (a a double constant).  Unary ops use a only.
#include <stdio.h>
#include <string.h>

#include <type_traits>

#include "blsq_dual.cuh"

using D = blsq_dual::Dual<2>;

static double val(double x) { return x; }
static double val(const D& x) { return x.v; }
static double der(const D& x, int k) { return x.d[k]; }

// the expression of `op` with unqualified calls, as a templated residual has them
template <class X, class Y>
static auto expr(const char* op, const X& x, const Y& y) {
    using R = decltype(x + y);
#define OP(name, e) if (!strcmp(op, name)) return R(e);
    OP("add", x + y) OP("sub", x - y) OP("mul", x * y) OP("div", x / y)
    OP("pow", pow(x, y)) OP("atan2", atan2(x, y)) OP("hypot", hypot(x, y))
    OP("fmin", fmin(x, y)) OP("fmax", fmax(x, y))
    OP("eq", x == y) OP("ne", x != y) OP("lt", x < y) OP("le", x <= y) OP("gt", x > y)
    OP("ge", x >= y)
    OP("neg", -x) OP("pos", +x) OP("lit", (2 * x + 1) / 3 - x * 4 + (x > 0 ? 1 : 2))
    OP("powi", pow(x, 3)) OP("exp", exp(x)) OP("expm1", expm1(x)) OP("log", log(x))
    OP("log1p", log1p(x)) OP("sqrt", sqrt(x)) OP("cbrt", cbrt(x)) OP("sin", sin(x))
    OP("cos", cos(x)) OP("tan", tan(x)) OP("atan", atan(x)) OP("sinh", sinh(x))
    OP("cosh", cosh(x)) OP("tanh", tanh(x)) OP("erf", erf(x)) OP("fabs", fabs(x))
#undef OP
    if constexpr (std::is_same<X, D>::value) {
        X t = x;
        if (!strcmp(op, "iadd")) return R(t += y);
        if (!strcmp(op, "isub")) return R(t -= y);
        if (!strcmp(op, "imul")) return R(t *= y);
        if (!strcmp(op, "idiv")) return R(t /= y);
    } else {   // compound assignments have a Dual on the left: never read
        X t = x;
        if (!strcmp(op, "iadd")) return R(t += val(y));
        if (!strcmp(op, "isub")) return R(t -= val(y));
        if (!strcmp(op, "imul")) return R(t *= val(y));
        if (!strcmp(op, "idiv")) return R(t /= val(y));
    }
    fprintf(stderr, "unknown op %s\n", op);
    return R(0.0);
}

int main() {
    char op[32], form[8];
    double a, b;
    while (scanf("%31s %7s %la %la", op, form, &a, &b) == 4) {
        D A(a), B(b);
        A.d[0] = 1.0;
        B.d[1] = 1.0;
        const double vv = val(expr(op, a, b));
        double vd, d0 = 0.0, d1 = 0.0;
        if (!strcmp(form, "DD")) {
            const D r = expr(op, A, B);
            vd = r.v, d0 = der(r, 0), d1 = der(r, 1);
        } else if (!strcmp(form, "Dd")) {
            const D r = expr(op, A, b);
            vd = r.v, d0 = der(r, 0);
        } else {
            const D r = expr(op, a, B);
            vd = r.v, d1 = der(r, 1);
        }
        printf("%a %a %a %a\n", vd, vv, d0, d1);
    }
    return 0;
}
