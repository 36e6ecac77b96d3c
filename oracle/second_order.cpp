/*
 * oracle/second_order.cpp — TEST INFRASTRUCTURE ONLY (never imported by the product path).
 *
 * Second derivatives of the RK4 step, the checker of mpcf_step_rk4_hess_batch / mpcf_step_rk4_hvp_batch: the restatement
 * (core.inc.h: ABA, fatigue ODE, RK4) instantiated a fourth time with SC = a hyper-dual number (value, two tangents a and b, and
 * the mixed second derivative ab), so one sweep gives d2 x+ / dz_a dz_b exactly to rounding.  Unlike the CUDA kernels, which
 * write the fatigue rows and columns in closed form, this sweeps ALL P (P + 1) / 2 pairs of z = (q, qd, tau, f, dt), P = 4n + 1,
 * the fatigue inputs included, so the closed form is checked against an independent sweep.
 */
#include <cmath>
#include <cstdlib>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "mpcf_oracle.h"

namespace {

struct HD {
    double v, a, b, ab;
    HD() {}
    HD(double x) : v(x), a(0), b(0), ab(0) {}
    HD(double v_, double a_, double b_, double ab_) : v(v_), a(a_), b(b_), ab(ab_) {}
};
inline HD operator+(const HD &x, const HD &y) { return HD(x.v + y.v, x.a + y.a, x.b + y.b, x.ab + y.ab); }
inline HD operator-(const HD &x, const HD &y) { return HD(x.v - y.v, x.a - y.a, x.b - y.b, x.ab - y.ab); }
inline HD operator*(const HD &x, const HD &y)
{
    return HD(x.v * y.v, x.v * y.a + x.a * y.v, x.v * y.b + x.b * y.v, x.v * y.ab + x.a * y.b + x.b * y.a + x.ab * y.v);
}
inline HD operator-(const HD &x) { return HD(-x.v, -x.a, -x.b, -x.ab); }
inline HD operator+(const HD &x, double y) { return HD(x.v + y, x.a, x.b, x.ab); }
inline HD operator+(double x, const HD &y) { return y + x; }
inline HD operator-(const HD &x, double y) { return HD(x.v - y, x.a, x.b, x.ab); }
inline HD operator-(double x, const HD &y) { return HD(x - y.v, -y.a, -y.b, -y.ab); }
inline HD operator*(const HD &x, double y) { return HD(x.v * y, x.a * y, x.b * y, x.ab * y); }
inline HD operator*(double x, const HD &y) { return y * x; }
// 1 / y: r' = -y' r^2, r'' = -y'' r^2 + 2 y'_a y'_b r^3
inline HD hd_recip(const HD &y)
{
    const double r = 1.0 / y.v, r2 = r * r;
    return HD(r, -y.a * r2, -y.b * r2, -y.ab * r2 + 2.0 * y.a * y.b * r2 * r);
}
inline HD operator/(const HD &x, const HD &y) { return x * hd_recip(y); }
inline HD operator/(double x, const HD &y) { return x * hd_recip(y); }
inline HD operator/(const HD &x, double y) { return x * (1.0 / y); }
inline HD &operator+=(HD &x, const HD &y) { x = x + y; return x; }
inline HD &operator-=(HD &x, const HD &y) { x = x - y; return x; }
inline HD &operator+=(HD &x, double y) { x.v += y; return x; }
inline bool operator==(const HD &x, double y) { return x.v == y; }
inline HD hd_sin(const HD &x) { const double s = std::sin(x.v), c = std::cos(x.v); return HD(s, c * x.a, c * x.b, c * x.ab - s * x.a * x.b); }
inline HD hd_cos(const HD &x) { const double s = std::sin(x.v), c = std::cos(x.v); return HD(c, -s * x.a, -s * x.b, -s * x.ab - c * x.a * x.b); }
inline HD hd_exp(const HD &x) { const double e = std::exp(x.v); return HD(e, e * x.a, e * x.b, e * (x.ab + x.a * x.b)); }
inline HD hd_expm1(const HD &x) { const double e = std::exp(x.v); return HD(std::expm1(x.v), e * x.a, e * x.b, e * (x.ab + x.a * x.b)); }

#define SC HD
#define SUF(x) x##_h
#define SIN hd_sin
#define COS hd_cos
#define EXP hd_exp
#define EXPM1 hd_expm1
#include "core.inc.h"
#undef SC
#undef SUF
#undef SIN
#undef COS
#undef EXP
#undef EXPM1

inline double at(const double *p, long i) { return p ? p[i] : 0.0; }

// One step of unit u with direction a of z on the first tangent and, on the second, direction b (b >= 0) or the vector v (b < 0;
// v = (vq, vqd, vtau, vf, vdt)); returns sum_r lambda_r x+_r.ab and leaves x+ in xn.
int sweep(const mpcfo_model *m, long U, long u, const double *const *z, double hv, const double *const *lam, int a, int b,
          const double *const *v, HD *xn, double *s)
{
    const int n = m->n;
    auto seed = [&](int c, long k) {  // input c of z at plane offset k
        return HD(c < 4 * n ? z[c / n][k] : hv, a == c ? 1.0 : 0.0, b >= 0 ? (b == c ? 1.0 : 0.0) : at(v[c / n], k), 0.0);
    };
    HD x[3 * MPCFO_MAXN], t[MPCFO_MAXN];
    for (int i = 0; i < n; ++i) {
        const long k = (long)i * U + u;
        x[i] = seed(i, k);
        x[n + i] = seed(n + i, k);
        t[i] = seed(2 * n + i, k);
        x[2 * n + i] = seed(3 * n + i, k);
    }
    const HD h = seed(4 * n, u);
    const int rc = step_rk4_h(m, x, t, h, xn);
    double acc = 0.0;
    for (int r = 0; r < 3 * n; ++r) acc += at(lam[r / n], (long)(r % n) * U + u) * xn[r].ab;
    *s = acc;
    return rc;
}

}  // namespace

/* H [4n+1][4n+1][U] (plane r*(4n+1)+c) = d2(lambda^T x+)/dz dz, z = (q, qd, tau, f, dt); lq/lqd/lf NULL = 0.  Every pair a <= b is
 * swept; both triangles are written. */
extern "C" int mpcfo_step_rk4_hess_batch(const mpcfo_model *m, long U, const double *q, const double *qd, const double *tau,
                                         const double *f, double dt, const double *dt_u, const double *lq, const double *lqd,
                                         const double *lf, double *H)
{
    const int n = m->n, P = 4 * n + 1;
    const double *z[4] = {q, qd, tau, f}, *lam[3] = {lq, lqd, lf};
    const long npair = (long)P * (P + 1) / 2;
    int rc = 0;
#pragma omp parallel for schedule(dynamic, 16) reduction(| : rc)
    for (long w = 0; w < npair * U; ++w) {
        const long u = w % U, k = w / U;
        int a = 0;
        long off = 0;
        while (off + (P - a) <= k) { off += P - a; ++a; }
        const int b = a + (int)(k - off);
        HD xn[3 * MPCFO_MAXN];
        double s;
        rc |= sweep(m, U, u, z, dt_u ? dt_u[u] : dt, lam, a, b, nullptr, xn, &s) != 0;
        H[((long)a * P + b) * U + u] = s;
        H[((long)b * P + a) * U + u] = s;
    }
    return rc ? -3 : 0;
}

/* hq, hqd, htau, hf [n][U], hdt [U] = H v with v = (vq, vqd, vtau, vf, vdt) (NULL = 0), one sweep per input; jq, jqd, jf [n][U] =
 * J v (NULL to skip). */
extern "C" int mpcfo_step_rk4_hvp_batch(const mpcfo_model *m, long U, const double *q, const double *qd, const double *tau,
                                        const double *f, double dt, const double *dt_u, const double *lq, const double *lqd,
                                        const double *lf, const double *vq, const double *vqd, const double *vtau, const double *vf,
                                        const double *vdt, double *hq, double *hqd, double *htau, double *hf, double *hdt,
                                        double *jq, double *jqd, double *jf)
{
    const int n = m->n, P = 4 * n + 1;
    const double *z[4] = {q, qd, tau, f}, *lam[3] = {lq, lqd, lf}, *v[5] = {vq, vqd, vtau, vf, vdt};
    double *out[5] = {hq, hqd, htau, hf, hdt}, *jv[3] = {jq, jqd, jf};
    int rc = 0;
#pragma omp parallel for schedule(dynamic, 16) reduction(| : rc)
    for (long w = 0; w < (long)P * U; ++w) {
        const long u = w % U;
        const int a = (int)(w / U);
        HD xn[3 * MPCFO_MAXN];
        double s;
        rc |= sweep(m, U, u, z, dt_u ? dt_u[u] : dt, lam, a, -1, v, xn, &s) != 0;
        out[a / n][(long)(a % n) * U + u] = s;
        if (a == 0 && jq)
            for (int r = 0; r < 3 * n; ++r) jv[r / n][(long)(r % n) * U + u] = xn[r].b;
    }
    return rc ? -3 : 0;
}
