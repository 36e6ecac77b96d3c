/*
 * oracle/forward_mode.cpp — TEST INFRASTRUCTURE / CPU BASELINE ONLY (never imported by the product path).
 *
 * The CPU baseline bench.py times beside the GPU: the same restatement (core.inc.h: ABA, fatigue ODE, RK4) instantiated a
 * third time with SC = a forward-mode "multi-dual" number that carries all 3n + 1 tangent directions (q, qd, tau, dt) of
 * one unit as SIMD lanes next to the value.  This is the algorithm class of the reference's CPU path — CasADi differentiates
 * the traced Pinocchio graph by forward/reverse sweeps over the same operations (nlpsol's jac_g,
 * python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:195-197) — compiled, vectorised and run on all host cores, i.e. at least
 * as fast as CasADi's single-threaded SX interpreter.  The n fatigue columns are closed form (d(q+, qd+)/df = 0,
 * df+/df = diag RK4 amplification), exactly as the CUDA path writes them.
 *
 * The complex-step instantiation in mpcf_oracle.c stays the parity CHECKER (it shares no derivative code with anything);
 * tests/test_oracle_consistency.py checks this file against it.
 */
#include <cmath>
#include <cstdlib>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "mpcf_oracle.h"

namespace {

constexpr int LANES = 24;  // up to 3n + 1 = 19 directions for n = 6, padded to three 512-bit vectors
typedef double vd __attribute__((vector_size(LANES * 8 / 3)));  // 8 doubles

struct MDual {
    double v;
    vd d[3];
    MDual() {}
    MDual(double x) : v(x) { d[0] = d[1] = d[2] = vd{0, 0, 0, 0, 0, 0, 0, 0}; }
};
#define LOOP3 for (int k = 0; k < 3; ++k)
inline MDual operator+(const MDual &a, const MDual &b) { MDual r; r.v = a.v + b.v; LOOP3 r.d[k] = a.d[k] + b.d[k]; return r; }
inline MDual operator-(const MDual &a, const MDual &b) { MDual r; r.v = a.v - b.v; LOOP3 r.d[k] = a.d[k] - b.d[k]; return r; }
inline MDual operator*(const MDual &a, const MDual &b) { MDual r; r.v = a.v * b.v; LOOP3 r.d[k] = a.v * b.d[k] + b.v * a.d[k]; return r; }
inline MDual operator-(const MDual &a) { MDual r; r.v = -a.v; LOOP3 r.d[k] = -a.d[k]; return r; }
inline MDual operator+(const MDual &a, double b) { MDual r = a; r.v += b; return r; }
inline MDual operator+(double a, const MDual &b) { MDual r = b; r.v += a; return r; }
inline MDual operator-(const MDual &a, double b) { MDual r = a; r.v -= b; return r; }
inline MDual operator-(double a, const MDual &b) { MDual r; r.v = a - b.v; LOOP3 r.d[k] = -b.d[k]; return r; }
inline MDual operator*(const MDual &a, double b) { MDual r; r.v = a.v * b; LOOP3 r.d[k] = a.d[k] * b; return r; }
inline MDual operator*(double a, const MDual &b) { return b * a; }
inline MDual operator/(double a, const MDual &b) { const double iv = 1.0 / b.v; MDual r; r.v = a * iv; const double s = -r.v * iv; LOOP3 r.d[k] = s * b.d[k]; return r; }
inline MDual operator/(const MDual &a, double b) { return a * (1.0 / b); }
inline MDual operator/(const MDual &a, const MDual &b) { const double iv = 1.0 / b.v; MDual r; r.v = a.v * iv; LOOP3 r.d[k] = (a.d[k] - r.v * b.d[k]) * iv; return r; }
inline MDual &operator+=(MDual &a, const MDual &b) { a.v += b.v; LOOP3 a.d[k] += b.d[k]; return a; }
inline MDual &operator-=(MDual &a, const MDual &b) { a.v -= b.v; LOOP3 a.d[k] -= b.d[k]; return a; }
inline MDual &operator+=(MDual &a, double b) { a.v += b; return a; }
inline bool operator==(const MDual &a, double b) { return a.v == b; }
inline MDual md_sin(const MDual &a) { MDual r; const double c = std::cos(a.v); r.v = std::sin(a.v); LOOP3 r.d[k] = c * a.d[k]; return r; }
inline MDual md_cos(const MDual &a) { MDual r; const double s = -std::sin(a.v); r.v = std::cos(a.v); LOOP3 r.d[k] = s * a.d[k]; return r; }
inline MDual md_exp(const MDual &a) { MDual r; r.v = std::exp(a.v); LOOP3 r.d[k] = r.v * a.d[k]; return r; }
inline MDual md_expm1(const MDual &a) { MDual r; const double e = std::exp(a.v); r.v = std::expm1(a.v); LOOP3 r.d[k] = e * a.d[k]; return r; }
inline void seed(MDual &a, int lane) { reinterpret_cast<double *>(a.d)[lane] = 1.0; }
inline double tangent(const MDual &a, int lane) { return reinterpret_cast<const double *>(a.d)[lane]; }

#define SC MDual
#define SUF(x) x##_m
#define SIN md_sin
#define COS md_cos
#define EXP md_exp
#define EXPM1 md_expm1
#include "core.inc.h"
#undef SC
#undef SUF
#undef SIN
#undef COS
#undef EXP
#undef EXPM1

}  // namespace

/* Same contract as mpcfo_step_rk4_jvp_batch (jac: [3n][4n+1][U], rows (q+, qd+, f+), columns (q, qd, tau, f, dt)); one
 * forward-mode sweep per unit with every direction in the SIMD lanes.  n <= 7 (3n + 1 <= 24 lanes - 2). */
extern "C" int mpcfo_step_rk4_jvp_forward_batch(const mpcfo_model *m, long U, const double *q, const double *qd, const double *tau,
                                                const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn,
                                                double *jac)
{
    if (m->n <= 0 || 3 * m->n + 1 > LANES) return -1;
    const int n = m->n, P = 4 * n + 1;
    int rc = 0;
#pragma omp parallel for schedule(static) reduction(| : rc)
    for (long u = 0; u < U; ++u) {
        MDual x[3 * MPCFO_MAXN], t[MPCFO_MAXN], xn[3 * MPCFO_MAXN];
        for (int i = 0; i < n; ++i) {
            x[i] = MDual(q[i * U + u]); seed(x[i], i);
            x[n + i] = MDual(qd[i * U + u]); seed(x[n + i], n + i);
            x[2 * n + i] = MDual(f[i * U + u]);
            t[i] = MDual(tau[i * U + u]); seed(t[i], 2 * n + i);
        }
        const double hv = dt_u ? dt_u[u] : dt;
        MDual h(hv);
        seed(h, 3 * n);
        rc |= step_rk4_m(m, x, t, h, xn) != 0;
        for (int r = 0; r < 3 * n; ++r) {
            for (int d = 0; d < 3 * n; ++d) jac[((long)r * P + d) * U + u] = tangent(xn[r], d);
            jac[((long)r * P + 4 * n) * U + u] = tangent(xn[r], 3 * n);
            for (int j = 0; j < n; ++j) {  // fatigue columns: closed form (RK4 amplification of the linear compartment)
                const double z = m->fat[4 * j] * hv;
                jac[((long)r * P + 3 * n + j) * U + u] = (r == 2 * n + j) ? 1.0 + z * (-1.0 + z * (0.5 + z * (-1.0 / 6.0 + z / 24.0))) : 0.0;
            }
        }
        if (qn)
            for (int i = 0; i < n; ++i) { qn[i * U + u] = xn[i].v; qdn[i * U + u] = xn[n + i].v; fn[i * U + u] = xn[2 * n + i].v; }
    }
    return rc ? -3 : 0;
}

extern "C" int mpcfo_fwd_set_threads(int nthreads)
{
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
    return omp_get_max_threads();
#else
    (void)nthreads;
    return 1;
#endif
}
