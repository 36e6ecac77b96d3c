/*
 * oracle/mpcf_oracle.c — TEST INFRASTRUCTURE ONLY (see mpcf_oracle.h).
 *
 * Batch drivers around core.inc.h.  Build: `make -C oracle` (gcc -O2 -ffp-contract=off for the
 * reproducible checker `libmpcf_oracle.so`; -O3 -march=native for the timing build
 * `libmpcf_oracle_fast.so` used by bench.py's cpu_baseline leg).
 */
#include "mpcf_oracle.h"

#include <complex.h>
#include <math.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* real instantiation */
#define SC double
#define SUF(x) x##_r
#define SIN sin
#define COS cos
#define EXP exp
#define EXPM1 expm1
#include "core.inc.h"
#undef SC
#undef SUF
#undef SIN
#undef COS
#undef EXP
#undef EXPM1

/* exp(z) - 1 for complex z = x + i y without the cancellation of cexp(z) - 1 at small |z|:
 * e^x cos y - 1 = expm1(x) cos y - 2 sin^2(y / 2) */
static inline double complex cexpm1(double complex z)
{
    const double x = creal(z), y = cimag(z), s = sin(0.5 * y);
    return CMPLX(expm1(x) * cos(y) - 2.0 * s * s, exp(x) * sin(y));
}

/* complex instantiation (complex-step derivatives) */
#define SC double complex
#define SUF(x) x##_c
#define SIN csin
#define COS ccos
#define EXP cexp
#define EXPM1 cexpm1
#include "core.inc.h"
#undef SC
#undef SUF
#undef SIN
#undef COS
#undef EXP
#undef EXPM1

static int g_threads = 0;

int mpcfo_set_threads(int nthreads)
{
#ifdef _OPENMP
    if (nthreads > 0) { g_threads = nthreads; omp_set_num_threads(nthreads); }
    return g_threads > 0 ? g_threads : omp_get_max_threads();
#else
    (void)nthreads;
    return 1;
#endif
}

#define CHECK_N(m) do { if ((m)->n <= 0 || (m)->n > MPCFO_MAXN) return -1; } while (0)

int mpcfo_rnea_batch(const mpcfo_model *m, long U, const double *q, const double *qd, const double *qdd,
                     double *tau)
{
    CHECK_N(m);
    int n = m->n;
#pragma omp parallel for schedule(static)
    for (long u = 0; u < U; ++u) {
        double a[MPCFO_MAXN], b[MPCFO_MAXN], c[MPCFO_MAXN], t[MPCFO_MAXN];
        for (int i = 0; i < n; ++i) { a[i] = q[i * U + u]; b[i] = qd[i * U + u]; c[i] = qdd ? qdd[i * U + u] : 0.0; }
        rnea_r(m, a, b, c, t);
        for (int i = 0; i < n; ++i) tau[i * U + u] = t[i];
    }
    return 0;
}

int mpcfo_fk_batch(const mpcfo_model *m, int frame, long U, const double *q, double *pos, double *rot)
{
    CHECK_N(m);
    if (frame < 0 || frame >= m->nframes) return -2;
    int n = m->n;
#pragma omp parallel for schedule(static)
    for (long u = 0; u < U; ++u) {
        double a[MPCFO_MAXN], p[3], R[9];
        for (int i = 0; i < n; ++i) a[i] = q[i * U + u];
        frame_fk_r(m, frame, a, p, R);
        for (int k = 0; k < 3; ++k) pos[k * U + u] = p[k];
        for (int k = 0; k < 9; ++k) rot[k * U + u] = R[k];
    }
    return 0;
}

int mpcfo_jac_batch(const mpcfo_model *m, int frame, long U, const double *q, double *J)
{
    CHECK_N(m);
    if (frame < 0 || frame >= m->nframes) return -2;
    int n = m->n;
#pragma omp parallel for schedule(static)
    for (long u = 0; u < U; ++u) {
        double a[MPCFO_MAXN], Jl[6 * MPCFO_MAXN];
        for (int i = 0; i < n; ++i) a[i] = q[i * U + u];
        frame_jacobian_r(m, frame, a, Jl);
        for (int k = 0; k < 6 * n; ++k) J[k * U + u] = Jl[k];
    }
    return 0;
}

int mpcfo_crba(const mpcfo_model *m, const double *q, double *M)
{
    CHECK_N(m);
    crba_r(m, q, M);
    return 0;
}

int mpcfo_aba_batch(const mpcfo_model *m, long U, const double *q, const double *qd, const double *tau,
                    double *qdd)
{
    CHECK_N(m);
    int n = m->n, rc = 0;
#pragma omp parallel for schedule(static) reduction(| : rc)
    for (long u = 0; u < U; ++u) {
        double a[MPCFO_MAXN], b[MPCFO_MAXN], c[MPCFO_MAXN], t[MPCFO_MAXN];
        for (int i = 0; i < n; ++i) { a[i] = q[i * U + u]; b[i] = qd[i * U + u]; c[i] = tau[i * U + u]; }
        rc |= aba_r(m, a, b, c, t) != 0;
        for (int i = 0; i < n; ++i) qdd[i * U + u] = t[i];
    }
    return rc ? -3 : 0;
}

int mpcfo_node_eval_ref_batch(const mpcfo_model *m, int nee, const int *ee_frames, double wsign, long U,
                              const double *q, const double *qd, const double *qdd, const double *W,
                              const double *T, double h, double *tau, double *qnext, double *Tnext)
{
    CHECK_N(m);
    if (nee < 0 || nee > 8) return -2;
    for (int e = 0; e < nee; ++e)
        if (ee_frames[e] < 0 || ee_frames[e] >= m->nframes) return -2;
    int n = m->n;
#pragma omp parallel for schedule(static)
    for (long u = 0; u < U; ++u) {
        double a[MPCFO_MAXN], b[MPCFO_MAXN], c[MPCFO_MAXN], Tl[MPCFO_MAXN], Wl[48];
        double t[MPCFO_MAXN], qn[MPCFO_MAXN], Tn[MPCFO_MAXN];
        for (int i = 0; i < n; ++i) {
            a[i] = q[i * U + u]; b[i] = qd[i * U + u];
            c[i] = qdd ? qdd[i * U + u] : 0.0;
            Tl[i] = T ? T[i * U + u] : 0.0;
        }
        for (int k = 0; k < 6 * nee; ++k) Wl[k] = W[k * U + u];
        node_eval_ref_r(m, nee, ee_frames, wsign, a, b, c, Wl, Tl, h, t, qn, Tn);
        for (int i = 0; i < n; ++i) {
            tau[i * U + u] = t[i];
            if (qnext) qnext[i * U + u] = qn[i];
            if (Tnext) Tnext[i * U + u] = Tn[i];
        }
    }
    return 0;
}

int mpcfo_step_rk4_batch(const mpcfo_model *m, long U, const double *q, const double *qd, const double *tau,
                         const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn)
{
    CHECK_N(m);
    int n = m->n, rc = 0;
#pragma omp parallel for schedule(static) reduction(| : rc)
    for (long u = 0; u < U; ++u) {
        double x[3 * MPCFO_MAXN], t[MPCFO_MAXN], xn[3 * MPCFO_MAXN];
        for (int i = 0; i < n; ++i) {
            x[i] = q[i * U + u]; x[n + i] = qd[i * U + u]; x[2 * n + i] = f[i * U + u]; t[i] = tau[i * U + u];
        }
        rc |= step_rk4_r(m, x, t, dt_u ? dt_u[u] : dt, xn) != 0;
        for (int i = 0; i < n; ++i) {
            qn[i * U + u] = xn[i]; qdn[i * U + u] = xn[n + i]; fn[i * U + u] = xn[2 * n + i];
        }
    }
    return rc ? -3 : 0;
}

int mpcfo_step_rk4_jvp_batch(const mpcfo_model *m, long U, const double *q, const double *qd,
                             const double *tau, const double *f, double dt, const double *dt_u, double *qn,
                             double *qdn, double *fn, double *jac)
{
    CHECK_N(m);
    const int n = m->n, P = 4 * n + 1;
    const double hstep = 1e-40;
    int rc = 0;
#pragma omp parallel for schedule(static) reduction(| : rc)
    for (long u = 0; u < U; ++u) {
        double complex x[3 * MPCFO_MAXN], t[MPCFO_MAXN], xn[3 * MPCFO_MAXN], h;
        for (int d = 0; d < P; ++d) {
            for (int i = 0; i < n; ++i) {
                x[i] = q[i * U + u]; x[n + i] = qd[i * U + u]; x[2 * n + i] = f[i * U + u]; t[i] = tau[i * U + u];
            }
            h = dt_u ? dt_u[u] : dt;
            /* seed direction d of (q, qd, tau, f, dt) */
            if (d < 2 * n) x[d] += hstep * I;
            else if (d < 3 * n) t[d - 2 * n] += hstep * I;
            else if (d < 4 * n) x[d - n] += hstep * I; /* f lives at x[2n..3n) */
            else h += hstep * I;
            rc |= step_rk4_c(m, x, t, h, xn) != 0;
            for (int r = 0; r < 3 * n; ++r) jac[((long)r * P + d) * U + u] = cimag(xn[r]) / hstep;
            if (d == 0 && qn)
                for (int i = 0; i < n; ++i) {
                    qn[i * U + u] = creal(xn[i]); qdn[i * U + u] = creal(xn[n + i]); fn[i * U + u] = creal(xn[2 * n + i]);
                }
        }
    }
    return rc ? -3 : 0;
}

int mpcfo_step_rk4_coupled_batch(const mpcfo_model *m, const mpcfo_coupling *cp, long U, const double *q, const double *qd,
                                 const double *tau, const double *f, double dt, const double *dt_u, double *qn, double *qdn,
                                 double *fn)
{
    CHECK_N(m);
    int n = m->n, rc = 0;
#pragma omp parallel for schedule(static) reduction(| : rc)
    for (long u = 0; u < U; ++u) {
        double x[3 * MPCFO_MAXN], t[MPCFO_MAXN], xn[3 * MPCFO_MAXN];
        for (int i = 0; i < n; ++i) {
            x[i] = q[i * U + u]; x[n + i] = qd[i * U + u]; x[2 * n + i] = f[i * U + u]; t[i] = tau[i * U + u];
        }
        rc |= step_rk4_coupled_r(m, cp, x, t, dt_u ? dt_u[u] : dt, xn) != 0;
        for (int i = 0; i < n; ++i) {
            qn[i * U + u] = xn[i]; qdn[i * U + u] = xn[n + i]; fn[i * U + u] = xn[2 * n + i];
        }
    }
    return rc ? -3 : 0;
}

int mpcfo_step_rk4_coupled_jvp_batch(const mpcfo_model *m, const mpcfo_coupling *cp, long U, const double *q, const double *qd,
                                     const double *tau, const double *f, double dt, const double *dt_u, double *qn, double *qdn,
                                     double *fn, double *jac)
{
    CHECK_N(m);
    const int n = m->n, P = 4 * n + 1;
    const double hstep = 1e-40;
    int rc = 0;
#pragma omp parallel for schedule(static) reduction(| : rc)
    for (long u = 0; u < U; ++u) {
        double complex x[3 * MPCFO_MAXN], t[MPCFO_MAXN], xn[3 * MPCFO_MAXN], h;
        for (int d = 0; d < P; ++d) {
            for (int i = 0; i < n; ++i) {
                x[i] = q[i * U + u]; x[n + i] = qd[i * U + u]; x[2 * n + i] = f[i * U + u]; t[i] = tau[i * U + u];
            }
            h = dt_u ? dt_u[u] : dt;
            if (d < 2 * n) x[d] += hstep * I;
            else if (d < 3 * n) t[d - 2 * n] += hstep * I;
            else if (d < 4 * n) x[d - n] += hstep * I;
            else h += hstep * I;
            rc |= step_rk4_coupled_c(m, cp, x, t, h, xn) != 0;
            for (int r = 0; r < 3 * n; ++r) jac[((long)r * P + d) * U + u] = cimag(xn[r]) / hstep;
            if (d == 0 && qn)
                for (int i = 0; i < n; ++i) {
                    qn[i * U + u] = creal(xn[i]); qdn[i * U + u] = creal(xn[n + i]); fn[i * U + u] = creal(xn[2 * n + i]);
                }
        }
    }
    return rc ? -3 : 0;
}

int mpcfo_ocp_rows_batch(const mpcfo_model *m, const mpcfo_rows_opts *o, long B, int N, const double *q, const double *qd,
                         const double *F, const double *T, const double *q_last, const double *T_last, const double *rel_pos0,
                         const double *rel_ori0, double *rows, double *cost, double *kin_jac)
{
    CHECK_N(m);
    if (o->narm < 1 || o->narm > 2) return -2;
    const int n = m->n, narm = o->narm, kin = narm == 2 ? 26 : 3, nrows = kin + 3 * n, nd = n + 3 * narm;
    const long U = B * N;
    const double hstep = 1e-40;
#pragma omp parallel for schedule(static)
    for (long u = 0; u < U; ++u) {
        const long b = u % B;
        const int k = (int)(u / B);
        double ql[MPCFO_MAXN], qdl[MPCFO_MAXN], Tl[MPCFO_MAXN], qn[MPCFO_MAXN], Tn[MPCFO_MAXN], Fl[6], relprev[3] = {0, 0, 0}, ori0[3] = {0, 0, 0};
        double r[26 + 3 * MPCFO_MAXN], c;
        for (int i = 0; i < n; ++i) {
            ql[i] = q[i * U + u]; qdl[i] = qd[i * U + u]; Tl[i] = T ? T[i * U + u] : 0.0;
            qn[i] = k + 1 < N ? q[i * U + u + B] : (q_last ? q_last[i * B + b] : 0.0);
            Tn[i] = T ? (k + 1 < N ? T[i * U + u + B] : (T_last ? T_last[i * B + b] : 0.0)) : 0.0;
        }
        for (int i = 0; i < 3 * narm; ++i) Fl[i] = F[i * U + u];
        if (narm == 2) {
            if (k == 0) { for (int i = 0; i < 3; ++i) relprev[i] = rel_pos0 ? rel_pos0[i * B + b] : 0.0; }
            else {
                double qp[MPCFO_MAXN], pL[3], RL[9], pR[3], RR[9], dm[3];
                for (int i = 0; i < n; ++i) qp[i] = q[i * U + u - B];
                frame_fk_r(m, o->ee_frame[0], qp, pL, RL);
                frame_fk_r(m, o->ee_frame[1], qp, pR, RR);
                for (int i = 0; i < 3; ++i) dm[i] = pR[i] - pL[i];
                mtv_r(RL, dm, relprev);
            }
            for (int i = 0; i < 3; ++i) ori0[i] = rel_ori0 ? rel_ori0[i * B + b] : 0.0;
        }
        const int have_qn = k + 1 < N || q_last != NULL, have_Tn = T && (k + 1 < N || T_last != NULL);
        ocp_rows_r(m, o, ql, qdl, Fl, T ? Tl : NULL, have_qn ? qn : NULL, have_Tn ? Tn : NULL, relprev, ori0, r, &c);
        for (int i = 0; i < nrows; ++i) rows[i * U + u] = r[i];
        cost[u] = c;
        if (kin_jac) {
            double complex qc[MPCFO_MAXN], qdc[MPCFO_MAXN], Fc[6], rc[26 + 3 * MPCFO_MAXN], cc, rp[3] = {0, 0, 0};
            const double z3[3] = {0, 0, 0};
            for (int d = 0; d < nd; ++d) {
                for (int i = 0; i < n; ++i) { qc[i] = ql[i]; qdc[i] = qdl[i]; }
                for (int i = 0; i < 3 * narm; ++i) Fc[i] = Fl[i];
                if (d < n) qc[d] += hstep * I; else Fc[d - n] += hstep * I;
                ocp_rows_c(m, o, qc, qdc, Fc, NULL, NULL, NULL, rp, z3, rc, &cc);
                for (int i = 0; i < kin; ++i) kin_jac[((long)i * nd + d) * U + u] = cimag(rc[i]) / hstep;
            }
        }
    }
    return 0;
}

int mpcfo_fatigue_zoh_batch(const mpcfo_model *m, long U, const double *T, const double *tau, const double *qd,
                            double h, double *Tnext)
{
    CHECK_N(m);
    int n = m->n;
#pragma omp parallel for schedule(static)
    for (long u = 0; u < U; ++u)
        for (int i = 0; i < n; ++i)
            Tnext[i * U + u] = fatigue_zoh_r(m, i, T[i * U + u], tau[i * U + u], qd[i * U + u], h);
    return 0;
}

int mpcfo_fatigue_rhs_batch(const mpcfo_model *m, long U, const double *f, const double *tau, const double *qd,
                            double *fdot)
{
    CHECK_N(m);
    int n = m->n;
    for (long u = 0; u < U; ++u)
        for (int i = 0; i < n; ++i)
            fdot[i * U + u] = fatigue_rhs_r(m, i, f[i * U + u], tau[i * U + u], qd[i * U + u]);
    return 0;
}

/* Forward-dynamics derivatives at (q, qd, tau): A = d qdd/d q, B = d qdd/d qd (complex-step through aba_c),
 * C = M^-1 = d qdd/d tau.  Outputs are [n*n][U] planes, plane index row*n + col. */
int mpcfo_fd_derivs_batch(const mpcfo_model *m, long U, const double *q, const double *qd, const double *tau,
                          double *A, double *B, double *Cm)
{
    CHECK_N(m);
    const int n = m->n;
    const double hstep = 1e-40;
    int rc = 0;
#pragma omp parallel for schedule(static) reduction(| : rc)
    for (long u = 0; u < U; ++u) {
        double complex a[MPCFO_MAXN], b[MPCFO_MAXN], c[MPCFO_MAXN], t[MPCFO_MAXN];
        for (int d = 0; d < 3 * n; ++d) {
            for (int i = 0; i < n; ++i) { a[i] = q[i * U + u]; b[i] = qd[i * U + u]; c[i] = tau[i * U + u]; }
            if (d < n) a[d] += hstep * I;
            else if (d < 2 * n) b[d - n] += hstep * I;
            else c[d - 2 * n] += hstep * I;
            rc |= aba_c(m, a, b, c, t) != 0;
            double *out = d < n ? A : (d < 2 * n ? B : Cm);
            int col = d % n;
            for (int r = 0; r < n; ++r) out[((long)r * n + col) * U + u] = cimag(t[r]) / hstep;
        }
    }
    return rc ? -3 : 0;
}

/* Inverse-dynamics derivatives at (q, qd, qdd) by complex-step through rnea_c: Dq = d tau/d q, Dv = d tau/d qd,
 * M = d tau/d qdd; outputs [n*n][U], plane row*n + col. */
int mpcfo_rnea_derivs_batch(const mpcfo_model *m, long U, const double *q, const double *qd, const double *qdd,
                            double *Dq, double *Dv, double *M)
{
    CHECK_N(m);
    const int n = m->n;
    const double hstep = 1e-40;
#pragma omp parallel for schedule(static)
    for (long u = 0; u < U; ++u) {
        double complex a[MPCFO_MAXN], b[MPCFO_MAXN], c[MPCFO_MAXN], t[MPCFO_MAXN];
        for (int d = 0; d < 3 * n; ++d) {
            for (int i = 0; i < n; ++i) { a[i] = q[i * U + u]; b[i] = qd[i * U + u]; c[i] = qdd ? qdd[i * U + u] : 0.0; }
            if (d < n) a[d] += hstep * I;
            else if (d < 2 * n) b[d - n] += hstep * I;
            else c[d - 2 * n] += hstep * I;
            rnea_c(m, a, b, c, t);
            double *out = d < n ? Dq : (d < 2 * n ? Dv : M);
            int col = d % n;
            for (int r = 0; r < n; ++r) out[((long)r * n + col) * U + u] = cimag(t[r]) / hstep;
        }
    }
    return 0;
}

/* d tau/d q and d tau/d qd of the reference-mode torque tau = RNEA + wsign * sum J^T W, complex-step through node_eval_ref_c */
int mpcfo_node_eval_ref_jvp_batch(const mpcfo_model *m, int nee, const int *ee_frames, double wsign, long U, const double *q,
                                  const double *qd, const double *qdd, const double *W, double *Dq, double *Dv)
{
    CHECK_N(m);
    if (nee < 0 || nee > 8) return -2;
    const int n = m->n;
    const double hstep = 1e-40;
#pragma omp parallel for schedule(static)
    for (long u = 0; u < U; ++u) {
        double complex a[MPCFO_MAXN], b[MPCFO_MAXN], c[MPCFO_MAXN], Tl[MPCFO_MAXN], Wl[48], t[MPCFO_MAXN], qn[MPCFO_MAXN], Tn[MPCFO_MAXN];
        for (int d = 0; d < 2 * n; ++d) {
            for (int i = 0; i < n; ++i) { a[i] = q[i * U + u]; b[i] = qd[i * U + u]; c[i] = qdd ? qdd[i * U + u] : 0.0; Tl[i] = 0.0; }
            for (int k = 0; k < 6 * nee; ++k) Wl[k] = W[k * U + u];
            if (d < n) a[d] += hstep * I; else b[d - n] += hstep * I;
            node_eval_ref_c(m, nee, ee_frames, wsign, a, b, c, Wl, Tl, 0.0, t, qn, Tn);
            double *out = d < n ? Dq : Dv;
            for (int r = 0; r < n; ++r) out[((long)r * n + d % n) * U + u] = cimag(t[r]) / hstep;
        }
    }
    return 0;
}
