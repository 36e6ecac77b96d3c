// kernels_jvp.cu — RK4 step with forward-mode Jacobians.
#include "launch.cuh"

namespace mpcf {

// Forward-mode Jacobian of the RK4 step.  blockIdx.y = seed direction d in [0, 3n]:
//   d < 2n : state seed (q, qd)   2n <= d < 3n : tau seed   d = 3n : dt seed
// The n fatigue columns need no sweep: d(q+, qd+)/df = 0 and df+/df = diag(1 - z + z^2/2 - z^3/6 + z^4/24),
// z = lambda dt (RK4 amplification of the linear compartment); the dt block writes them.
struct StepJvpBody {
    template <class MP>
    // cnt (the kernel wrapper's guard) units are evaluated; U is the plane stride of the input / state arrays, UJ of jac
    static MPCF_DI void run(const MP &m, long u, long /*cnt*/, long U, long UJ, const double *q, const double *qd, const double *tau,
                            const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn, double *jac)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        constexpr int UNR3 = MP::kStatic ? 3 * MP::MAXN : 1;
        const int n = m.n();
        const int d = blockIdx.y;
        const long P = 4 * n + 1;
        Dual x[3 * MP::MAXN], t[MP::MAXN], xn[3 * MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            x[i] = Dual(q[i * U + u], d == i ? 1.0 : 0.0);
            x[n + i] = Dual(qd[i * U + u], d == n + i ? 1.0 : 0.0);
            x[2 * n + i] = Dual(f[i * U + u], 0.0);
            t[i] = Dual(tau[i * U + u], d == 2 * n + i ? 1.0 : 0.0);
        }
        const double hv = dt_u ? dt_u[u] : dt;
        const Dual h(hv, d == 3 * n ? 1.0 : 0.0);
        Dyn<Dual, MP>::step_rk4(m, x, t, h, xn);
        const long col = d < 3 * n ? d : 4 * n;
#pragma unroll UNR3
        for (int r = 0; r < 3 * n; ++r) jac[((long)r * P + col) * UJ + u] = xn[r].d;
        if (d == 0 && qn) {
#pragma unroll UNR
            for (int i = 0; i < n; ++i) {
                qn[i * U + u] = xn[i].v;
                qdn[i * U + u] = xn[n + i].v;
                fn[i * U + u] = xn[2 * n + i].v;
            }
        }
        if (d == 3 * n) {
#pragma unroll UNR
            for (int j = 0; j < n; ++j) {
                const double z = m.fat(j, 0) * hv;
                const double g = 1.0 + z * (-1.0 + z * (0.5 + z * (-1.0 / 6.0 + z * (1.0 / 24.0))));
#pragma unroll UNR3
                for (int r = 0; r < 3 * n; ++r) jac[((long)r * P + 3 * n + j) * UJ + u] = (r == 2 * n + j) ? g : 0.0;
            }
        }
    }
};

// Vector-Jacobian product by the same sweeps: blockIdx.y = input direction d in [0, 3n] as above, and the block writes
// sum_r lambda_r d xn_r / d z_d (+ the addend for the state directions).  The fatigue inputs need no sweep: g_f,j = lambda_f,j
// amp(lambda_j h) (+ addend), written by the dt block, which skips its sweep when g_dt is not requested.  The path of run-time
// models with n > 40, as for the Jacobian.
struct StepVjpDualBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long /*cnt*/, long U, const double *q, const double *qd, const double *tau, const double *f,
                            double dt, const double *dt_u, const VjpArgs a, double *qn, double *qdn, double *fn)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n();
        const int d = blockIdx.y;
        const double hv = dt_u ? dt_u[u] : dt;
        auto lam = [&](int r) {
            const double *p = r < n ? a.lq : (r < 2 * n ? a.lqd : a.lf);
            return p ? p[(r % n) * a.ldl + u] : 0.0;
        };
        if (d == 3 * n) {
#pragma unroll UNR
            for (int j = 0; j < n; ++j) {
                const double z = m.fat(j, 0) * hv;
                const double g = 1.0 + z * (-1.0 + z * (0.5 + z * (-1.0 / 6.0 + z * (1.0 / 24.0))));
                a.gf[j * a.ldg + u] = fma(lam(2 * n + j), g, a.af ? a.af[j * a.lda + u] : 0.0);
            }
            if (!a.gdt) return;
        }
        Dual x[3 * MP::MAXN], t[MP::MAXN], xn[3 * MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            x[i] = Dual(q[i * U + u], d == i ? 1.0 : 0.0);
            x[n + i] = Dual(qd[i * U + u], d == n + i ? 1.0 : 0.0);
            x[2 * n + i] = Dual(f[i * U + u], 0.0);
            t[i] = Dual(tau[i * U + u], d == 2 * n + i ? 1.0 : 0.0);
        }
        const Dual h(hv, d == 3 * n ? 1.0 : 0.0);
        Dyn<Dual, MP>::step_rk4(m, x, t, h, xn);
        double g = 0.0;
        for (int r = 0; r < 3 * n; ++r) g = fma(lam(r), xn[r].d, g);
        if (d < n) a.gq[d * a.ldg + u] = g + (a.aq ? a.aq[d * a.lda + u] : 0.0);
        else if (d < 2 * n) a.gqd[(d - n) * a.ldg + u] = g + (a.aqd ? a.aqd[(d - n) * a.lda + u] : 0.0);
        else if (d < 3 * n) a.gtau[(d - 2 * n) * a.ldgt + u] = g;
        else a.gdt[u] = g;
        if (d == 0 && qn) {
#pragma unroll UNR
            for (int i = 0; i < n; ++i) {
                qn[i * U + u] = xn[i].v;
                qdn[i * U + u] = xn[n + i].v;
                fn[i * U + u] = xn[2 * n + i].v;
            }
        }
    }
};

cudaError_t launch_step_vjp_dual(const LaunchModel &m, long U, long cnt, const double *q, const double *qd, const double *tau, const double *f,
                                 double dt, const double *dt_u, const VjpArgs &a, double *qn, double *qdn, double *fn, cudaStream_t s)
{
    return dispatch_generic<StepVjpDualBody>(m, cnt, 3 * m.n + 1, s, U, q, qd, tau, f, dt, dt_u, a, qn, qdn, fn);
}

cudaError_t launch_step_jvp(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, const double *f,
                            double dt, const double *dt_u, double *qn, double *qdn, double *fn, double *jac, cudaStream_t s, long cnt, long UJ)
{
    if (cnt < 0) cnt = U;
    if (UJ <= 0) UJ = U;
    return dispatch<StepJvpBody>(m, cnt, 3 * m.n + 1, s, U, UJ, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac);
}

}  // namespace mpcf
