// kernels_ilqr.cu — closed-loop rollouts of the iLQR solver (DESIGN.md §4g): the line-search pass (one thread per (step length,
// scenario)) and the accept pass (one thread per scenario, trajectory and the Riccati inputs of the tracking cost written).
//
// Both bodies run the values-only RK4 step of RolloutBody with the state in registers, under the feedback law
//   tau_k = taubar_k + alpha k_k + K_k (x_k - xbar_k),   x_{k+1} = RK4(x_k, tau_k, dt),   x_0 = x0,
// and accumulate the tracking cost through the one node-cost function below, in the same order, so the two passes give the same
// bits for the same alpha.  alpha == 0 reads no gain: tau_k = taubar_k exactly.
#include "launch.cuh"

namespace mpcf {

namespace {

MPCF_DI double ld_or0(const double *p, long i) { return p ? __ldg(p + i) : 0.0; }
// (d)+ that keeps a NaN: NaN <= 0 is false
MPCF_DI double pos(double d) { return d <= 0.0 ? 0.0 : d; }

// Riccati inputs of one node, written when the pointers are set (all or none): unit u of planes with stride ld
struct NodeDerivs {
    double *gx, *gu, *wx, *wu;
    long u, ld;
};

// One node's term of the tracking cost (k < N: running, k == N: terminal, t unused).  x [3n], t [n]; unit ux of the x_ref planes
// (stride UX), ut of the tau_ref planes (stride U).  Every operation is an explicit round-to-nearest intrinsic, so the term has the
// same bits wherever the function is inlined.  With d.gx set: the gradient and the Gauss-Newton curvature of the term.
template <class MP>
MPCF_DI double node_cost(const TrackCost &c, int n, int k, int N, const double *x, const double *t, long ux, long UX, long ut, long U,
                         const NodeDerivs *d)
{
    constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
    const bool term = k == N;
    const double *w = term ? c.wN : c.wx;
    double s = 0.0;
#pragma unroll UNR
    for (int i = 0; i < 3 * n; ++i) {
        const double e = __dsub_rn(x[i], ld_or0(c.x_ref, (long)i * UX + ux));
        const double wi = ld_or0(w, i);
        s = __fma_rn(__dmul_rn(wi, e), e, s);
        double g = __dmul_rn(wi, e), h = wi;
        if (i >= 2 * n) {  // fatigue penalty
            const double p = pos(__dsub_rn(x[i], c.f_max));
            s = __fma_rn(__dmul_rn(c.rho_f, p), p, s);
            g = __fma_rn(c.rho_f, p, g);
            if (p > 0.0) h = __dadd_rn(h, c.rho_f);
        }
        if (d) {
            d->gx[(long)i * d->ld + d->u] = g;
            d->wx[(long)i * d->ld + d->u] = h;
        }
    }
    if (!term) {
#pragma unroll UNR
        for (int j = 0; j < n; ++j) {
            const double e = __dsub_rn(t[j], ld_or0(c.tau_ref, (long)j * U + ut));
            const double wj = ld_or0(c.wu, j);
            s = __fma_rn(__dmul_rn(wj, e), e, s);
            double g = __dmul_rn(wj, e), h = wj;
            if (c.bound) {
                const double *lu = c.bound + 2 * ((long)k * n + j);
                const double pl = pos(__dsub_rn(__ldg(lu), t[j])), pu = pos(__dsub_rn(t[j], __ldg(lu + 1)));
                s = __fma_rn(__dmul_rn(c.rho_tau, pl), pl, s);
                s = __fma_rn(__dmul_rn(c.rho_tau, pu), pu, s);
                g = __fma_rn(c.rho_tau, __dsub_rn(pu, pl), g);
                if (pl > 0.0 || pu > 0.0) h = __dadd_rn(h, c.rho_tau);
            }
            if (d) {
                d->gu[(long)j * d->ld + d->u] = g;
                d->wu[(long)j * d->ld + d->u] = h;
            }
        }
    }
    return __dmul_rn(0.5, s);
}

// tau_k of scenario b under the feedback law (alpha != 0: K and xbar are read); u = k B + b, a unit of both the [.][N B] planes and
// the xbar planes [3n][(N+1) B]
template <class MP>
MPCF_DI void feedback(int n, const IlqrArgs &a, double alpha, long u, const double *x, double *t)
{
    constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
    const long U = (long)a.N * a.B, UX = U + a.B;
    const int ldk = 3 * n + 1;
#pragma unroll UNR
    for (int j = 0; j < n; ++j) t[j] = __ldg(a.taubar + (long)j * U + u);
    if (alpha == 0.0) return;
    double dx[3 * MP::MAXN];
#pragma unroll UNR
    for (int i = 0; i < 3 * n; ++i) dx[i] = __dsub_rn(x[i], __ldg(a.xbar + (long)i * UX + u));
#pragma unroll UNR
    for (int j = 0; j < n; ++j) {
        const double *Kj = a.K + (long)j * ldk * U + u;
        double s = 0.0;
#pragma unroll UNR
        for (int i = 0; i < 3 * n; ++i) s = __fma_rn(__ldg(Kj + (long)i * U), dx[i], s);
        t[j] = __dadd_rn(__fma_rn(alpha, __ldg(Kj + (long)(3 * n) * U), t[j]), s);
    }
}

}  // namespace

// Line-search pass: thread (candidate c, scenario b) = c B + b; J [na][B]
struct IlqrCostsBody {
    static constexpr int kGenericMinBlocks = 3;
    template <class MP>
    static MPCF_DI void run(const MP &m, long tid, long, const IlqrArgs a)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n(), N = a.N;
        const long B = a.B, U = (long)N * B, UX = U + B;
        const long ci = tid / B, b = tid - ci * B;
        double alpha = 0.0;
#pragma unroll
        for (int i = 0; i < kIlqrMaxAlphas; ++i)
            if (i == ci) alpha = a.alphas[i];
        if (!a.K) alpha = 0.0;
        double x[3 * MP::MAXN], t[MP::MAXN], xn[3 * MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < 3 * n; ++i) x[i] = __ldg(a.x0 + (long)i * B + b);
        double J = 0.0;
#pragma unroll 1
        for (int k = 0; k < N; ++k) {
            const long u = (long)k * B + b;
            feedback<MP>(n, a, alpha, u, x, t);
            J = __dadd_rn(J, node_cost<MP>(a.cost, n, k, N, x, t, u, UX, u, U, nullptr));
            Dyn<double, MP>::step_rk4(m, x, t, a.dt, xn);
#pragma unroll UNR
            for (int i = 0; i < 3 * n; ++i) x[i] = xn[i];
        }
        J = __dadd_rn(J, node_cost<MP>(a.cost, n, N, N, x, t, U + b, UX, 0, U, nullptr));
        a.J[tid] = J;
    }
};

// Accept pass: thread = scenario; x [3n][(N+1) B], tau [n][N B], J [B] and, with a.gx set, the Riccati inputs of the cost
struct FeedbackRolloutBody {
    static constexpr int kGenericMinBlocks = 3;
    template <class MP>
    static MPCF_DI void run(const MP &m, long b, long B, const IlqrArgs a)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n(), N = a.N;
        const long U = (long)N * B, UX = U + B;
        const double alpha = a.K ? __ldg(a.alpha + b) : 0.0;
        double x[3 * MP::MAXN], t[MP::MAXN], xn[3 * MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < 3 * n; ++i) {
            x[i] = __ldg(a.x0 + (long)i * B + b);
            a.x[(long)i * UX + b] = x[i];
        }
        NodeDerivs d{a.gx, a.gu, a.wxo, a.wuo, 0, U};
        double J = 0.0;
#pragma unroll 1
        for (int k = 0; k < N; ++k) {
            const long u = (long)k * B + b;
            feedback<MP>(n, a, alpha, u, x, t);
#pragma unroll UNR
            for (int j = 0; j < n; ++j) a.tau[(long)j * U + u] = t[j];
            d.u = u;
            J = __dadd_rn(J, node_cost<MP>(a.cost, n, k, N, x, t, u, UX, u, U, a.gx ? &d : nullptr));
            Dyn<double, MP>::step_rk4(m, x, t, a.dt, xn);
#pragma unroll UNR
            for (int i = 0; i < 3 * n; ++i) {
                x[i] = xn[i];
                a.x[(long)i * UX + u + B] = x[i];
            }
        }
        NodeDerivs dN{a.gN, nullptr, a.wNo, nullptr, b, B};
        J = __dadd_rn(J, node_cost<MP>(a.cost, n, N, N, x, t, U + b, UX, 0, U, a.gx ? &dN : nullptr));
        a.J[b] = J;
    }
};

cudaError_t launch_ilqr_costs(const LaunchModel &m, const IlqrArgs &a, cudaStream_t s)
{
    return dispatch<IlqrCostsBody>(m, (long)a.na * a.B, 1, s, a);
}

cudaError_t launch_feedback_rollout(const LaunchModel &m, const IlqrArgs &a, cudaStream_t s)
{
    return dispatch<FeedbackRolloutBody>(m, a.B, 1, s, a);
}

}  // namespace mpcf
