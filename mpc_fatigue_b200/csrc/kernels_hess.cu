// kernels_hess.cu — second derivatives of the RK4 step by hyper-dual sweeps (DESIGN.md §4e).
//
// z = (q, qd, tau, f, dt), P = 4n + 1; lambda = (lq, lqd, lf); H = d2(lambda^T x+)/dz dz.  The swept directions are the 3n + 1 inputs
// d in D = (q, qd, tau, dt), numbered as the Jacobian's seeds (d < 3n: q, qd, tau; d = 3n: dt).  The fatigue inputs need no sweep:
// f+_i = amp(Lambda_i h) f_i + (terms free of f), so the only non-zero second derivatives involving f are
// H[f_i][dt] = lf_i Lambda_i amp'(Lambda_i h), amp'(z) = -1 + z - z^2/2 + z^3/6.
#include "launch.cuh"

namespace mpcf {

namespace {

MPCF_DI double amp_prime(double z) { return -1.0 + z * (1.0 - z * (0.5 - z * (1.0 / 6.0))); }

MPCF_DI double at(const double *p, long i) { return p ? p[i] : 0.0; }

// column of swept direction d in z
MPCF_DI long zcol(int d, int n) { return d < 3 * n ? d : 4 * n; }

// one hyper-dual step: direction a on the first tangent; on the second, direction b (b >= 0) or, for b < 0, the vector v of `h`
template <class MP>
MPCF_DI void sweep(const MP &m, long u, long U, const double *q, const double *qd, const double *tau, const double *f, double hv,
                   int a, int b, const HessArgs &h, HDual *xn)
{
    constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
    const int n = m.n();
    const bool vec = b < 0;
    HDual x[3 * MP::MAXN], t[MP::MAXN];
#pragma unroll UNR
    for (int i = 0; i < n; ++i) {
        const long k = i * U + u;
        x[i] = HDual(q[k], a == i ? 1.0 : 0.0, vec ? at(h.vq, k) : (b == i ? 1.0 : 0.0), 0.0);
        x[n + i] = HDual(qd[k], a == n + i ? 1.0 : 0.0, vec ? at(h.vqd, k) : (b == n + i ? 1.0 : 0.0), 0.0);
        x[2 * n + i] = HDual(f[k], 0.0, vec ? at(h.vf, k) : 0.0, 0.0);
        t[i] = HDual(tau[k], a == 2 * n + i ? 1.0 : 0.0, vec ? at(h.vtau, k) : (b == 2 * n + i ? 1.0 : 0.0), 0.0);
    }
    const HDual dt(hv, a == 3 * n ? 1.0 : 0.0, vec ? at(h.vdt, u) : (b == 3 * n ? 1.0 : 0.0), 0.0);
    Dyn<HDual, MP>::step_rk4(m, x, t, dt, xn);
}

// sum_r lambda_r x+_r.ab
template <class MP>
MPCF_DI double contract(const MP &m, long u, long U, const HessArgs &h, const HDual *xn)
{
    const int n = m.n();
    double s = 0.0;
    for (int r = 0; r < 3 * n; ++r) {
        const double *p = r < n ? h.lq : (r < 2 * n ? h.lqd : h.lf);
        if (p) s = fma(p[(r % n) * U + u], xn[r].ab, s);
    }
    return s;
}

}  // namespace

// Dense Hessian.  blockIdx.y = k < D(D+1)/2: the pair a <= b of swept directions (row-major over the upper triangle), written to
// both H[a][b] and H[b][a]; k = D(D+1)/2: the f rows and columns in closed form.
struct StepHessBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, const double *q, const double *qd, const double *tau, const double *f, double dt,
                            const double *dt_u, const HessArgs h)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n(), D = 3 * n + 1;
        const long P = 4 * n + 1;
        const int k = blockIdx.y;
        const double hv = dt_u ? dt_u[u] : dt;
        if (k == D * (D + 1) / 2) {
#pragma unroll UNR
            for (int i = 0; i < n; ++i) {
                const long fi = 3 * n + i;
                for (long c = 0; c < P; ++c) {
                    const double e = c == 4 * n ? at(h.lf, i * U + u) * m.fat(i, 0) * amp_prime(m.fat(i, 0) * hv) : 0.0;
                    h.H[(fi * P + c) * U + u] = e;
                    h.H[(c * P + fi) * U + u] = e;
                }
            }
            return;
        }
        // k -> (a, b): row a of the upper triangle starts at a D - a (a - 1) / 2
        int a = (int)((2.0 * D + 1.0 - sqrt((2.0 * D + 1.0) * (2.0 * D + 1.0) - 8.0 * k)) * 0.5);
        while (a > 0 && a * D - a * (a - 1) / 2 > k) --a;
        while ((a + 1) * D - (a + 1) * a / 2 <= k) ++a;
        const int b = a + (k - (a * D - a * (a - 1) / 2));
        HDual xn[3 * MP::MAXN];
        sweep(m, u, U, q, qd, tau, f, hv, a, b, h, xn);
        const double s = contract(m, u, U, h, xn);
        const long ca = zcol(a, n), cb = zcol(b, n);
        h.H[(ca * P + cb) * U + u] = s;
        h.H[(cb * P + ca) * U + u] = s;
    }
};

// Hessian-vector product.  blockIdx.y = a in D writes (H v)_a; the dt block also writes the f entries (H v)_f_i = lf_i Lambda_i
// amp'(Lambda_i h) vdt and skips its sweep when hdt is not requested; block 0 writes J v = x+.b when asked.
struct StepHvpBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, const double *q, const double *qd, const double *tau, const double *f, double dt,
                            const double *dt_u, const HessArgs h)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n();
        const int a = blockIdx.y;
        const double hv = dt_u ? dt_u[u] : dt;
        if (a == 3 * n) {
            const double vdt = at(h.vdt, u);
#pragma unroll UNR
            for (int i = 0; i < n; ++i)
                h.hf[i * U + u] = at(h.lf, i * U + u) * m.fat(i, 0) * amp_prime(m.fat(i, 0) * hv) * vdt;
            if (!h.hdt) return;
        }
        HDual xn[3 * MP::MAXN];
        sweep(m, u, U, q, qd, tau, f, hv, a, -1, h, xn);
        const double s = contract(m, u, U, h, xn);
        if (a < n) h.hq[a * U + u] = s;
        else if (a < 2 * n) h.hqd[(a - n) * U + u] = s;
        else if (a < 3 * n) h.htau[(a - 2 * n) * U + u] = s;
        else h.hdt[u] = s;
        if (a == 0 && h.jq) {
#pragma unroll UNR
            for (int i = 0; i < n; ++i) {
                h.jq[i * U + u] = xn[i].b;
                h.jqd[i * U + u] = xn[n + i].b;
                h.jf[i * U + u] = xn[2 * n + i].b;
            }
        }
    }
};

cudaError_t launch_step_hess(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, const double *f,
                             double dt, const double *dt_u, const HessArgs &h, cudaStream_t s)
{
    const int D = 3 * m.n + 1;
    return dispatch<StepHessBody>(m, U, D * (D + 1) / 2 + 1, s, q, qd, tau, f, dt, dt_u, h);
}

cudaError_t launch_step_hvp(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, const double *f,
                            double dt, const double *dt_u, const HessArgs &h, cudaStream_t s)
{
    return dispatch<StepHvpBody>(m, U, 3 * m.n + 1, s, q, qd, tau, f, dt, dt_u, h);
}

}  // namespace mpcf
