// kernels_basic.cu — RNEA, frame FK, frame Jacobian, reference-mode node evaluation, cost/residual reduction.
#include "frames.cuh"

namespace mpcf {

std::atomic<long> g_launches{0};
long launch_count() { return g_launches.load(); }

struct RneaBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, const double *q, const double *qd, const double *qdd, double *tau)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n();
        double a[MP::MAXN], b[MP::MAXN], c[MP::MAXN], t[MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            a[i] = q[i * U + u];
            b[i] = qd[i * U + u];
            c[i] = qdd ? qdd[i * U + u] : 0.0;
        }
        Dyn<double, MP>::rnea(m, a, b, c, t);
#pragma unroll UNR
        for (int i = 0; i < n; ++i) tau[i * U + u] = t[i];
    }
};

struct FkBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, FrameArg f, const double *q, double *pos, double *rot)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n();
        double a[MP::MAXN], oR[MP::MAXN][9], op[MP::MAXN][3], p[3], R[9];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) a[i] = q[i * U + u];
        Dyn<double, MP>::fk_all(m, a, oR, op);
        Dyn<double, MP>::frame_pose(f.joint, f.R, f.p, oR, op, p, R);
#pragma unroll
        for (int k = 0; k < 3; ++k) pos[k * U + u] = p[k];
#pragma unroll
        for (int k = 0; k < 9; ++k) rot[k * U + u] = R[k];
    }
};

struct JacBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, FrameArg f, const double *q, double *J)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n();
        double a[MP::MAXN], oR[MP::MAXN][9], op[MP::MAXN][3], p[3], R[9];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) a[i] = q[i * U + u];
        Dyn<double, MP>::fk_all(m, a, oR, op);
        Dyn<double, MP>::frame_pose(f.joint, f.R, f.p, oR, op, p, R);
        int cur = f.joint;
#pragma unroll UNR
        for (int i = n - 1; i >= 0; --i) {
            double col[6] = {0, 0, 0, 0, 0, 0};
            if (i == cur) {
                jac_column(m, i, oR, op, p, col);
                cur = m.parent(i);
            }
#pragma unroll
            for (int r = 0; r < 6; ++r) J[(long)(r * n + i) * U + u] = col[r];
        }
    }
};

// Reference-mode node evaluation, one launch:
//   tau = RNEA(q, qd, qdd) + wsign * sum_e J_e^T W_e ; qnext = q + h qd ; Tnext = ZOH(T; tau, qd, h)
// (python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:290-293,463 ; python/Centauro_script/mpc_principal.py:267-301)
// jtw_only: skip RNEA and the integrators and write only J^T W (mpcf_frame_jac_t_wrench_batch).
// Run-time trees carry the wrenches through the RNEA sweep (frames.cuh: WrenchExtTree).
struct NodeEvalBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, EeArgs ee, double wsign, const double *q, const double *qd,
                            const double *qdd, const double *W, const double *T, double h, ZohArg zoh, double *tau,
                            double *qnext, double *Tnext, bool jtw_only)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n();
        double a[MP::MAXN], b[MP::MAXN], c[MP::MAXN], t[MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            a[i] = q[i * U + u];
            b[i] = (!jtw_only && qd) ? qd[i * U + u] : 0.0;
            c[i] = (!jtw_only && qdd) ? qdd[i * U + u] : 0.0;
            t[i] = 0.0;
        }
        JointVar<double> jv[MP::MAXN];  // one sincos per joint, shared by the dynamics and the frame kinematics
        bool wrenches_done = false;
        if constexpr (!MP::kStatic) {
            if (!jtw_only) {  // run-time trees: the wrenches ride the RNEA sweep as external link forces
                WrenchExtTree<MP> ext;
                ext.nee = ee.nee;
                ext.wsign = wsign;
                for (int e = 0; e < ee.nee; ++e) {
                    ext.je[e] = ee.f[e].joint;  // -1 (world-fixed frame) never matches a link
#pragma unroll
                    for (int r = 0; r < 6; ++r) ext.Wl[e][r] = W[(long)(6 * e + r) * U + u];
#pragma unroll
                    for (int r = 0; r < 3; ++r) ext.pl[e][r] = ee.f[e].p[r];
                }
                Dyn<double, MP>::template rnea_impl<false>(m, a, jv, b, c, t, ext);
                wrenches_done = true;
            }
        }
        if (!wrenches_done) {
#pragma unroll UNR
            for (int i = 0; i < n; ++i) Dyn<double, MP>::joint_var(m, i, a[i], jv[i]);
            if (!jtw_only) Dyn<double, MP>::rnea_jv(m, jv, b, c, t);
        }
        if (ee.nee > 0 && !wrenches_done) {
            double oR[MP::MAXN][9], op[MP::MAXN][3];
            Dyn<double, MP>::fk_all_jv(m, jv, oR, op);
            for (int e = 0; e < ee.nee; ++e) {
                double pf[3], Rf[9], w[6];
                Dyn<double, MP>::frame_pose(ee.f[e].joint, ee.f[e].R, ee.f[e].p, oR, op, pf, Rf);
#pragma unroll
                for (int r = 0; r < 6; ++r) w[r] = W[(long)(6 * e + r) * U + u];
                int cur = ee.f[e].joint;
#pragma unroll UNR
                for (int i = n - 1; i >= 0; --i) {
                    if (i == cur) {
                        double col[6];
                        jac_column(m, i, oR, op, pf, col);
                        double acc = 0.0;
#pragma unroll
                        for (int r = 0; r < 6; ++r) acc += col[r] * w[r];
                        t[i] += wsign * acc;
                        cur = m.parent(i);
                    }
                }
            }
        }
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            tau[i * U + u] = t[i];
            if (jtw_only) continue;
            if (qnext) qnext[i * U + u] = a[i] + h * b[i];
            if (Tnext) {
                const double P = m.fat(i, 2) * t[i] * t[i] + m.fat(i, 3) * b[i] * b[i];
                const double Ti = T[i * U + u];
                const double lam = m.fat(i, 0);
                Tnext[i * U + u] = (lam == 0.0) ? Ti + h * m.fat(i, 1) * P : zoh.a[i] * Ti + (1.0 - zoh.a[i]) * (m.fat(i, 1) / lam) * P;
            }
        }
    }
};

// First derivatives of the reference-mode joint torque tau = RNEA(q, qd, qdd) + wsign * sum_e J_e^T W_e with respect to
// q and qd: one dual-number sweep per seed (blockIdx.y in [0, 2n)).  d tau/d W_e = wsign * J_e^T comes from the frame
// Jacobian kernel.  These are the Jacobian blocks of the torque-bound rows of the reference's OCPs
// (python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:134-148).
struct NodeEvalJvpBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, EeArgs ee, double wsign, const double *q, const double *qd,
                            const double *qdd, const double *W, double *dtau_dq, double *dtau_dqd)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        using D = Dyn<Dual, MP>;
        const int n = m.n();
        const int d = blockIdx.y;
        Dual a[MP::MAXN], b[MP::MAXN], c[MP::MAXN], t[MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            a[i] = Dual(q[i * U + u], d == i ? 1.0 : 0.0);
            b[i] = Dual(qd[i * U + u], d == n + i ? 1.0 : 0.0);
            c[i] = Dual(qdd ? qdd[i * U + u] : 0.0, 0.0);
        }
        JointVar<Dual> jv[MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) D::joint_var(m, i, a[i], jv[i]);
        D::rnea_jv(m, jv, b, c, t);
        if (ee.nee > 0 && d < n) {  // J^T W depends on q only
            Dual oR[MP::MAXN][9], op[MP::MAXN][3];
            D::fk_all_jv(m, jv, oR, op);
            for (int e = 0; e < ee.nee; ++e) {
                Dual pf[3], Rf[9];
                D::frame_pose(ee.f[e].joint, ee.f[e].R, ee.f[e].p, oR, op, pf, Rf);
                double w[6];
#pragma unroll
                for (int r = 0; r < 6; ++r) w[r] = W[(long)(6 * e + r) * U + u];
                int cur = ee.f[e].joint;
#pragma unroll UNR
                for (int i = n - 1; i >= 0; --i) {
                    if (i == cur) {
                        const Dual z[3] = {oR[i][2], oR[i][5], oR[i][8]};
                        Dual acc;
                        if (!m.prismatic(i)) {
                            const Dual dd[3] = {pf[0] - op[i][0], pf[1] - op[i][1], pf[2] - op[i][2]};
                            Dual lin[3];
                            cross3(z, dd, lin);
                            acc = lin[0] * w[0] + lin[1] * w[1] + lin[2] * w[2] + z[0] * w[3] + z[1] * w[4] + z[2] * w[5];
                        } else {
                            acc = z[0] * w[0] + z[1] * w[1] + z[2] * w[2];
                        }
                        t[i] += wsign * acc;
                        cur = m.parent(i);
                    }
                }
            }
        }
        double *out = d < n ? dtau_dq : dtau_dqd;
        const int col = d % n;
#pragma unroll UNR
        for (int r = 0; r < n; ++r) out[(size_t)(r * n + col) * U + u] = t[r].d;
    }
};

// ---------------------------------------------------------------------------------------------
// per-scenario cost / residual reduction: thread b walks the N nodes of scenario b (u = k*B + b,
// coalesced across b) and writes (cost, defect, torque-bound, fatigue-bound) into out[4][B]
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cost_residual_kernel(int n, long B, int N, const double *q, const double *qd, const double *f,
                                                          const double *tau, const double *qn, const double *qdn, const double *fn,
                                                          CostArgs c, double *out)
{
    const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const long U = B * N;
    double cost = 0.0, r0 = 0.0, r1 = 0.0, r2 = 0.0;
    for (int k = 0; k < N; ++k) {
        const long u = (long)k * B + b;
        const double bound = fmax(c.tau0 * exp(-c.alpha * k * c.dt), c.tau_floor);
        for (int i = 0; i < n; ++i) {
            const long o = (long)i * U + u;
            const double v = qd[o], t = tau[o];
            cost += c.w_qd * v * v + c.w_tau * t * t;
            r1 = fmax(r1, fabs(t) - bound);
            r2 = fmax(r2, fn[o] - c.f_max);
            if (k + 1 < N) {
                const long o1 = o + B;
                r0 = fmax(r0, fabs(qn[o] - q[o1]));
                r0 = fmax(r0, fabs(qdn[o] - qd[o1]));
                r0 = fmax(r0, fabs(fn[o] - f[o1]));
            }
        }
    }
    out[b] = cost;
    out[B + b] = r0;
    out[2 * B + b] = r1;
    out[3 * B + b] = r2;
}

// Same reduction with a per-node, per-joint bound table [N][n][2] = (lb, ub) instead of the closed-form F0 schedule, which
// covers all three torque-limit mechanisms of the reference: F0 decaying (force_optimization_pilz_6DOF.py:136-148: lb = -b_k,
// ub = b_k), F2 stepwise over segments of the horizon (both_robots_torque_limited_2_pilz.py:129-147, Box_Pilz_6DOF2.py:303-433)
// and F3 joint switch-off (Centauro_dynamics.py:327-348: |tau_i| <= C_i after the first third for the joints selected by S).
// The table (2 n N doubles) is staged in shared memory once per block.  resid[1] = max violation max(lb - tau, tau - ub, 0).
__global__ void __launch_bounds__(256) cost_residual_table_kernel(int n, long B, int N, const double *q, const double *qd, const double *f,
                                                                const double *tau, const double *qn, const double *qdn,
                                                                const double *fn, double w_qd, double w_tau, double f_max,
                                                                const double *__restrict__ table, double *out, long ld_out)
{
    extern __shared__ double tb[];
    for (int k = threadIdx.x; k < 2 * n * N; k += blockDim.x) tb[k] = table[k];
    __syncthreads();
    const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const long U = B * N;
    double cost = 0.0, r0 = 0.0, r1 = 0.0, r2 = 0.0;
    for (int k = 0; k < N; ++k) {
        const long u = (long)k * B + b;
        for (int i = 0; i < n; ++i) {
            const long o = (long)i * U + u;
            const double v = qd[o], t = tau[o];
            cost += w_qd * v * v + w_tau * t * t;
            r1 = fmax(r1, fmax(tb[2 * (k * n + i)] - t, t - tb[2 * (k * n + i) + 1]));
            r2 = fmax(r2, fn[o] - f_max);
            if (k + 1 < N) {
                const long o1 = o + B;
                r0 = fmax(r0, fabs(qn[o] - q[o1]));
                r0 = fmax(r0, fabs(qdn[o] - qd[o1]));
                r0 = fmax(r0, fabs(fn[o] - f[o1]));
            }
        }
    }
    out[b] = cost;
    out[ld_out + b] = r0;
    out[2 * ld_out + b] = r1;
    out[3 * ld_out + b] = r2;
}

cudaError_t launch_cost_residual_table(int n, long B, int N, const double *q, const double *qd, const double *f, const double *tau,
                                       const double *qn, const double *qdn, const double *fn, double w_qd, double w_tau, double f_max,
                                       const double *table, double *out, long ld_out, cudaStream_t s)
{
    if (B <= 0) return cudaSuccess;
    constexpr int kMaxSmem = 200 * 1024;
    const size_t smem = (size_t)2 * n * N * sizeof(double);
    if (smem > kMaxSmem) return cudaErrorInvalidValue;
    if (smem > 48 * 1024) {  // one limit for every table size: the largest accepted
        const cudaError_t e = raise_smem_limit<cost_residual_table_kernel>(kMaxSmem);
        if (e != cudaSuccess) return e;
    }
    cost_residual_table_kernel<<<(unsigned)((B + 255) / 256), 256, smem, s>>>(n, B, N, q, qd, f, tau, qn, qdn, fn, w_qd, w_tau, f_max, table, out,
                                                                            ld_out);
    g_launches.fetch_add(1);
    return cudaGetLastError();
}

// Packs selected planes of an SoA array into a contiguous staging buffer: dst[k][u] = src[map[k]][u].  The host-facing
// pipeline uses it so that everything a chunk sends back to the host (states + the structurally non-zero Jacobian planes)
// leaves the device in ONE large copy.  Pure HBM traffic (16-byte accesses when the plane length allows).
__global__ void __launch_bounds__(256) gather_planes_kernel(const double *__restrict__ src, double *__restrict__ dst,
                                                           const int *__restrict__ map, long U, long ld_src)
{
    const double *s = src + (size_t)map[blockIdx.y] * ld_src;
    double *d = dst + (size_t)blockIdx.y * U;
    const long stride = (long)gridDim.x * blockDim.x;
    if (((U | ld_src) & 1) == 0) {
        const double2 *s2 = reinterpret_cast<const double2 *>(s);
        double2 *d2 = reinterpret_cast<double2 *>(d);
        for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < U / 2; i += stride) __stcs(d2 + i, __ldcs(s2 + i));
    } else {
        for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < U; i += stride) d[i] = s[i];
    }
}

cudaError_t launch_gather_planes(const double *src, double *dst, const int *map, int nplanes, long U, long ld_src, cudaStream_t s)
{
    if (nplanes <= 0 || U <= 0) return cudaSuccess;
    long bx = (U / 2 + 255) / 256;
    if (bx > 148 * 4) bx = 148 * 4;
    if (bx < 1) bx = 1;
    gather_planes_kernel<<<dim3((unsigned)bx, (unsigned)nplanes), 256, 0, s>>>(src, dst, map, U, ld_src);
    g_launches.fetch_add(1);
    return cudaGetLastError();
}

// FP64 pipe probe: 8 independent DFMA chains per thread; the roofline denominator of bench.py
// (MEASURED_PEAKS.json carries no FP64 figure).  flops = blocks * threads * iters * 8 * 2.
__global__ void __launch_bounds__(256) fp64_probe_kernel(long iters, double *out)
{
    double x0 = threadIdx.x * 1e-3, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    const double a = 0.999999, b = 1e-7;
    for (long i = 0; i < iters; ++i) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    out[(long)blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}
cudaError_t launch_fp64_probe(long iters, int blocks, double *out, cudaStream_t s)
{
    fp64_probe_kernel<<<blocks, 256, 0, s>>>(iters, out);
    g_launches.fetch_add(1);
    return cudaGetLastError();
}

cudaError_t launch_rnea(const LaunchModel &m, long U, const double *q, const double *qd, const double *qdd, double *tau, cudaStream_t s)
{
    return dispatch<RneaBody>(m, U, 1, s, q, qd, qdd, tau);
}
// ---------------------------------------------------------------------------------------------
// Frame kinematics of ONE serial chain of a static family, register resident (no per-link pose arrays, no run-time
// indexing): the chain is walked link by link with the running world pose (R, o) and stops at the frame's joint fj
// (uniform over the launch).  q points at the chain's planes; c0 / ntot place the chain inside a forest's outputs.
// ---------------------------------------------------------------------------------------------
template <class MP>
MPCF_DI void chain_link_pose(const MP &m, int i, double c, double s, double *R, double *o)
{
    double Rl[9], Rn[9], on[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        Rl[3 * r + 0] = m.Rp(i, 3 * r) * c + m.Rp(i, 3 * r + 1) * s;
        Rl[3 * r + 1] = m.Rp(i, 3 * r + 1) * c - m.Rp(i, 3 * r) * s;
        Rl[3 * r + 2] = m.Rp(i, 3 * r + 2);
    }
    if (i == 0) {
#pragma unroll
        for (int k = 0; k < 9; ++k) Rn[k] = Rl[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) on[k] = m.pp(i, k);
    } else {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
            for (int cc = 0; cc < 3; ++cc) Rn[3 * r + cc] = R[3 * r] * Rl[cc] + R[3 * r + 1] * Rl[3 + cc] + R[3 * r + 2] * Rl[6 + cc];
            on[r] = o[r] + R[3 * r] * m.pp(i, 0) + R[3 * r + 1] * m.pp(i, 1) + R[3 * r + 2] * m.pp(i, 2);
        }
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = Rn[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) o[k] = on[k];
}

// ee_pos, ee_rot of a frame carried by chain joint f.joint (bridge.hpp:106-111)
template <int N>
__global__ void __launch_bounds__(kThreads) fk_chain_kernel(const __grid_constant__ StaticParams<N> P, long U, FrameArg f, const double *q,
                                                           double *pos, double *rot)
{
    const StaticModel<N, N> m{P};
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    double R[9], o[3];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        if (i > f.joint) break;
        double s, c;
        sincos(q[i * U + u], &s, &c);
        chain_link_pose(m, i, c, s, R, o);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        pos[r * U + u] = o[r] + R[3 * r] * f.p[0] + R[3 * r + 1] * f.p[1] + R[3 * r + 2] * f.p[2];
#pragma unroll
        for (int c = 0; c < 3; ++c) rot[(3 * r + c) * U + u] = R[3 * r] * f.R[c] + R[3 * r + 1] * f.R[3 + c] + R[3 * r + 2] * f.R[6 + c];
    }
}

// 6 x ntot LOCAL_WORLD_ALIGNED frame Jacobian (bridge.hpp:138-146): column c0 + i = [z_i x (p_f - o_i) ; z_i] for the chain
// joints up to the frame's, zero elsewhere (other chains of a forest included)
template <int N>
__global__ void __launch_bounds__(kThreads) jac_chain_kernel(const __grid_constant__ StaticParams<N> P, long U, FrameArg f, const double *q,
                                                            double *J, int ntot, int c0)
{
    const StaticModel<N, N> m{P};
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    double R[9], o[3], z[N][3], oj[N][3];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        if (i > f.joint) break;
        double s, c;
        sincos(q[i * U + u], &s, &c);
        chain_link_pose(m, i, c, s, R, o);
#pragma unroll
        for (int r = 0; r < 3; ++r) { z[i][r] = R[3 * r + 2]; oj[i][r] = o[r]; }
    }
    double pf[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) pf[r] = o[r] + R[3 * r] * f.p[0] + R[3 * r + 1] * f.p[1] + R[3 * r + 2] * f.p[2];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        double col[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        if (i <= f.joint) {
            const double d[3] = {pf[0] - oj[i][0], pf[1] - oj[i][1], pf[2] - oj[i][2]};
            cross3(z[i], d, col);
            col[3] = z[i][0]; col[4] = z[i][1]; col[5] = z[i][2];
        }
#pragma unroll
        for (int r = 0; r < 6; ++r) J[(long)(r * ntot + c0 + i) * U + u] = col[r];
    }
#pragma unroll 1
    for (int i = 0; i < ntot; ++i)
        if (i < c0 || i >= c0 + N)
#pragma unroll
            for (int r = 0; r < 6; ++r) J[(long)(r * ntot + i) * U + u] = 0.0;
}

// out = J^T W without materialising J (SURVEY.md §8 a3): the wrench, turned into the frame link's coordinates
// ([R^T F ; R^T n + p x R^T F]: rotation chain only), is carried down the chain like a link force of the RNEA's inward
// sweep and leaves its joint-axis component at every joint.  Rows of other chains are zero.
template <int N>
__global__ void __launch_bounds__(kThreads) jtw_chain_kernel(const __grid_constant__ StaticParams<N> P, long U, FrameArg f, const double *q,
                                                            const double *W, double *out, int ntot, int c0)
{
    const StaticModel<N, N> m{P};
    using D = Dyn<double, StaticModel<N, N>>;
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    JointVar<double> jv[N];
    double R[9], o[3];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        if (i > f.joint) break;
        sincos(q[i * U + u], &jv[i].s, &jv[i].c);
        chain_link_pose(m, i, jv[i].c, jv[i].s, R, o);
    }
    double w[6], fl[6], t[3];
#pragma unroll
    for (int r = 0; r < 6; ++r) w[r] = W[(long)r * U + u];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        fl[c] = R[c] * w[0] + R[3 + c] * w[1] + R[6 + c] * w[2];
        fl[3 + c] = R[c] * w[3] + R[3 + c] * w[4] + R[6 + c] * w[5];
    }
    cross3(f.p, fl, t);
#pragma unroll
    for (int c = 0; c < 3; ++c) fl[3 + c] += t[c];
#pragma unroll
    for (int i = N - 1; i >= 0; --i) {
        if (i > f.joint) {
            out[(long)(c0 + i) * U + u] = 0.0;
            continue;
        }
        out[(long)(c0 + i) * U + u] = fl[5];
        if (i > 0) {
            double fp[6];
            D::force_to_parent(m, i, jv[i], fl, fp);
#pragma unroll
            for (int r = 0; r < 6; ++r) fl[r] = fp[r];
        }
    }
#pragma unroll 1
    for (int i = 0; i < ntot; ++i)
        if (i < c0 || i >= c0 + N) out[(long)i * U + u] = 0.0;
}

// A frame on a chain of a static family goes to that chain's kernel (chain f.joint / L, joint index made chain-relative); a
// world-fixed frame (f.joint < 0) has a constant pose and takes the generic body.
cudaError_t launch_fk(const LaunchModel &m, const FrameArg &f, long U, const double *q, double *pos, double *rot, cudaStream_t s)
{
    if (U <= 0) return cudaSuccess;
    if (f.joint >= 0 && with_chains(m, [&](auto L, const auto *chains, auto) {
            FrameArg fc = f;
            fc.joint = f.joint % L;
            const int c0 = f.joint - fc.joint;
            fk_chain_kernel<L><<<(unsigned)((U + kThreads - 1) / kThreads), kThreads, 0, s>>>(chains[c0 / L], U, fc, q + (size_t)c0 * U, pos, rot);
            g_launches.fetch_add(1);
        }))
        return cudaGetLastError();
    return dispatch<FkBody>(m, U, 1, s, f, q, pos, rot);
}
cudaError_t launch_jac(const LaunchModel &m, const FrameArg &f, long U, const double *q, double *J, cudaStream_t s)
{
    if (U <= 0) return cudaSuccess;
    if (f.joint >= 0 && with_chains(m, [&](auto L, const auto *chains, auto) {
            FrameArg fc = f;
            fc.joint = f.joint % L;
            const int c0 = f.joint - fc.joint;
            jac_chain_kernel<L><<<(unsigned)((U + kThreads - 1) / kThreads), kThreads, 0, s>>>(chains[c0 / L], U, fc, q + (size_t)c0 * U, J, m.n, c0);
            g_launches.fetch_add(1);
        }))
        return cudaGetLastError();
    return dispatch<JacBody>(m, U, 1, s, f, q, J);
}
// Contact wrenches as external link forces of the RNEA (serial chain): W_e = [F ; n] is given in world axes at the frame
// point carried by chain joint je[e] (LOCAL_WORLD_ALIGNED, bridge.hpp:144), so in the coordinates of that link it is
// [R^T F ; R^T n + p x R^T F] with R the link's world orientation and p the frame's offset in the link — only the rotation
// chain is needed, and it advances inside the RNEA's own forward sweep.  tau = ID + wsign * sum_e J_e^T W_e.
template <int N, int NEE>
struct WrenchExt {
    double R[9];  // world orientation of the link the sweep is at
    int je[NEE > 0 ? NEE : 1];
    double Wl[NEE > 0 ? NEE : 1][6], pl[NEE > 0 ? NEE : 1][3];
    double wsign;
    MPCF_DI void link(const StaticModel<N, N> &m, int i, const JointVar<double> &jv, double *f)
    {
        if constexpr (NEE > 0) {
            double Rl[9], Rn[9];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                Rl[3 * r + 0] = m.Rp(i, 3 * r) * jv.c + m.Rp(i, 3 * r + 1) * jv.s;
                Rl[3 * r + 1] = m.Rp(i, 3 * r + 1) * jv.c - m.Rp(i, 3 * r) * jv.s;
                Rl[3 * r + 2] = m.Rp(i, 3 * r + 2);
            }
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    Rn[3 * r + c] = (i == 0) ? Rl[3 * r + c] : R[3 * r] * Rl[c] + R[3 * r + 1] * Rl[3 + c] + R[3 * r + 2] * Rl[6 + c];
#pragma unroll
            for (int k = 0; k < 9; ++k) R[k] = Rn[k];
#pragma unroll
            for (int e = 0; e < NEE; ++e)
                if (je[e] == i) {
                    double Fl[3], nl[3], t[3];
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        Fl[c] = R[c] * Wl[e][0] + R[3 + c] * Wl[e][1] + R[6 + c] * Wl[e][2];
                        nl[c] = R[c] * Wl[e][3] + R[3 + c] * Wl[e][4] + R[6 + c] * Wl[e][5];
                    }
                    cross3(pl[e], Fl, t);
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        f[c] += wsign * Fl[c];
                        f[3 + c] += wsign * (nl[c] + t[c]);
                    }
                }
        }
    }
};

// Reference-mode node for ONE serial chain of a static family (joints [c0, c0 + N) of the model; the pointers already address
// the chain's planes): tau = ID(q, qd, qdd) + wsign * sum_e J_e^T W_e, q+ = q + h qd, thermal ZOH — one RNEA sweep pair with
// the wrenches injected as external link forces (WrenchExt).  NEE = number of wrenches handled (ee.nee <= NEE).
template <int N, int NEE>
__global__ void __launch_bounds__(kThreads, 3) node_eval_chain_kernel(const __grid_constant__ StaticParams<N> P, long U, EeArgs ee, double wsign,
                                                                     const double *q, const double *qd, const double *qdd, const double *W,
                                                                     const double *T, double h, ZohArg zoh, double *tau, double *qnext,
                                                                     double *Tnext, int c0)
{
    const StaticModel<N, N> m{P};
    using D = Dyn<double, StaticModel<N, N>>;
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    double a[N], b[N], c[N], t[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        a[i] = q[i * U + u];
        b[i] = qd ? qd[i * U + u] : 0.0;
        c[i] = qdd ? qdd[i * U + u] : 0.0;
    }
    if (Tnext) {  // the temperatures are read after the dynamics: start their loads now (no registers held)
#pragma unroll
        for (int i = 0; i < N; ++i) asm volatile("prefetch.global.L1 [%0];" ::"l"(T + i * U + u));
    }
    WrenchExt<N, NEE> ext;
    ext.wsign = wsign;
#pragma unroll
    for (int e = 0; e < NEE; ++e) {
        const int j = e < ee.nee ? ee.f[e].joint - c0 : -1;
        ext.je[e] = (e < ee.nee && ee.f[e].joint >= 0 && j >= 0 && j < N) ? j : -1;  // world-fixed frame / other chain: no term
#pragma unroll
        for (int r = 0; r < 6; ++r) ext.Wl[e][r] = ext.je[e] >= 0 ? W[(long)(6 * e + r) * U + u] : 0.0;
#pragma unroll
        for (int r = 0; r < 3; ++r) ext.pl[e][r] = ee.f[e].p[r];
    }
    JointVar<double> jv[N];
    D::template rnea_impl<false>(m, a, jv, b, c, t, ext);
#pragma unroll
    for (int i = 0; i < N; ++i) {
        tau[i * U + u] = t[i];
        if (qnext) qnext[i * U + u] = a[i] + h * b[i];
        if (Tnext) {
            const double Pl = m.fat(i, 2) * t[i] * t[i] + m.fat(i, 3) * b[i] * b[i];
            const double Ti = T[i * U + u];
            const double lam = m.fat(i, 0), za = zoh.a[c0 + i];
            Tnext[i * U + u] = (lam == 0.0) ? Ti + h * m.fat(i, 1) * Pl : za * Ti + (1.0 - za) * (m.fat(i, 1) / lam) * Pl;
        }
    }
}

cudaError_t launch_node_eval(const LaunchModel &m, const EeArgs &ee, double wsign, long U, const double *q, const double *qd,
                             const double *qdd, const double *W, const double *T, double h, const ZohArg &zoh, double *tau,
                             double *qnext, double *Tnext, bool jtw_only, cudaStream_t s)
{
    if (U <= 0) return cudaSuccess;
    const unsigned gb = (unsigned)((U + kThreads - 1) / kThreads);
    const FrameArg &f = ee.f[0];
    if (jtw_only && ee.nee == 1 && wsign == 1.0 && f.joint >= 0 && with_chains(m, [&](auto L, const auto *chains, auto) {
            FrameArg fc = f;
            fc.joint = f.joint % L;
            const int c0 = f.joint - fc.joint;
            jtw_chain_kernel<L><<<gb, kThreads, 0, s>>>(chains[c0 / L], U, fc, q + (size_t)c0 * U, W, tau, m.n, c0);
            g_launches.fetch_add(1);
        }))
        return cudaGetLastError();
    if (!jtw_only && with_chains(m, [&](auto L, const auto *chains, auto nchains) {
            for (int c = 0; c < nchains; ++c) {
                const size_t off = (size_t)c * L * U;
                auto at = [off](auto *p) { return p ? p + off : p; };
                auto go = [&](auto kern) {
                    kern<<<gb, kThreads, 0, s>>>(chains[c], U, ee, wsign, q + off, at(qd), at(qdd), W, at(T), h, zoh, tau + off, at(qnext), at(Tnext), c * L);
                };
                if (ee.nee == 0) go(node_eval_chain_kernel<L, 0>);
                else if (ee.nee == 1) go(node_eval_chain_kernel<L, 1>);
                else if (ee.nee == 2) go(node_eval_chain_kernel<L, 2>);
                else go(node_eval_chain_kernel<L, MPCF_MAX_EE>);
                g_launches.fetch_add(1);
            }
        }))
        return cudaGetLastError();
    return dispatch<NodeEvalBody>(m, U, 1, s, ee, wsign, q, qd, qdd, W, T, h, zoh, tau, qnext, Tnext, jtw_only);
}
cudaError_t launch_node_eval_jvp_dual(const LaunchModel &m, const EeArgs &ee, double wsign, long U, const double *q, const double *qd,
                                 const double *qdd, const double *W, double *dtau_dq, double *dtau_dqd, cudaStream_t s)
{
    return dispatch_generic<NodeEvalJvpBody>(m, U, 2 * m.n, s, ee, wsign, q, qd, qdd, W, dtau_dq, dtau_dqd);
}
cudaError_t launch_cost_residual(int n, long B, int N, const double *q, const double *qd, const double *f, const double *tau,
                                 const double *qn, const double *qdn, const double *fn, const CostArgs &c, double *out,
                                 cudaStream_t s)
{
    if (B <= 0) return cudaSuccess;
    cost_residual_kernel<<<(unsigned)((B + 255) / 256), 256, 0, s>>>(n, B, N, q, qd, f, tau, qn, qdn, fn, c, out);
    g_launches.fetch_add(1);
    return cudaGetLastError();
}


}  // namespace mpcf
