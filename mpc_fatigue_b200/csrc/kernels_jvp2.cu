// kernels_jvp2.cu — analytic Jacobian pipeline of the RK4 dynamics+fatigue step for static chain families
// (chain3 / chain6 / chain7; forests of two such chains run the pipeline once per chain).  Three kernels per chunk of
// units, staged through a caller-provided workspace (all planes SoA `[row][chunk]`, coalesced):
//
//   K1 step_stages   thread = unit            primal RK4 (forward dynamics through M = L D L^T) -> x+, and per stage
//                                             (q_s, qd_s, qdd_s, fdot_s) and C_s = M^-1                      -> workspace
//   K2 stage_derivs  thread = (unit, stage)   A_s = dqdd/dq = -C dID/dq, B_s = dqdd/dqd = -C dID/dqd, column by column as
//                                             the backward pass completes them (derivs.cuh: run_cols)        -> workspace
//   K3 chain_rule    warp = (32 units, column) forward accumulation of d x+/d (q, qd, tau, dt) through the four stages.
//                    Persistent CTAs; one producer thread streams each (tile, stage) chunk of the workspace into a
//                    shared-memory ring with cp.async.bulk (TMA) + mbarriers; consumer warps read A_s/B_s/C_s from
//                    shared memory with conflict-free LDS.64 (lane = unit).
//
// Workspace layout (AoSoA, tile = 32 units): tile t, stage s -> one contiguous chunk of (3 n^2 + 4 n) planes x 32
// doubles: first the A, B, C planes (row*n + col), then q_s, qd_s, qdd_s, fdot_s.  Every plane offset inside a chunk is
// a compile-time constant, so loads/stores carry immediates, and a chunk is a single bulk copy.
//
// Cost per unit drops from 19 dual-number sweeps of RK4(ABA) (v1, kernels_jvp.cu) to one primal sweep, four
// derivative evaluations and 19 cheap column recursions.  Generic (run-time tree) models keep the v1 kernel.
#include <atomic>
#include <cstdlib>
#include <mutex>
#include <vector>

#include "derivs.cuh"
#include "launch.cuh"

namespace mpcf {

template <int N>
struct WsLayout {
    static constexpr int kTile = 32;
    static constexpr int kPlanes2 = 3 * N * N;                       // A, B, C
    static constexpr int kPlanes1 = 4 * N;                           // qd_s, qdd_s, fdot_s, q_s
    // plane offsets inside the stage-state block; q_s comes last: the chain-rule kernel does not use it and leaves it out
    // of its bulk copies
    static constexpr int kQd = 0, kQdd = N, kFd = 2 * N, kQ = 3 * N;
    static constexpr int kStageDoubles = (kPlanes2 + kPlanes1) * kTile;
    static constexpr unsigned kStageBytes = kStageDoubles * sizeof(double);
    static constexpr int kRingDoubles = (kPlanes2 + 3 * N) * kTile;  // what one ring slot of the chain-rule kernel holds
    static constexpr unsigned kRingBytes = kRingDoubles * sizeof(double);
    static constexpr int kUnitDoubles = 4 * (kPlanes2 + kPlanes1);
    // chunk of (tile, stage)
    static MPCF_DI size_t chunk(long tile, int s) { return ((size_t)tile * 4 + s) * kStageDoubles; }
};

// ------------------------------------------------------------------------------------------------ K1
template <int N, int L>
__global__ void __launch_bounds__(kThreads) k_step_stages(const __grid_constant__ StaticParams<N> P, long U, long u0, long cnt,
                                                         const double *q, const double *qd, const double *tau, const double *theat,
                                                         long UT, const double *f, double dt, const double *dt_u, double *qn, double *qdn,
                                                         double *fn, double *ws)
{
    // theat: the torque that heats the windings (fatigue right-hand side); equals tau unless the model couples the arms'
    // fatigue through a shared load (kernels_couple.cu), in which case the dynamics still see tau
    static_assert(N == L, "the pipeline runs one serial chain at a time (forests: one launch per chain)");
    const StaticModel<N, L> m{P};
    using D = Dyn<double, StaticModel<N, L>>;
    using W = WsLayout<N>;
    const long lu = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (lu >= cnt) return;
    const long u = u0 + lu;
    double x[3 * N], t[N], th[N], xs[3 * N], xn[3 * N], k[3 * N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        x[i] = q[i * U + u];
        x[N + i] = qd[i * U + u];
        x[2 * N + i] = f[i * U + u];
        t[i] = tau[i * U + u];
        th[i] = theat[i * UT + u];
    }
    const double h = dt_u ? dt_u[u] : dt;
#pragma unroll
    for (int i = 0; i < 3 * N; ++i) { xs[i] = x[i]; xn[i] = x[i]; }
#pragma unroll 1
    for (int s = 0; s < 4; ++s) {
        const double cs = s < 2 ? 0.5 : (s == 2 ? 1.0 : 0.0);
        const double wt = (s == 0 || s == 3) ? 1.0 / 6.0 : 1.0 / 3.0;
        double *w = ws + W::chunk(lu / 32, s) + W::kPlanes2 * 32 + (lu & 31);
        {   // forward dynamics through M; C = M^-1 goes straight to the stage chunk (K2 reads it, K3 consumes it)
            double Cs[N * (N + 1) / 2];
            D::template fd_crba<L, true>(m, xs, xs + N, t, k + N, Cs);
#pragma unroll
            for (int i = 0; i < N; ++i) {
                k[i] = xs[N + i];
                k[2 * N + i] = D::fatigue_rhs(m, i, xs[2 * N + i], th[i], xs[N + i]);
            }
            double *c = ws + W::chunk(lu / 32, s) + 2 * N * N * 32 + (lu & 31);
#pragma unroll
            for (int r = 0; r < N; ++r)
#pragma unroll
                for (int cc = 0; cc < N; ++cc) __stcs(c + (r * N + cc) * 32, Cs[r >= cc ? r * (r + 1) / 2 + cc : cc * (cc + 1) / 2 + r]);
        }
#pragma unroll
        for (int i = 0; i < N; ++i) {
            __stcs(w + (W::kQ + i) * 32, xs[i]);
            __stcs(w + (W::kQd + i) * 32, xs[N + i]);
            __stcs(w + (W::kQdd + i) * 32, k[N + i]);
            __stcs(w + (W::kFd + i) * 32, k[2 * N + i]);
        }
        const double a = h * wt, c = h * cs;
#pragma unroll
        for (int i = 0; i < 3 * N; ++i) {
            xn[i] += a * k[i];
            xs[i] = x[i] + c * k[i];
        }
    }
    if (qn) {
#pragma unroll
        for (int i = 0; i < N; ++i) {
            qn[i * U + u] = xn[i];
            qdn[i * U + u] = xn[N + i];
            fn[i * U + u] = xn[2 * N + i];
        }
    }
}

// ------------------------------------------------------------------------------------------------ K2
constexpr int kSmCountHint = 148;  // B200; only tunes how far ahead k_stage_derivs prefetches
MPCF_DI void cp_async8(double *smem, const double *gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
// where k_stage_derivs finds C = M^-1 (lower triangle): its own column of the shared-memory slab, or the stage chunk
struct CFromShared {
    double *base;
    int stride;
    MPCF_DI void ready() const { asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory"); }
    MPCF_DI double operator()(int r, int c) const { return base[(r * (r + 1) / 2 + c) * stride]; }
};
template <int N>
struct CFromGlobal {
    const double *o;
    MPCF_DI void ready() const {}
    MPCF_DI double operator()(int r, int c) const { return o[(2 * N * N + r * N + c) * 32]; }
};

// C held by the caller (a lambda over its register array)
template <class F>
struct CFromRegisters {
    F f;
    MPCF_DI void ready() const {}
    MPCF_DI double operator()(int r, int c) const { return f(r, c); }
};

template <int N, int L, bool KSMEM>
__global__ void __launch_bounds__(kThreads) k_stage_derivs(const __grid_constant__ StaticParams<N> P, long cnt, double *ws)
{
    const StaticModel<N, L> m{P};
    using W = WsLayout<N>;
    const long lu = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (lu >= cnt) return;
    const int s = blockIdx.y;
    double *o = ws + W::chunk(lu / 32, s) + (lu & 31);
    const double *w = o + W::kPlanes2 * 32;
    double q[N], qd[N], qdd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        q[i] = __ldcs(w + (W::kQ + i) * 32);
        qd[i] = __ldcs(w + (W::kQd + i) * 32);
        qdd[i] = __ldcs(w + (W::kQdd + i) * 32);
    }
    {   // pull the inputs of the block that is dispatched one wave of resident blocks later (blocks are dispatched in
        // linear order, two per SM) into L2: its first loads then cost an L2 hit instead of a DRAM round trip
        const long lin = (long)blockIdx.y * gridDim.x + blockIdx.x + 2 * kSmCountHint;
        if (lin < 4l * gridDim.x) {
            const long lu2 = (lin % gridDim.x) * blockDim.x + threadIdx.x;
            if (lu2 < cnt) {
                const double *o2 = ws + W::chunk(lu2 / 32, (int)(lin / gridDim.x)) + (lu2 & 31);
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(o2 + (W::kPlanes2 + W::kQ + i) * 32));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(o2 + (W::kPlanes2 + W::kQd + i) * 32));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(o2 + (W::kPlanes2 + W::kQdd + i) * 32));
                }
#pragma unroll
                for (int r = 0; r < N; ++r)
#pragma unroll
                    for (int c = 0; c <= r; ++c) asm volatile("prefetch.global.L2 [%0];" ::"l"(o2 + (2 * N * N + r * N + c) * 32));
            }
        }
    }
    // streaming stores: the workspace is consumed once by the next kernel; keep L2 for this kernel's spill lines
    auto emit = [&](int mat, int r, int c, double v) { __stcs(o + (mat * N * N + r * N + c) * 32, v); };
    // M^-1 of this stage was written by k_step_stages
    if (KSMEM) {
        // slab: (S, xi, eta) of links 0 .. N-2, then the lower triangle of C, copied asynchronously (no registers, its
        // DRAM latency hides under the forward pass); every thread touches only its own column of the slab
        extern __shared__ double k2_slab[];
        SharedLinkStore ks{k2_slab + threadIdx.x, (int)blockDim.x};
        CFromShared Cs{k2_slab + 18 * (N - 1) * blockDim.x + threadIdx.x, (int)blockDim.x};
#pragma unroll
        for (int r = 0; r < N; ++r)
#pragma unroll
            for (int c = 0; c <= r; ++c) cp_async8(Cs.base + (r * (r + 1) / 2 + c) * Cs.stride, o + (2 * N * N + r * N + c) * 32);
        FdDerivs<StaticModel<N, L>, L>::run_cols(m, q, qd, qdd, Cs, emit, ks);
    } else {
        LocalLinkStore<N> ks;
        CFromGlobal<N> Cs{o};
        FdDerivs<StaticModel<N, L>, L>::run_cols(m, q, qd, qdd, Cs, emit, ks);
    }
}

// public fd-derivs entry for static families, one serial chain per launch (joints [c0, c0 + N) of an ntot-joint forest; q, qd,
// tau point at the chain's planes): forward dynamics through M = L D L^T, which also yields C = M^-1, then the
// column-streamed derivative pass (run_cols) with C in registers.  Entries between different chains are written as 0.
template <int N>
__global__ void __launch_bounds__(kThreads) k_fd_derivs(const __grid_constant__ StaticParams<N> P, long U, const double *q, const double *qd,
                                                       const double *tau, double *Ao, double *Bo, double *Co, int ntot, int c0)
{
    const StaticModel<N, N> m{P};
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    double a[N], b[N], c[N], qdd[N], Cv[N * (N + 1) / 2];
#pragma unroll
    for (int i = 0; i < N; ++i) { a[i] = q[i * U + u]; b[i] = qd[i * U + u]; c[i] = tau[i * U + u]; }
    Dyn<double, StaticModel<N, N>>::template fd_crba<N, true>(m, a, b, c, qdd, Cv);
    auto at = [&](int r, int cc) { return (size_t)((c0 + r) * ntot + c0 + cc) * U + u; };
#pragma unroll
    for (int r = 0; r < N; ++r)
#pragma unroll
        for (int cc = 0; cc < N; ++cc) Co[at(r, cc)] = Cv[r >= cc ? r * (r + 1) / 2 + cc : cc * (cc + 1) / 2 + r];
    auto cget = [&](int r, int cc) { return Cv[r * (r + 1) / 2 + cc]; };
    CFromRegisters<decltype(cget)> Cs{cget};
    auto emit = [&](int mat, int r, int cc, double v) { (mat == 0 ? Ao : Bo)[at(r, cc)] = v; };
    extern __shared__ double link_slab[];
    SharedLinkStore ks{link_slab + threadIdx.x, (int)blockDim.x};
    FdDerivs<StaticModel<N, N>, N>::run_cols(m, a, b, qdd, Cs, emit, ks);
#pragma unroll 1
    for (int r = 0; r < N; ++r)
#pragma unroll 1
        for (int cc = 0; cc < ntot; ++cc)
            if (cc < c0 || cc >= c0 + N) {
                const size_t k = (size_t)((c0 + r) * ntot + cc) * U + u;
                Ao[k] = 0.0; Bo[k] = 0.0; Co[k] = 0.0;
            }
}

// inverse-dynamics derivatives for static families, one serial chain per launch (joints [c0, c0 + N) of an ntot-joint
// forest): dtau/dq, dtau/dqd, M at (q, qd, qdd), streamed entry by entry (run_id_stream); thread = unit
template <int N>
__global__ void __launch_bounds__(kThreads) k_rnea_derivs(const __grid_constant__ StaticParams<N> P, long U, const double *q, const double *qd,
                                                         const double *qdd, double *Dq, double *Dv, double *Mo, int ntot, int c0)
{
    const StaticModel<N, N> m{P};
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    double a[N], b[N], c[N];
#pragma unroll
    for (int i = 0; i < N; ++i) { a[i] = q[i * U + u]; b[i] = qd[i * U + u]; c[i] = qdd ? qdd[i * U + u] : 0.0; }
    extern __shared__ double link_slab[];
    SharedLinkStore ks{link_slab + threadIdx.x, (int)blockDim.x};
    struct Hooks {
        double *Dq, *Dv, *Mo;
        long U, u;
        int ntot, c0;
        MPCF_DI size_t at(int r, int cc) const { return (size_t)((c0 + r) * ntot + c0 + cc) * U + u; }
        MPCF_DI void link(int, const double *, const double *) const {}
        MPCF_DI void pair(int k, int j, const LinkFwd &, const LinkFwd &, double dqkj, double dqjk, double dvkj, double dvjk, double mkj) const
        {
            Dq[at(k, j)] = dqkj;
            Dv[at(k, j)] = dvkj;
            Mo[at(k, j)] = mkj;
            if (j < k) {
                Dq[at(j, k)] = dqjk;
                Dv[at(j, k)] = dvjk;
                Mo[at(j, k)] = mkj;
            }
        }
    } hooks{Dq, Dv, Mo, U, u, ntot, c0};
    FdDerivs<StaticModel<N, N>, N>::run_id_stream(m, a, b, c, hooks, ks);
#pragma unroll 1
    for (int r = 0; r < N; ++r)
#pragma unroll 1
        for (int cc = 0; cc < ntot; ++cc)  // entries between different chains are structurally zero
            if (cc < c0 || cc >= c0 + N) {
                const size_t k = (size_t)((c0 + r) * ntot + cc) * U + u;
                Dq[k] = 0.0; Dv[k] = 0.0; Mo[k] = 0.0;
            }
}

// Reference-mode torque rows tau = ID(q, qd, qdd) + wsign * sum_e J_e^T W_e (force_optimization_pilz_6DOF.py:134,
// Box_Pilz_6DOF2.py:292-293, mpc_principal.py:269), first derivatives w.r.t. q and qd, analytic, thread = unit.
// ID part: the world-frame pairing pass of derivs.cuh.  External part: with S_i = [o_i x z_i ; z_i] and the wrench moved to the
// world origin, Wo = [F ; n + p_f x F] (F, n fixed in world axes, p_f attached to the frame's link),
//   J_e^T W |_i = S_i . Wo,    d/dq_j = [j < i] (S_j x S_i) . Wo + ang(S_i) . ((lin(S_j) + ang(S_j) x p_f) x F),   i, j on the path to e
template <int N, int NEE>
struct NodeEvalJvpHooks {
    static constexpr int NE = NEE > 0 ? NEE : 1;
    // one serial chain = joints [c0, c0 + N) of an ntot-joint forest; wrench e acts on the frame carried by chain joint je[e]
    // (-1: not on this chain) at the world point pf[e]; Wo[e] = [F ; n + pf x F] is the wrench moved to the world origin
    double *Dq, *Dv;
    long U, u;
    int ntot, c0;
    double wsign;
    int je[NE];
    double pl[NE][3], pf[NE][3], Wo[NE][6];
    MPCF_DI void link(int i, const double *R, const double *o)
    {
#pragma unroll
        for (int e = 0; e < NEE; ++e)
            if (je[e] == i) {
#pragma unroll
                for (int r = 0; r < 3; ++r) pf[e][r] = o[r] + R[3 * r] * pl[e][0] + R[3 * r + 1] * pl[e][1] + R[3 * r + 2] * pl[e][2];
                double t[3];
                cross3(pf[e], Wo[e], t);  // Wo[3..5] held the moment n so far
#pragma unroll
                for (int r = 0; r < 3; ++r) Wo[e][3 + r] += t[r];
            }
    }
    // h_j = (lin(S_j) + ang(S_j) x pf) x F
    MPCF_DI void hvec(const LinkFwd &Kj, int e, double *h) const
    {
        double t[3], dp[3];
        cross3(Kj.S + 3, pf[e], t);
#pragma unroll
        for (int r = 0; r < 3; ++r) dp[r] = Kj.S[r] + t[r];
        cross3(dp, Wo[e], h);
    }
    MPCF_DI void pair(int k, int j, const LinkFwd &Kk, const LinkFwd &Kj, double dqkj, double dqjk, double dvkj, double dvjk, double) const
    {
#pragma unroll
        for (int e = 0; e < NEE; ++e)
            if (k <= je[e]) {  // both joints carry the frame (j <= k)
                double hj[3];
                hvec(Kj, e, hj);
                double vkj = dot3(Kk.S + 3, hj);
                if (j < k) {
                    double x[6], hk[3];
                    mxm(Kj.S, Kk.S, x);
                    vkj += dot6(x, Wo[e]);
                    hvec(Kk, e, hk);
                    dqjk += wsign * dot3(Kj.S + 3, hk);
                }
                dqkj += wsign * vkj;
            }
        Dq[(size_t)((c0 + k) * ntot + c0 + j) * U + u] = dqkj;
        Dv[(size_t)((c0 + k) * ntot + c0 + j) * U + u] = dvkj;
        if (j < k) {
            Dq[(size_t)((c0 + j) * ntot + c0 + k) * U + u] = dqjk;
            Dv[(size_t)((c0 + j) * ntot + c0 + k) * U + u] = dvjk;
        }
    }
};

template <int N, int NEE>
__global__ void __launch_bounds__(kThreads) k_node_eval_jvp(const __grid_constant__ StaticParams<N> P, long U, EeArgs ee, double wsign,
                                                           const double *q, const double *qd, const double *qdd, const double *W,
                                                           double *Dq, double *Dv, int ntot, int c0)
{
    // one serial chain of N joints = joints [c0, c0 + N) of an ntot-joint forest (q, qd, qdd already point at the chain's planes)
    const StaticModel<N, N> m{P};
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    double a[N], b[N], c[N];
#pragma unroll
    for (int i = 0; i < N; ++i) { a[i] = q[i * U + u]; b[i] = qd[i * U + u]; c[i] = qdd ? qdd[i * U + u] : 0.0; }
    // NEE = number of wrenches the instantiation handles (ee.nee <= NEE; missing ones are inert)
    NodeEvalJvpHooks<N, NEE> hooks;
    hooks.Dq = Dq; hooks.Dv = Dv; hooks.U = U; hooks.u = u; hooks.ntot = ntot; hooks.c0 = c0; hooks.wsign = wsign;
#pragma unroll
    for (int e = 0; e < NEE; ++e) {
        const int j = e < ee.nee ? ee.f[e].joint - c0 : -1;
        hooks.je[e] = (e < ee.nee && ee.f[e].joint >= 0 && j >= 0 && j < N) ? j : -1;  // world-fixed frames / other chains: no term
#pragma unroll
        for (int r = 0; r < 3; ++r) { hooks.pl[e][r] = ee.f[e].p[r]; hooks.pf[e][r] = 0.0; }
#pragma unroll
        for (int r = 0; r < 6; ++r) hooks.Wo[e][r] = (hooks.je[e] >= 0) ? W[(long)(6 * e + r) * U + u] : 0.0;
    }
    extern __shared__ double link_slab[];
    SharedLinkStore ks{link_slab + threadIdx.x, (int)blockDim.x};
    FdDerivs<StaticModel<N, N>, N>::run_id_stream(m, a, b, c, hooks, ks);
#pragma unroll 1
    for (int r = 0; r < N; ++r)
#pragma unroll 1
        for (int cc = 0; cc < ntot; ++cc)  // entries between different chains are structurally zero
            if (cc < c0 || cc >= c0 + N) { Dq[(size_t)((c0 + r) * ntot + cc) * U + u] = 0.0; Dv[(size_t)((c0 + r) * ntot + cc) * U + u] = 0.0; }
}

// generic fallback: one dual-number RNEA sweep per seed direction (blockIdx.y in [0, 3n): q, qd, qdd seeds)
struct RneaDerivsDualBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, const double *q, const double *qd, const double *qdd, double *Dq, double *Dv,
                            double *Mo)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n();
        const int d = blockIdx.y;
        Dual a[MP::MAXN], b[MP::MAXN], c[MP::MAXN], t[MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            a[i] = Dual(q[i * U + u], d == i ? 1.0 : 0.0);
            b[i] = Dual(qd[i * U + u], d == n + i ? 1.0 : 0.0);
            c[i] = Dual(qdd ? qdd[i * U + u] : 0.0, d == 2 * n + i ? 1.0 : 0.0);
        }
        Dyn<Dual, MP>::rnea(m, a, b, c, t);
        double *out = d < n ? Dq : (d < 2 * n ? Dv : Mo);
        const int col = d % n;
#pragma unroll UNR
        for (int r = 0; r < n; ++r) out[(size_t)(r * n + col) * U + u] = t[r].d;
    }
};

// generic fallback for fd-derivs: one dual-number ABA sweep per seed direction (blockIdx.y in [0, 3n))
struct FdDerivsDualBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, const double *q, const double *qd, const double *tau, double *Ao, double *Bo,
                            double *Co)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n();
        const int d = blockIdx.y;
        Dual a[MP::MAXN], b[MP::MAXN], c[MP::MAXN], t[MP::MAXN];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            a[i] = Dual(q[i * U + u], d == i ? 1.0 : 0.0);
            b[i] = Dual(qd[i * U + u], d == n + i ? 1.0 : 0.0);
            c[i] = Dual(tau[i * U + u], d == 2 * n + i ? 1.0 : 0.0);
        }
        Dyn<Dual, MP>::aba(m, a, b, c, t);
        double *out = d < n ? Ao : (d < 2 * n ? Bo : Co);
        const int col = d % n;
#pragma unroll UNR
        for (int r = 0; r < n; ++r) out[(size_t)(r * n + col) * U + u] = t[r].d;
    }
};

// ------------------------------------------------------------------------------------------------ K3
// Column recursion.  With Y_s := dt K_s (+ k_s in the dt column):  X_{s+1} = X_1 + c_s Y_s,  out = X_1 + sum_s w_s Y_s.
// Per thread: one Jacobian column of one unit = 7 n doubles of state (X, accumulators, new qd-rows).
template <int N, int L>
struct ColumnState {
    double Xq[N], Xv[N], Xf[N], aq[N], av[N], af[N];
    int jq, jv, jt;
    bool isdt;
    double ktau;  // tau columns: d(fatigue rhs_jt)/d tau_jt = 2 kappa c_tau tau_jt (one scalar: the column's own joint)
    double xq1;  // the single non-zero of X_2[q] (stage index 1) for q and qd columns

    MPCF_DI void set_tau(const StaticParams<N> &P, double tauj)
    {
        ktau = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i)
            if (i == jt) ktau = 2.0 * P.fat[i][1] * P.fat[i][2] * tauj;
    }
    MPCF_DI void init(int col)
    {
        jq = col < N ? col : -1;
        jv = (col >= N && col < 2 * N) ? col - N : -1;
        jt = (col >= 2 * N && col < 3 * N) ? col - 2 * N : -1;
        isdt = col == 3 * N;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            Xq[i] = (i == jq) ? 1.0 : 0.0;
            Xv[i] = (i == jv) ? 1.0 : 0.0;
            Xf[i] = 0.0;
            aq[i] = Xq[i]; av[i] = Xv[i]; af[i] = 0.0;
        }
        xq1 = 0.0;
    }
    // second half of a stage: fatigue rows, accumulators, next stage state
    MPCF_DI void finish(const StaticParams<N> &P, int s, const double *w1, double h, const double *nv)
    {
        const double cs = s < 2 ? 0.5 : (s == 2 ? 1.0 : 0.0);
        const double wt = (s == 0 || s == 3) ? 1.0 / 6.0 : 1.0 / 3.0;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const double qds = w1[(WsLayout<N>::kQd + i) * 32];
            double kf = 2.0 * P.fat[i][1] * P.fat[i][3] * qds * Xv[i] - P.fat[i][0] * Xf[i];
            if (i == jt) kf += ktau;
            double yq = h * Xv[i], yf = h * kf, yv = h * nv[i];
            if (isdt) {
                yq += qds;
                yv += w1[(WsLayout<N>::kQdd + i) * 32];
                yf += w1[(WsLayout<N>::kFd + i) * 32];
            }
            aq[i] = fma(wt, yq, aq[i]);
            av[i] = fma(wt, yv, av[i]);
            af[i] = fma(wt, yf, af[i]);
            Xq[i] = ((i == jq) ? 1.0 : 0.0) + cs * yq;
            Xv[i] = ((i == jv) ? 1.0 : 0.0) + cs * yv;
            Xf[i] = cs * yf;
            if (s == 0 && (i == jq || i == jv)) xq1 = Xq[i];
        }
    }
    // one RK4 stage for ONE column; w points at this lane's element of plane 0 of the (tile, stage) chunk
    MPCF_DI void stage(const StaticParams<N> &P, int s, const double *w, double h)
    {
        // the three cases are separate straight-line blocks (one branch per stage, not per row): the scheduler batches the
        // shared-memory loads of a whole block, which is what hides their latency at 19 warps per SM
        double nv[N];
        if (s == 0) {  // X_1 is a unit vector (or zero): the product is a single entry of A_1 / B_1
#pragma unroll
            for (int r = 0; r < N; ++r) {
                double kv = 0.0;
                if (jq >= 0 && jq / L == r / L) kv = w[(r * N + jq) * 32];
                if (jv >= 0 && jv / L == r / L) kv = w[(N * N + r * N + jv) * 32];
                nv[r] = kv;
            }
        } else if (s == 1 && !isdt) {
            // X_2[q] = X_1[q] + (dt/2) X_1[qd] still has a single non-zero (q and qd columns) or none (tau columns)
            const int js = jq >= 0 ? jq : jv;
#pragma unroll
            for (int r = 0; r < N; ++r) {
                double kv = 0.0;
                if (js >= 0 && js / L == r / L) kv = w[(r * N + js) * 32] * xq1;
#pragma unroll
                for (int c = 0; c < N; ++c) {
                    if (r / L != c / L) continue;
                    kv = fma(w[(N * N + r * N + c) * 32], Xv[c], kv);
                }
                nv[r] = kv;
            }
        } else {
#pragma unroll
            for (int r = 0; r < N; ++r) {
                double kv = 0.0;
#pragma unroll
                for (int c = 0; c < N; ++c) {
                    if (r / L != c / L) continue;
                    kv = fma(w[(r * N + c) * 32], Xq[c], kv);
                    kv = fma(w[(N * N + r * N + c) * 32], Xv[c], kv);
                }
                nv[r] = kv;
            }
        }
        if (jt >= 0) {
#pragma unroll
            for (int r = 0; r < N; ++r)
                if (jt / L == r / L) nv[r] += w[(2 * N * N + r * N + jt) * 32];
        }
        finish(P, s, w + 3 * N * N * 32, h, nv);
    }
    // one RK4 stage for TWO columns of the same unit: every A/B entry is read once and feeds both recursions
    static MPCF_DI void stage2(ColumnState &a, ColumnState &b, const StaticParams<N> &P, int s, const double *w, double h)
    {
        double na[N], nb[N];
#pragma unroll
        for (int r = 0; r < N; ++r) {
            double ka = 0.0, kb = 0.0;
#pragma unroll
            for (int c = 0; c < N; ++c) {
                if (r / L != c / L) continue;
                const double A = w[(r * N + c) * 32], B = w[(N * N + r * N + c) * 32];
                ka = fma(A, a.Xq[c], ka);
                kb = fma(A, b.Xq[c], kb);
                ka = fma(B, a.Xv[c], ka);
                kb = fma(B, b.Xv[c], kb);
            }
            if (a.jt >= 0 && a.jt / L == r / L) ka += w[(2 * N * N + r * N + a.jt) * 32];
            if (b.jt >= 0 && b.jt / L == r / L) kb += w[(2 * N * N + r * N + b.jt) * 32];
            na[r] = ka;
            nb[r] = kb;
        }
        a.finish(P, s, w + 3 * N * N * 32, h, na);
        b.finish(P, s, w + 3 * N * N * 32, h, nb);
    }
    // Write this column into the Jacobian of the WHOLE model (ntot joints; this chain owns joints c0 .. c0+N-1): own rows
    // get the values, the rows of the other chains are structurally zero.  The dt column is shared by all chains, so
    // there only the own rows are written (every chain's launch writes its part).
    // WHOLE: the chain is the whole model (ntot = N, c0 = 0) and every offset is a compile-time constant
    template <bool WHOLE>
    MPCF_DI void store(const StaticParams<N> &P, int col, double h, long U, long u, double *jac, int ntot_, int c0_) const  // U = plane stride of jac
    {
        const int ntot = WHOLE ? N : ntot_, c0 = WHOLE ? 0 : c0_;
        const long PC = 4 * ntot + 1;
        const long ocol = isdt ? 4 * ntot : (col / N) * ntot + c0 + col % N;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            __stcs(jac + ((size_t)(c0 + i) * PC + ocol) * U + u, aq[i]);
            __stcs(jac + ((size_t)(ntot + c0 + i) * PC + ocol) * U + u, av[i]);
            __stcs(jac + ((size_t)(2 * ntot + c0 + i) * PC + ocol) * U + u, af[i]);
        }
        // (forests: the structural zeros between different chains are written by k_forest_fill_cross, coalesced, once per call)
        if (isdt) {  // the fatigue columns of this chain in closed form (see kernels_jvp.cu), own rows
#pragma unroll
            for (int j = 0; j < N; ++j) {
                const double z = P.fat[j][0] * h;
                const double g = 1.0 + z * (-1.0 + z * (0.5 + z * (-1.0 / 6.0 + z * (1.0 / 24.0))));
                if (WHOLE) {
#pragma unroll
                    for (int r = 0; r < 3 * N; ++r) __stcs(jac + ((size_t)r * PC + 3 * N + j) * U + u, (r == 2 * N + j) ? g : 0.0);
                } else {
#pragma unroll
                    for (int blk = 0; blk < 3; ++blk)
#pragma unroll
                        for (int i = 0; i < N; ++i)
                            __stcs(jac + ((size_t)(blk * ntot + c0 + i) * PC + 3 * ntot + c0 + j) * U + u, (blk == 2 && i == j) ? g : 0.0);
                }
            }
        }
    }
};

// ------------------------------------------------------------------------------------------------ reverse sweep
// Vector-Jacobian product of the step, thread = unit, in place of K3 (DESIGN.md §4d).  Stages walked 4 -> 1 with
// rho_s = w_s lambda + c_s J_{s+1}^T r_{s+1}, r_s = h rho_s:
//   J_s^T r = (A_s^T r_v, r_q + B_s^T r_v + 2 kappa cv qd_s r_f, -Lambda r_f),   g_tau += C_s r_v + 2 kappa ctau tau r_f,
//   g_x = lambda + sum_s J_s^T r_s (+ addend),   g_dt = sum_s rho_s^T k_s.
// Every workspace load is one coalesced warp access (lane = unit of the 32-unit tile); 3 n^2 FMAs per stage.
// gdt_add: a forest's second chain adds its share of g_dt to the first chain's (stream order, no atomics).
template <int N, int L>
__global__ void __launch_bounds__(kThreads) k_step_vjp(const __grid_constant__ StaticParams<N> P, long U, long u0, long cnt,
                                                      const double *__restrict__ tau, double dt, const double *__restrict__ dt_u,
                                                      const VjpArgs a, int gdt_add, const double *__restrict__ ws)
{
    static_assert(N == L, "the reverse sweep runs one serial chain at a time (forests: one launch per chain)");
    using W = WsLayout<N>;
    const long lu = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (lu >= cnt) return;
    const long u = u0 + lu;
    const double h = dt_u ? dt_u[u] : dt;
    double lam[3 * N], gx[3 * N], ad[3 * N], gt[N], kt[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        lam[i] = a.lq ? a.lq[i * a.ldl + u] : 0.0;
        lam[N + i] = a.lqd ? a.lqd[i * a.ldl + u] : 0.0;
        lam[2 * N + i] = a.lf ? a.lf[i * a.ldl + u] : 0.0;
        gx[i] = lam[i] + (a.aq ? a.aq[i * a.lda + u] : 0.0);
        gx[N + i] = lam[N + i] + (a.aqd ? a.aqd[i * a.lda + u] : 0.0);
        gx[2 * N + i] = lam[2 * N + i] + (a.af ? a.af[i * a.lda + u] : 0.0);
        kt[i] = 2.0 * P.fat[i][1] * P.fat[i][2] * tau[i * U + u];
        gt[i] = 0.0;
    }
#pragma unroll
    for (int i = 0; i < 3 * N; ++i) ad[i] = 0.0;
    double gh = 0.0;
#pragma unroll 1
    for (int s = 3; s >= 0; --s) {
        const double cs = s < 2 ? 0.5 : (s == 2 ? 1.0 : 0.0);  // x_{s+1} = x + c_s h k_s (ad = 0 at the last stage)
        const double wt = (s == 0 || s == 3) ? 1.0 / 6.0 : 1.0 / 3.0;
        const double *w = ws + W::chunk(lu / 32, s) + (lu & 31);
        const double *v = w + W::kPlanes2 * 32;
        double rq[N], rv[N], rf[N], nq[N], nv[N];
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const double qds = __ldcs(v + (W::kQd + i) * 32);
            const double pq = fma(wt, lam[i], cs * ad[i]), pv = fma(wt, lam[N + i], cs * ad[N + i]),
                         pf = fma(wt, lam[2 * N + i], cs * ad[2 * N + i]);
            gh = fma(pq, qds, gh);
            gh = fma(pv, __ldcs(v + (W::kQdd + i) * 32), gh);
            gh = fma(pf, __ldcs(v + (W::kFd + i) * 32), gh);
            rq[i] = h * pq;
            rv[i] = h * pv;
            rf[i] = h * pf;
            nq[i] = 0.0;
            nv[i] = fma(2.0 * P.fat[i][1] * P.fat[i][3] * qds, rf[i], rq[i]);
            gt[i] = fma(kt[i], rf[i], gt[i]);
        }
        // one basic block per row (the never-taken fence, cf. StaticModel::skip): ptxas would otherwise hoist all 3 n^2 loads of the
        // stage and take the whole register file
#pragma unroll
        for (int r = 0; r < N; ++r) {
            if (P.fence0 > r) continue;
            const double x = rv[r];
#pragma unroll
            for (int c = 0; c < N; ++c) {
                nq[c] = fma(__ldcs(w + (r * N + c) * 32), x, nq[c]);
                nv[c] = fma(__ldcs(w + (N * N + r * N + c) * 32), x, nv[c]);
                gt[c] = fma(__ldcs(w + (2 * N * N + r * N + c) * 32), x, gt[c]);
            }
        }
#pragma unroll
        for (int i = 0; i < N; ++i) {
            ad[i] = nq[i];
            ad[N + i] = nv[i];
            ad[2 * N + i] = -P.fat[i][0] * rf[i];
            gx[i] += ad[i];
            gx[N + i] += ad[N + i];
            gx[2 * N + i] += ad[2 * N + i];
        }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) {
        a.gq[i * a.ldg + u] = gx[i];
        a.gqd[i * a.ldg + u] = gx[N + i];
        a.gf[i * a.ldg + u] = gx[2 * N + i];
        a.gtau[i * a.ldgt + u] = gt[i];
    }
    if (a.gdt) a.gdt[u] = gdt_add ? a.gdt[u] + gh : gh;
}

// ---- mbarrier / bulk-copy primitives (PTX ISA 8.0, sm_90+; forms as in <cuda/ptx>) ----
MPCF_DI unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
MPCF_DI void mbar_init(unsigned long long *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
MPCF_DI void mbar_arrive(unsigned long long *bar)
{
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
MPCF_DI void mbar_arrive_expect_tx(unsigned long long *bar, unsigned bytes)
{
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.release.cta.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
MPCF_DI void mbar_wait(unsigned long long *bar, unsigned parity)
{
    unsigned done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
    } while (!done);
}
MPCF_DI void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// item -> (tile, stage) -> ring slot: wait until the slot is free, arm its `full` barrier, start the bulk copy
template <class W, int NBUF>
MPCF_DI void tma_issue(unsigned item, double *buf, unsigned long long *full, unsigned long long *empty, const double *ws, unsigned bid,
                       unsigned nblk)
{
    const unsigned slot = item % NBUF, round = item / NBUF;
    const long t = bid + (long)(item / 4) * nblk;
    mbar_wait(&empty[slot], (round & 1) ^ 1);
    mbar_arrive_expect_tx(&full[slot], W::kRingBytes);
    bulk_g2s(buf + (size_t)slot * W::kRingDoubles, ws + W::chunk(t, item & 3), W::kRingBytes, &full[slot]);
}

// Persistent chain-rule kernel for N <= 6.  CPW = Jacobian columns per consumer thread (1 or 2); NW consumer warps.
// No dedicated producer warp: lane 0 of warp 0 refills the ring slot that was released NBUF-1 stages ago before it
// starts its own stage (the slot is free by then unless the whole CTA is memory-starved).
template <int N, int L, int NBUF, int CPW, bool WHOLE>
__global__ void __launch_bounds__(32 * ((3 * N + CPW) / CPW), 1)
    k_chain_rule_tma(const __grid_constant__ StaticParams<N> P, long U, long u0, long cnt, const double *__restrict__ tau, long UT, double dt,
                     const double *__restrict__ dt_u, const double *__restrict__ ws, double *__restrict__ jac, long UJ, int ntot, int c0)
{
    using W = WsLayout<N>;
    constexpr int NC = 3 * N + 1;
    constexpr int NW = (NC + CPW - 1) / CPW;  // consumer warps
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *buf = reinterpret_cast<double *>(smem_raw);
    unsigned long long *full = reinterpret_cast<unsigned long long *>(smem_raw + (size_t)NBUF * W::kRingBytes);
    unsigned long long *empty = full + NBUF;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long ntiles = (cnt + 31) / 32;
    const long my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const unsigned nitems = (unsigned)(my_tiles * 4);
    const bool producer = threadIdx.x == 0;
    if (producer) {
        for (int i = 0; i < NBUF; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], NW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (unsigned i = 0; i < NBUF - 1 && i < nitems; ++i)  // prologue: fill all but one slot
            tma_issue<W, NBUF>(i, buf, full, empty, ws, blockIdx.x, gridDim.x);
    }
    __syncthreads();
    const int col0 = warp, col1 = warp + NW;
    const bool two = CPW == 2 && col1 < NC;
    unsigned it = 0;
    for (long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const long lu = t * 32 + lane;
        const bool live = lu < cnt;
        const long u = u0 + (live ? lu : 0);
        const double h = dt_u ? dt_u[u] : dt;
        ColumnState<N, L> a, b;
        a.init(col0);
        a.set_tau(P, a.jt >= 0 ? tau[(size_t)a.jt * UT + u] : 0.0);  // tau here = the heating torque (plane stride UT)
        if (CPW == 2) {
            b.init(two ? col1 : col0);
            b.set_tau(P, b.jt >= 0 ? tau[(size_t)b.jt * UT + u] : 0.0);
        }
#pragma unroll 1
        for (int s = 0; s < 4; ++s, ++it) {
            if (producer && it + NBUF - 1 < nitems) tma_issue<W, NBUF>(it + NBUF - 1, buf, full, empty, ws, blockIdx.x, gridDim.x);
            const unsigned slot = it % NBUF, round = it / NBUF;
            mbar_wait(&full[slot], round & 1);
            const double *w = buf + (size_t)slot * W::kRingDoubles + lane;
            if (CPW == 2) ColumnState<N, L>::stage2(a, b, P, s, w, h);
            else a.stage(P, s, w, h);
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[slot]);
        }
        if (live) {
            a.template store<WHOLE>(P, col0, h, UJ, u, jac, ntot, c0);
            if (two) b.template store<WHOLE>(P, col1, h, UJ, u, jac, ntot, c0);
        }
    }
}

// Fallback for larger models (a stage chunk does not fit the shared-memory ring): same recursion, operands read
// straight from the workspace tile with immediate plane offsets.
template <int N, int L, int NCY>
__global__ void __launch_bounds__(32 * NCY, 2)
    k_chain_rule_ldg(const __grid_constant__ StaticParams<N> P, long U, long u0, long cnt, const double *__restrict__ tau, long UT, double dt,
                     const double *__restrict__ dt_u, const double *__restrict__ ws, double *__restrict__ jac, long UJ, int ntot, int c0)
{
    using W = WsLayout<N>;
    const long lu = (long)blockIdx.x * 32 + threadIdx.x;
    if (lu >= cnt) return;
    const long u = u0 + lu;
    const double h = dt_u ? dt_u[u] : dt;
    constexpr int NC = 3 * N + 1;
    for (int col = threadIdx.y; col < NC; col += blockDim.y) {
        ColumnState<N, L> st;
        st.init(col);
        st.set_tau(P, st.jt >= 0 ? tau[(size_t)st.jt * UT + u] : 0.0);
#pragma unroll 1
        for (int s = 0; s < 4; ++s) st.stage(P, s, ws + W::chunk(blockIdx.x, s) + threadIdx.x, h);
        st.template store<false>(P, col, h, UJ, u, jac, ntot, c0);
    }
}

// ------------------------------------------------------------------------------------------------ launchers
// Optional per-kernel timing (bench.py roofline): when enabled, every kernel of the pipeline is bracketed by CUDA
// events on the launch stream; jvp_profile_read() synchronises and returns the accumulated milliseconds per kernel.
// The event list is shared by all host threads that launch while profiling is on: guarded by a mutex (taken only when
// profiling is enabled; the flag itself is atomic).
struct ProfEvent { cudaEvent_t a, b; int k; };
static std::atomic<bool> g_prof_on{false};
static std::mutex g_prof_mu;
static std::vector<ProfEvent> g_prof;
void jvp_profile_enable(bool on) { g_prof_on.store(on); }
// returns the event to record at the end of the bracket (nullptr when profiling is off)
static cudaEvent_t prof_begin(int k, cudaStream_t s)
{
    if (!g_prof_on.load(std::memory_order_relaxed)) return nullptr;
    ProfEvent e;
    cudaEventCreate(&e.a);
    cudaEventCreate(&e.b);
    e.k = k;
    cudaEventRecord(e.a, s);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.push_back(e);
    return e.b;
}
static void prof_end(cudaEvent_t b, cudaStream_t s)
{
    if (b) cudaEventRecord(b, s);
}
int jvp_profile_read(double *ms3, long *launches)
{
    std::lock_guard<std::mutex> lk(g_prof_mu);
    ms3[0] = ms3[1] = ms3[2] = 0.0;
    *launches = (long)g_prof.size();
    for (auto &e : g_prof) {
        float t = 0.f;
        cudaEventSynchronize(e.b);
        cudaEventElapsedTime(&t, e.a, e.b);
        ms3[e.k] += t;
        cudaEventDestroy(e.a);
        cudaEventDestroy(e.b);
    }
    g_prof.clear();
    return 0;
}

static int current_device()
{
    int dev = 0;
    cudaGetDevice(&dev);
    return dev >= 0 && dev < 64 ? dev : 0;
}
static int sm_count()
{
    static int n[64] = {};
    const int dev = current_device();
    if (!n[dev]) {
        cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev);
        if (n[dev] <= 0) n[dev] = 148;
    }
    return n[dev];
}

// K2 launch shape: 2 blocks per SM with the link slab in shared memory
template <int N, int L>
struct K2Config {
    static constexpr int kThreadsK2 = (2 * (18 * (N - 1) + N * (N + 1) / 2) * kThreads * (int)sizeof(double) <= 227 * 1024) ? kThreads : 96;
    static constexpr int kSlab = (18 * (N - 1) + N * (N + 1) / 2) * kThreadsK2 * (int)sizeof(double);
    static constexpr bool kSmem = N == L && 2 * kSlab <= 227 * 1024;
};

// K1 + K2 of one chunk of units [u0, u0 + cnt): what the Jacobian (K3) and the reverse sweep (k_step_vjp) read
template <int N, int L>
static cudaError_t launch_stages_derivs(const StaticParams<N> &P, long U, long u0, long cnt, const double *q, const double *qd, const double *tau,
                                 const double *theat, long UT, const double *f, double dt, const double *dt_u, double *qn, double *qdn,
                                 double *fn, double *ws, cudaStream_t s)
{
    using K2 = K2Config<N, L>;
    static const int k2smem = getenv("MPCF_K2_SMEM") ? atoi(getenv("MPCF_K2_SMEM")) : 1;
    if constexpr (K2::kSmem) {
        if (k2smem) {
            const cudaError_t e = raise_smem_limit<k_stage_derivs<N, L, true>>(K2::kSlab);
            if (e != cudaSuccess) return e;
        }
    }
    const unsigned gb = (unsigned)((cnt + kThreads - 1) / kThreads);
    cudaEvent_t pe = prof_begin(0, s);
    k_step_stages<N, L><<<gb, kThreads, 0, s>>>(P, U, u0, cnt, q, qd, tau, theat, UT, f, dt, dt_u, qn, qdn, fn, ws);
    prof_end(pe, s);
    pe = prof_begin(1, s);
    bool k2done = false;
    if constexpr (K2::kSmem) {
        if (k2smem) {
            k_stage_derivs<N, L, true><<<dim3((unsigned)((cnt + K2::kThreadsK2 - 1) / K2::kThreadsK2), 4), K2::kThreadsK2, K2::kSlab, s>>>(P, cnt, ws);
            k2done = true;
        }
    }
    if (!k2done) k_stage_derivs<N, L, false><<<dim3(gb, 4), kThreads, 0, s>>>(P, cnt, ws);
    prof_end(pe, s);
    return cudaSuccess;
}

template <int N, int L>
static cudaError_t run_jvp2(const StaticParams<N> &P, long U, long Ucnt, const double *q, const double *qd, const double *tau, const double *theat,
                            long UT, const double *f,
                            double dt, const double *dt_u, double *qn, double *qdn, double *fn, double *jac, long UJ, double *ws, long Uc,
                            cudaStream_t s, int ntot, int c0)
{
    using W = WsLayout<N>;
    // chain-rule kernel: bulk-copy ring of up to 5 slots (a deeper ring takes the shared-memory carve-out from L1, which the
    // streaming Jacobian stores want); 3 N + 1 column warps of 96 registers fit the register file up to N = 6, longer chains
    // run two columns per thread
    constexpr bool kTma = N <= 7;
    constexpr int kRingMax = (227 * 1024 - 256) / (int)W::kRingBytes;
    constexpr int NBUF = kTma ? (kRingMax > 5 ? 5 : kRingMax) : 0;  // measured on chain6: 5 slots 11.74 ms, 4: 11.89, 6: 12.08, 7: 12.93 (L1 gets what the ring leaves)
    constexpr int kCpwDefault = (3 * N + 1 <= 19) ? 1 : 2;
    constexpr size_t smem = (size_t)NBUF * W::kRingBytes + 2 * NBUF * sizeof(unsigned long long);
    if constexpr (kTma) {
        cudaError_t e = cudaSuccess;
        if constexpr (kCpwDefault == 1) {
            if ((e = raise_smem_limit<k_chain_rule_tma<N, L, NBUF, 1, true>>((int)smem)) != cudaSuccess) return e;
            if ((e = raise_smem_limit<k_chain_rule_tma<N, L, NBUF, 1, false>>((int)smem)) != cudaSuccess) return e;
        }
        if ((e = raise_smem_limit<k_chain_rule_tma<N, L, NBUF, 2, true>>((int)smem)) != cudaSuccess) return e;
        if ((e = raise_smem_limit<k_chain_rule_tma<N, L, NBUF, 2, false>>((int)smem)) != cudaSuccess) return e;
    }
    for (long u0 = 0; u0 < Ucnt; u0 += Uc) {
        const long cnt = (Ucnt - u0) < Uc ? (Ucnt - u0) : Uc;
        const long ntiles = (cnt + 31) / 32;
        const cudaError_t e = launch_stages_derivs<N, L>(P, U, u0, cnt, q, qd, tau, theat, UT, f, dt, dt_u, qn, qdn, fn, ws, s);
        if (e != cudaSuccess) return e;
        cudaEvent_t pe = prof_begin(2, s);
        if constexpr (kTma) {
            const unsigned g3 = (unsigned)(ntiles < sm_count() ? ntiles : sm_count());
            static const int cpw_env = getenv("MPCF_K3_CPW") ? atoi(getenv("MPCF_K3_CPW")) : 1;
            const int cpw = kCpwDefault == 2 ? 2 : cpw_env;
            if (cpw == 2) {
                (ntot == N ? k_chain_rule_tma<N, L, NBUF, 2, true> : k_chain_rule_tma<N, L, NBUF, 2, false>)<<<g3, 32 * ((3 * N + 2) / 2), smem, s>>>(
                    P, U, u0, cnt, theat, UT, dt, dt_u, ws, jac, UJ, ntot, c0);
            } else if constexpr (kCpwDefault == 1) {
                (ntot == N ? k_chain_rule_tma<N, L, NBUF, 1, true> : k_chain_rule_tma<N, L, NBUF, 1, false>)<<<g3, 32 * (3 * N + 1), smem, s>>>(
                    P, U, u0, cnt, theat, UT, dt, dt_u, ws, jac, UJ, ntot, c0);
            }
        } else {
            k_chain_rule_ldg<N, L, 10><<<(unsigned)ntiles, dim3(32, 10), 0, s>>>(P, U, u0, cnt, theat, UT, dt, dt_u, ws, jac, UJ, ntot, c0);
        }
        prof_end(pe, s);
        g_launches.fetch_add(3);
    }
    return cudaGetLastError();
}

// Forest Jacobians: every entry between joints of different chains is structurally zero (columns q, qd, tau, f; the dt column
// is dense).  One coalesced pass: thread = unit, blockIdx.y = Jacobian row, loop over the columns of the other chains.
template <int L, class V>
__global__ void __launch_bounds__(256) k_forest_fill_cross(int ntot, long cntv, long UJ, double *jac)
{
    const long uv = (long)blockIdx.x * blockDim.x + threadIdx.x;  // unit (V = double) or pair of units (V = double2)
    if (uv >= cntv) return;
    const int r = blockIdx.y, rc = (r % ntot) / L, nch = ntot / L;
    const long PC = 4 * ntot + 1;
    V zero;
    memset(&zero, 0, sizeof(V));
    double *row = jac + (size_t)r * PC * UJ;
    for (int b = 0; b < 4; ++b)
        for (int oc = 0; oc < nch; ++oc) {
            if (oc == rc) continue;
            double *p = row + (size_t)(b * ntot + oc * L) * UJ;
#pragma unroll
            for (int i = 0; i < L; ++i) __stcs(reinterpret_cast<V *>(p + (size_t)i * UJ) + uv, zero);
        }
}

bool jvp2_supported(const LaunchModel &m) { return family_chain_len(m.fam) > 0; }

size_t jvp_ws_bytes_per_unit(const LaunchModel &m)
{
    size_t bytes = 0;
    with_chains(m, [&](auto L, const auto *, auto) { bytes = WsLayout<L>::kUnitDoubles * sizeof(double); });
    return bytes;
}

// units per chunk of the pipeline in ws_bytes of workspace: whole 32-unit tiles
static long jvp_chunk_units(const LaunchModel &m, size_t ws_bytes)
{
    const long Uc = (long)(ws_bytes / jvp_ws_bytes_per_unit(m));
    return Uc - Uc % 32;
}

// Forests: the chains are dynamically decoupled, so each runs the single-chain pipeline on its own input planes and writes its
// block of the whole-model Jacobian; k_forest_fill_cross then writes the zeros of the cross blocks.
cudaError_t launch_step_jvp_ws(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, const double *f,
                               double dt, const double *dt_u, double *qn, double *qdn, double *fn, double *jac, double *ws,
                               size_t ws_bytes, cudaStream_t s, long cnt, long UJ, const double *theat, long UT)
{
    if (!theat) { theat = tau; UT = U; }  // uncoupled model: the commanded torque is what heats the windings
    // cnt units are evaluated; U is the plane stride of the input / state arrays, UJ that of the Jacobian planes (callers
    // evaluating a unit range of a larger batch pass base pointers shifted to the range and a chunk-local Jacobian buffer)
    if (cnt < 0) cnt = U;
    if (UJ <= 0) UJ = U;
    if (cnt <= 0) return cudaSuccess;
    const long Uc = jvp_chunk_units(m, ws_bytes);
    if (Uc < 32) return cudaErrorInvalidValue;
    cudaError_t e = cudaErrorInvalidValue;
    with_chains(m, [&](auto L, const auto *chains, auto nchains) {
        for (int c = 0; c < nchains; ++c) {
            const size_t off = (size_t)c * L * U;
            e = run_jvp2<L, L>(chains[c], U, cnt, q + off, qd + off, tau + off, theat + (size_t)c * L * UT, UT, f + off, dt, dt_u,
                               qn ? qn + off : nullptr, qdn ? qdn + off : nullptr, fn ? fn + off : nullptr, jac, UJ, ws, Uc, s, m.n, c * L);
            if (e != cudaSuccess) return;
        }
        if constexpr (decltype(nchains)::value > 1) {
            if (cnt % 2 == 0 && UJ % 2 == 0 && (reinterpret_cast<size_t>(jac) & 15) == 0)
                k_forest_fill_cross<L, double2><<<dim3((unsigned)((cnt / 2 + 255) / 256), 3 * m.n), 256, 0, s>>>(m.n, cnt / 2, UJ, jac);
            else
                k_forest_fill_cross<L, double><<<dim3((unsigned)((cnt + 255) / 256), 3 * m.n), 256, 0, s>>>(m.n, cnt, UJ, jac);
            g_launches.fetch_add(1);
            e = cudaGetLastError();
        }
    });
    return e;
}

// Reverse sweep of one serial chain: K1 and K2 unchanged over the same chunks as run_jvp2, then k_step_vjp in place of K3.
// gdt_add: this chain's g_dt is added to what an earlier chain's launch wrote.
template <int N, int L>
static cudaError_t run_vjp2(const StaticParams<N> &P, long U, long Ucnt, const double *q, const double *qd, const double *tau, const double *f,
                            double dt, const double *dt_u, const VjpArgs &a, int gdt_add, double *qn, double *qdn, double *fn, double *ws, long Uc,
                            cudaStream_t s)
{
    for (long u0 = 0; u0 < Ucnt; u0 += Uc) {
        const long cnt = (Ucnt - u0) < Uc ? (Ucnt - u0) : Uc;
        const cudaError_t e = launch_stages_derivs<N, L>(P, U, u0, cnt, q, qd, tau, tau, U, f, dt, dt_u, qn, qdn, fn, ws, s);
        if (e != cudaSuccess) return e;
        k_step_vjp<N, L><<<(unsigned)((cnt + kThreads - 1) / kThreads), kThreads, 0, s>>>(P, U, u0, cnt, tau, dt, dt_u, a, gdt_add, ws);
        g_launches.fetch_add(3);
    }
    return cudaGetLastError();
}

cudaError_t launch_step_vjp_ws(const LaunchModel &m, long U, long cnt, const double *q, const double *qd, const double *tau, const double *f,
                               double dt, const double *dt_u, const VjpArgs &a, double *qn, double *qdn, double *fn, double *ws,
                               size_t ws_bytes, cudaStream_t s)
{
    if (cnt <= 0) return cudaSuccess;
    const long Uc = jvp_chunk_units(m, ws_bytes);
    if (Uc < 32) return cudaErrorInvalidValue;
    cudaError_t e = cudaErrorInvalidValue;
    with_chains(m, [&](auto L, const auto *chains, auto nchains) {
        for (int c = 0; c < nchains; ++c) {
            const size_t off = (size_t)c * L * U;
            e = run_vjp2<L, L>(chains[c], U, cnt, q + off, qd + off, tau + off, f + off, dt, dt_u, a.rows(c * L), c > 0, qn ? qn + off : nullptr,
                               qdn ? qdn + off : nullptr, fn ? fn + off : nullptr, ws, Uc, s);
            if (e != cudaSuccess) return;
        }
    });
    return e;
}

// shared-memory slab of the streaming derivative kernels: (S, xi, eta) of links 0 .. n-2, one column per thread
static constexpr int link_slab_bytes(int n) { return 18 * (n - 1) * kThreads * (int)sizeof(double); }

cudaError_t launch_node_eval_jvp(const LaunchModel &m, const EeArgs &ee, double wsign, long U, const double *q, const double *qd,
                                 const double *qdd, const double *W, double *dtau_dq, double *dtau_dqd, cudaStream_t s)
{
    if (U <= 0) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    if (with_chains(m, [&](auto L, const auto *chains, auto nchains) {
            auto go = [&](auto nee) {
                constexpr auto kern = k_node_eval_jvp<L, decltype(nee)::value>;
                if ((e = raise_smem_limit<kern>(link_slab_bytes(L))) != cudaSuccess) return;
                for (int c = 0; c < nchains; ++c) {
                    const size_t off = (size_t)c * L * U;
                    kern<<<(unsigned)((U + kThreads - 1) / kThreads), kThreads, link_slab_bytes(L), s>>>(
                        chains[c], U, ee, wsign, q + off, qd + off, qdd ? qdd + off : nullptr, W, dtau_dq, dtau_dqd, m.n, c * L);
                    g_launches.fetch_add(1);
                }
                e = cudaGetLastError();
            };
            using std::integral_constant;
            if (ee.nee == 0) go(integral_constant<int, 0>{});
            else if (ee.nee == 1) go(integral_constant<int, 1>{});
            else if (ee.nee == 2) go(integral_constant<int, 2>{});
            else go(integral_constant<int, MPCF_MAX_EE>{});
        }))
        return e;
    return launch_node_eval_jvp_dual(m, ee, wsign, U, q, qd, qdd, W, dtau_dq, dtau_dqd, s);
}

cudaError_t launch_rnea_derivs(const LaunchModel &m, long U, const double *q, const double *qd, const double *qdd, double *Dq, double *Dv,
                               double *M, cudaStream_t s)
{
    if (U <= 0) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    if (with_chains(m, [&](auto L, const auto *chains, auto nchains) {
            if ((e = raise_smem_limit<k_rnea_derivs<L>>(link_slab_bytes(L))) != cudaSuccess) return;
            for (int c = 0; c < nchains; ++c) {
                const size_t off = (size_t)c * L * U;
                k_rnea_derivs<L><<<(unsigned)((U + kThreads - 1) / kThreads), kThreads, link_slab_bytes(L), s>>>(
                    chains[c], U, q + off, qd + off, qdd ? qdd + off : nullptr, Dq, Dv, M, m.n, c * L);
                g_launches.fetch_add(1);
            }
            e = cudaGetLastError();
        }))
        return e;
    return dispatch_generic<RneaDerivsDualBody>(m, U, 3 * m.n, s, q, qd, qdd, Dq, Dv, M);
}

cudaError_t launch_fd_derivs(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, double *A, double *B,
                             double *C, cudaStream_t s)
{
    if (U <= 0) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    if (with_chains(m, [&](auto L, const auto *chains, auto nchains) {
            if ((e = raise_smem_limit<k_fd_derivs<L>>(link_slab_bytes(L))) != cudaSuccess) return;
            for (int c = 0; c < nchains; ++c) {
                const size_t off = (size_t)c * L * U;
                k_fd_derivs<L><<<(unsigned)((U + kThreads - 1) / kThreads), kThreads, link_slab_bytes(L), s>>>(
                    chains[c], U, q + off, qd + off, tau + off, A, B, C, m.n, c * L);
                g_launches.fetch_add(1);
            }
            e = cudaGetLastError();
        }))
        return e;
    return dispatch_generic<FdDerivsDualBody>(m, U, 3 * m.n, s, q, qd, tau, A, B, C);
}

}  // namespace mpcf
