// kernels_tree.cu — analytic Jacobian pipeline of the RK4 dynamics+fatigue step for RUN-TIME TREES (branched models with
// revolute / prismatic joints, n <= 40: config C4's 37-joint tree), replacing the 3n + 1 dual-number sweeps for these models.
// Same mathematics as the static-chain pipeline (kernels_jvp2.cu, DESIGN.md §4) with ancestor relations instead of chain
// relations (tree_derivs.cuh), and a different chain-rule mapping, because at n = 37 the per-unit products are real matrix
// products ([37 x 74] . [74 x 112] per stage) and the per-unit matrices do not fit a thread:
//
//   T1 k_tree_stages     thread = unit           primal RK4 (ABA), per stage (q_s, qd_s, qdd_s) and the fatigue-row coefficients
//   T2 k_tree_derivs     thread = (unit, stage)  dID/dq, dID/dqd and M on the ancestor pattern (packed: 5 npat values per stage
//                                                instead of 3 n^2)
//      k_tree_factor     warp = (unit, stage)    M = L^T D L and L^-1 in place, in shared memory
//   T3 k_tree_chain_tc   CTA = (unit, slab of 64 Jacobian columns), FP64 tensor cores (mma.sync m8n8k4), per stage
//                          Z = [dID/dq | dID/dqd] [X[q]; X[qd]],   K = L^-1 D^-1 L^-T (E_tau - Z)   (two triangular products)
//                        X in shared memory (warp-private columns), accumulators in register fragments; units handed out by an
//                        atomic counter so that neighbouring units (which share 32-byte sectors of the outputs) stay in L2
//      k_tree_chain      the DFMA variant (CTA = unit, thread = column, triangular solves with L), MPCF_TREE_CHAIN=scalar:
//                        kept as an independent cross-check of the tensor-core path
//      k_tree_fill_fatigue_cols  the closed-form fatigue columns, coalesced
//
// Workspace: one contiguous block per (unit, stage); the four values of a pattern entry (dID/dq_kj, dID/dqd_kj, dID/dq_jk,
// dID/dqd_jk) are adjacent = one 32-byte sector per entry for the thread-per-unit writer, whole sectors for the CTA-per-unit
// reader (cp.async scatter copies into the dense shared-memory matrices, issued one stage ahead of the arithmetic).
//
// Accumulator identities that keep the per-column state small (checked on the host by tests/hostcheck, same formulas as plain
// loops, and on the GPU against the oracle):
//   Yv_s = h K_s (+ qdd_s in the dt column),  P = Yv_1 + Yv_2 + Yv_3
//   d q+ /dz = X1[q] + h X1[qd] + (h/6) P (+ sum_s w_s qd_s in the dt column)
//   d qd+/dz = X1[qd] + (2 P - Yv_1 + Yv_4) / 6
//   d f+_i/dz = sum_{s<=3} fnext_s[i] Yv_s[i] (+ closed-form terms), fnext_s = c_s gamma_{s+1}(lambda_i h) (h/6) 2 kappa_i cv_i qd_{s+1,i}
//               with gamma = (1 - z + z^2/2 - z^3/4, 2 - z + z^2/2, 2 - z, 1): the RK4 response of the linear fatigue rows
//               to a forcing applied at stage s, so the rows need no per-column recursion state.
#include <cstdlib>

#include "launch.cuh"
#include "tree_derivs.cuh"

#ifndef MPCF_T1_BLOCKS
#define MPCF_T1_BLOCKS 2
#endif
#ifndef MPCF_T2_BLOCKS
#define MPCF_T2_BLOCKS 2
#endif

namespace mpcf {

// ------------------------------------------------------------------------------------------------ workspace layout
struct TreeWs {
    int n, npat, NE;  // NE doubles per (unit, stage) block, a multiple of 4 (blocks stay 32-byte aligned)
    MPCF_HD static int planes(int n, int npat) { return (5 * npat + 5 * n + 3) & ~3; }
    // A (unit, stage) block is contiguous: the chain kernels (CTA = unit) then read whole 32-byte sectors, and the four values of
    // a pattern entry are adjacent, so the thread-per-unit writer stores one full sector per entry.
    MPCF_HD size_t at(long u, int s) const { return ((size_t)u * 4 + s) * NE; }
    // element indices inside a block
    MPCF_HD int dqkj(int e) const { return 4 * e; }
    MPCF_HD int dvkj(int e) const { return 4 * e + 1; }
    MPCF_HD int dqjk(int e) const { return 4 * e + 2; }
    MPCF_HD int dvjk(int e) const { return 4 * e + 3; }
    MPCF_HD int lf(int e) const { return 4 * npat + e; }
    MPCF_HD int vec(int slot, int i) const { return 5 * npat + slot * n + i; }  // 0 qd_s, 1 qdd_s, 2 fnext_s, 3 q_s, 4 extra_s
};
size_t tree_ws_doubles_per_unit(int n, int npat) { return (size_t)4 * TreeWs::planes(n, npat); }

// ------------------------------------------------------------------------------------------------ T1
template <int MAXN>
__global__ void __launch_bounds__(kThreads, MPCF_T1_BLOCKS) k_tree_stages(GenericBlob blob, TreeWs W, long U, long cnt, const double *q, const double *qd,
                                                            const double *tau, const double *f, double dt, const double *dt_u, double *qn,
                                                            double *qdn, double *fn, double *ws)
{
    extern __shared__ double smem[];
    const int n = blob.n;
    const int nd = 27 * n + 3;
    int *si = reinterpret_cast<int *>(smem + nd);
    for (int k = threadIdx.x; k < nd; k += blockDim.x) smem[k] = blob.dbl[k];
    for (int k = threadIdx.x; k < blob_ints(n); k += blockDim.x) si[k] = blob.ints[k];
    __syncthreads();
    const GenericModel<MAXN> m{n, smem, si};
    using D = Dyn<double, GenericModel<MAXN>>;
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= cnt) return;
    double x[3 * MAXN], t[MAXN], xs[3 * MAXN], xn[3 * MAXN], k[3 * MAXN];
    double fsum[MAXN], gdt[MAXN], qdbar[MAXN];
    for (int i = 0; i < n; ++i) {
        x[i] = q[i * U + u];
        x[n + i] = qd[i * U + u];
        x[2 * n + i] = f[i * U + u];
        t[i] = tau[i * U + u];
        fsum[i] = 0.0; gdt[i] = 0.0; qdbar[i] = 0.0;
    }
    const double h = dt_u ? dt_u[u] : dt;
    for (int i = 0; i < 3 * n; ++i) { xs[i] = x[i]; xn[i] = x[i]; }
#pragma unroll 1
    for (int s = 0; s < 4; ++s) {
        const double cs = s < 2 ? 0.5 : (s == 2 ? 1.0 : 0.0);
        const double cprev = s == 3 ? 1.0 : 0.5;  // c_{s-1}
        const double wt = (s == 0 || s == 3) ? 1.0 / 6.0 : 1.0 / 3.0;
        D::aba(m, xs, xs + n, t, k + n);
        double *w = ws + W.at(u, s);
        double *wprev = ws + W.at(u, s > 0 ? s - 1 : 0);
        for (int i = 0; i < n; ++i) {
            const double qdi = xs[n + i];
            k[i] = qdi;
            k[2 * n + i] = D::fatigue_rhs(m, i, xs[2 * n + i], t[i], qdi);
            w[W.vec(0, i)] = qdi;
            w[W.vec(1, i)] = k[n + i];
            w[W.vec(3, i)] = xs[i];
            const double z = m.fat(i, 0) * h;
            const double gam = s == 0 ? 1.0 + z * (-1.0 + z * (0.5 - 0.25 * z)) : (s == 1 ? 2.0 + z * (-1.0 + 0.5 * z) : (s == 2 ? 2.0 - z : 1.0));
            const double fcoef = gam * (h / 6.0) * 2.0 * m.fat(i, 1) * m.fat(i, 3) * qdi;
            fsum[i] += fcoef;
            gdt[i] += gam * (1.0 / 6.0) * k[2 * n + i];
            qdbar[i] += wt * qdi;
            if (s > 0) wprev[W.vec(2, i)] = fcoef * cprev;
        }
        const double a = h * wt, c = h * cs;
        for (int i = 0; i < 3 * n; ++i) {
            xn[i] += a * k[i];
            xs[i] = x[i] + c * k[i];
        }
    }
    for (int i = 0; i < n; ++i) {
        ws[W.at(u, 0) + (size_t)W.vec(4, i)] = gdt[i];
        ws[W.at(u, 1) + (size_t)W.vec(4, i)] = fsum[i];
        ws[W.at(u, 3) + (size_t)W.vec(4, i)] = qdbar[i];
        if (qn) {
            qn[i * U + u] = xn[i];
            qdn[i * U + u] = xn[n + i];
            fn[i * U + u] = xn[2 * n + i];
        }
    }
}

// ------------------------------------------------------------------------------------------------ T2
struct TreePackedOut {
    double *o;  // the (unit, stage) block
    TreeWs W;
    MPCF_HD void pair(int, int, int e, double dqkj, double dvkj, double dqjk, double dvjk) const
    {
        double2 *p = reinterpret_cast<double2 *>(o + 4 * (size_t)e);  // one 32-byte sector
        p[0] = make_double2(dqkj, dvkj);
        p[1] = make_double2(dqjk, dvjk);
    }
};

template <int MAXN>
__global__ void __launch_bounds__(kThreads, MPCF_T2_BLOCKS) k_tree_derivs(GenericBlob blob, TreeWs W, long cnt, double *ws)
{
    extern __shared__ double smem[];
    const int n = blob.n;
    const int nd = 27 * n + 3;
    int *si = reinterpret_cast<int *>(smem + nd);
    for (int k = threadIdx.x; k < nd; k += blockDim.x) smem[k] = blob.dbl[k];
    for (int k = threadIdx.x; k < blob_ints(n); k += blockDim.x) si[k] = blob.ints[k];
    __syncthreads();
    const GenericModel<MAXN> m{n, smem, si};
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= cnt) return;
    const int s = blockIdx.y;
    double *o = ws + W.at(u, s);
    double q[MAXN], qd[MAXN], qdd[MAXN];
    for (int i = 0; i < n; ++i) {
        q[i] = o[(size_t)W.vec(3, i)];
        qd[i] = o[(size_t)W.vec(0, i)];
        qdd[i] = o[(size_t)W.vec(1, i)];
    }
    TreeRec rec[MAXN];
    TreeComp comp[MAXN];
    TreePackedOut out{o, W};
    TreeDerivs<GenericModel<MAXN>>::forward(m, q, qd, qdd, rec, comp);
    // M goes straight to its place in the (unit, stage) block (the thread's own contiguous run of sectors): k_tree_factor
    // factorises and inverts it there, a warp per block, in shared memory
    TreeDerivs<GenericModel<MAXN>>::backward(m, rec, comp, o + W.lf(0), out);
}

// ------------------------------------------------------------------------------------------------ T2b
// M = L^T D L on the packed ancestor pattern, then L^-1 (same pattern), one WARP per (unit, stage), all in shared memory.  The
// thread-per-unit versions (tree_derivs.cuh: factorize, invert_unit_factor — same arithmetic in the same order, kept for the
// host check) were a third of k_tree_derivs' local-memory traffic (k_tree_derivs 4.3 -> 3.3 ms per 33 k units without them; a
// thread-per-unit kernel with the matrix in shared memory fits only two warps per SM and takes 3.8 ms, this one 1.1 ms).  Both
// loops expose their parallelism through tables built once per (persistent) block:
//   factorisation, step k = n-1 .. 0: the updates M_ij -= (M_ki / D_k) M_kj over all pairs j <= i of ancestors of k are
//     independent (they read row k, which the step only rescales afterwards): lanes over the dk (dk + 1) / 2 pairs;
//   inversion: Linv_id = -L_id - sum_{d < e < depth(i)} L_ie Linv_{anc_e(i), d} needs only entries with a smaller ancestor distance
//     depth(i) - d, so all entries of one distance are independent: lanes over the entries, bucketed by distance.
// Output in place: strictly-lower entries L^-1 (or L when want_linv == 0), diagonal 1 / D_k (NaN for a non-positive pivot).
template <int MAXN>
__global__ void __launch_bounds__(256) k_tree_factor(GenericBlob blob, TreeWs W, long cnt, double *ws, int want_linv)
{
    extern __shared__ __align__(16) unsigned char fsm[];
    const int n = blob.n, npat = W.npat, t = threadIdx.x, w = t >> 5, l = t & 31;
    double *Mw = reinterpret_cast<double *>(fsm) + (size_t)w * 2 * npat, *Lw = Mw + npat;
    unsigned short *arow = reinterpret_cast<unsigned short *>(reinterpret_cast<double *>(fsm) + (size_t)8 * 2 * npat);  // [n][n]: row offset of the ancestor of k at depth a
    unsigned short *order = arow + n * n, *bstart = order + npat, *rowp = bstart + (n + 2);
    unsigned char *tri = reinterpret_cast<unsigned char *>(rowp + (n + 1));  // [n (n + 1) / 2][2]
    unsigned char *erow = tri + n * (n + 1), *edep = erow + npat, *dep = edep + npat;
    __shared__ int s_maxd;
    {
        const int *parent = blob.ints, *depth = blob.ints + 3 * n, *rowptr = blob.ints + 4 * n;
        for (int k = t; k <= n; k += 256) rowp[k] = (unsigned short)rowptr[k];
        for (int k = t; k < n; k += 256) {
            dep[k] = (unsigned char)depth[k];
            for (int j = k; j >= 0; j = parent[j]) {
                arow[k * n + depth[j]] = (unsigned short)rowptr[j];
                const int e = rowptr[k] + depth[j];
                erow[e] = (unsigned char)k;
                edep[e] = (unsigned char)depth[j];
            }
        }
        for (int idx = t; idx < n * (n + 1) / 2; idx += 256) {
            int a = 0;
            while ((a + 1) * (a + 2) / 2 <= idx) ++a;
            tri[2 * idx] = (unsigned char)a;
            tri[2 * idx + 1] = (unsigned char)(idx - a * (a + 1) / 2);
        }
        __syncthreads();
        if (t == 0) {  // strictly-lower entries bucketed by ancestor distance (counting sort, once per block)
            int md = 0;
            for (int k = 0; k < n; ++k) md = depth[k] > md ? depth[k] : md;
            s_maxd = md;
            for (int d = 0; d <= n + 1; ++d) bstart[d] = 0;
            for (int e = 0; e < npat; ++e) {
                const int dist = dep[erow[e]] - edep[e];
                if (dist > 0) ++bstart[dist + 1];
            }
            for (int d = 1; d <= n + 1; ++d) bstart[d] = (unsigned short)(bstart[d] + bstart[d - 1]);
            for (int e = 0; e < npat; ++e) {
                const int dist = dep[erow[e]] - edep[e];
                if (dist > 0) order[bstart[dist]++] = (unsigned short)e;
            }
            for (int d = n + 1; d > 0; --d) bstart[d] = bstart[d - 1];  // bucket d = [bstart[d], bstart[d + 1])
            bstart[0] = 0;
        }
        __syncthreads();
    }
    const int maxd = s_maxd;
    const double nanv = nan_value();
    for (long item = (long)blockIdx.x * 8 + w; item < cnt * 4; item += (long)gridDim.x * 8) {
        double *o = ws + W.at(item >> 2, (int)(item & 3)) + W.lf(0);
        for (int e = l; e < npat; e += 32) Mw[e] = o[e];
        __syncwarp();
        for (int k = n - 1; k >= 0; --k) {
            const int rk = rowp[k], dk = dep[k];
            double d = Mw[rk + dk];
            if (!(d > 0.0)) d = nanv;
            const double dinv = 1.0 / d;
            for (int idx = l; idx < dk * (dk + 1) / 2; idx += 32) {
                const int a = tri[2 * idx], b = tri[2 * idx + 1];  // b <= a < dk
                Mw[arow[k * n + a] + b] -= (Mw[rk + a] * dinv) * Mw[rk + b];
            }
            __syncwarp();
            for (int a = l; a < dk; a += 32) Mw[rk + a] *= dinv;
            if (l == 0) Mw[rk + dk] = d;
            __syncwarp();
        }
        if (want_linv) {
            for (int dist = 1; dist <= maxd; ++dist) {
                for (int i = bstart[dist] + l; i < bstart[dist + 1]; i += 32) {
                    const int e = order[i], r = erow[e], d = edep[e], rr = rowp[r], dr = dep[r];
                    double sum = -Mw[rr + d];
                    for (int ee = d + 1; ee < dr; ++ee) sum -= Mw[rr + ee] * Lw[arow[r * n + ee] + d];
                    Lw[rr + d] = sum;
                }
                __syncwarp();
            }
        }
        for (int e = l; e < npat; e += 32) {
            const bool diag = edep[e] == dep[erow[e]];
            o[e] = diag ? 1.0 / Mw[e] : (want_linv ? Lw[e] : Mw[e]);
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------ reverse sweep
// Vector-Jacobian product of the step (DESIGN.md §4d), thread = unit, over the unit's contiguous (unit, stage) blocks after T1, T2
// and k_tree_factor (with L^-1).  Per stage, with r = h rho and r_v its qd part:
//   mu = M^-1 r_v = L^-1 D^-1 L^-T r_v        two triangular matvecs on the packed ancestor pattern
//   A^T r_v = -(dID/dq)^T mu,  B^T r_v = -(dID/dqd)^T mu,  C r_v = mu
// O(npat) work per stage.  The fatigue states of the stages are recomputed from f, tau and the stored qd_s with the same
// arithmetic as T1 (the rows are per joint and linear in f).
template <int MAXN>
__global__ void __launch_bounds__(kThreads) k_tree_vjp(GenericBlob blob, TreeWs W, long U, long u0, long cnt, const double *tau, const double *f,
                                                       double dt, const double *dt_u, const VjpArgs a, const double *ws)
{
    extern __shared__ double smem[];
    const int n = blob.n;
    const int nd = 27 * n + 3;
    int *si = reinterpret_cast<int *>(smem + nd);
    for (int k = threadIdx.x; k < nd; k += blockDim.x) smem[k] = blob.dbl[k];
    for (int k = threadIdx.x; k < blob_ints(n); k += blockDim.x) si[k] = blob.ints[k];
    __syncthreads();
    const GenericModel<MAXN> m{n, smem, si};
    using D = Dyn<double, GenericModel<MAXN>>;
    const long lu = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (lu >= cnt) return;
    const long u = u0 + lu;
    const double h = dt_u ? dt_u[u] : dt;
    double lam[3 * MAXN], gx[3 * MAXN], ad[3 * MAXN], gt[MAXN], y[MAXN], fd[4 * MAXN];
    for (int i = 0; i < n; ++i) {
        lam[i] = a.lq ? a.lq[i * a.ldl + u] : 0.0;
        lam[n + i] = a.lqd ? a.lqd[i * a.ldl + u] : 0.0;
        lam[2 * n + i] = a.lf ? a.lf[i * a.ldl + u] : 0.0;
        gx[i] = lam[i] + (a.aq ? a.aq[i * a.lda + u] : 0.0);
        gx[n + i] = lam[n + i] + (a.aqd ? a.aqd[i * a.lda + u] : 0.0);
        gx[2 * n + i] = lam[2 * n + i] + (a.af ? a.af[i * a.lda + u] : 0.0);
        ad[i] = 0.0; ad[n + i] = 0.0; ad[2 * n + i] = 0.0;
        gt[i] = 0.0;
        // stage fatigue derivatives fdot_s, as T1 forms them: f_1 = f, f_{s+1} = f + (c_s h) fdot_s
        const double ti = tau[i * U + u], fi = f[i * U + u];
        double fs = fi;
        for (int s = 0; s < 4; ++s) {
            const double cs = s < 2 ? 0.5 : (s == 2 ? 1.0 : 0.0);
            const double k = D::fatigue_rhs(m, i, fs, ti, ws[W.at(lu, s) + (size_t)W.vec(0, i)]);
            fd[s * n + i] = k;
            fs = fi + (h * cs) * k;
        }
    }
    double gh = 0.0;
#pragma unroll 1
    for (int s = 3; s >= 0; --s) {
        const double cs = s < 2 ? 0.5 : (s == 2 ? 1.0 : 0.0);
        const double wt = (s == 0 || s == 3) ? 1.0 / 6.0 : 1.0 / 3.0;
        const double *o = ws + W.at(lu, s);  // the workspace is chunk-local
        // rho_s and r_s = h rho_s (r overwrites ad), g_dt += rho_s^T k_s
        for (int i = 0; i < n; ++i) {
            const double pq = fma(wt, lam[i], cs * ad[i]), pv = fma(wt, lam[n + i], cs * ad[n + i]), pf = fma(wt, lam[2 * n + i], cs * ad[2 * n + i]);
            gh = fma(pq, o[W.vec(0, i)], gh);
            gh = fma(pv, o[W.vec(1, i)], gh);
            gh = fma(pf, fd[s * n + i], gh);
            ad[i] = h * pq;
            ad[n + i] = h * pv;
            ad[2 * n + i] = h * pf;
        }
        // y = L^-T r_v (scatter to the ancestors), then D^-1 (diagonal entries hold 1 / D_k)
        for (int k = 0; k < n; ++k) y[k] = ad[n + k];
        for (int k = 0; k < n; ++k) {
            const double rk = ad[n + k];
            const int rp = m.rowptr(k);
            for (int j = m.parent(k); j >= 0; j = m.parent(j)) y[j] = fma(o[W.lf(rp + m.depth(j))], rk, y[j]);
        }
        for (int k = 0; k < n; ++k) y[k] *= o[W.lf(m.rowptr(k) + m.depth(k))];
        // mu = L^-1 y, in place from the leaves up (row k reads only its ancestors, which come earlier)
        for (int k = n - 1; k >= 0; --k) {
            double acc = y[k];
            const int rp = m.rowptr(k);
            for (int j = m.parent(k); j >= 0; j = m.parent(j)) acc = fma(o[W.lf(rp + m.depth(j))], y[j], acc);
            y[k] = acc;
        }
        // J_s^T r: own-joint terms, then the ancestor-pattern scatter of -(dID/dq)^T mu and -(dID/dqd)^T mu
        for (int i = 0; i < n; ++i) {
            const double rf = ad[2 * n + i];
            gt[i] += fma(2.0 * m.fat(i, 1) * m.fat(i, 2) * tau[i * U + u], rf, y[i]);
            ad[n + i] = fma(2.0 * m.fat(i, 1) * m.fat(i, 3) * o[W.vec(0, i)], rf, ad[i]);
            ad[2 * n + i] = -m.fat(i, 0) * rf;
            ad[i] = 0.0;
        }
        for (int k = 0; k < n; ++k) {
            const int rp = m.rowptr(k);
            const double mk = y[k];
            for (int j = k; j >= 0; j = m.parent(j)) {
                const int e = rp + m.depth(j);
                ad[j] -= o[W.dqkj(e)] * mk;
                ad[n + j] -= o[W.dvkj(e)] * mk;
                if (j != k) {
                    ad[k] -= o[W.dqjk(e)] * y[j];
                    ad[n + k] -= o[W.dvjk(e)] * y[j];
                }
            }
        }
        for (int i = 0; i < 3 * n; ++i) gx[i] += ad[i];
    }
    for (int i = 0; i < n; ++i) {
        a.gq[i * a.ldg + u] = gx[i];
        a.gqd[i * a.ldg + u] = gx[n + i];
        a.gf[i * a.ldg + u] = gx[2 * n + i];
        a.gtau[i * a.ldgt + u] = gt[i];
    }
    if (a.gdt) a.gdt[u] = gh;
}

// ------------------------------------------------------------------------------------------------ T3
MPCF_DI void cp_async8s(unsigned smem_addr, const double *gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_addr), "l"(gmem) : "memory");
}
MPCF_DI void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
MPCF_DI void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct TreeChainArgs {
    TreeWs W;
    long U, UJ, cnt;         // plane strides of the inputs / of jac, units in this launch
    const double *tau, *dt_u;
    double dt;
    const double *ws;
    double *jac;
    double *scratch;         // [gridDim.x][2][n][128]: fatigue-row sums and P per column (L2-resident, coalesced)
    const double *fat;       // device blob: fat[n][4]
    const int *ints;         // device blob ints: parent n | jtype n | keep n | depth n | rowptr n + 1
    int fence0;              // always 0: `if (a.fence0 > i) continue;` is never taken but cuts the unrolled triangular solves into one
                             // basic block per column (cf. StaticModel::skip); in one block ptxas hoists ~800 loads and spills 6.7 KB
};

// NR: padded row count (even, n <= NR); XS: column stride of the X arrays
template <int NR>
__global__ void __launch_bounds__(128, 2) k_tree_chain(TreeChainArgs a)
{
    const TreeWs W = a.W;
    const int n = W.n, npat = W.npat;
    const int NC = 3 * n + 1;
    const int XS = (NC + 15) & ~15;
    extern __shared__ __align__(16) double sm[];
    double *DqT = sm, *DvT = DqT + n * NR, *LT = DvT + n * NR;      // column-major: column c at c * NR; LT is NR x NR (padding = 0)
    double *V = LT + NR * NR;                                      // 2 buffers x 4 vectors x NR: qd_s, qdd_s, fnext_s, extra_s
    double *Xq = V + 2 * 4 * NR, *Xv = Xq + n * XS;
    unsigned short *okj = reinterpret_cast<unsigned short *>(Xv + n * XS), *ojk = okj + npat;
    const int t = threadIdx.x;
    const bool active = t < NC;
    // ---- once per CTA: zero the dense matrices, build the packed-entry -> dense-offset tables ----
    for (int i = t; i < 2 * n * NR + NR * NR; i += 128) sm[i] = 0.0;
    for (int i = t; i < 2 * 4 * NR; i += 128) V[i] = 0.0;
    {
        const int *parent = a.ints, *depth = a.ints + 3 * n, *rowptr = a.ints + 4 * n;
        for (int k = t; k < n; k += 128)
            for (int j = k; j >= 0; j = parent[j]) {
                const int e = rowptr[k] + depth[j];
                okj[e] = (unsigned short)(j * NR + k);  // entry (row k, col j)
                ojk[e] = (unsigned short)(k * NR + j);  // entry (row j, col k)
            }
    }
    __syncthreads();
    const int jq = t < n ? t : -1, jv = (t >= n && t < 2 * n) ? t - n : -1, jt = (t >= 2 * n && t < 3 * n) ? t - 2 * n : -1;
    const bool isdt = t == 3 * n;
    const unsigned sDq = (unsigned)__cvta_generic_to_shared(DqT), sDv = (unsigned)__cvta_generic_to_shared(DvT),
                   sLT = (unsigned)__cvta_generic_to_shared(LT), sV = (unsigned)__cvta_generic_to_shared(V);
    // group A of (unit u, stage s): dID/dq, dID/dqd entries + the four vectors (into vector buffer s & 1); group B: the factor
    auto issue_A = [&](long u, int s) {
        const double *w = a.ws + W.at(u, s);
        for (int e = t; e < npat; e += 128) {
            const unsigned kj = okj[e] * 8u, jk = ojk[e] * 8u;
            cp_async8s(sDq + kj, w + (size_t)W.dqkj(e));
            cp_async8s(sDv + kj, w + (size_t)W.dvkj(e));
            if (kj != jk) {
                cp_async8s(sDq + jk, w + (size_t)W.dqjk(e));
                cp_async8s(sDv + jk, w + (size_t)W.dvjk(e));
            }
        }
        const unsigned vb = sV + (unsigned)((s & 1) * 4 * NR) * 8u;
        for (int i = t; i < n; i += 128) {
            cp_async8s(vb + (unsigned)(0 * NR + i) * 8u, w + (size_t)W.vec(0, i));
            cp_async8s(vb + (unsigned)(1 * NR + i) * 8u, w + (size_t)W.vec(1, i));
            cp_async8s(vb + (unsigned)(2 * NR + i) * 8u, w + (size_t)W.vec(2, i));
            cp_async8s(vb + (unsigned)(3 * NR + i) * 8u, w + (size_t)W.vec(4, i));
        }
        cp_async_commit();
    };
    auto issue_B = [&](long u, int s) {
        const double *w = a.ws + W.at(u, s);
        for (int e = t; e < npat; e += 128) cp_async8s(sLT + okj[e] * 8u, w + (size_t)W.lf(e));  // L_kj at (row k, col j); diagonal: 1 / D_k
        cp_async_commit();
    };
    double *AF = a.scratch + (size_t)blockIdx.x * 2 * n * 128 + t, *Ps = AF + (size_t)n * 128;
    long u = blockIdx.x;
    if (u < a.cnt) { issue_A(u, 0); issue_B(u, 0); }
    for (; u < a.cnt; u += gridDim.x) {
        const double h = a.dt_u ? a.dt_u[u] : a.dt;
        double acc[NR];
        if (active)
            for (int c = 0; c < n; ++c) { Xq[c * XS + t] = (c == jq) ? 1.0 : 0.0; Xv[c * XS + t] = (c == jv) ? 1.0 : 0.0; }
        const long PC = 4 * n + 1;
        const long ocol = isdt ? 4 * n : t;
        double *jq_out = a.jac + (size_t)ocol * a.UJ + u;  // + row * PC * UJ
#pragma unroll 1
        for (int s = 0; s < 4; ++s) {
            const long un = u + gridDim.x;  // the item after (u, 3) is (un, 0)
            const bool more = s < 3 || un < a.cnt;
            const long u2 = s < 3 ? u : un;
            const int s2 = s < 3 ? s + 1 : 0;
            cp_async_wait<1>();  // group A of this stage has landed (B may still be in flight)
            __syncthreads();
            // ---- phase 1: acc = dID/dq X[q] + dID/dqd X[qd] ----
            if (s == 0) {
#pragma unroll
                for (int r = 0; r < NR; ++r) acc[r] = jq >= 0 ? DqT[jq * NR + r] : (jv >= 0 ? DvT[jv * NR + r] : 0.0);
            } else {
#pragma unroll
                for (int r = 0; r < NR; ++r) acc[r] = 0.0;
                if (active) {
#pragma unroll 1
                    for (int c = 0; c < n; ++c) {
                        const double xq = Xq[c * XS + t], xv = Xv[c * XS + t];
                        const double2 *dq = reinterpret_cast<const double2 *>(DqT + c * NR);
                        const double2 *dv = reinterpret_cast<const double2 *>(DvT + c * NR);
                        // two half-columns: all broadcast loads of a half first (80 staging registers), then its FMAs.  Left to
                        // itself ptxas funnels every load through one register and each DFMA waits for its own LDS; the never-taken
                        // branch keeps the halves in separate basic blocks so the loads are not sunk back into the FMA stream
#pragma unroll
                        for (int b = 0; b < NR / 2; b += NR / 4) {
                            double2 A[NR / 4], B[NR / 4];
#pragma unroll
                            for (int i = 0; i < NR / 4; ++i) { A[i] = dq[b + i]; B[i] = dv[b + i]; }
#pragma unroll
                            for (int i = 0; i < NR / 4; ++i) {
                                const int r2 = b + i;
                                acc[2 * r2] = fma(A[i].x, xq, acc[2 * r2]);
                                acc[2 * r2 + 1] = fma(A[i].y, xq, acc[2 * r2 + 1]);
                                acc[2 * r2] = fma(B[i].x, xv, acc[2 * r2]);
                                acc[2 * r2 + 1] = fma(B[i].y, xv, acc[2 * r2 + 1]);
                            }
                            if (a.fence0 > b) break;
                        }
                    }
                }
            }
            __syncthreads();  // every thread is done with this stage's dID/dq, dID/dqd: the next stage's may land
            if (more) issue_A(u2, s2); else cp_async_commit();
            cp_async_wait<1>();  // group B of this stage has landed (the A just issued may still be in flight)
            __syncthreads();
            // ---- phase 2: rhs = -acc (+ e_j in the tau columns); M k = rhs with M = L^T D L ----
#pragma unroll
            for (int r = 0; r < NR; ++r) acc[r] = ((r == jt) ? 1.0 : 0.0) - acc[r];
#pragma unroll
            for (int i = NR - 2; i >= 0; --i) {  // L^T y = rhs: y_i = rhs_i - sum_{k > i} L_ki y_k   (column i of L is contiguous)
                if (a.fence0 > i) continue;
                const double *col = LT + i * NR;
                constexpr int kMaxPairs = NR / 2;
                double2 Lc[kMaxPairs];
                const int k0 = (i + 2) & ~1;  // first aligned pair; an odd start contributes one scalar term
                double s0 = ((i + 1) & 1) ? col[i + 1] * acc[i + 1] : 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
                for (int k = k0; k < NR; k += 2) Lc[(k - k0) / 2] = *reinterpret_cast<const double2 *>(col + k);
#pragma unroll
                for (int k = k0; k < NR; k += 2) {
                    const double2 L2 = Lc[(k - k0) / 2];
                    if (((k - k0) / 2) & 1) { s2 = fma(L2.x, acc[k], s2); s3 = fma(L2.y, acc[k + 1], s3); }
                    else { s0 = fma(L2.x, acc[k], s0); s1 = fma(L2.y, acc[k + 1], s1); }
                }
                acc[i] -= (s0 + s1) + (s2 + s3);
            }
#pragma unroll
            for (int i = 0; i < NR; ++i) acc[i] *= LT[i * NR + i];  // 1 / D_i (0 in the padding rows)
#pragma unroll
            for (int j = 0; j < NR - 1; ++j) {  // L x = w, column-oriented
                if (a.fence0 > j) continue;
                const double *col = LT + j * NR;
                const double xj = -acc[j];
                const int i0 = (j + 2) & ~1;
                double2 Lc[NR / 2];
#pragma unroll
                for (int i = i0; i < NR; i += 2) Lc[(i - i0) / 2] = *reinterpret_cast<const double2 *>(col + i);
                if ((j + 1) & 1) acc[j + 1] = fma(col[j + 1], xj, acc[j + 1]);
#pragma unroll
                for (int i = i0; i < NR; i += 2) {
                    acc[i] = fma(Lc[(i - i0) / 2].x, xj, acc[i]);
                    acc[i + 1] = fma(Lc[(i - i0) / 2].y, xj, acc[i + 1]);
                }
            }
            __syncthreads();  // every thread is done with this stage's factor
            if (more) issue_B(u2, s2); else cp_async_commit();
            // ---- update: Yv, accumulators (scratch, fire-and-forget), next stage's X (column-private) ----
            const double cs = s < 2 ? 0.5 : (s == 2 ? 1.0 : 0.0);
            const double *Vs = V + (s & 1) * 4 * NR;
            if (active) {
#pragma unroll
                for (int r = 0; r < NR; ++r) {
                    if (r < n) {
                        const double yv = h * acc[r] + (isdt ? Vs[1 * NR + r] : 0.0);
                        acc[r] = yv;
                        const double xvold = Xv[r * XS + t];
                        if (s == 0) {
                            jq_out[(size_t)(n + r) * PC * a.UJ] = ((r == jv) ? 1.0 : 0.0) - yv * (1.0 / 6.0);
                            Ps[r * 128] = yv;
                            AF[r * 128] = Vs[2 * NR + r] * yv + (isdt ? Vs[3 * NR + r] : 0.0);  // dt column: + sum_s gamma_s / 6 fdot_s
                        } else if (s < 3) {
                            atomicAdd(Ps + r * 128, yv);
                            // qd column j, row j: the X1[qd] term sum_s fcoef_s travels with stage 1
                            atomicAdd(AF + r * 128, Vs[2 * NR + r] * yv + ((s == 1 && r == jv) ? Vs[3 * NR + r] : 0.0));
                        }
                        const double yq = h * xvold + (isdt ? Vs[0 * NR + r] : 0.0);
                        Xq[r * XS + t] = ((r == jq) ? 1.0 : 0.0) + cs * yq;
                        Xv[r * XS + t] = ((r == jv) ? 1.0 : 0.0) + cs * yv;
                    }
                }
            }
            if (s == 3 && active) {
                // ---- epilogue of this column, in four row blocks: a block's scratch loads first (independent, one round trip),
                // then its stores.  (All rows at once would need 240 registers here, and a kernel whose first schedule does not fit
                // the register file makes ptxas re-schedule EVERY region for minimum pressure: each DFMA then waits for its own LDS.)
#pragma unroll
                for (int b = 0; b < NR; b += NR / 4) {
                    double Pv[NR / 4], Av[NR / 4];
#pragma unroll
                    for (int i = 0; i < NR / 4; ++i)
                        if (b + i < n) { Pv[i] = Ps[(b + i) * 128]; Av[i] = AF[(b + i) * 128]; }
#pragma unroll
                    for (int i = 0; i < NR / 4; ++i) {
                        const int r = b + i;
                        if (r < n) {
                            const double aq = ((r == jq) ? 1.0 : 0.0) + h * ((r == jv) ? 1.0 : 0.0) + (h * (1.0 / 6.0)) * Pv[i] + (isdt ? Vs[3 * NR + r] : 0.0);
                            jq_out[(size_t)r * PC * a.UJ] = aq;
                            atomicAdd(jq_out + (size_t)(n + r) * PC * a.UJ, (2.0 * Pv[i] + acc[r]) * (1.0 / 6.0));
                            double af = Av[i];
                            if (r == jt) {
                                const double z = a.fat[4 * r] * h;
                                af += 2.0 * a.fat[4 * r + 1] * a.fat[4 * r + 2] * a.tau[(size_t)r * a.U + u] * h * (1.0 + z * (-0.5 + z * (1.0 / 6.0 - z * (1.0 / 24.0))));
                            }
                            jq_out[(size_t)(2 * n + r) * PC * a.UJ] = af;
                        }
                    }
                    if (a.fence0 > b) break;
                }
            }
        }
        // ---- the n fatigue columns: closed form (d(q+, qd+)/df = 0, df+/df = diag RK4 amplification) ----
        for (int idx = t; idx < 3 * n * n; idx += 128) {
            const int r = idx / n, j = idx - r * n;
            double v = 0.0;
            if (r == 2 * n + j) {
                const double z = a.fat[4 * j] * h;
                v = 1.0 + z * (-1.0 + z * (0.5 + z * (-1.0 / 6.0 + z * (1.0 / 24.0))));
            }
            a.jac[((size_t)r * PC + 3 * n + j) * a.UJ + u] = v;
        }
    }
    cp_async_wait<0>();
}


// ------------------------------------------------------------------------------------------------ T3 on the FP64 tensor cores
// Same recursion with every per-stage product as DMMA (mma.sync m8n8k4 f64) GEMMs.  CTA = (unit, slab of 64 Jacobian
// columns), 4 warps x 16 columns, two CTAs per SM; all column state of a warp is warp-private, so the only block-wide
// barriers are the ones that swap the stage matrices:
//   Z = [dID/dq | dID/dqd] . [X[q] ; X[qd]]     M = NR, K = 2 NR, N = 64   (stage 1: Z is a column of the matrices, no product)
//   T = D^-1 L^-T (E_tau - Z),  K = L^-1 T      with L^-1 from k_tree_derivs (invert_unit_factor: same ancestor pattern as L), so
//                                               M^-1 = L^-1 D^-1 L^-T is two TRIANGULAR products (only the tiles on or below /
//                                               above the diagonal are issued); the B operands come straight from the previous
//                                               product's accumulator fragments through warp shuffles
// Accumulators P and the fatigue-row sums are register fragments (2 n-tiles x MT m-tiles per warp = 4 MT doubles each per
// thread), X lives in shared memory k-major (row stride 68 = 4 mod 16: conflict-free B-fragment loads), the matrices row-major
// with strides 2 NR + 4 / NR + 4 (conflict-free A-fragment loads, both of L^-1 and of its transpose).
MPCF_DI void dmma884(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
MPCF_DI void red_add(double *p, double v) { asm volatile("red.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory"); }

template <int NR>
struct TcLayout {
    static constexpr int MT = NR / 8, RSA = 2 * NR + 4, RSL = NR + 4, XS = 68, KS1 = NR / 2, KS2 = NR / 4;
    static constexpr int oDA = 0, oLI = oDA + NR * RSA, oDI = oLI + NR * RSL, oV = oDI + NR, oTF = oV + 2 * 4 * NR, oX = oTF + NR, oY1 = oX + 2 * NR * XS, nD = oY1 + 4 * MT * 128;
    static size_t bytes(int npat) { return (size_t)nD * sizeof(double) + (size_t)3 * npat * sizeof(unsigned short); }
};

// NJ: n-tiles (8 Jacobian columns each) per warp; 8 / NJ warps per CTA cover the slab's 64 columns
template <int NR, int NJ>
__global__ void __launch_bounds__(256 / NJ, 2) k_tree_chain_tc(TreeChainArgs a)
{
    using Ly = TcLayout<NR>;
    constexpr int NTH = 256 / NJ;
    constexpr int MT = Ly::MT, RSA = Ly::RSA, RSL = Ly::RSL, XS = Ly::XS, KS1 = Ly::KS1, KS2 = Ly::KS2;
    const TreeWs W = a.W;
    const int n = W.n, npat = W.npat;
    const int NC = 3 * n + 1;
    extern __shared__ __align__(16) double sm[];
    double *DA = sm + Ly::oDA, *LI = sm + Ly::oLI, *DI = sm + Ly::oDI, *V = sm + Ly::oV, *TF = sm + Ly::oTF, *Xs = sm + Ly::oX, *Y1 = sm + Ly::oY1;
    unsigned short *okj = reinterpret_cast<unsigned short *>(sm + Ly::nD), *ojk = okj + npat, *okl = ojk + npat;
    const int t = threadIdx.x, w = t >> 5, l = t & 31, g = l >> 2, tq = l & 3;
    const int slab = blockIdx.y;
    for (int i = t; i < Ly::oX; i += NTH) sm[i] = 0.0;
    __syncthreads();
    {
        const int *parent = a.ints, *depth = a.ints + 3 * n, *rowptr = a.ints + 4 * n;
        for (int k = t; k < n; k += NTH) {
            LI[k * RSL + k] = 1.0;  // unit diagonal of L^-1 (the padding rows stay 0, so the padding rows of every product are 0)
            for (int j = k; j >= 0; j = parent[j]) {
                const int e = rowptr[k] + depth[j];
                okj[e] = (unsigned short)(k * RSA + j);  // entry (row k, col j) of [dID/dq | dID/dqd], row-major
                ojk[e] = (unsigned short)(j * RSA + k);
                okl[e] = (unsigned short)(j == k ? NR * RSL + k : k * RSL + j);  // L^-1_kj, or 1 / D_k into the vector behind the matrix
            }
        }
    }
    __syncthreads();
    const unsigned sDA = (unsigned)__cvta_generic_to_shared(DA), sLI = (unsigned)__cvta_generic_to_shared(LI), sV = (unsigned)__cvta_generic_to_shared(V);
    auto issue_A = [&](long u, int s) {
        const double *ws = a.ws + W.at(u, s);
        for (int e = t; e < npat; e += NTH) {
            const unsigned kj = okj[e] * 8u, jk = ojk[e] * 8u;
            cp_async8s(sDA + kj, ws + (size_t)W.dqkj(e));
            cp_async8s(sDA + kj + (unsigned)NR * 8u, ws + (size_t)W.dvkj(e));
            if (kj != jk) {
                cp_async8s(sDA + jk, ws + (size_t)W.dqjk(e));
                cp_async8s(sDA + jk + (unsigned)NR * 8u, ws + (size_t)W.dvjk(e));
            }
        }
        const unsigned vb = sV + (unsigned)((s & 1) * 4 * NR) * 8u;
        for (int i = t; i < n; i += NTH) {
            cp_async8s(vb + (unsigned)(0 * NR + i) * 8u, ws + (size_t)W.vec(0, i));
            cp_async8s(vb + (unsigned)(1 * NR + i) * 8u, ws + (size_t)W.vec(1, i));
            cp_async8s(vb + (unsigned)(2 * NR + i) * 8u, ws + (size_t)W.vec(2, i));
            cp_async8s(vb + (unsigned)(3 * NR + i) * 8u, ws + (size_t)W.vec(4, i));
        }
        cp_async_commit();
    };
    auto issue_B = [&](long u, int s) {
        const double *ws = a.ws + W.at(u, s);
        for (int e = t; e < npat; e += NTH) cp_async8s(sLI + okl[e] * 8u, ws + (size_t)W.lf(e));
        cp_async_commit();
    };
    // this thread's fragment elements: rows 8 mt + g, columns cb + 8 j + 2 tq + e (cb = the warp's first column)
    const int cb = 64 * slab + 8 * NJ * w;
    const long PC = 4 * n + 1;
    unsigned mq = 0, mv = 0, mt_ = 0;  // bit (mt * NJ + j) * 2 + e: X1[q] = 1, X1[qd] = 1, tau-column unit entry
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int j = 0; j < NJ; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int r = 8 * mt + g, c = cb + 8 * j + 2 * tq + e, bit = (mt * NJ + j) * 2 + e;
                if (r < n && c == r) mq |= 1u << bit;
                if (r < n && c == n + r) mv |= 1u << bit;
                if (r < n && c == 2 * n + r) mt_ |= 1u << bit;
            }
    bool dtf[NJ][2];
#pragma unroll
    for (int j = 0; j < NJ; ++j) { dtf[j][0] = cb + 8 * j + 2 * tq == 3 * n; dtf[j][1] = cb + 8 * j + 2 * tq + 1 == 3 * n; }
    unsigned sp = 0;  // bit mt * NJ + j: some lane of this warp has a special entry in tile (mt, j) -> warp-uniform
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int tile = mt * NJ + j;
            const bool mine = (((mq | mv | mt_) >> (tile * 2)) & 3u) != 0 || dtf[j][0] || dtf[j][1];
            if (__any_sync(0xffffffffu, mine)) sp |= 1u << tile;
        }
    auto isdt = [&](int j, int e) { return dtf[j][e]; };
    const double *Xcol = Xs + 8 * NJ * w;  // this warp's columns
    // Units are handed out dynamically (one counter per slab, zeroed by the launcher) instead of strided by CTA: units u .. u + 3
    // share every 32-byte sector of the AoSoA workspace and of the [plane][unit] Jacobian, and only units that are in flight at
    // about the same time meet in L2 (with a static stride the CTAs drift apart: 36 GB of DRAM reads per 32k units instead of 5).
    __shared__ unsigned long long s_unit[2];
    unsigned long long *counter = reinterpret_cast<unsigned long long *>(a.scratch) + slab;
    if (t == 0) s_unit[0] = atomicAdd(counter, 1ull);
    __syncthreads();
    long u = (long)s_unit[0];
    int par = 0;
    if (u < a.cnt) { issue_A(u, 0); issue_B(u, 0); }
    for (; u < a.cnt; par ^= 1) {
        if (t == 0) s_unit[par ^ 1] = atomicAdd(counter, 1ull);  // the unit after this one: read behind the stage barriers
        long un = a.cnt;
        const double h = a.dt_u ? a.dt_u[u] : a.dt;
        // closed-form tau-column term of the fatigue rows (row r, column tau_r), one value per joint
        double tf = 0.0;
        if (t < n) {
            const double z = a.fat[4 * t] * h;
            tf = 2.0 * a.fat[4 * t + 1] * a.fat[4 * t + 2] * a.tau[(size_t)t * a.U + u] * h * (1.0 + z * (-0.5 + z * (1.0 / 6.0 - z * (1.0 / 24.0))));
        }
        double acc[MT][NJ][2], yv[MT][NJ][2], Pq[MT][NJ][2], AF[MT][NJ][2];
#pragma unroll 1
        for (int s = 0; s < 4; ++s) {
            // copy groups in flight here: this stage's matrices (A) and, at stage 1 only, its factor (B, issued behind the previous
            // unit's last product); the factor of stages 2-4 is issued right below, once every warp has left the previous update
            if (s == 0) cp_async_wait<1>(); else cp_async_wait<0>();
            __syncthreads();
            if (s == 3) un = (long)s_unit[par ^ 1];
            const bool more = s < 3 || un < a.cnt;
            const long u2 = s < 3 ? u : un;
            const int s2 = s < 3 ? s + 1 : 0;
            if (s > 0) issue_B(u, s);
            if (s == 0 && t < n) TF[t] = tf;  // every warp has left the previous unit's epilogue; read after many barriers
            // ---- Z ----
            if (s == 0) {  // X1 = unit columns: Z is a column of dID/dq (q columns), of dID/dqd (qd columns) or 0
#pragma unroll
                for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                    for (int j = 0; j < NJ; ++j)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int c = cb + 8 * j + 2 * tq + e;
                            const int cc = c < n ? c : (c < 2 * n ? NR + c - n : -1);
                            acc[mt][j][e] = cc >= 0 ? DA[(8 * mt + g) * RSA + cc] : 0.0;
                        }
            } else {
#pragma unroll
                for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                    for (int j = 0; j < NJ; ++j) { acc[mt][j][0] = 0.0; acc[mt][j][1] = 0.0; }
                const double *ap = DA + g * RSA + tq, *bp = Xcol + tq * XS + g;
                double af[MT], bf[NJ], af2[MT], bf2[NJ];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) af[mt] = ap[8 * mt * RSA];
                for (int j = 0; j < NJ; ++j) bf[j] = bp[8 * j];
#pragma unroll 1
                for (int ks = 0; ks < KS1; ks += 2) {  // two k-steps per trip, the next one's fragments loaded ahead of this one's DMMA
                    const double *ap1 = ap + 4 * (ks + 1), *bp1 = bp + 4 * (ks + 1) * XS;
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) af2[mt] = ap1[8 * mt * RSA];
                    for (int j = 0; j < NJ; ++j) bf2[j] = bp1[8 * j];
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                        for (int j = 0; j < NJ; ++j) dmma884(acc[mt][j][0], acc[mt][j][1], af[mt], bf[j]);
                    if (ks + 2 < KS1) {
                        const double *ap2 = ap + 4 * (ks + 2), *bp2 = bp + 4 * (ks + 2) * XS;
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) af[mt] = ap2[8 * mt * RSA];
                        for (int j = 0; j < NJ; ++j) bf[j] = bp2[8 * j];
                    }
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                        for (int j = 0; j < NJ; ++j) dmma884(acc[mt][j][0], acc[mt][j][1], af2[mt], bf2[j]);
                }
            }
            __syncthreads();
            if (more) issue_A(u2, s2); else cp_async_commit();
            cp_async_wait<1>();
            __syncthreads();
            // ---- rhs = E_tau - Z, staged in this warp's (dead) X[q] rows so that the next product reads its B fragments with the same
            //      conflict-free loads as the first one ----
            double *xw = Xs + 8 * NJ * w + 2 * tq;
            const double *bq = Xcol + tq * XS + g;
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const double r0 = (((mt_ >> ((mt * NJ + j) * 2)) & 1) ? 1.0 : 0.0) - acc[mt][j][0];
                    const double r1 = (((mt_ >> ((mt * NJ + j) * 2 + 1)) & 1) ? 1.0 : 0.0) - acc[mt][j][1];
                    *reinterpret_cast<double2 *>(xw + (8 * mt + g) * XS + 8 * j) = make_double2(r0, r1);
                    yv[mt][j][0] = 0.0; yv[mt][j][1] = 0.0;
                }
            __syncwarp();
            // ---- T = D^-1 L^-T rhs: A(r, k) = L^-1[k][r], only the tiles with 4 ks + 3 >= 8 mt ----
#pragma unroll
            for (int ks = 0; ks < KS2; ++ks) {
                double bb[NJ];
#pragma unroll
                for (int j = 0; j < NJ; ++j) bb[j] = bq[4 * ks * XS + 8 * j];
#pragma unroll
                for (int mt = 0; mt <= ks / 2 && mt < MT; ++mt) {
                    const double af = LI[(4 * ks + tq) * RSL + 8 * mt + g];
#pragma unroll
                    for (int j = 0; j < NJ; ++j) dmma884(yv[mt][j][0], yv[mt][j][1], af, bb[j]);
                }
            }
            __syncwarp();
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const double di = DI[8 * mt + g];
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    *reinterpret_cast<double2 *>(xw + (8 * mt + g) * XS + 8 * j) = make_double2(yv[mt][j][0] * di, yv[mt][j][1] * di);
                    acc[mt][j][0] = 0.0; acc[mt][j][1] = 0.0;
                }
            }
            __syncwarp();
            // ---- K = L^-1 T: A(r, k) = L^-1[r][k], only the tiles with 4 ks <= 8 mt + 7 ----
#pragma unroll
            for (int ks = 0; ks < KS2; ++ks) {
                double bb[NJ];
#pragma unroll
                for (int j = 0; j < NJ; ++j) bb[j] = bq[4 * ks * XS + 8 * j];
#pragma unroll
                for (int mt = ks / 2; mt < MT; ++mt) {
                    const double af = LI[(8 * mt + g) * RSL + 4 * ks + tq];
#pragma unroll
                    for (int j = 0; j < NJ; ++j) dmma884(acc[mt][j][0], acc[mt][j][1], af, bb[j]);
                }
            }
            __syncwarp();
            if (s == 3) {  // the next unit's first factor: its stage 1 has no product to hide the copy behind
                __syncthreads();
                if (more) issue_B(u2, 0); else cp_async_commit();
            }
            // ---- update: Yv, accumulators, next stage's X (warp-private columns).  Per 8 x 8 tile one warp-uniform branch: only the
            //      few tiles that hold a unit entry of X1, a tau-column unit entry or the dt column take the general form ----
            const double cs = s < 2 ? 0.5 : (s == 2 ? 1.0 : 0.0);
            const double csh = cs * h;
            const double *Vs = V + (s & 1) * 4 * NR;
            double *y1 = Y1 + t;
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const int r = 8 * mt + g;
                const double fn = Vs[2 * NR + r];
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int tile = mt * NJ + j;
                    double2 xvold = make_double2(0.0, 0.0);
                    if (s > 0) xvold = *reinterpret_cast<const double2 *>(xw + (NR + r) * XS + 8 * j);
                    double xqn[2], xvn[2];
                    if ((sp >> tile) & 1) {
                        const double qdd_r = Vs[1 * NR + r], qd_r = Vs[0 * NR + r], ex_r = Vs[3 * NR + r];
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int bit = tile * 2 + e;
                            const double x1q = ((mq >> bit) & 1) ? 1.0 : 0.0, x1v = ((mv >> bit) & 1) ? 1.0 : 0.0;
                            const bool dtc = isdt(j, e);
                            const double y = fma(h, acc[mt][j][e], dtc ? qdd_r : 0.0);
                            acc[mt][j][e] = y;
                            if (s == 0) {
                                Pq[mt][j][e] = y;
                                AF[mt][j][e] = fma(fn, y, dtc ? ex_r : 0.0);
                                y1[bit * NTH] = y;
                            } else if (s < 3) {
                                Pq[mt][j][e] += y;
                                AF[mt][j][e] = fma(fn, y, AF[mt][j][e] + ((s == 1 && x1v != 0.0) ? ex_r : 0.0));
                            }
                            const double xo = s > 0 ? (e == 0 ? xvold.x : xvold.y) : x1v;
                            xqn[e] = fma(cs, fma(h, xo, dtc ? qd_r : 0.0), x1q);
                            xvn[e] = fma(cs, y, x1v);
                        }
                    } else {
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const double y = h * acc[mt][j][e];
                            acc[mt][j][e] = y;
                            if (s == 0) {
                                Pq[mt][j][e] = y;
                                AF[mt][j][e] = fn * y;
                                y1[(tile * 2 + e) * NTH] = y;
                            } else if (s < 3) {
                                Pq[mt][j][e] += y;
                                AF[mt][j][e] = fma(fn, y, AF[mt][j][e]);
                            }
                            xqn[e] = csh * (e == 0 ? xvold.x : xvold.y);
                            xvn[e] = cs * y;
                        }
                    }
                    if (s < 3) {
                        *reinterpret_cast<double2 *>(xw + r * XS + 8 * j) = make_double2(xqn[0], xqn[1]);
                        *reinterpret_cast<double2 *>(xw + (NR + r) * XS + 8 * j) = make_double2(xvn[0], xvn[1]);
                    }
                }
            }
            if (s == 3) {
                // ---- Jacobian rows, column by column: one pointer per column, stepped by 8 rows per m-tile ----
                const size_t RSJ = (size_t)PC * a.UJ;  // one Jacobian row (all columns, plane stride UJ)
                const double h6 = h * (1.0 / 6.0);
#pragma unroll
                for (int j = 0; j < NJ; ++j)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int c = cb + 8 * j + 2 * tq + e;
                        const bool dtc = isdt(j, e);
                        if (c < NC) {
                            double *p = a.jac + (size_t)(dtc ? 4 * n : c) * a.UJ + u + (size_t)g * RSJ;
#pragma unroll
                            for (int mt = 0; mt < MT; ++mt, p += 8 * RSJ) {
                                const int r = 8 * mt + g, tile = mt * NJ + j, bit = tile * 2 + e;
                                if (r < n) {
                                    double jq = h6 * Pq[mt][j][e];
                                    double jv = (2.0 * Pq[mt][j][e] - y1[bit * NTH] + acc[mt][j][e]) * (1.0 / 6.0);
                                    double jf = AF[mt][j][e];
                                    if ((sp >> tile) & 1) {
                                        const double x1q = ((mq >> bit) & 1) ? 1.0 : 0.0, x1v = ((mv >> bit) & 1) ? 1.0 : 0.0;
                                        jq += x1q + h * x1v + (dtc ? Vs[3 * NR + r] : 0.0);
                                        jv += x1v;
                                        jf += ((mt_ >> bit) & 1) ? TF[r] : 0.0;
                                    }
                                    __stcs(p, jq);
                                    __stcs(p + (size_t)n * RSJ, jv);
                                    __stcs(p + (size_t)2 * n * RSJ, jf);
                                }
                            }
                        }
                    }
            }
            __syncwarp();
        }
        u = un;
    }
    cp_async_wait<0>();
}

// The n fatigue columns of the Jacobian in closed form (d(q+, qd+)/df = 0, df+/df = diag of the RK4 amplification of the linear
// fatigue rows): 3n x n planes per unit, written coalesced (thread = unit, blockIdx.y = Jacobian row) beside the chain kernel.
__global__ void __launch_bounds__(256) k_tree_fill_fatigue_cols(int n, long cnt, long UJ, const double *fat, double dt, const double *dt_u, double *jac)
{
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= cnt) return;
    const int r = blockIdx.y;
    const long PC = 4 * n + 1;
    double *p = jac + ((size_t)r * PC + 3 * n) * UJ + u;
    double v = 0.0;
    if (r >= 2 * n) {
        const double z = fat[4 * (r - 2 * n)] * (dt_u ? dt_u[u] : dt);
        v = 1.0 + z * (-1.0 + z * (0.5 + z * (-1.0 / 6.0 + z * (1.0 / 24.0))));
    }
    for (int j = 0; j < n; ++j) __stcs(p + (size_t)j * UJ, (j == r - 2 * n) ? v : 0.0);
}

// ------------------------------------------------------------------------------------------------ launcher
#ifndef MPCF_TC_NJ
#define MPCF_TC_NJ 2
#endif
static constexpr int TC_NJ = MPCF_TC_NJ;  // n-tiles per warp of the tensor-core chain kernel: 1 -> 8 warps per CTA, 2 -> 4 warps

bool tree_jvp_supported(const LaunchModel &m) { return (m.fam == FAM_GENERIC16 || m.fam == FAM_GENERIC64) && m.n <= 40; }

static size_t tree_factor_smem(int n, int npat)
{
    return (size_t)8 * 2 * npat * sizeof(double) + ((size_t)n * n + npat + (n + 2) + (n + 1)) * sizeof(unsigned short) + (size_t)n * (n + 1) + 2 * npat + n + 16;
}
static constexpr int tree_factor_smem_limit(int maxn) { return maxn > 16 ? 128 * 1024 : 48 * 1024; }
static size_t tree_chain_smem(int n, int NR, int npat)
{
    const int NC = 3 * n + 1, XS = (NC + 15) & ~15;
    return ((size_t)2 * n * NR + (size_t)NR * NR + 2 * 4 * NR + (size_t)2 * n * XS) * sizeof(double) + (size_t)2 * npat * sizeof(unsigned short);
}

template <int MAXN, int NR>
static cudaError_t run_tree(const LaunchModel &m, int npat, long U, long cnt, const double *q, const double *qd, const double *tau, const double *f,
                            double dt, const double *dt_u, double *qn, double *qdn, double *fn, double *jac, long UJ, double *ws, size_t ws_bytes,
                            cudaStream_t s)
{
    const int n = m.n;
    TreeWs W{n, npat, TreeWs::planes(n, npat)};
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    const size_t smem3 = tree_chain_smem(n, NR, npat);
    // n <= 38 fits two CTAs per SM (<= 113 KB each); n = 39, 40 run one CTA per SM
    cudaError_t e;
    if ((e = raise_smem_limit<k_tree_chain<NR>>(NR > 16 ? 160 * 1024 : 56 * 1024)) != cudaSuccess) return e;
    if ((e = raise_smem_limit<k_tree_factor<MAXN>>(tree_factor_smem_limit(MAXN))) != cudaSuccess) return e;
    if ((e = raise_smem_limit<k_tree_chain_tc<NR, TC_NJ>>(NR > 16 ? 113 * 1024 : 56 * 1024)) != cudaSuccess) return e;
    const int ctas_per_sm = smem3 <= 113 * 1024 ? 2 : 1;
    const long grid3_max = (long)nsm * ctas_per_sm;
    // workspace = [stage data of the chunk][fatigue-row scratch of the chain kernel's CTAs]
    const size_t scratch_bytes = (size_t)grid3_max * 2 * 40 * 128 * sizeof(double);
    if (ws_bytes <= scratch_bytes) return cudaErrorInvalidValue;
    const size_t per_unit = tree_ws_doubles_per_unit(n, npat) * sizeof(double);
    long Uc = (long)((ws_bytes - scratch_bytes) / per_unit);
    Uc -= Uc % 32;
    if (Uc < 32) return cudaErrorInvalidValue;
    // whole waves of the derivative kernel (thread = (unit, stage), MPCF_T2_BLOCKS 128-thread blocks per SM): a chunk that ends
    // in a partly filled wave wastes it (measured: 28,416-unit chunks +2.5 % over 32,768 on 148 SMs)
    const long wave = (long)nsm * MPCF_T2_BLOCKS * 32;
    if (Uc > wave) Uc -= Uc % wave;
    double *scratch = ws + (size_t)Uc * tree_ws_doubles_per_unit(n, npat);
    const size_t smem12 = blob_smem_bytes(n);
    for (long u0 = 0; u0 < cnt; u0 += Uc) {
        const long c = (cnt - u0) < Uc ? (cnt - u0) : Uc;
        const unsigned gb = (unsigned)((c + kThreads - 1) / kThreads);
        k_tree_stages<MAXN><<<gb, kThreads, smem12, s>>>(m.blob, W, U, c, q + u0, qd + u0, tau + u0, f + u0, dt, dt_u ? dt_u + u0 : nullptr,
                                                        qn ? qn + u0 : nullptr, qdn ? qdn + u0 : nullptr, fn ? fn + u0 : nullptr, ws);
        // default: the tensor-core chain kernel; MPCF_TREE_CHAIN=scalar selects the DFMA kernel (kept as a cross-check: same
        // recursion with triangular solves instead of the products with L^-1)
        const char *env = getenv("MPCF_TREE_CHAIN");
        const bool use_tc = !(env && env[0] == 's');
        k_tree_derivs<MAXN><<<dim3(gb, 4), kThreads, smem12, s>>>(m.blob, W, c, ws);
        {
            const long blocks = (c * 4 + 7) / 8;
            const long cap = (long)nsm * 4;
            k_tree_factor<MAXN><<<(unsigned)(blocks < cap ? blocks : cap), 256, tree_factor_smem(n, npat), s>>>(m.blob, W, c, ws, use_tc ? 1 : 0);
            g_launches.fetch_add(1);
        }
        TreeChainArgs a{W, U, UJ, c, tau + u0, dt_u ? dt_u + u0 : nullptr, dt, ws, jac + u0, scratch, m.blob.dbl + 23 * n, m.blob.ints, 0};
        if (use_tc) {
            const int nslab = (3 * n + 1 + 63) / 64;
            const long gx_max = (long)nsm * 2 / nslab;
            const unsigned gx = (unsigned)(c < gx_max ? c : gx_max);
            cudaMemsetAsync(scratch, 0, 64, s);  // the per-slab unit counters
            k_tree_chain_tc<NR, TC_NJ><<<dim3(gx, nslab), 256 / TC_NJ, TcLayout<NR>::bytes(npat), s>>>(a);
            k_tree_fill_fatigue_cols<<<dim3((unsigned)((c + 255) / 256), 3 * n), 256, 0, s>>>(n, c, UJ, a.fat, dt, a.dt_u, a.jac);
            g_launches.fetch_add(1);
        } else {
            const unsigned g3 = (unsigned)(c < grid3_max ? c : grid3_max);
            k_tree_chain<NR><<<g3, 128, smem3, s>>>(a);
        }
        g_launches.fetch_add(3);
    }
    return cudaGetLastError();
}

// Reverse sweep: T1, T2 and k_tree_factor (with L^-1) unchanged, then k_tree_vjp.  It needs no chain-kernel scratch and no fatigue
// columns, so the whole workspace holds stage data.
template <int MAXN>
static cudaError_t run_tree_vjp(const LaunchModel &m, int npat, long U, long cnt, const double *q, const double *qd, const double *tau,
                                const double *f, double dt, const double *dt_u, const VjpArgs &a, double *qn, double *qdn, double *fn, double *ws,
                                size_t ws_bytes, cudaStream_t s)
{
    const int n = m.n;
    TreeWs W{n, npat, TreeWs::planes(n, npat)};
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    const cudaError_t e = raise_smem_limit<k_tree_factor<MAXN>>(tree_factor_smem_limit(MAXN));
    if (e != cudaSuccess) return e;
    const size_t per_unit = tree_ws_doubles_per_unit(n, npat) * sizeof(double);
    long Uc = (long)(ws_bytes / per_unit);
    Uc -= Uc % 32;
    if (Uc < 32) return cudaErrorInvalidValue;
    const long wave = (long)nsm * MPCF_T2_BLOCKS * 32;  // whole waves of the derivative kernel (see run_tree)
    if (Uc > wave) Uc -= Uc % wave;
    const size_t smem12 = blob_smem_bytes(n);
    for (long u0 = 0; u0 < cnt; u0 += Uc) {
        const long c = (cnt - u0) < Uc ? (cnt - u0) : Uc;
        const unsigned gb = (unsigned)((c + kThreads - 1) / kThreads);
        k_tree_stages<MAXN><<<gb, kThreads, smem12, s>>>(m.blob, W, U, c, q + u0, qd + u0, tau + u0, f + u0, dt, dt_u ? dt_u + u0 : nullptr,
                                                        qn ? qn + u0 : nullptr, qdn ? qdn + u0 : nullptr, fn ? fn + u0 : nullptr, ws);
        k_tree_derivs<MAXN><<<dim3(gb, 4), kThreads, smem12, s>>>(m.blob, W, c, ws);
        const long blocks = (c * 4 + 7) / 8, cap = (long)nsm * 4;
        k_tree_factor<MAXN><<<(unsigned)(blocks < cap ? blocks : cap), 256, tree_factor_smem(n, npat), s>>>(m.blob, W, c, ws, 1);
        k_tree_vjp<MAXN><<<gb, kThreads, smem12, s>>>(m.blob, W, U, u0, c, tau, f, dt, dt_u, a, ws);
        g_launches.fetch_add(4);
    }
    return cudaGetLastError();
}

cudaError_t launch_step_vjp_tree(const LaunchModel &m, int npat, long U, long cnt, const double *q, const double *qd, const double *tau,
                                 const double *f, double dt, const double *dt_u, const VjpArgs &a, double *qn, double *qdn, double *fn,
                                 double *ws, size_t ws_bytes, cudaStream_t s)
{
    if (cnt <= 0) return cudaSuccess;
    if (m.n <= 16) return run_tree_vjp<16>(m, npat, U, cnt, q, qd, tau, f, dt, dt_u, a, qn, qdn, fn, ws, ws_bytes, s);
    if (m.n <= 40) return run_tree_vjp<40>(m, npat, U, cnt, q, qd, tau, f, dt, dt_u, a, qn, qdn, fn, ws, ws_bytes, s);
    return cudaErrorInvalidValue;
}

size_t tree_jvp_workspace_bytes(int n, int npat, long U)
{
    long units = U < (1L << 15) ? U : (1L << 15);  // chunks of at most 32768 units (1.9 GB for the 37-joint tree) ...
    units = (units + 31) / 32 * 32;
    int dev = 0, nsm = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    const long wave = (long)nsm * MPCF_T2_BLOCKS * 32;  // ... cut to whole waves of the derivative kernel (see run_tree)
    if (units > wave) units -= units % wave;
    const size_t scratch = (size_t)148 * 4 * 2 * 40 * 128 * sizeof(double);  // generous: up to 2x the CTAs of a 148-SM part
    return (size_t)units * tree_ws_doubles_per_unit(n, npat) * sizeof(double) + scratch;
}

cudaError_t launch_step_jvp_tree(const LaunchModel &m, int npat, long U, long cnt, const double *q, const double *qd, const double *tau,
                                 const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn, double *jac, long UJ,
                                 double *ws, size_t ws_bytes, cudaStream_t s)
{
    if (cnt <= 0) return cudaSuccess;
    if (m.n <= 16) return run_tree<16, 16>(m, npat, U, cnt, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, UJ, ws, ws_bytes, s);
    if (m.n <= 40) return run_tree<40, 40>(m, npat, U, cnt, q, qd, tau, f, dt, dt_u, qn, qdn, fn, jac, UJ, ws, ws_bytes, s);
    return cudaErrorInvalidValue;
}

}  // namespace mpcf
