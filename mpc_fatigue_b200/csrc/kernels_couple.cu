// kernels_couple.cu — coupled fatigue of a two-arm model carrying one box (config C3: dual-arm 2 x Pilz 6-DOF "with coupled
// fatigue states").  Builder-defined (the reference has no dynamics-mode fatigue; what it has is the box equilibrium
// F_L,z + F_R,z = m g, python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:197,272-274, and tau = ID - J^T F, :292-293); the oracle twin is
// oracle/core.inc.h: step_rk4_coupled.  Zero-order hold over the step, like tau itself:
//
//   Phi_c   = sum of the fatigue states of arm c at the start of the step
//   s_c     = Phi_other / (Phi_0 + Phi_1)          share of the box weight arm c carries (the less fatigued arm takes more)
//   g_c(q)  = J_ee,c(q)^T [0, 0, w, 0, 0, 0]       torque holding the whole box weight w at arm c's end-effector
//   theat_i = tau_i + s_c g_i(q(t_k))              torque the motor of joint i delivers: what heats its winding
//
// The dynamics see tau, the fatigue right-hand side sees theat, so the Jacobian pipeline runs unchanged with theat in the
// fatigue terms, and because theat is constant over the step and RK4 is linear in a constant forcing, the extra Jacobian
// blocks are closed form.  With Hd_i := d f+_i / d theat_i = 2 kappa_i ctau_i theat_i h phi(lambda_i h),
// phi(z) = 1 - z/2 + z^2/6 - z^3/24 (RK4 response of y' = -lambda y + c):
//
//   d f+_i / d q_j  += Hd_i s_c dg_i/dq_j          j on the same arm
//   d f+_i / d f_j   = [i = j] amp(lambda_i h) + Hd_i g_i ds_c/df_j      every j of BOTH arms: the cross-arm block
//   dg_i/dq_j = F . (z_j x (z_i x d_i))  (j <= i),  F . (z_i x (z_j x d_j))  (j > i),   d_i = p_ee - o_i, F = (0, 0, w)
//
// One thread per unit; mode 0 writes theat before the pipeline, mode 1 patches the Jacobian after it.
#include "launch.cuh"

namespace mpcf {

template <int L>
struct ArmKin {
    double z[L][3], o[L][3], pf[3];
    // world joint axes / origins of one serial arm and the end-effector point (frame on joint `ej`, offset `ep` in that joint's frame)
    MPCF_DI void run(const StaticParams<L> &P, const double *q, int ej, const double *ep)
    {
        double R[9], pos[3];
#pragma unroll
        for (int i = 0; i < L; ++i) {
            double s, c;
            sincos(q[i], &s, &c);
            double Rl[9];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                Rl[3 * r + 0] = P.Rp[i][3 * r] * c + P.Rp[i][3 * r + 1] * s;
                Rl[3 * r + 1] = P.Rp[i][3 * r + 1] * c - P.Rp[i][3 * r] * s;
                Rl[3 * r + 2] = P.Rp[i][3 * r + 2];
            }
            if (i == 0) {
#pragma unroll
                for (int k = 0; k < 9; ++k) R[k] = Rl[k];
#pragma unroll
                for (int k = 0; k < 3; ++k) pos[k] = P.pp[i][k];
            } else {
                double Rn[9];
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    pos[r] += R[3 * r] * P.pp[i][0] + R[3 * r + 1] * P.pp[i][1] + R[3 * r + 2] * P.pp[i][2];
#pragma unroll
                    for (int cc = 0; cc < 3; ++cc) Rn[3 * r + cc] = R[3 * r] * Rl[cc] + R[3 * r + 1] * Rl[3 + cc] + R[3 * r + 2] * Rl[6 + cc];
                }
#pragma unroll
                for (int k = 0; k < 9; ++k) R[k] = Rn[k];
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) { z[i][k] = R[3 * k + 2]; o[i][k] = pos[k]; }
            if (i == ej) {
#pragma unroll
                for (int r = 0; r < 3; ++r) pf[r] = pos[r] + R[3 * r] * ep[0] + R[3 * r + 1] * ep[1] + R[3 * r + 2] * ep[2];
            }
        }
    }
    // g_i = F . (z_i x d_i), F = (0, 0, w); joints past the end-effector joint do not carry the box
    MPCF_DI double g(int i, int ej, double w) const
    {
        if (i > ej) return 0.0;
        const double dx = pf[0] - o[i][0], dy = pf[1] - o[i][1];
        return w * (z[i][0] * dy - z[i][1] * dx);
    }
    MPCF_DI double dg(int i, int j, int ej, double w) const
    {
        if (i > ej || j > ej) return 0.0;
        const int a = j <= i ? j : i, b = j <= i ? i : j;  // F . (z_a x (z_b x d_b)), a = min, b = max
        const double d[3] = {pf[0] - o[b][0], pf[1] - o[b][1], pf[2] - o[b][2]};
        double t[3], v[3];
        cross3(z[b], d, t);
        cross3(z[a], t, v);
        return w * v[2];
    }
};

struct CoupleArgs {
    double weight;
    int ee_joint[2];   // end-effector joint, local to its arm
    double ee_p[2][3]; // end-effector point in that joint's frame
};

template <int L>
__global__ void __launch_bounds__(kThreads) k_couple(const __grid_constant__ StaticParams<L> P0, const __grid_constant__ StaticParams<L> P1,
                                                    CoupleArgs ca, long cnt, long ld, const double *q, const double *f, const double *tau,
                                                    double *theat, long ld_t, int mode, double dt, const double *dt_u, double *jac, long UJ)
{
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= cnt) return;
    constexpr int n = 2 * L;
    double Phi[2] = {0.0, 0.0};
#pragma unroll
    for (int i = 0; i < n; ++i) Phi[i / L] += f[(long)i * ld + u];
    const double S = Phi[0] + Phi[1], iS = 1.0 / S;
    const double share[2] = {Phi[1] * iS, Phi[0] * iS};
    // d share_c / d f_j: -share_c / S for j on arm c, (1 - share_c) / S for j on the other arm
    const double h = dt_u ? dt_u[u] : dt;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const StaticParams<L> &P = c == 0 ? P0 : P1;
        double qa[L];
#pragma unroll
        for (int i = 0; i < L; ++i) qa[i] = q[(long)(c * L + i) * ld + u];
        ArmKin<L> K;
        K.run(P, qa, ca.ee_joint[c], ca.ee_p[c]);
        if (mode == 0) {
#pragma unroll
            for (int i = 0; i < L; ++i) theat[(long)(c * L + i) * ld_t + u] = tau[(long)(c * L + i) * ld + u] + share[c] * K.g(i, ca.ee_joint[c], ca.weight);
            continue;
        }
        const long PC = 4 * n + 1;
#pragma unroll
        for (int i = 0; i < L; ++i) {
            const double gi = K.g(i, ca.ee_joint[c], ca.weight);
            const double T = tau[(long)(c * L + i) * ld + u] + share[c] * gi;
            const double zl = P.fat[i][0] * h;
            const double phi = 1.0 + zl * (-0.5 + zl * (1.0 / 6.0 - zl * (1.0 / 24.0)));
            const double amp = 1.0 + zl * (-1.0 + zl * (0.5 + zl * (-1.0 / 6.0 + zl * (1.0 / 24.0))));
            const double Hd = 2.0 * P.fat[i][1] * P.fat[i][2] * T * h * phi;
            double *row = jac + (size_t)(2 * n + c * L + i) * PC * UJ + u;
#pragma unroll
            for (int j = 0; j < L; ++j) row[(size_t)(c * L + j) * UJ] += Hd * share[c] * K.dg(i, j, ca.ee_joint[c], ca.weight);
#pragma unroll
            for (int j = 0; j < n; ++j) {
                const double ds = (j / L == c) ? -share[c] * iS : (1.0 - share[c]) * iS;
                row[(size_t)(3 * n + j) * UJ] = ((j == c * L + i) ? amp : 0.0) + Hd * gi * ds;
            }
        }
    }
}

// mode 0: theat[n][ld_t] = tau + share * g(q).  mode 1: patch the fatigue rows of jac (plane stride UJ) after the pipeline.
cudaError_t launch_couple(const LaunchModel &m, const CoupleHost &ch, long cnt, long ld, const double *q, const double *f, const double *tau,
                          double *theat, long ld_t, int mode, double dt, const double *dt_u, double *jac, long UJ, cudaStream_t s)
{
    if (cnt <= 0) return cudaSuccess;
    CoupleArgs ca;
    ca.weight = ch.weight;
    for (int c = 0; c < 2; ++c) {
        ca.ee_joint[c] = ch.ee_joint[c];
        for (int k = 0; k < 3; ++k) ca.ee_p[c][k] = ch.ee_p[c][k];
    }
    cudaError_t e = cudaErrorInvalidValue;  // the two-arm families only
    with_chains(m, [&](auto L, const auto *chains, auto nchains) {
        if constexpr (decltype(nchains)::value == 2) {
            k_couple<L><<<(unsigned)((cnt + kThreads - 1) / kThreads), kThreads, 0, s>>>(chains[0], chains[1], ca, cnt, ld, q, f, tau, theat, ld_t,
                                                                                        mode, dt, dt_u, jac, UJ);
            g_launches.fetch_add(1);
            e = cudaGetLastError();
        }
    });
    return e;
}

}  // namespace mpcf
