// kernels_rows.cu — fused reference-mode OCP node rows: every constraint row and the running cost that the reference's
// scripts build per shooting node around the bridge Functions, in ONE launch per batch, plus the first derivatives of the
// kinematic rows.  One thread per (scenario, node) unit, node-major units u = k * B + b.
//
//   one arm  (python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:130-177, python/Pilz_3_DOF/*.py): rows
//        [0,3)      ee_pos - p_ref                 (the line constraint uses its x, y components, :152-156)
//        [3,3+n)    tau = ID(q, qd, 0) + wsign J^T [F; 0]                                          (:134)
//        then n     Euler defect q + h qd - q_next                                                 (:160,170)
//        then n     thermal defect T+ - T_next  (zero-order hold, mpc_principal.py:296-301,325)
//        cost       w_F F.F + w_qd qd.qd        (w_F = -1: the script's -F^T F, :177)
//   two arms (python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:244-293,454-475; python/Centauro_script/mpc_principal.py:229-327;
//             RepeatedMPCwithThermal_confriction.py:251-273): rows
//        [0,3)      force equilibrium     F_L + F_R - fdes                                         (mpc_principal.py:229)
//        [3,6)      moment equilibrium    (pL - pR) x F_L + (pR - pL) x F_R                        (:234)
//        [6]        |pL - pR|^2 - dist2_ref                                                        (Box_Pilz_6DOF2.py:283-285)
//        [7,10)     relative position     R_L^T (pR - pL) - (the same at the previous node | rel_pos0)   (:241-246)
//        [10,13)    relative orientation  e(R_L R_R^T) - rel_ori0,  e = (S21, S20, S10), S = (Ro - Ro^T)/2   (:248-258)
//        [13,23)    friction cones        A1 (-R_L^T F_L), A2 (-R_R^T F_R)  <= 0                   (confriction.py:251-273)
//        [23,26)    p_box - p_ref,  p_box = (pL + pR) / 2
//        then tau (n), Euler defect (n), thermal defect (n) as above, with tau = ID + wsign (J_L^T [F_L;0] + J_R^T [F_R;0])
//        cost       w_box |p_box - p_ref|^2 + w_qd qd.qd + w_F (F_L.F_L + F_R.F_R)                 (mpc_principal.py:281-284)
//
// One pair of thread-per-unit bodies serves every kernel family through dispatch: the compile-time chains and forests and
// the run-time trees (branched trees, prismatic and continuous joints, shared ancestors such as a torso joint under both
// arms).  Arm c's frame sits on joint a.ee_joint[c] (global index, -1 = world-fixed: constant pose, zero Jacobian).
//   RowsBody runs ONE RNEA sweep with the forces injected as external link forces (frames.cuh: WrenchExtTree, which also
//   captures both frame poses on the way), so tau = ID + wsign (J_L^T [F_L;0] + J_R^T [F_R;0]) sums both terms on shared
//   ancestors without an explicit Jacobian; the previous node's relative position walks the two frames' ancestor paths only.
//   RowsJacBody (launched only when dtau_dF or kin_jac is requested) computes the poses of the frames' ancestors once, takes
//   their Jacobian columns (d tau / d F = wsign J_c,lin^T, non-zero in both arm blocks on shared ancestors) and evaluates the
//   kinematic rows (box_kin_rows, generic over double | Dual) once per direction in (q, F), seeded with the pose tangent
//   (q_j: dp_c = J_c,lin[:, j], dR_c = [J_c,ang[:, j]]x R_c, zero when j is not an ancestor of frame c; F: the force entry
//   itself) — no frame kinematics per direction.
// The torque rows' derivatives in (q, qd) come from mpcf_node_eval_ref_jvp_batch (analytic); d tau / d F and d T+ / d tau are
// emitted here in closed form.
// Oracle twin: oracle/core.inc.h: ocp_rows.
#include "frames.cuh"

namespace mpcf {

struct RowsArgs {
    int narm, n, N;
    long B;
    int ee_joint[2];     // end-effector joint: global index, -1 = world-fixed frame
    double ee_p[2][3], ee_R[2][9];
    double wsign, fdes[3], dist2_ref, mu, p_ref[3], w_box, w_qd, w_F, h;
};

// the 26 kinematic rows of the two-arm node (header comment) from the two end-effector poses and the two forces
template <class T>
MPCF_DI void box_kin_rows(const RowsArgs &a, const T *pL, const T *RL, const T *pR, const T *RR, const T *FL, const T *FR, const T *relprev,
                          const double *ori0, T *g)
{
    T d[3] = {pL[0] - pR[0], pL[1] - pR[1], pL[2] - pR[2]};
#pragma unroll
    for (int k = 0; k < 3; ++k) g[k] = FL[k] + FR[k] - a.fdes[k];
    T dF[3] = {FL[0] - FR[0], FL[1] - FR[1], FL[2] - FR[2]};  // (pL - pR) x F_L + (pR - pL) x F_R = (pL - pR) x (F_L - F_R)
    cross3(d, dF, g + 3);
    g[6] = d[0] * d[0] + d[1] * d[1] + d[2] * d[2] - a.dist2_ref;
#pragma unroll
    for (int k = 0; k < 3; ++k) g[7 + k] = -(RL[k] * d[0] + RL[3 + k] * d[1] + RL[6 + k] * d[2]) - relprev[k];  // R_L^T (pR - pL)
    // Ro = R_L R_R^T ; e = ((Ro21 - Ro12)/2, (Ro20 - Ro02)/2, (Ro10 - Ro01)/2)
    auto Ro = [&](int r, int c) { return RL[3 * r] * RR[3 * c] + RL[3 * r + 1] * RR[3 * c + 1] + RL[3 * r + 2] * RR[3 * c + 2]; };
    g[10] = 0.5 * (Ro(2, 1) - Ro(1, 2)) - ori0[0];
    g[11] = 0.5 * (Ro(2, 0) - Ro(0, 2)) - ori0[1];
    g[12] = 0.5 * (Ro(1, 0) - Ro(0, 1)) - ori0[2];
    // friction cones on the forces the environment exerts, in the end-effector frames: f1 = -R_L^T F_L, f2 = -R_R^T F_R
    T f1[3], f2[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        f1[k] = -(RL[k] * FL[0] + RL[3 + k] * FL[1] + RL[6 + k] * FL[2]);
        f2[k] = -(RR[k] * FR[0] + RR[3 + k] * FR[1] + RR[6 + k] * FR[2]);
    }
    const double mu = a.mu;
    g[13] = -f1[1];
    g[14] = f1[2] - mu * f1[1];
    g[15] = -f1[2] - mu * f1[1];
    g[16] = f1[0] - mu * f1[1];
    g[17] = -f1[0] - mu * f1[1];
    g[18] = f2[1];
    g[19] = f2[0] + mu * f2[1];
    g[20] = -f2[0] + mu * f2[1];
    g[21] = f2[2] + mu * f2[1];
    g[22] = -f2[2] + mu * f2[1];
#pragma unroll
    for (int k = 0; k < 3; ++k) g[23 + k] = 0.5 * (pL[k] + pR[k]) - a.p_ref[k];
}

// the arm count: fixed by a compile-time family (one per serial chain), so its instantiations carry no code for the other
template <class MP>
MPCF_DI int arms(const RowsArgs &a)
{
    if constexpr (MP::kStatic) return MP::MAXN / MP::kChain;
    else return a.narm;
}

// rows, cost and (optional) d T+ / d tau: one RNEA sweep with the forces as external link forces
struct RowsBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, RowsArgs a, const double *q, const double *qd, const double *F, const double *T,
                            const double *q_last, const double *T_last, const double *rel_pos0, const double *rel_ori0, double *rows,
                            double *cost, double *dT_dtau)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n(), narm = arms<MP>(a), KIN = narm == 2 ? 26 : 3;
        const long b = u % a.B;
        const int k = (int)(u / a.B);
        double qa[MP::MAXN], qda[MP::MAXN], zero[MP::MAXN], tau[MP::MAXN];
        double cqd = 0.0, cF = 0.0, ckin = 0.0;
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            qa[i] = q[(long)i * U + u];
            qda[i] = qd[(long)i * U + u];
            zero[i] = 0.0;
            cqd += qda[i] * qda[i];
        }
        double Fv[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            Fv[i] = i < 3 * narm ? F[(long)i * U + u] : 0.0;
            cF += Fv[i] * Fv[i];
        }
        WrenchExtTree<MP, true> ext;
        ext.nee = narm;
        ext.wsign = a.wsign;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            if (c >= narm) break;
            ext.je[c] = a.ee_joint[c];  // -1 (world-fixed frame) never matches a link: no torque, the constant pose stays
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                ext.Wl[c][r] = Fv[3 * c + r];
                ext.Wl[c][3 + r] = 0.0;
                ext.pl[c][r] = a.ee_p[c][r];
                ext.Pw[c][r] = a.ee_p[c][r];
            }
#pragma unroll
            for (int r = 0; r < 9; ++r) { ext.Rf[c][r] = a.ee_R[c][r]; ext.Rw[c][r] = a.ee_R[c][r]; }
        }
        JointVar<double> jv[MP::MAXN];
        Dyn<double, MP>::template rnea_impl<false>(m, qa, jv, qda, zero, tau, ext);
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            const double t = tau[i];
            // static models re-read q, qd rather than hold every joint's in registers across the sweep (forests spill less)
            const double qi = MP::kStatic ? q[(long)i * U + u] : qa[i], qdi = MP::kStatic ? qd[(long)i * U + u] : qda[i];
            rows[(long)(KIN + i) * U + u] = t;
            // Euler defect against the next node's q (last node: the trailing q_N)
            const double qn = qi + a.h * qdi;
            const double qnext = k + 1 < a.N ? q[(long)i * U + u + a.B] : (q_last ? q_last[(long)i * a.B + b] : qn);
            rows[(long)(KIN + n + i) * U + u] = qn - qnext;
            double Tdef = 0.0, dTdt = 0.0;
            if (T) {
                const double lam = m.fat(i, 0), kap = m.fat(i, 1);
                const double Pl = m.fat(i, 2) * t * t + m.fat(i, 3) * qdi * qdi;
                const double Ti = T[(long)i * U + u];
                const double za = exp(-lam * a.h);
                // expm1: 1 - za cancels as lam h -> 0 (lam h = 1e-12: ~1e-4 relative), and the gain must meet h kap there
                const double gain = lam == 0.0 ? a.h * kap : -expm1(-lam * a.h) * (kap / lam);
                const double Tn = za * Ti + gain * Pl;
                const double Tnext = k + 1 < a.N ? T[(long)i * U + u + a.B] : (T_last ? T_last[(long)i * a.B + b] : Tn);
                Tdef = Tn - Tnext;
                dTdt = gain * 2.0 * m.fat(i, 2) * t;
            }
            rows[(long)(KIN + 2 * n + i) * U + u] = Tdef;
            if (dT_dtau) dT_dtau[(long)i * U + u] = dTdt;
        }
        if (narm == 2) {
            double relprev[3], ori0[3], g[26];
            if (k == 0) {
#pragma unroll
                for (int r = 0; r < 3; ++r) relprev[r] = rel_pos0 ? rel_pos0[(long)r * a.B + b] : 0.0;
            } else {  // the same quantity at the previous node (unit u - B): the two frames' ancestor paths only
                double pL[3], RL[9], pR[3], RR[9];
                frame_pose_walk(m, a.ee_joint[0], a.ee_R[0], a.ee_p[0], q, U, u - a.B, pL, RL);
                frame_pose_walk(m, a.ee_joint[1], a.ee_R[1], a.ee_p[1], q, U, u - a.B, pR, RR);
#pragma unroll
                for (int r = 0; r < 3; ++r) relprev[r] = RL[r] * (pR[0] - pL[0]) + RL[3 + r] * (pR[1] - pL[1]) + RL[6 + r] * (pR[2] - pL[2]);
            }
#pragma unroll
            for (int r = 0; r < 3; ++r) ori0[r] = rel_ori0 ? rel_ori0[(long)r * a.B + b] : 0.0;
            box_kin_rows<double>(a, ext.Pw[0], ext.Rw[0], ext.Pw[1], ext.Rw[1], Fv, Fv + 3, relprev, ori0, g);
#pragma unroll
            for (int r = 0; r < 26; ++r) rows[(long)r * U + u] = g[r];
            ckin = g[23] * g[23] + g[24] * g[24] + g[25] * g[25];
        } else {
#pragma unroll
            for (int r = 0; r < 3; ++r) rows[(long)r * U + u] = ext.Pw[0][r] - a.p_ref[r];
        }
        cost[u] = a.w_box * ckin + a.w_qd * cqd + a.w_F * cF;
    }
};

// dtau_dF [n][3 narm][U] and kin_jac [KIN][n + 3 narm][U] (either may be NULL): frame kinematics of the two frames' ancestors
// once, then one box_kin_rows<Dual> per direction seeded with the pose tangent
struct RowsJacBody {
    template <class MP>
    static MPCF_DI void run(const MP &m, long u, long U, RowsArgs a, const double *q, const double *F, double *dtau_dF, double *kin_jac)
    {
        constexpr int UNR = MP::kStatic ? MP::MAXN : 1;
        const int n = m.n(), narm = arms<MP>(a), KIN = narm == 2 ? 26 : 3, ND = n + 3 * narm;
        unsigned long long anc[2] = {0ull, 0ull};  // ancestor sets of the frames (bit j: joint j moves frame c)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            if (c >= narm) break;
            for (int j = a.ee_joint[c]; j >= 0; j = m.parent(j)) anc[c] |= 1ull << j;
        }
        const unsigned long long both = anc[0] | anc[1];
        double oR[MP::MAXN][9], op[MP::MAXN][3];
        fk_subset(m, both, q, U, u, oR, op);
        double pe[2][3], Re[2][9], Fv[6];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const int cc = c < narm ? c : 0;
            Dyn<double, MP>::frame_pose(a.ee_joint[cc], a.ee_R[cc], a.ee_p[cc], oR, op, pe[c], Re[c]);
        }
#pragma unroll
        for (int i = 0; i < 6; ++i) Fv[i] = i < 3 * narm ? F[(long)i * U + u] : 0.0;
        if (dtau_dF) {
#pragma unroll UNR
            for (int j = 0; j < n; ++j) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    if (c >= narm) break;
                    double col[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
                    if ((anc[c] >> j) & 1ull) jac_column(m, j, oR, op, pe[c], col);
#pragma unroll
                    for (int r = 0; r < 3; ++r) dtau_dF[((long)j * 3 * narm + 3 * c + r) * U + u] = a.wsign * col[r];
                }
            }
        }
        if (!kin_jac) return;
        const long ld = (long)ND * U;  // stride between the rows of one direction
        const Dual relprev[3] = {Dual(0.0), Dual(0.0), Dual(0.0)};
        const double ori0[3] = {0.0, 0.0, 0.0};
#pragma unroll 1
        for (int d = 0; d < ND; ++d) {
            double *out = kin_jac + (long)d * U + u;
            if (d < n && !((both >> d) & 1ull)) {  // joint d moves neither frame
                for (int r = 0; r < KIN; ++r) out[r * ld] = 0.0;
                continue;
            }
            if (narm == 1) {  // rows p - p_ref: J_lin, nothing in F
                double col[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
                if (d < n) jac_column(m, d, oR, op, pe[0], col);
#pragma unroll
                for (int r = 0; r < 3; ++r) out[r * ld] = col[r];
                continue;
            }
            Dual pd[2][3], Rd[2][9], Fd[6], g[26];
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                double col[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
                if (d < n && ((anc[c] >> d) & 1ull)) jac_column(m, d, oR, op, pe[c], col);
#pragma unroll
                for (int r = 0; r < 3; ++r) pd[c][r] = Dual(pe[c][r], col[r]);
#pragma unroll
                for (int cc = 0; cc < 3; ++cc) {  // d R = [w]x R, column by column
                    const double rc[3] = {Re[c][cc], Re[c][3 + cc], Re[c][6 + cc]};
                    double dr[3];
                    cross3(col + 3, rc, dr);
#pragma unroll
                    for (int r = 0; r < 3; ++r) Rd[c][3 * r + cc] = Dual(Re[c][3 * r + cc], dr[r]);
                }
            }
#pragma unroll
            for (int i = 0; i < 6; ++i) Fd[i] = Dual(Fv[i], d == n + i ? 1.0 : 0.0);
            box_kin_rows<Dual>(a, pd[0], Rd[0], pd[1], Rd[1], Fd, Fd + 3, relprev, ori0, g);
#pragma unroll
            for (int r = 0; r < 26; ++r) out[r * ld] = g[r].d;
        }
    }
};

cudaError_t launch_ocp_rows(const LaunchModel &m, const RowsHost &h, const double *q, const double *qd, const double *F, const double *T,
                            const double *q_last, const double *T_last, const double *rel_pos0, const double *rel_ori0, double *rows,
                            double *cost, double *dtau_dF, double *dT_dtau, double *kin_jac, cudaStream_t s)
{
    if (h.B <= 0 || h.N <= 0) return cudaSuccess;
    RowsArgs a;
    a.narm = h.narm; a.n = m.n; a.N = h.N; a.B = h.B;
    for (int c = 0; c < 2; ++c) {
        a.ee_joint[c] = h.ee_joint[c];
        for (int k = 0; k < 3; ++k) a.ee_p[c][k] = h.ee_p[c][k];
        for (int k = 0; k < 9; ++k) a.ee_R[c][k] = h.ee_R[c][k];
    }
    a.wsign = h.wsign; a.dist2_ref = h.dist2_ref; a.mu = h.mu; a.w_box = h.w_box; a.w_qd = h.w_qd; a.w_F = h.w_F; a.h = h.h;
    for (int k = 0; k < 3; ++k) { a.fdes[k] = h.fdes[k]; a.p_ref[k] = h.p_ref[k]; }
    const long U = a.B * a.N;
    cudaError_t e = dispatch<RowsBody>(m, U, 1, s, a, q, qd, F, T, q_last, T_last, rel_pos0, rel_ori0, rows, cost, dT_dtau);
    if (e != cudaSuccess || !(dtau_dF || kin_jac)) return e;
    return dispatch<RowsJacBody>(m, U, 1, s, a, q, F, dtau_dF, kin_jac);
}

}  // namespace mpcf
