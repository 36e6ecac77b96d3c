// frames.cuh — frame kinematics shared by the reference-mode node evaluation (kernels_basic.cu) and the fused OCP rows
// (kernels_rows.cu): Jacobian columns, contact wrenches riding the RNEA sweep, and frame poses by ancestor walk.
#pragma once
#include "launch.cuh"

namespace mpcf {

// column i of the LOCAL_WORLD_ALIGNED frame Jacobian: [z_i x (p_f - o_i); z_i] (revolute), [z_i; 0] (prismatic)
template <class MP>
MPCF_DI void jac_column(const MP &m, int i, double (*oR)[9], double (*op)[3], const double *pf, double *col)
{
    const double z[3] = {oR[i][2], oR[i][5], oR[i][8]};
    if (!m.prismatic(i)) {
        const double d[3] = {pf[0] - op[i][0], pf[1] - op[i][1], pf[2] - op[i][2]};
        cross3(z, d, col);
        col[3] = z[0]; col[4] = z[1]; col[5] = z[2];
    } else {
        col[0] = z[0]; col[1] = z[1]; col[2] = z[2];
        col[3] = 0.0; col[4] = 0.0; col[5] = 0.0;
    }
}

// Contact wrenches as external link forces for run-time trees and the OCP rows of every family (cf. WrenchExt): the world
// orientation of every link advances inside the RNEA's forward sweep — carried in registers along chain segments, parked in
// a local array only for links that others branch off (m.keep) — and the wrench of end-effector e, given in world axes
// at its frame point, enters link je[e] as [R^T F ; R^T n + p x R^T F].
// kPose: the sweep also carries the link origins the same way and captures the world pose (Pw, Rw) of every end-effector
// frame whose link it visits (frame placement pl / Rf in link coordinates); frames on no link (je = -1) are left untouched.
template <int MAXN, bool kPose>
struct PoseTrack {};  // empty: the plain sweep keeps its frame size
template <int MAXN>
struct PoseTrack<MAXN, true> {
    double p[3];                                       // origin of the current link
    double pk[MAXN][3];                                // origins of the links others branch off
    double Rf[MPCF_MAX_EE][9];                         // frame orientation in link coordinates (inputs)
    double Pw[MPCF_MAX_EE][3], Rw[MPCF_MAX_EE][9];     // captured world frame poses (outputs)
};
template <class MP, bool kPose = false>
struct WrenchExtTree : PoseTrack<MP::MAXN, kPose> {
    double R[9];
    double Rk[MP::MAXN][9];
    int nee;
    int je[MPCF_MAX_EE];
    double Wl[MPCF_MAX_EE][6], pl[MPCF_MAX_EE][3];
    double wsign;
    MPCF_DI void link(const MP &m, int i, const JointVar<double> &jv, double *f)
    {
        if (nee == 0) return;
        const int par = m.parent(i);
        double Rp_[9], Rl[9], Rn[9];
        if (par >= 0 && par != i - 1) {
#pragma unroll
            for (int k = 0; k < 9; ++k) Rp_[k] = Rk[par][k];
        } else {
#pragma unroll
            for (int k = 0; k < 9; ++k) Rp_[k] = R[k];
        }
        if (!m.prismatic(i)) {
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                Rl[3 * r + 0] = m.Rp(i, 3 * r) * jv.c + m.Rp(i, 3 * r + 1) * jv.s;
                Rl[3 * r + 1] = m.Rp(i, 3 * r + 1) * jv.c - m.Rp(i, 3 * r) * jv.s;
                Rl[3 * r + 2] = m.Rp(i, 3 * r + 2);
            }
        } else {
#pragma unroll
            for (int k = 0; k < 9; ++k) Rl[k] = m.Rp(i, k);
        }
        if constexpr (kPose) {  // o_i = o_par + R_par t_i, t_i = pp_i (+ q_i Rp_i e_z for a prismatic joint)
            double t[3], pn[3];
#pragma unroll
            for (int r = 0; r < 3; ++r) t[r] = m.prismatic(i) ? m.pp(i, r) + m.Rp(i, 3 * r + 2) * jv.c : m.pp(i, r);
            if (par < 0) {
#pragma unroll
                for (int r = 0; r < 3; ++r) pn[r] = t[r];
            } else {
                const double *pp_ = par != i - 1 ? this->pk[par] : this->p;
#pragma unroll
                for (int r = 0; r < 3; ++r) pn[r] = pp_[r] + Rp_[3 * r] * t[0] + Rp_[3 * r + 1] * t[1] + Rp_[3 * r + 2] * t[2];
            }
#pragma unroll
            for (int r = 0; r < 3; ++r) this->p[r] = pn[r];
            if (m.keep(i)) {
#pragma unroll
                for (int r = 0; r < 3; ++r) this->pk[i][r] = pn[r];
            }
        }
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c)
                Rn[3 * r + c] = (par < 0) ? Rl[3 * r + c] : Rp_[3 * r] * Rl[c] + Rp_[3 * r + 1] * Rl[3 + c] + Rp_[3 * r + 2] * Rl[6 + c];
#pragma unroll
        for (int k = 0; k < 9; ++k) R[k] = Rn[k];
        if (m.keep(i)) {
#pragma unroll
            for (int k = 0; k < 9; ++k) Rk[i][k] = Rn[k];
        }
        auto frame = [&](int e) {
            double Fl[3], nl[3], t[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                Fl[c] = Rn[c] * Wl[e][0] + Rn[3 + c] * Wl[e][1] + Rn[6 + c] * Wl[e][2];
                nl[c] = Rn[c] * Wl[e][3] + Rn[3 + c] * Wl[e][4] + Rn[6 + c] * Wl[e][5];
            }
            cross3(pl[e], Fl, t);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                f[c] += wsign * Fl[c];
                f[3 + c] += wsign * (nl[c] + t[c]);
            }
            if constexpr (kPose) {
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    this->Pw[e][r] = this->p[r] + Rn[3 * r] * pl[e][0] + Rn[3 * r + 1] * pl[e][1] + Rn[3 * r + 2] * pl[e][2];
#pragma unroll
                    for (int c = 0; c < 3; ++c)
                        this->Rw[e][3 * r + c] = Rn[3 * r] * this->Rf[e][c] + Rn[3 * r + 1] * this->Rf[e][3 + c] + Rn[3 * r + 2] * this->Rf[e][6 + c];
                }
            }
        };
        if constexpr (MP::kStatic) {  // a fixed trip count: the frame arrays index at compile time and stay in registers
#pragma unroll
            for (int e = 0; e < MPCF_MAX_EE; ++e)
                if (e < nee && je[e] == i) frame(e);
        } else {
            for (int e = 0; e < nee; ++e)
                if (je[e] == i) frame(e);
        }
    }
};

// Placement liMi_j(q_j) = (Rl, t) of joint j in its parent's coordinates: Rp Rz(q) and pp (revolute), Rp and pp + q Rp e_z
// (prismatic); the same two stages as Dyn::fk_all_jv.
template <class MP>
MPCF_DI void joint_placement(const MP &m, int j, double qj, double *Rl, double *t)
{
    if (!m.prismatic(j)) {
        double s, c;
        sincos(qj, &s, &c);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            Rl[3 * r + 0] = m.Rp(j, 3 * r) * c + m.Rp(j, 3 * r + 1) * s;
            Rl[3 * r + 1] = m.Rp(j, 3 * r + 1) * c - m.Rp(j, 3 * r) * s;
            Rl[3 * r + 2] = m.Rp(j, 3 * r + 2);
            t[r] = m.pp(j, r);
        }
    } else {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
            for (int c = 0; c < 3; ++c) Rl[3 * r + c] = m.Rp(j, 3 * r + c);
            t[r] = m.pp(j, r) + m.Rp(j, 3 * r + 2) * qj;
        }
    }
}

// World pose of a frame (parent joint j, placement fR / fp in the joint's coordinates; j = -1: world-fixed) at unit v of the
// SoA plane q[i * U + v], by walking its ancestor path from the frame up to the root: X <- liMi_j(q_j) X.  Touches only the
// ancestors (depth of the frame), not all n links.
template <class MP>
MPCF_DI void frame_pose_walk(const MP &m, int j, const double *fR, const double *fp, const double *q, long U, long v, double *pos, double *rot)
{
#pragma unroll
    for (int k = 0; k < 9; ++k) rot[k] = fR[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) pos[k] = fp[k];
#pragma unroll 1
    for (; j >= 0; j = m.parent(j)) {
        double Rl[9], t[3], Rn[9], pn[3];
        joint_placement(m, j, q[(long)j * U + v], Rl, t);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            pn[r] = t[r] + Rl[3 * r] * pos[0] + Rl[3 * r + 1] * pos[1] + Rl[3 * r + 2] * pos[2];
#pragma unroll
            for (int c = 0; c < 3; ++c) Rn[3 * r + c] = Rl[3 * r] * rot[c] + Rl[3 * r + 1] * rot[3 + c] + Rl[3 * r + 2] * rot[6 + c];
        }
#pragma unroll
        for (int k = 0; k < 9; ++k) rot[k] = Rn[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) pos[k] = pn[k];
    }
}

// World placements (oR, op) of the links in `mask` (bit i = link i; closed under parents, n <= 64) at unit v, top-down as in
// Dyn::fk_all_jv; the other links' entries are left unwritten.
template <class MP>
MPCF_DI void fk_subset(const MP &m, unsigned long long mask, const double *q, long U, long v, double (*oR)[9], double (*op)[3])
{
    const int n = m.n();
#pragma unroll 1
    for (int i = 0; i < n; ++i) {
        if (!((mask >> i) & 1ull)) continue;
        double Rl[9], t[3];
        joint_placement(m, i, q[(long)i * U + v], Rl, t);
        const int par = m.parent(i);
        if (par < 0) {
#pragma unroll
            for (int k = 0; k < 9; ++k) oR[i][k] = Rl[k];
#pragma unroll
            for (int k = 0; k < 3; ++k) op[i][k] = t[k];
        } else {
#pragma unroll
            for (int r = 0; r < 3; ++r) {
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    oR[i][3 * r + c] = oR[par][3 * r] * Rl[c] + oR[par][3 * r + 1] * Rl[3 + c] + oR[par][3 * r + 2] * Rl[6 + c];
                op[i][r] = op[par][r] + oR[par][3 * r] * t[0] + oR[par][3 * r + 1] * t[1] + oR[par][3 * r + 2] * t[2];
            }
        }
    }
}

}  // namespace mpcf
