/*
 * oracle/core.inc.h — TEST INFRASTRUCTURE ONLY (never imported by the product path).
 *
 * Scalar-generic CPU restatement of the hot path of ADVRHumanoids/mpc_fatigue.  This file is
 * included twice by mpcf_oracle.c: once with SC = double (suffix _r) and once with
 * SC = double complex (suffix _c); the complex instantiation gives exact forward-mode
 * derivatives by complex-step differentiation (Im f(x + i h d) / h, h = 1e-40).
 *
 * What it restates (reference file:line):
 *   rnea            pinocchio::rnea as traced by src/casadi_pinocchio_bridge.hpp:76
 *   frame_fk        framesForwardKinematics + oMf[frame]   src/casadi_pinocchio_bridge.hpp:106-108
 *   frame_jacobian  getFrameJacobian(LOCAL_WORLD_ALIGNED)   src/casadi_pinocchio_bridge.hpp:141-144
 *   thermal_zoh     python/Centauro_script/mpc_principal.py:296-301, python/Libraries/TemperatureModel.py:77
 *   node_eval_ref   python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:290-293,463 ; python/Centauro_script/mpc_principal.py:267-301
 *   crba / aba / step_rk4: north-star additions (no reference code; Featherstone RBDA ch. 6-7,
 *   Pinocchio 2.x conventions: [linear; angular] ordering, body-local frames, gravity as base accel).
 *
 * Pinocchio itself is not in /root/reference (third-party, version unpinned; API implies 2.x >= 2.2),
 * so the algorithms are restated from the published formulation (SURVEY.md Appendix E).
 */

#define MAXN MPCFO_MAXN

static inline void SUF(cross)(const SC *a, const SC *b, SC *o)
{
    SC x = a[1] * b[2] - a[2] * b[1];
    SC y = a[2] * b[0] - a[0] * b[2];
    SC z = a[0] * b[1] - a[1] * b[0];
    o[0] = x; o[1] = y; o[2] = z;
}
static inline void SUF(mv)(const SC *R, const SC *v, SC *o) /* o = R v */
{
    SC x = R[0] * v[0] + R[1] * v[1] + R[2] * v[2];
    SC y = R[3] * v[0] + R[4] * v[1] + R[5] * v[2];
    SC z = R[6] * v[0] + R[7] * v[1] + R[8] * v[2];
    o[0] = x; o[1] = y; o[2] = z;
}
static inline void SUF(mtv)(const SC *R, const SC *v, SC *o) /* o = R^T v */
{
    SC x = R[0] * v[0] + R[3] * v[1] + R[6] * v[2];
    SC y = R[1] * v[0] + R[4] * v[1] + R[7] * v[2];
    SC z = R[2] * v[0] + R[5] * v[1] + R[8] * v[2];
    o[0] = x; o[1] = y; o[2] = z;
}
static inline void SUF(mm)(const SC *A, const SC *B, SC *o) /* o = A B (3x3) */
{
    SC t[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c)
            t[3 * r + c] = A[3 * r] * B[c] + A[3 * r + 1] * B[3 + c] + A[3 * r + 2] * B[6 + c];
    for (int k = 0; k < 9; ++k) o[k] = t[k];
}
static inline void SUF(mmt)(const SC *A, const SC *B, SC *o) /* o = A B^T */
{
    SC t[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c)
            t[3 * r + c] = A[3 * r] * B[3 * c] + A[3 * r + 1] * B[3 * c + 1] + A[3 * r + 2] * B[3 * c + 2];
    for (int k = 0; k < 9; ++k) o[k] = t[k];
}

/* liMi(q) = jointPlacement * Rz(q) (revolute-z) or jointPlacement * Tz(q) (prismatic-z). */
static void SUF(joint_xform)(const mpcfo_model *m, int i, SC q, SC *R, SC *p)
{
    const double *Rp = m->Rp + 9 * i, *pp = m->pp + 3 * i;
    if (m->jtype[i] == 0) {
        SC c = COS(q), s = SIN(q);
        for (int r = 0; r < 3; ++r) {
            R[3 * r + 0] = Rp[3 * r + 0] * c + Rp[3 * r + 1] * s;
            R[3 * r + 1] = Rp[3 * r + 1] * c - Rp[3 * r + 0] * s;
            R[3 * r + 2] = Rp[3 * r + 2];
            p[r] = pp[r];
        }
    } else {
        for (int r = 0; r < 3; ++r) {
            R[3 * r + 0] = Rp[3 * r + 0];
            R[3 * r + 1] = Rp[3 * r + 1];
            R[3 * r + 2] = Rp[3 * r + 2];
            p[r] = pp[r] + Rp[3 * r + 2] * q;
        }
    }
}
#define SIDX(m, i) ((m)->jtype[i] == 0 ? 5 : 2)

/* Motion actInv: parent coords -> child coords. [R^T (v - p x w); R^T w] */
static inline void SUF(m_actinv)(const SC *R, const SC *p, const SC *mp, SC *mc)
{
    SC t[3], u[3];
    SUF(cross)(p, mp + 3, t);
    u[0] = mp[0] - t[0]; u[1] = mp[1] - t[1]; u[2] = mp[2] - t[2];
    SUF(mtv)(R, u, mc);
    SUF(mtv)(R, mp + 3, mc + 3);
}
/* Force act: child coords -> parent coords. [R f; R n + p x (R f)] */
static inline void SUF(f_act)(const SC *R, const SC *p, const SC *fc, SC *fp)
{
    SC t[3];
    SUF(mv)(R, fc, fp);
    SUF(mv)(R, fc + 3, fp + 3);
    SUF(cross)(p, fp, t);
    fp[3] += t[0]; fp[4] += t[1]; fp[5] += t[2];
}
/* Rigid-body inertia times motion: [m v - mc x w ; Io w + mc x v] */
static inline void SUF(inertia_mul)(const mpcfo_model *m, int i, const SC *mo, SC *f)
{
    const double *Io = m->Io + 6 * i;
    SC mc[3] = {m->mc[3 * i], m->mc[3 * i + 1], m->mc[3 * i + 2]};
    SC t[3], u[3];
    SUF(cross)(mc, mo + 3, t);
    SUF(cross)(mc, mo, u);
    f[0] = m->mass[i] * mo[0] - t[0];
    f[1] = m->mass[i] * mo[1] - t[1];
    f[2] = m->mass[i] * mo[2] - t[2];
    f[3] = Io[0] * mo[3] + Io[1] * mo[4] + Io[2] * mo[5] + u[0];
    f[4] = Io[1] * mo[3] + Io[3] * mo[4] + Io[4] * mo[5] + u[1];
    f[5] = Io[2] * mo[3] + Io[4] * mo[4] + Io[5] * mo[5] + u[2];
}
/* v x* f = [w x f ; w x n + v x f] */
static inline void SUF(crossf)(const SC *v, const SC *f, SC *o)
{
    SC a[3], b[3], c[3];
    SUF(cross)(v + 3, f, a);
    SUF(cross)(v + 3, f + 3, b);
    SUF(cross)(v, f, c);
    o[0] = a[0]; o[1] = a[1]; o[2] = a[2];
    o[3] = b[0] + c[0]; o[4] = b[1] + c[1]; o[5] = b[2] + c[2];
}
/* c = v x (S qd) for S = e5 (revolute) or e2 (prismatic) */
static inline void SUF(bias_c)(int jtype, const SC *v, SC qd, SC *c)
{
    if (jtype == 0) {
        c[0] = v[1] * qd; c[1] = -v[0] * qd; c[2] = 0;
        c[3] = v[4] * qd; c[4] = -v[3] * qd; c[5] = 0;
    } else {
        c[0] = v[4] * qd; c[1] = -v[3] * qd; c[2] = 0;
        c[3] = 0; c[4] = 0; c[5] = 0;
    }
}

/* ---- RNEA: tau = M(q) qdd + C(q,qd) qd + g(q)  (+ armature * qdd) ---- */
static void SUF(rnea)(const mpcfo_model *m, const SC *q, const SC *qd, const SC *qdd, SC *tau)
{
    int n = m->n;
    SC R[MAXN][9], p[MAXN][3], v[MAXN][6], a[MAXN][6], f[MAXN][6];
    for (int i = 0; i < n; ++i) {
        int par = m->parent[i], s = SIDX(m, i);
        SC vp[6] = {0, 0, 0, 0, 0, 0}, ap[6] = {-m->grav[0], -m->grav[1], -m->grav[2], 0, 0, 0};
        if (par >= 0)
            for (int k = 0; k < 6; ++k) { vp[k] = v[par][k]; ap[k] = a[par][k]; }
        SUF(joint_xform)(m, i, q[i], R[i], p[i]);
        SUF(m_actinv)(R[i], p[i], vp, v[i]);
        v[i][s] += qd[i];
        SUF(m_actinv)(R[i], p[i], ap, a[i]);
        SC c[6];
        SUF(bias_c)(m->jtype[i], v[i], qd[i], c);
        for (int k = 0; k < 6; ++k) a[i][k] += c[k];
        a[i][s] += qdd[i];
        SC h[6], fa[6], fb[6];
        SUF(inertia_mul)(m, i, v[i], h);
        SUF(inertia_mul)(m, i, a[i], fa);
        SUF(crossf)(v[i], h, fb);
        for (int k = 0; k < 6; ++k) f[i][k] = fa[k] + fb[k];
    }
    for (int i = n - 1; i >= 0; --i) {
        int par = m->parent[i], s = SIDX(m, i);
        tau[i] = f[i][s] + m->arm[i] * qdd[i];
        if (par >= 0) {
            SC fp[6];
            SUF(f_act)(R[i], p[i], f[i], fp);
            for (int k = 0; k < 6; ++k) f[par][k] += fp[k];
        }
    }
}

/* ---- world placements oMi of every joint ---- */
static void SUF(fk_all)(const mpcfo_model *m, const SC *q, SC (*oR)[9], SC (*op)[3])
{
    for (int i = 0; i < m->n; ++i) {
        SC R[9], p[3];
        int par = m->parent[i];
        SUF(joint_xform)(m, i, q[i], R, p);
        if (par < 0) {
            for (int k = 0; k < 9; ++k) oR[i][k] = R[k];
            for (int k = 0; k < 3; ++k) op[i][k] = p[k];
        } else {
            SC t[3];
            SUF(mm)(oR[par], R, oR[i]);
            SUF(mv)(oR[par], p, t);
            for (int k = 0; k < 3; ++k) op[i][k] = op[par][k] + t[k];
        }
    }
}

/* ---- frame FK: ee_pos[3], ee_rot[9] row-major (element (i,j) = R[i][j]) ---- */
static void SUF(frame_fk)(const mpcfo_model *m, int frame, const SC *q, SC *pos, SC *rot)
{
    SC oR[MAXN][9], op[MAXN][3];
    SUF(fk_all)(m, q, oR, op);
    int j = m->fparent[frame];
    const double *fR = m->fR + 9 * frame, *fp = m->fp + 3 * frame;
    SC fRs[9], fps[3];
    for (int k = 0; k < 9; ++k) fRs[k] = fR[k];
    for (int k = 0; k < 3; ++k) fps[k] = fp[k];
    if (j < 0) {
        for (int k = 0; k < 9; ++k) rot[k] = fRs[k];
        for (int k = 0; k < 3; ++k) pos[k] = fps[k];
    } else {
        SC t[3];
        SUF(mm)(oR[j], fRs, rot);
        SUF(mv)(oR[j], fps, t);
        for (int k = 0; k < 3; ++k) pos[k] = op[j][k] + t[k];
    }
}

/* ---- frame Jacobian, LOCAL_WORLD_ALIGNED, J[6][n] row-major ---- */
static void SUF(frame_jacobian)(const mpcfo_model *m, int frame, const SC *q, SC *J)
{
    int n = m->n;
    SC oR[MAXN][9], op[MAXN][3], pos[3], rot[9];
    SUF(fk_all)(m, q, oR, op);
    SUF(frame_fk)(m, frame, q, pos, rot);
    for (int k = 0; k < 6 * n; ++k) J[k] = 0;
    for (int i = m->fparent[frame]; i >= 0; i = m->parent[i]) {
        SC z[3] = {oR[i][2], oR[i][5], oR[i][8]};
        if (m->jtype[i] == 0) {
            SC d[3] = {pos[0] - op[i][0], pos[1] - op[i][1], pos[2] - op[i][2]}, lin[3];
            SUF(cross)(z, d, lin);
            for (int r = 0; r < 3; ++r) { J[r * n + i] = lin[r]; J[(3 + r) * n + i] = z[r]; }
        } else {
            for (int r = 0; r < 3; ++r) J[r * n + i] = z[r];
        }
    }
}

/* ---- CRBA: dense joint-space inertia M[n][n] (armature on the diagonal) ---- */
static void SUF(crba)(const mpcfo_model *m, const SC *q, SC *M)
{
    int n = m->n;
    SC R[MAXN][9], p[MAXN][3];
    SC cm[MAXN], cmc[MAXN][3], cI[MAXN][9]; /* composite mass, mass*com, inertia about origin (full 3x3) */
    for (int i = 0; i < n; ++i) {
        SUF(joint_xform)(m, i, q[i], R[i], p[i]);
        const double *Io = m->Io + 6 * i;
        cm[i] = m->mass[i];
        for (int k = 0; k < 3; ++k) cmc[i][k] = m->mc[3 * i + k];
        cI[i][0] = Io[0]; cI[i][1] = Io[1]; cI[i][2] = Io[2];
        cI[i][3] = Io[1]; cI[i][4] = Io[3]; cI[i][5] = Io[4];
        cI[i][6] = Io[2]; cI[i][7] = Io[4]; cI[i][8] = Io[5];
    }
    for (int k = 0; k < n * n; ++k) M[k] = 0;
    for (int i = n - 1; i >= 0; --i) {
        int par = m->parent[i];
        /* column i: F = Yc_i S_i */
        SC F[6];
        if (m->jtype[i] == 0) {
            F[0] = -cmc[i][1]; F[1] = cmc[i][0]; F[2] = 0;
            F[3] = cI[i][2]; F[4] = cI[i][5]; F[5] = cI[i][8];
        } else {
            F[0] = 0; F[1] = 0; F[2] = cm[i];
            F[3] = cmc[i][1]; F[4] = -cmc[i][0]; F[5] = 0;
        }
        M[i * n + i] = F[SIDX(m, i)] + m->arm[i];
        for (int j = i; m->parent[j] >= 0;) {
            SC Fp[6];
            SUF(f_act)(R[j], p[j], F, Fp);
            for (int k = 0; k < 6; ++k) F[k] = Fp[k];
            j = m->parent[j];
            M[i * n + j] = F[SIDX(m, j)];
            M[j * n + i] = F[SIDX(m, j)];
        }
        if (par >= 0) {
            /* composite inertia of i expressed in the parent frame, added to the parent */
            SC a[3], RI[9], RIRt[9];
            SUF(mv)(R[i], cmc[i], a); /* a = R * (m c) */
            SUF(mm)(R[i], cI[i], RI);
            SUF(mmt)(RI, R[i], RIRt);
            SC ap = a[0] * p[i][0] + a[1] * p[i][1] + a[2] * p[i][2];
            SC pp = p[i][0] * p[i][0] + p[i][1] * p[i][1] + p[i][2] * p[i][2];
            SC dg = 2 * ap + cm[i] * pp;
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c) {
                    SC e = RIRt[3 * r + c] - (a[r] * p[i][c] + p[i][r] * a[c] + cm[i] * p[i][r] * p[i][c]);
                    if (r == c) e += dg;
                    cI[par][3 * r + c] += e;
                }
            for (int k = 0; k < 3; ++k) cmc[par][k] += a[k] + cm[i] * p[i][k];
            cm[par] += cm[i];
        }
    }
}

/* ---- ABA: qdd = M^-1 (tau - h(q,qd)), three passes, armature added to D_i ---- */
static int SUF(aba)(const mpcfo_model *m, const SC *q, const SC *qd, const SC *tau, SC *qdd)
{
    int n = m->n;
    SC R[MAXN][9], p[MAXN][3], v[MAXN][6], c[MAXN][6], pA[MAXN][6], IA[MAXN][36];
    SC U[MAXN][6], Dinv[MAXN], u[MAXN], a[MAXN][6];
    for (int i = 0; i < n; ++i) {
        int par = m->parent[i], s = SIDX(m, i);
        SC vp[6] = {0, 0, 0, 0, 0, 0};
        if (par >= 0)
            for (int k = 0; k < 6; ++k) vp[k] = v[par][k];
        SUF(joint_xform)(m, i, q[i], R[i], p[i]);
        SUF(m_actinv)(R[i], p[i], vp, v[i]);
        v[i][s] += qd[i];
        SUF(bias_c)(m->jtype[i], v[i], qd[i], c[i]);
        SC h[6];
        SUF(inertia_mul)(m, i, v[i], h);
        SUF(crossf)(v[i], h, pA[i]);
        /* IA = rigid-body inertia as a 6x6: [[m 1, -[mc]x],[[mc]x, Io]] */
        const double *Io = m->Io + 6 * i, *mc = m->mc + 3 * i;
        double ms = m->mass[i];
        SC *I6 = IA[i];
        for (int k = 0; k < 36; ++k) I6[k] = 0;
        I6[0] = ms; I6[7] = ms; I6[14] = ms;
        /* -[mc]x block (rows 0-2, cols 3-5) */
        I6[0 * 6 + 4] = mc[2];  I6[0 * 6 + 5] = -mc[1];
        I6[1 * 6 + 3] = -mc[2]; I6[1 * 6 + 5] = mc[0];
        I6[2 * 6 + 3] = mc[1];  I6[2 * 6 + 4] = -mc[0];
        /* [mc]x block (rows 3-5, cols 0-2) */
        I6[3 * 6 + 1] = -mc[2]; I6[3 * 6 + 2] = mc[1];
        I6[4 * 6 + 0] = mc[2];  I6[4 * 6 + 2] = -mc[0];
        I6[5 * 6 + 0] = -mc[1]; I6[5 * 6 + 1] = mc[0];
        I6[3 * 6 + 3] = Io[0]; I6[3 * 6 + 4] = Io[1]; I6[3 * 6 + 5] = Io[2];
        I6[4 * 6 + 3] = Io[1]; I6[4 * 6 + 4] = Io[3]; I6[4 * 6 + 5] = Io[4];
        I6[5 * 6 + 3] = Io[2]; I6[5 * 6 + 4] = Io[4]; I6[5 * 6 + 5] = Io[5];
    }
    for (int i = n - 1; i >= 0; --i) {
        int par = m->parent[i], s = SIDX(m, i);
        SC *I6 = IA[i];
        for (int k = 0; k < 6; ++k) U[i][k] = I6[k * 6 + s];
        SC D = U[i][s] + m->arm[i];
        if (D == 0) return -(i + 1); /* singular: zero joint-space inertia without armature */
        Dinv[i] = 1.0 / D;
        u[i] = tau[i] - pA[i][s];
        if (par >= 0) {
            SC Ia[36], pa[6];
            for (int r = 0; r < 6; ++r)
                for (int cc = 0; cc < 6; ++cc) Ia[r * 6 + cc] = I6[r * 6 + cc] - U[i][r] * Dinv[i] * U[i][cc];
            for (int r = 0; r < 6; ++r) {
                SC acc = pA[i][r] + U[i][r] * Dinv[i] * u[i];
                for (int cc = 0; cc < 6; ++cc) acc += Ia[r * 6 + cc] * c[i][cc];
                pa[r] = acc;
            }
            /* IA_par += X_F Ia X_M^-1 with blocks A (ll), B (la), C (aa): see DESIGN.md */
            SC A[9], B[9], C[9], Bt[9], t9[9];
            for (int r = 0; r < 3; ++r)
                for (int cc = 0; cc < 3; ++cc) {
                    A[3 * r + cc] = Ia[r * 6 + cc];
                    B[3 * r + cc] = Ia[r * 6 + 3 + cc];
                    C[3 * r + cc] = Ia[(3 + r) * 6 + 3 + cc];
                }
            SUF(mm)(R[i], A, t9); SUF(mmt)(t9, R[i], A);
            SUF(mm)(R[i], B, t9); SUF(mmt)(t9, R[i], B);
            SUF(mm)(R[i], C, t9); SUF(mmt)(t9, R[i], C);
            SC P[9] = {0, -p[i][2], p[i][1], p[i][2], 0, -p[i][0], -p[i][1], p[i][0], 0};
            SC AP[9], B2[9], PB2[9], BtP[9];
            SUF(mm)(A, P, AP);
            for (int k = 0; k < 9; ++k) B2[k] = B[k] - AP[k]; /* B'' = B' - A'P */
            for (int r = 0; r < 3; ++r)
                for (int cc = 0; cc < 3; ++cc) Bt[3 * r + cc] = B[3 * cc + r];
            SUF(mm)(Bt, P, BtP);
            SUF(mm)(P, B2, PB2);
            SC *Ip = IA[par];
            for (int r = 0; r < 3; ++r)
                for (int cc = 0; cc < 3; ++cc) {
                    Ip[r * 6 + cc] += A[3 * r + cc];
                    Ip[r * 6 + 3 + cc] += B2[3 * r + cc];
                    Ip[(3 + cc) * 6 + r] += B2[3 * r + cc];
                    Ip[(3 + r) * 6 + 3 + cc] += C[3 * r + cc] - BtP[3 * r + cc] + PB2[3 * r + cc];
                }
            SC fp[6];
            SUF(f_act)(R[i], p[i], pa, fp);
            for (int k = 0; k < 6; ++k) pA[par][k] += fp[k];
        }
    }
    for (int i = 0; i < n; ++i) {
        int par = m->parent[i], s = SIDX(m, i);
        SC ap[6] = {-m->grav[0], -m->grav[1], -m->grav[2], 0, 0, 0};
        if (par >= 0)
            for (int k = 0; k < 6; ++k) ap[k] = a[par][k];
        SUF(m_actinv)(R[i], p[i], ap, a[i]);
        SC acc = u[i];
        for (int k = 0; k < 6; ++k) { a[i][k] += c[i][k]; acc -= U[i][k] * a[i][k]; }
        qdd[i] = Dinv[i] * acc;
        a[i][s] += qdd[i];
    }
    return 0;
}

/* ---- fatigue (K = 1 compartment per joint): fdot = -lambda f + kappa (ctau tau^2 + cv qd^2) ---- */
static inline SC SUF(fatigue_rhs)(const mpcfo_model *m, int i, SC f, SC tau, SC qd)
{
    const double *c = m->fat + 4 * i;
    return -c[0] * f + c[1] * (c[2] * tau * tau + c[3] * qd * qd);
}
/* exact zero-order-hold map over h (the reference's T_next line, mpc_principal.py:301).  The gain (1 - a) kappa / lambda is
 * formed as -expm1(-lambda h) kappa / lambda: 1 - exp(-lambda h) loses all but a few digits as lambda h -> 0 (lambda h = 1e-12:
 * ~1e-4 relative), while expm1 keeps the gain continuous into the lambda = 0 branch. */
static inline SC SUF(fatigue_zoh)(const mpcfo_model *m, int i, SC f, SC tau, SC qd, SC h)
{
    const double *c = m->fat + 4 * i;
    SC P = c[2] * tau * tau + c[3] * qd * qd;
    if (c[0] == 0.0) return f + h * c[1] * P;
    SC a = EXP(-c[0] * h);
    return a * f + (-EXPM1(-c[0] * h)) * (c[1] / c[0]) * P;
}

/* xdot = (qd, ABA(q,qd,tau), fatigue_rhs) */
static int SUF(xdot)(const mpcfo_model *m, const SC *x, const SC *tau, SC *k)
{
    int n = m->n;
    int rc = SUF(aba)(m, x, x + n, tau, k + n);
    for (int i = 0; i < n; ++i) {
        k[i] = x[n + i];
        k[2 * n + i] = SUF(fatigue_rhs)(m, i, x[2 * n + i], tau[i], x[n + i]);
    }
    return rc;
}

/* ---- classical RK4 over x = (q, qd, f) with tau held over the step ---- */
static int SUF(step_rk4)(const mpcfo_model *m, const SC *x, const SC *tau, SC dt, SC *xn)
{
    int n3 = 3 * m->n, rc = 0;
    SC k1[3 * MAXN], k2[3 * MAXN], k3[3 * MAXN], k4[3 * MAXN], xs[3 * MAXN];
    rc |= SUF(xdot)(m, x, tau, k1);
    for (int i = 0; i < n3; ++i) xs[i] = x[i] + 0.5 * dt * k1[i];
    rc |= SUF(xdot)(m, xs, tau, k2);
    for (int i = 0; i < n3; ++i) xs[i] = x[i] + 0.5 * dt * k2[i];
    rc |= SUF(xdot)(m, xs, tau, k3);
    for (int i = 0; i < n3; ++i) xs[i] = x[i] + dt * k3[i];
    rc |= SUF(xdot)(m, xs, tau, k4);
    for (int i = 0; i < n3; ++i) xn[i] = x[i] + dt / 6.0 * (k1[i] + 2.0 * k2[i] + 2.0 * k3[i] + k4[i]);
    return rc;
}

/* ---- coupled fatigue of a two-arm model carrying one box (config C3; builder-defined, PARITY UNPINNED: the reference has no
 * dynamics-mode fatigue at all — what it has is the box equilibrium F_L,z + F_R,z = m g of python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:197,272-274
 * and tau = ID - J^T F of :292-293).  Definition, zero-order hold over the step like tau itself:
 *   Phi_c   = sum of the fatigue states of arm c at the start of the step
 *   s_c     = Phi_other / (Phi_0 + Phi_1)            share of the box weight arm c carries: the less fatigued arm takes more
 *   g_c(q)  = J_ee,c(q)^T [0, 0, w, 0, 0, 0]         torque that holds the whole box weight w = m g at arm c's end-effector
 *   theat_i = tau_i + s_c(i) g_i(q(t_k))             torque the motor of joint i delivers (motion + payload feed-forward)
 * and the step is x+ = RK4 of (qd, ABA(q, qd, tau), fatigue_rhs(f, theat, qd)): the dynamics see tau, the windings heat with theat.
 * The two arms are coupled through s_c (d f+_L / d f_R != 0) and the fatigue rows depend on q through g. */
static int SUF(xdot_heat)(const mpcfo_model *m, const SC *x, const SC *tau, const SC *theat, SC *k)
{
    int n = m->n;
    int rc = SUF(aba)(m, x, x + n, tau, k + n);
    for (int i = 0; i < n; ++i) {
        k[i] = x[n + i];
        k[2 * n + i] = SUF(fatigue_rhs)(m, i, x[2 * n + i], theat[i], x[n + i]);
    }
    return rc;
}
static void SUF(coupled_heat_torque)(const mpcfo_model *m, const mpcfo_coupling *cp, const SC *q, const SC *f, const SC *tau, SC *theat)
{
    int n = m->n;
    SC Phi[2] = {0, 0}, J[6 * MAXN];
    for (int i = 0; i < n; ++i) Phi[cp->chain_of[i]] += f[i];
    SC S = Phi[0] + Phi[1];
    SC share[2] = {Phi[1] / S, Phi[0] / S};
    for (int i = 0; i < n; ++i) theat[i] = tau[i];
    for (int c = 0; c < 2; ++c) {
        SUF(frame_jacobian)(m, cp->ee_frame[c], q, J);
        for (int i = 0; i < n; ++i)
            if (cp->chain_of[i] == c) theat[i] += share[c] * (J[2 * n + i] * cp->weight);
    }
}
static int SUF(step_rk4_coupled)(const mpcfo_model *m, const mpcfo_coupling *cp, const SC *x, const SC *tau, SC dt, SC *xn)
{
    int n = m->n, n3 = 3 * m->n, rc = 0;
    SC k1[3 * MAXN], k2[3 * MAXN], k3[3 * MAXN], k4[3 * MAXN], xs[3 * MAXN], theat[MAXN];
    SUF(coupled_heat_torque)(m, cp, x, x + 2 * n, tau, theat);
    rc |= SUF(xdot_heat)(m, x, tau, theat, k1);
    for (int i = 0; i < n3; ++i) xs[i] = x[i] + 0.5 * dt * k1[i];
    rc |= SUF(xdot_heat)(m, xs, tau, theat, k2);
    for (int i = 0; i < n3; ++i) xs[i] = x[i] + 0.5 * dt * k2[i];
    rc |= SUF(xdot_heat)(m, xs, tau, theat, k3);
    for (int i = 0; i < n3; ++i) xs[i] = x[i] + dt * k3[i];
    rc |= SUF(xdot_heat)(m, xs, tau, theat, k4);
    for (int i = 0; i < n3; ++i) xn[i] = x[i] + dt / 6.0 * (k1[i] + 2.0 * k2[i] + 2.0 * k3[i] + k4[i]);
    return rc;
}

/* ---- reference-mode node evaluation (pinned by the plotter fixtures):
 *   tau   = RNEA(q, qd, qdd) + wsign * sum_e J_e^T W_e         (Box_Pilz_6DOF2.py:292-293: wsign=-1;
 *                                                               mpc_principal.py:269: wsign=+1)
 *   qnext = q + h qd                                            (Box_Pilz_6DOF2.py:463)
 *   Tnext = a T + (1-a) (kappa/lambda) P(tau, qd)               (mpc_principal.py:296-301)
 */
static void SUF(node_eval_ref)(const mpcfo_model *m, int nee, const int *ee_frames, double wsign,
                               const SC *q, const SC *qd, const SC *qdd, const SC *W, const SC *T, SC h,
                               SC *tau, SC *qnext, SC *Tnext)
{
    int n = m->n;
    SC J[6 * MAXN];
    SUF(rnea)(m, q, qd, qdd, tau);
    for (int e = 0; e < nee; ++e) {
        SUF(frame_jacobian)(m, ee_frames[e], q, J);
        for (int i = 0; i < n; ++i) {
            SC acc = 0;
            for (int r = 0; r < 6; ++r) acc += J[r * n + i] * W[6 * e + r];
            tau[i] += wsign * acc;
        }
    }
    for (int i = 0; i < n; ++i) {
        qnext[i] = q[i] + h * qd[i];
        Tnext[i] = SUF(fatigue_zoh)(m, i, T[i], tau[i], qd[i], h);
    }
}

/* ---- reference-mode OCP node rows (the fused kernel of csrc/kernels_rows.cu restated with the oracle's own frame FK,
 * frame Jacobian and RNEA): one arm  python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:130-177;  two arms
 * python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:244-293,454-475, python/Centauro_script/mpc_principal.py:229-327,
 * RepeatedMPCwithThermal_confriction.py:251-273.  Row order: see include/mpcf.h (mpcf_ocp_rows_batch).
 * qnext / Tnext: the next node's state (NULL: zero defect); relprev: R_L^T (pR - pL) at the previous node (or rel_pos0). */
static void SUF(ocp_rows)(const mpcfo_model *m, const mpcfo_rows_opts *o, const SC *q, const SC *qd, const SC *F, const SC *T,
                          const SC *qnext, const SC *Tnext, const SC *relprev, const double *ori0, SC *rows, SC *cost)
{
    int n = m->n, narm = o->narm, kin = narm == 2 ? 26 : 3;
    SC pe[2][3], Re[2][9], W[12], zero[MAXN], Tl[MAXN], tau[MAXN], qn[MAXN], Tn[MAXN];
    for (int i = 0; i < n; ++i) { zero[i] = 0; Tl[i] = T ? T[i] : 0; }
    for (int c = 0; c < narm; ++c) {
        SUF(frame_fk)(m, o->ee_frame[c], q, pe[c], Re[c]);
        for (int k = 0; k < 3; ++k) { W[6 * c + k] = F[3 * c + k]; W[6 * c + 3 + k] = 0; }
    }
    SUF(node_eval_ref)(m, narm, o->ee_frame, o->wsign, q, qd, zero, W, Tl, o->h, tau, qn, Tn);
    SC cF = 0, cqd = 0, ckin = 0;
    for (int i = 0; i < 3 * narm; ++i) cF += F[i] * F[i];
    for (int i = 0; i < n; ++i) {
        cqd += qd[i] * qd[i];
        rows[kin + i] = tau[i];
        rows[kin + n + i] = qnext ? qn[i] - qnext[i] : 0;
        rows[kin + 2 * n + i] = (T && Tnext) ? Tn[i] - Tnext[i] : 0;
    }
    if (narm == 1) {
        for (int k = 0; k < 3; ++k) rows[k] = pe[0][k] - o->p_ref[k];
    } else {
        const SC *pL = pe[0], *pR = pe[1], *RL = Re[0], *RR = Re[1], *FL = F, *FR = F + 3;
        SC d[3] = {pL[0] - pR[0], pL[1] - pR[1], pL[2] - pR[2]}, a1[3], a2[3], dm[3] = {pR[0] - pL[0], pR[1] - pL[1], pR[2] - pL[2]};
        for (int k = 0; k < 3; ++k) rows[k] = FL[k] + FR[k] - o->fdes[k];
        SUF(cross)(d, FL, a1);
        SUF(cross)(dm, FR, a2);
        for (int k = 0; k < 3; ++k) rows[3 + k] = a1[k] + a2[k];
        rows[6] = d[0] * d[0] + d[1] * d[1] + d[2] * d[2] - o->dist2_ref;
        SC rel[3], f1[3], f2[3], Ro[9];
        SUF(mtv)(RL, dm, rel);
        for (int k = 0; k < 3; ++k) rows[7 + k] = rel[k] - relprev[k];
        SUF(mmt)(RL, RR, Ro); /* R_L R_R^T */
        rows[10] = (Ro[7] - Ro[5]) / 2 - ori0[0];
        rows[11] = (Ro[6] - Ro[2]) / 2 - ori0[1];
        rows[12] = (Ro[3] - Ro[1]) / 2 - ori0[2];
        SUF(mtv)(RL, FL, f1);
        SUF(mtv)(RR, FR, f2);
        for (int k = 0; k < 3; ++k) { f1[k] = -f1[k]; f2[k] = -f2[k]; }
        const double A1[5][3] = {{0, -1, 0}, {0, -o->mu, 1}, {0, -o->mu, -1}, {1, -o->mu, 0}, {-1, -o->mu, 0}};
        const double A2[5][3] = {{0, 1, 0}, {1, o->mu, 0}, {-1, o->mu, 0}, {0, o->mu, 1}, {0, o->mu, -1}};
        for (int r = 0; r < 5; ++r) {
            rows[13 + r] = A1[r][0] * f1[0] + A1[r][1] * f1[1] + A1[r][2] * f1[2];
            rows[18 + r] = A2[r][0] * f2[0] + A2[r][1] * f2[1] + A2[r][2] * f2[2];
        }
        for (int k = 0; k < 3; ++k) {
            rows[23 + k] = (pL[k] + pR[k]) / 2 - o->p_ref[k];
            ckin += rows[23 + k] * rows[23 + k];
        }
    }
    *cost = o->w_box * ckin + o->w_qd * cqd + o->w_F * cF;
}

#undef MAXN
