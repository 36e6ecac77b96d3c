// dyn.cuh — device-side rigid-body dynamics + fatigue ODE, generic over
//   T  : scalar type (double, or Dual = value + one forward-mode tangent)
//   MP : model policy (compile-time topology with constants in the kernel-parameter constant bank,
//        or run-time topology with constants staged in shared memory)
//
// Conventions (Pinocchio 2.x, what the reference traces at src/casadi_pinocchio_bridge.hpp:76,106,141):
// spatial vectors are [linear; angular] in the body-local joint frame; every joint is revolute about /
// prismatic along its local +z; liMi(q) = (Rp, pp) * Rz(q)  or  (Rp, pp) * Tz(q); gravity enters as the
// base acceleration -g.  All joint transforms are applied in two stages — the variable stage (a planar
// rotation by (cos q, sin q), or a z-shift) and the constant stage (Rp, pp) — so only (c, s) is kept per
// link instead of a 3x3.
#pragma once

#include <cuda_runtime.h>

namespace mpcf {

#define MPCF_DI __device__ __forceinline__
// pure arithmetic shared with the host-side unit checks of the run-time-tree pipeline (tests/hostcheck): same source, compiled
// for the device in the product and, by the tests only, for the host
#define MPCF_HD __host__ __device__ __forceinline__

// ---------------------------------------------------------------------------------------------
// Dual numbers (one tangent direction)
// ---------------------------------------------------------------------------------------------
struct Dual {
    double v, d;
    MPCF_DI Dual() {}
    MPCF_DI Dual(double v_) : v(v_), d(0.0) {}
    MPCF_DI Dual(double v_, double d_) : v(v_), d(d_) {}
};
MPCF_DI Dual operator+(Dual a, Dual b) { return Dual(a.v + b.v, a.d + b.d); }
MPCF_DI Dual operator+(Dual a, double b) { return Dual(a.v + b, a.d); }
MPCF_DI Dual operator+(double a, Dual b) { return Dual(a + b.v, b.d); }
MPCF_DI Dual operator-(Dual a, Dual b) { return Dual(a.v - b.v, a.d - b.d); }
MPCF_DI Dual operator-(Dual a, double b) { return Dual(a.v - b, a.d); }
MPCF_DI Dual operator-(double a, Dual b) { return Dual(a - b.v, -b.d); }
MPCF_DI Dual operator-(Dual a) { return Dual(-a.v, -a.d); }
MPCF_DI Dual operator*(Dual a, Dual b) { return Dual(a.v * b.v, fma(a.v, b.d, a.d * b.v)); }
MPCF_DI Dual operator*(Dual a, double b) { return Dual(a.v * b, a.d * b); }
MPCF_DI Dual operator*(double a, Dual b) { return Dual(a * b.v, a * b.d); }
MPCF_DI Dual &operator+=(Dual &a, Dual b) { a.v += b.v; a.d += b.d; return a; }
MPCF_DI Dual &operator-=(Dual &a, Dual b) { a.v -= b.v; a.d -= b.d; return a; }
MPCF_DI Dual &operator+=(Dual &a, double b) { a.v += b; return a; }

MPCF_DI double recip(double a) { return 1.0 / a; }
MPCF_DI Dual recip(Dual a) { double r = 1.0 / a.v; return Dual(r, -a.d * r * r); }
MPCF_DI void sincos_t(double q, double &s, double &c) { sincos(q, &s, &c); }
MPCF_DI void sincos_t(Dual q, Dual &s, Dual &c)
{
    double sv, cv;
    sincos(q.v, &sv, &cv);
    s = Dual(sv, cv * q.d);
    c = Dual(cv, -sv * q.d);
}
// ---------------------------------------------------------------------------------------------
// Hyper-dual numbers: two tangent directions a, b and the mixed second derivative ab, exact to rounding (no truncation error)
// ---------------------------------------------------------------------------------------------
struct HDual {
    double v, a, b, ab;
    MPCF_DI HDual() {}
    MPCF_DI HDual(double v_) : v(v_), a(0.0), b(0.0), ab(0.0) {}
    MPCF_DI HDual(double v_, double a_, double b_, double ab_) : v(v_), a(a_), b(b_), ab(ab_) {}
};
MPCF_DI HDual operator+(HDual x, HDual y) { return HDual(x.v + y.v, x.a + y.a, x.b + y.b, x.ab + y.ab); }
MPCF_DI HDual operator+(HDual x, double y) { return HDual(x.v + y, x.a, x.b, x.ab); }
MPCF_DI HDual operator+(double x, HDual y) { return HDual(x + y.v, y.a, y.b, y.ab); }
MPCF_DI HDual operator-(HDual x, HDual y) { return HDual(x.v - y.v, x.a - y.a, x.b - y.b, x.ab - y.ab); }
MPCF_DI HDual operator-(HDual x, double y) { return HDual(x.v - y, x.a, x.b, x.ab); }
MPCF_DI HDual operator-(double x, HDual y) { return HDual(x - y.v, -y.a, -y.b, -y.ab); }
MPCF_DI HDual operator-(HDual x) { return HDual(-x.v, -x.a, -x.b, -x.ab); }
MPCF_DI HDual operator*(HDual x, HDual y)
{
    return HDual(x.v * y.v, fma(x.v, y.a, x.a * y.v), fma(x.v, y.b, x.b * y.v),
                 fma(x.v, y.ab, fma(x.a, y.b, fma(x.b, y.a, x.ab * y.v))));
}
MPCF_DI HDual operator*(HDual x, double y) { return HDual(x.v * y, x.a * y, x.b * y, x.ab * y); }
MPCF_DI HDual operator*(double x, HDual y) { return HDual(x * y.v, x * y.a, x * y.b, x * y.ab); }
MPCF_DI HDual &operator+=(HDual &x, HDual y) { x = x + y; return x; }
MPCF_DI HDual &operator-=(HDual &x, HDual y) { x = x - y; return x; }
MPCF_DI HDual &operator+=(HDual &x, double y) { x.v += y; return x; }
MPCF_DI HDual recip(HDual x)
{
    const double r = 1.0 / x.v, r2 = r * r;
    return HDual(r, -x.a * r2, -x.b * r2, fma(-x.ab, r2, 2.0 * (x.a * x.b) * (r2 * r)));
}
MPCF_DI void sincos_t(HDual q, HDual &s, HDual &c)
{
    double sv, cv;
    sincos(q.v, &sv, &cv);
    const double ab = q.a * q.b;
    s = HDual(sv, cv * q.a, cv * q.b, fma(cv, q.ab, -sv * ab));
    c = HDual(cv, -sv * q.a, -sv * q.b, fma(-sv, q.ab, -cv * ab));
}

MPCF_DI double nan_value() { return __longlong_as_double(0x7ff8000000000000ll); }
MPCF_DI double value_of(double a) { return a; }
MPCF_DI double value_of(Dual a) { return a.v; }
MPCF_DI double value_of(HDual a) { return a.v; }
MPCF_DI double tangent_of(double) { return 0.0; }
MPCF_DI double tangent_of(Dual a) { return a.d; }

// ---------------------------------------------------------------------------------------------
// small vector helpers (T or double operands mix freely through the overloads above)
// ---------------------------------------------------------------------------------------------
template <class A, class B, class O>
MPCF_HD void cross3(const A *a, const B *b, O *o)
{
    O x = a[1] * b[2] - a[2] * b[1];
    O y = a[2] * b[0] - a[0] * b[2];
    O z = a[0] * b[1] - a[1] * b[0];
    o[0] = x; o[1] = y; o[2] = z;
}

// Variable stage of a joint transform.
template <class T>
struct JointVar {
    T c, s;  // revolute: cos q, sin q.  prismatic: c = q (the shift), s unused
};

// ---------------------------------------------------------------------------------------------
// The algorithms.  MP provides: n(), parent(i), prismatic(i), Rp(i,k), pp(i,k), mass(i), mc(i,k),
// Io(i,k), arm(i), fat(i,k), grav(k), and static constexpr int MAXN.
// ---------------------------------------------------------------------------------------------
template <class T, class MP>
struct Dyn {
    static constexpr int MAXN = MP::MAXN;

    // ---- joint transform: motion parent -> child (actInv) ----
    static MPCF_DI void motion_to_child(const MP &m, int i, const JointVar<T> &jv, const T *mp, T *mc)
    {
        // constant stage: u = Rp^T (v - pp x w), w' = Rp^T w
        T t[3], u[3], w[3];
        double pp[3] = {m.pp(i, 0), m.pp(i, 1), m.pp(i, 2)};
        cross3(pp, mp + 3, t);
        t[0] = mp[0] - t[0]; t[1] = mp[1] - t[1]; t[2] = mp[2] - t[2];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            u[k] = m.Rp(i, k) * t[0] + m.Rp(i, 3 + k) * t[1] + m.Rp(i, 6 + k) * t[2];
            w[k] = m.Rp(i, k) * mp[3] + m.Rp(i, 3 + k) * mp[4] + m.Rp(i, 6 + k) * mp[5];
        }
        if (!m.prismatic(i)) {  // Rz(q)^T
            mc[0] = jv.c * u[0] + jv.s * u[1];
            mc[1] = jv.c * u[1] - jv.s * u[0];
            mc[2] = u[2];
            mc[3] = jv.c * w[0] + jv.s * w[1];
            mc[4] = jv.c * w[1] - jv.s * w[0];
            mc[5] = w[2];
        } else {  // shift by q along z: u - q z x w
            mc[0] = u[0] + jv.c * w[1];
            mc[1] = u[1] - jv.c * w[0];
            mc[2] = u[2];
            mc[3] = w[0]; mc[4] = w[1]; mc[5] = w[2];
        }
    }
    // ---- joint transform: force child -> parent (act) ----
    static MPCF_DI void force_to_parent(const MP &m, int i, const JointVar<T> &jv, const T *fc, T *fp)
    {
        T f[3], n[3];
        if (!m.prismatic(i)) {
            f[0] = jv.c * fc[0] - jv.s * fc[1];
            f[1] = jv.s * fc[0] + jv.c * fc[1];
            f[2] = fc[2];
            n[0] = jv.c * fc[3] - jv.s * fc[4];
            n[1] = jv.s * fc[3] + jv.c * fc[4];
            n[2] = fc[5];
        } else {  // n += (q z) x f
            f[0] = fc[0]; f[1] = fc[1]; f[2] = fc[2];
            n[0] = fc[3] - jv.c * fc[1];
            n[1] = fc[4] + jv.c * fc[0];
            n[2] = fc[5];
        }
        T t[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            fp[k] = m.Rp(i, 3 * k) * f[0] + m.Rp(i, 3 * k + 1) * f[1] + m.Rp(i, 3 * k + 2) * f[2];
            fp[3 + k] = m.Rp(i, 3 * k) * n[0] + m.Rp(i, 3 * k + 1) * n[1] + m.Rp(i, 3 * k + 2) * n[2];
        }
        double pp[3] = {m.pp(i, 0), m.pp(i, 1), m.pp(i, 2)};
        cross3(pp, fp, t);
        fp[3] += t[0]; fp[4] += t[1]; fp[5] += t[2];
    }
    static MPCF_DI void joint_var(const MP &m, int i, T q, JointVar<T> &jv)
    {
        if (!m.prismatic(i)) sincos_t(q, jv.s, jv.c);
        else { jv.c = q; jv.s = T(0.0); }
    }
    static MPCF_DI int sidx(const MP &m, int i) { return m.prismatic(i) ? 2 : 5; }

    // rigid-body inertia times motion: [m v - mc x w ; Io w + mc x v]
    static MPCF_DI void inertia_mul(const MP &m, int i, const T *mo, T *f)
    {
        double mc[3] = {m.mc(i, 0), m.mc(i, 1), m.mc(i, 2)};
        T t[3], u[3];
        cross3(mc, mo + 3, t);
        cross3(mc, mo, u);
        double ms = m.mass(i);
        f[0] = ms * mo[0] - t[0];
        f[1] = ms * mo[1] - t[1];
        f[2] = ms * mo[2] - t[2];
        f[3] = m.Io(i, 0) * mo[3] + m.Io(i, 1) * mo[4] + m.Io(i, 2) * mo[5] + u[0];
        f[4] = m.Io(i, 1) * mo[3] + m.Io(i, 3) * mo[4] + m.Io(i, 4) * mo[5] + u[1];
        f[5] = m.Io(i, 2) * mo[3] + m.Io(i, 4) * mo[4] + m.Io(i, 5) * mo[5] + u[2];
    }
    // v x* f
    static MPCF_DI void crossf(const T *v, const T *f, T *o)
    {
        T a[3], b[3], c[3];
        cross3(v + 3, f, a);
        cross3(v + 3, f + 3, b);
        cross3(v, f, c);
        o[0] = a[0]; o[1] = a[1]; o[2] = a[2];
        o[3] = b[0] + c[0]; o[4] = b[1] + c[1]; o[5] = b[2] + c[2];
    }
    // c = v x (S qd)
    static MPCF_DI void bias_c(const MP &m, int i, const T *v, T qd, T *c)
    {
        if (!m.prismatic(i)) {
            c[0] = v[1] * qd; c[1] = -(v[0] * qd); c[2] = T(0.0);
            c[3] = v[4] * qd; c[4] = -(v[3] * qd); c[5] = T(0.0);
        } else {
            c[0] = v[4] * qd; c[1] = -(v[3] * qd); c[2] = T(0.0);
            c[3] = T(0.0); c[4] = T(0.0); c[5] = T(0.0);
        }
    }

    // =========================================================================================
    // RNEA
    // =========================================================================================
    static MPCF_DI void rnea(const MP &m, const T *q, const T *qd, const T *qdd, T *tau)
    {
        JointVar<T> jv[MAXN];
        rnea_impl<false>(m, q, jv, qd, qdd, tau);
    }
    // same with the joint variables (cos q, sin q / shift) already evaluated, so callers that also need frame
    // kinematics share one sincos per joint
    static MPCF_DI void rnea_jv(const MP &m, const JointVar<T> *jv, const T *qd, const T *qdd, T *tau)
    {
        rnea_impl<true>(m, nullptr, const_cast<JointVar<T> *>(jv), qd, qdd, tau);
    }
    // Ext: external link forces.  ext.link(m, i, jv_i, f_i) is called once per link in the forward sweep, after the link's
    // net force f_i = I a + v x* I v (link coordinates, [force ; moment about the joint origin]) is formed; whatever it adds
    // to f_i is carried to the joints by the backward sweep like any other force (tau = ID - J^T f_ext).
    struct NoExt {
        MPCF_DI void link(const MP &, int, const JointVar<T> &, T *) {}
    };
    template <bool HAVE_JV>
    static MPCF_DI void rnea_impl(const MP &m, const T *q, JointVar<T> *jv, const T *qd, const T *qdd, T *tau)
    {
        NoExt none;
        rnea_impl<HAVE_JV>(m, q, jv, qd, qdd, tau, none);
    }
    template <bool HAVE_JV, class Ext>
    static MPCF_DI void rnea_impl(const MP &m, const T *q, JointVar<T> *jv, const T *qd, const T *qdd, T *tau, Ext &ext)
    {
        if constexpr (!MP::kStatic) {
            rnea_tree<HAVE_JV>(m, q, jv, qd, qdd, tau, ext);
            return;
        }
        const int n = m.n();
        constexpr int UNR = MP::kStatic ? MAXN : 1;
        T v[MAXN][6], a[MAXN][6], f[MAXN][6];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            if (!HAVE_JV) joint_var(m, i, q[i], jv[i]);  // interleaved with the link recursion: better ILP than hoisting all sincos
            const int par = m.parent(i), s = sidx(m, i);
            T vp[6], ap[6];
            if (par >= 0) {
#pragma unroll
                for (int k = 0; k < 6; ++k) { vp[k] = v[par][k]; ap[k] = a[par][k]; }
            } else {
#pragma unroll
                for (int k = 0; k < 6; ++k) { vp[k] = T(0.0); ap[k] = T(0.0); }
                ap[0] = T(-m.grav(0)); ap[1] = T(-m.grav(1)); ap[2] = T(-m.grav(2));
            }
            motion_to_child(m, i, jv[i], vp, v[i]);
            v[i][s] += qd[i];
            motion_to_child(m, i, jv[i], ap, a[i]);
            T c[6];
            bias_c(m, i, v[i], qd[i], c);
#pragma unroll
            for (int k = 0; k < 6; ++k) a[i][k] += c[k];
            a[i][s] += qdd[i];
            T h[6], fa[6], fb[6];
            inertia_mul(m, i, v[i], h);
            inertia_mul(m, i, a[i], fa);
            crossf(v[i], h, fb);
#pragma unroll
            for (int k = 0; k < 6; ++k) f[i][k] = fa[k] + fb[k];
            ext.link(m, i, jv[i], f[i]);
        }
#pragma unroll UNR
        for (int i = n - 1; i >= 0; --i) {
            const int par = m.parent(i), s = sidx(m, i);
            tau[i] = f[i][s] + m.arm(i) * qdd[i];
            if (par >= 0) {
                T fp[6];
                force_to_parent(m, i, jv[i], f[i], fp);
#pragma unroll
                for (int k = 0; k < 6; ++k) f[par][k] += fp[k];
            }
        }
    }

    // Run-time trees: the per-link arrays live in local memory (run-time indexing), and at 37 joints the sweeps are bound by
    // that traffic, not by arithmetic.  Links are numbered so that most parents are i - 1: the sweep keeps the current
    // link's (v, a) in registers, reads the arrays only when the parent is not the previous link and writes them only for
    // links some later link branches off (m.keep); the backward sweep likewise carries the force of link i in registers into
    // its parent when that is the next link visited.  Per chain-like link that leaves 6 doubles written and 6 read instead
    // of 18 written and 30 read.
    template <bool HAVE_JV, class Ext>
    static MPCF_DI void rnea_tree(const MP &m, const T *q, JointVar<T> *jv, const T *qd, const T *qdd, T *tau, Ext &ext)
    {
        const int n = m.n();
        T v[MAXN][6], a[MAXN][6], f[MAXN][6];
        T vc[6], ac[6];
#pragma unroll 1
        for (int i = 0; i < n; ++i) {
            if (!HAVE_JV) joint_var(m, i, q[i], jv[i]);
            const int par = m.parent(i), s = sidx(m, i);
            T vp[6], ap[6];
            if (par < 0) {
#pragma unroll
                for (int k = 0; k < 6; ++k) { vp[k] = T(0.0); ap[k] = T(0.0); }
                ap[0] = T(-m.grav(0)); ap[1] = T(-m.grav(1)); ap[2] = T(-m.grav(2));
            } else if (par == i - 1) {
#pragma unroll
                for (int k = 0; k < 6; ++k) { vp[k] = vc[k]; ap[k] = ac[k]; }
            } else {
#pragma unroll
                for (int k = 0; k < 6; ++k) { vp[k] = v[par][k]; ap[k] = a[par][k]; }
            }
            motion_to_child(m, i, jv[i], vp, vc);
            vc[s] += qd[i];
            motion_to_child(m, i, jv[i], ap, ac);
            T c[6];
            bias_c(m, i, vc, qd[i], c);
#pragma unroll
            for (int k = 0; k < 6; ++k) ac[k] += c[k];
            ac[s] += qdd[i];
            if (m.keep(i)) {
#pragma unroll
                for (int k = 0; k < 6; ++k) { v[i][k] = vc[k]; a[i][k] = ac[k]; }
            }
            T h[6], fa[6], fb[6], fi[6];
            inertia_mul(m, i, vc, h);
            inertia_mul(m, i, ac, fa);
            crossf(vc, h, fb);
#pragma unroll
            for (int k = 0; k < 6; ++k) fi[k] = fa[k] + fb[k];
            ext.link(m, i, jv[i], fi);
#pragma unroll
            for (int k = 0; k < 6; ++k) f[i][k] = fi[k];
        }
        T carry[6];  // force handed from link i + 1 to its parent i, when that is the link visited next
        bool have = false;
#pragma unroll 1
        for (int i = n - 1; i >= 0; --i) {
            const int par = m.parent(i), s = sidx(m, i);
            T fi[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) fi[k] = f[i][k] + (have ? carry[k] : T(0.0));
            tau[i] = fi[s] + m.arm(i) * qdd[i];
            have = false;
            if (par >= 0) {
                T fp[6];
                force_to_parent(m, i, jv[i], fi, fp);
                if (par == i - 1) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) carry[k] = fp[k];
                    have = true;
                } else {
#pragma unroll
                    for (int k = 0; k < 6; ++k) f[par][k] += fp[k];
                }
            }
        }
    }

    // =========================================================================================
    // World placements (FK) of joints 0..upto; oR row-major.
    // =========================================================================================
    static MPCF_DI void fk_all(const MP &m, const T *q, T (*oR)[9], T (*op)[3])
    {
        const int n = m.n();
        constexpr int UNR = MP::kStatic ? MAXN : 1;
        JointVar<T> jv[MAXN];
#pragma unroll UNR
        for (int i = 0; i < n; ++i) joint_var(m, i, q[i], jv[i]);
        fk_all_jv(m, jv, oR, op);
    }
    static MPCF_DI void fk_all_jv(const MP &m, const JointVar<T> *jvs, T (*oR)[9], T (*op)[3])
    {
        const int n = m.n();
        constexpr int UNR = MP::kStatic ? MAXN : 1;
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            const int par = m.parent(i);
            const JointVar<T> jv = jvs[i];
            // local liMi = (R, p)
            T R[9], p[3];
            if (!m.prismatic(i)) {
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    R[3 * r + 0] = m.Rp(i, 3 * r) * jv.c + m.Rp(i, 3 * r + 1) * jv.s;
                    R[3 * r + 1] = m.Rp(i, 3 * r + 1) * jv.c - m.Rp(i, 3 * r) * jv.s;
                    R[3 * r + 2] = T(m.Rp(i, 3 * r + 2));
                    p[r] = T(m.pp(i, r));
                }
            } else {
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    R[3 * r + 0] = T(m.Rp(i, 3 * r)); R[3 * r + 1] = T(m.Rp(i, 3 * r + 1)); R[3 * r + 2] = T(m.Rp(i, 3 * r + 2));
                    p[r] = m.pp(i, r) + m.Rp(i, 3 * r + 2) * jv.c;
                }
            }
            if (par < 0) {
#pragma unroll
                for (int k = 0; k < 9; ++k) oR[i][k] = R[k];
#pragma unroll
                for (int k = 0; k < 3; ++k) op[i][k] = p[k];
            } else {
#pragma unroll
                for (int r = 0; r < 3; ++r) {
#pragma unroll
                    for (int c = 0; c < 3; ++c)
                        oR[i][3 * r + c] = oR[par][3 * r] * R[c] + oR[par][3 * r + 1] * R[3 + c] + oR[par][3 * r + 2] * R[6 + c];
                    op[i][r] = op[par][r] + oR[par][3 * r] * p[0] + oR[par][3 * r + 1] * p[1] + oR[par][3 * r + 2] * p[2];
                }
            }
        }
    }

    // frame pose from joint placements; fj = parent joint (-1 world), (fR, fp) constant placement
    static MPCF_DI void frame_pose(int fj, const double *fR, const double *fp, T (*oR)[9], T (*op)[3], T *pos, T *rot)
    {
        if (fj < 0) {
#pragma unroll
            for (int k = 0; k < 9; ++k) rot[k] = T(fR[k]);
#pragma unroll
            for (int k = 0; k < 3; ++k) pos[k] = T(fp[k]);
            return;
        }
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
            for (int c = 0; c < 3; ++c)
                rot[3 * r + c] = oR[fj][3 * r] * fR[c] + oR[fj][3 * r + 1] * fR[3 + c] + oR[fj][3 * r + 2] * fR[6 + c];
            pos[r] = op[fj][r] + oR[fj][3 * r] * fp[0] + oR[fj][3 * r + 1] * fp[1] + oR[fj][3 * r + 2] * fp[2];
        }
    }

    // =========================================================================================
    // ABA.  Articulated inertia kept as symmetric blocks: A (lin-lin, sym 6), B (lin-ang, full 9),
    // C (ang-ang, sym 6); sym storage [xx xy xz yy yz zz].
    // =========================================================================================
    struct Art {
        T A[6], B[9], C[6];
    };
    static MPCF_DI T symget(const T *S, int r, int c)
    {
        const int idx[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};
        return S[idx[r][c]];
    }
    // rotate a symmetric 3x3 by Rz: S <- Rz S Rz^T, with c2 = c^2 - s^2, s2 = 2cs
    static MPCF_DI void rotz_sym(T *S, T c, T s, T c2, T s2)
    {
        T h = 0.5 * (S[0] + S[3]), d = 0.5 * (S[0] - S[3]);
        T e = d * c2 - S[1] * s2;
        T xy = d * s2 + S[1] * c2;
        T xz = c * S[2] - s * S[4];
        T yz = s * S[2] + c * S[4];
        S[0] = h + e; S[3] = h - e; S[1] = xy; S[2] = xz; S[4] = yz;
    }
    static MPCF_DI void rotz_full(T *B, T c, T s)
    {
#pragma unroll
        for (int k = 0; k < 3; ++k) {  // rows 0,1 mix
            T a = B[k], b = B[3 + k];
            B[k] = c * a - s * b;
            B[3 + k] = s * a + c * b;
        }
#pragma unroll
        for (int r = 0; r < 3; ++r) {  // cols 0,1 mix
            T a = B[3 * r], b = B[3 * r + 1];
            B[3 * r] = c * a - s * b;
            B[3 * r + 1] = s * a + c * b;
        }
    }
    // constant rotation: S <- R S R^T (sym), R row-major doubles via the model policy
    static MPCF_DI void rot_sym(const MP &m, int i, const T *S, T *O)
    {
        T t[9];  // t = R * S
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            double r0 = m.Rp(i, 3 * r), r1 = m.Rp(i, 3 * r + 1), r2 = m.Rp(i, 3 * r + 2);
            t[3 * r + 0] = r0 * S[0] + r1 * S[1] + r2 * S[2];
            t[3 * r + 1] = r0 * S[1] + r1 * S[3] + r2 * S[4];
            t[3 * r + 2] = r0 * S[2] + r1 * S[4] + r2 * S[5];
        }
        const int rr[6] = {0, 0, 0, 1, 1, 2}, cc[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
        for (int k = 0; k < 6; ++k)
            O[k] = t[3 * rr[k]] * m.Rp(i, 3 * cc[k]) + t[3 * rr[k] + 1] * m.Rp(i, 3 * cc[k] + 1) + t[3 * rr[k] + 2] * m.Rp(i, 3 * cc[k] + 2);
    }
    static MPCF_DI void rot_full(const MP &m, int i, const T *B, T *O)
    {
        T t[9];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c)
                t[3 * r + c] = m.Rp(i, 3 * r) * B[c] + m.Rp(i, 3 * r + 1) * B[3 + c] + m.Rp(i, 3 * r + 2) * B[6 + c];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c)
                O[3 * r + c] = t[3 * r] * m.Rp(i, 3 * c) + t[3 * r + 1] * m.Rp(i, 3 * c + 1) + t[3 * r + 2] * m.Rp(i, 3 * c + 2);
    }
    // translate blocks (already in the destination axes) by p:  B'' = B - A P ; C'' = C + (P B)^T + P B''
    template <class PT>
    static MPCF_DI void translate(T *A, T *B, T *C, const PT *p)
    {
        T G[9], H[9];  // G = P B (old B), H = P B''
#pragma unroll
        for (int c = 0; c < 3; ++c) {  // column c of P*M = p x M[:,c]
            G[c] = p[1] * B[6 + c] - p[2] * B[3 + c];
            G[3 + c] = p[2] * B[c] - p[0] * B[6 + c];
            G[6 + c] = p[0] * B[3 + c] - p[1] * B[c];
        }
#pragma unroll
        for (int r = 0; r < 3; ++r) {  // row r of A*P = A[r,:] x p
            T a0 = symget(A, r, 0), a1 = symget(A, r, 1), a2 = symget(A, r, 2);
            B[3 * r + 0] -= a1 * p[2] - a2 * p[1];
            B[3 * r + 1] -= a2 * p[0] - a0 * p[2];
            B[3 * r + 2] -= a0 * p[1] - a1 * p[0];
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            H[c] = p[1] * B[6 + c] - p[2] * B[3 + c];
            H[3 + c] = p[2] * B[c] - p[0] * B[6 + c];
            H[6 + c] = p[0] * B[3 + c] - p[1] * B[c];
        }
        const int rr[6] = {0, 0, 0, 1, 1, 2}, cc[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
        for (int k = 0; k < 6; ++k) C[k] += G[3 * cc[k] + rr[k]] + H[3 * rr[k] + cc[k]];
    }

    // Per-link quantities kept between the ABA passes.
    struct AbaLink {
        JointVar<T> jv;
        T v[6];
        T U[6];
        T Dinv, u;
    };

    // Generic ABA over a tree.  IA / pA are accumulated per link (needed for branches).
    // Returns false when some D_i == 0 (singular without armature).
    static MPCF_DI bool aba(const MP &m, const T *q, const T *qd, const T *tau, T *qdd)
    {
        if constexpr (!MP::kStatic) return aba_tree(m, q, qd, tau, qdd);
        const int n = m.n();
        constexpr int UNR = MP::kStatic ? MAXN : 1;
        AbaLink L[MAXN];
        Art IA[MAXN];
        T pA[MAXN][6];
        bool ok = true;
        // pass 1: velocities; zero the child-contribution accumulators
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            const int par = m.parent(i), s = sidx(m, i);
            joint_var(m, i, q[i], L[i].jv);
            if (par >= 0) motion_to_child(m, i, L[i].jv, L[par].v, L[i].v);
            else {
#pragma unroll
                for (int k = 0; k < 6; ++k) L[i].v[k] = T(0.0);
            }
            L[i].v[s] += qd[i];
#pragma unroll
            for (int k = 0; k < 6; ++k) { IA[i].A[k] = T(0.0); IA[i].C[k] = T(0.0); pA[i][k] = T(0.0); }
#pragma unroll
            for (int k = 0; k < 9; ++k) IA[i].B[k] = T(0.0);
        }
        // pass 2: articulated inertias leaf -> root
#pragma unroll UNR
        for (int i = n - 1; i >= 0; --i) {
            const int par = m.parent(i);
            const bool pr = m.prismatic(i);
            Art &I = IA[i];
            {   // add this link's own rigid-body inertia and bias force to what the children left
                const double ms = m.mass(i), cx = m.mc(i, 0), cy = m.mc(i, 1), cz = m.mc(i, 2);
                I.A[0] += ms; I.A[3] += ms; I.A[5] += ms;
                I.B[1] += cz;  I.B[2] += -cy;
                I.B[3] += -cz; I.B[5] += cx;
                I.B[6] += cy;  I.B[7] += -cx;
#pragma unroll
                for (int k = 0; k < 6; ++k) I.C[k] += m.Io(i, k);
                T h[6], pb[6];
                inertia_mul(m, i, L[i].v, h);
                crossf(L[i].v, h, pb);
#pragma unroll
                for (int k = 0; k < 6; ++k) pA[i][k] += pb[k];
            }
            // U = IA[:, s] as [lin(3); ang(3)],  D = IA[s][s] + armature
            T *U = L[i].U;
            T D;
            if (!pr) {
                U[0] = I.B[2]; U[1] = I.B[5]; U[2] = I.B[8];
                U[3] = I.C[2]; U[4] = I.C[4]; U[5] = I.C[5];
                D = I.C[5] + m.arm(i);
            } else {
                U[0] = I.A[2]; U[1] = I.A[4]; U[2] = I.A[5];
                U[3] = I.B[6]; U[4] = I.B[7]; U[5] = I.B[8];
                D = I.A[5] + m.arm(i);
            }
            if (!(value_of(D) > 0.0)) { ok = false; D = T(nan_value()); }  // singular: NaN outputs, never a plausible wrong number
            const T Dinv = recip(D);
            L[i].Dinv = Dinv;
            const T u = tau[i] - pA[i][pr ? 2 : 5];
            L[i].u = u;
            if (par >= 0) {
                T UD[6];
#pragma unroll
                for (int k = 0; k < 6; ++k) UD[k] = U[k] * Dinv;
                // Ia = IA - U Dinv U^T  (in place)
                const int rr[6] = {0, 0, 0, 1, 1, 2}, cc[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    I.A[k] -= UD[rr[k]] * U[cc[k]];
                    I.C[k] -= UD[3 + rr[k]] * U[3 + cc[k]];
                }
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int c = 0; c < 3; ++c) I.B[3 * r + c] -= UD[r] * U[3 + c];
                // pa = pA + Ia c + U Dinv u
                T cb[6], pa[6];
                bias_c(m, i, L[i].v, qd[i], cb);
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    pa[r] = pA[i][r] + UD[r] * u + symget(I.A, r, 0) * cb[0] + symget(I.A, r, 1) * cb[1] + symget(I.A, r, 2) * cb[2] +
                            I.B[3 * r] * cb[3] + I.B[3 * r + 1] * cb[4] + I.B[3 * r + 2] * cb[5];
                    pa[3 + r] = pA[i][3 + r] + UD[3 + r] * u + I.B[r] * cb[0] + I.B[3 + r] * cb[1] + I.B[6 + r] * cb[2] +
                                symget(I.C, r, 0) * cb[3] + symget(I.C, r, 1) * cb[4] + symget(I.C, r, 2) * cb[5];
                }
                // variable stage
                const JointVar<T> &jv = L[i].jv;
                if (!pr) {
                    T c2 = jv.c * jv.c - jv.s * jv.s, s2 = 2.0 * (jv.c * jv.s);
                    rotz_sym(I.A, jv.c, jv.s, c2, s2);
                    rotz_sym(I.C, jv.c, jv.s, c2, s2);
                    rotz_full(I.B, jv.c, jv.s);
                } else {
                    T pz[3] = {T(0.0), T(0.0), jv.c};
                    translate(I.A, I.B, I.C, pz);
                }
                // constant stage
                Art O;
                rot_sym(m, i, I.A, O.A);
                rot_sym(m, i, I.C, O.C);
                rot_full(m, i, I.B, O.B);
                double pp[3] = {m.pp(i, 0), m.pp(i, 1), m.pp(i, 2)};
                translate(O.A, O.B, O.C, pp);
                Art &Ip = IA[par];
#pragma unroll
                for (int k = 0; k < 6; ++k) { Ip.A[k] += O.A[k]; Ip.C[k] += O.C[k]; }
#pragma unroll
                for (int k = 0; k < 9; ++k) Ip.B[k] += O.B[k];
                T fp[6];
                force_to_parent(m, i, jv, pa, fp);
#pragma unroll
                for (int k = 0; k < 6; ++k) pA[par][k] += fp[k];
            }
        }
        // pass 3: accelerations root -> leaf.  pA[i] is reused to hold a_i.
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            const int par = m.parent(i), s = sidx(m, i);
            T ap[6], a[6], cb[6];
            if (par >= 0) {
#pragma unroll
                for (int k = 0; k < 6; ++k) ap[k] = pA[par][k];
            } else {
                ap[0] = T(-m.grav(0)); ap[1] = T(-m.grav(1)); ap[2] = T(-m.grav(2));
                ap[3] = T(0.0); ap[4] = T(0.0); ap[5] = T(0.0);
            }
            motion_to_child(m, i, L[i].jv, ap, a);
            bias_c(m, i, L[i].v, qd[i], cb);
            T acc = L[i].u;
#pragma unroll
            for (int k = 0; k < 6; ++k) { a[k] += cb[k]; acc -= L[i].U[k] * a[k]; }
            const T qa = L[i].Dinv * acc;
            qdd[i] = qa;
            a[s] += qa;
#pragma unroll
            for (int k = 0; k < 6; ++k) pA[i][k] = a[k];
        }
        return ok;
    }

    // ABA for run-time trees.  Same arithmetic as aba(); what changes is where the per-link data live (cf. rnea_tree): the
    // articulated inertia and bias force a link hands to its parent travel in registers when the parent is the link
    // visited next (par == i - 1), the accumulator arrays IA / pA are touched only by links whose parent is elsewhere and
    // are initialised only for links that have such children (m.keep), and the outward acceleration sweep keeps the
    // current link's acceleration in registers.  Local-memory traffic per chain-like link drops from ~160 to ~45 doubles.
    static MPCF_DI bool aba_tree(const MP &m, const T *q, const T *qd, const T *tau, T *qdd)
    {
        const int n = m.n();
        AbaLink L[MAXN];
        Art IA[MAXN];
        T pA[MAXN][6];
        bool ok = true;
        {
            T vc[6];
#pragma unroll 1
            for (int i = 0; i < n; ++i) {
                const int par = m.parent(i), s = sidx(m, i);
                JointVar<T> jv;
                joint_var(m, i, q[i], jv);
                L[i].jv = jv;
                T vp[6];
                if (par < 0) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) vp[k] = T(0.0);
                } else if (par == i - 1) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) vp[k] = vc[k];
                } else {
#pragma unroll
                    for (int k = 0; k < 6; ++k) vp[k] = L[par].v[k];
                }
                if (par >= 0) motion_to_child(m, i, jv, vp, vc);
                else {
#pragma unroll
                    for (int k = 0; k < 6; ++k) vc[k] = T(0.0);
                }
                vc[s] += qd[i];
#pragma unroll
                for (int k = 0; k < 6; ++k) L[i].v[k] = vc[k];
                if (m.keep(i)) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) { IA[i].A[k] = T(0.0); IA[i].C[k] = T(0.0); pA[i][k] = T(0.0); }
#pragma unroll
                    for (int k = 0; k < 9; ++k) IA[i].B[k] = T(0.0);
                }
            }
        }
        {
            Art cI;    // what link i + 1 hands to link i
            T cp[6];
            bool have = false;
#pragma unroll 1
            for (int i = n - 1; i >= 0; --i) {
                const int par = m.parent(i);
                const bool pr = m.prismatic(i);
                Art I;
                T p[6], v[6];
                if (m.keep(i)) {
                    I = IA[i];
#pragma unroll
                    for (int k = 0; k < 6; ++k) p[k] = pA[i][k];
                } else {
#pragma unroll
                    for (int k = 0; k < 6; ++k) { I.A[k] = T(0.0); I.C[k] = T(0.0); p[k] = T(0.0); }
#pragma unroll
                    for (int k = 0; k < 9; ++k) I.B[k] = T(0.0);
                }
                if (have) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) { I.A[k] += cI.A[k]; I.C[k] += cI.C[k]; p[k] += cp[k]; }
#pragma unroll
                    for (int k = 0; k < 9; ++k) I.B[k] += cI.B[k];
                }
                have = false;
#pragma unroll
                for (int k = 0; k < 6; ++k) v[k] = L[i].v[k];
                {
                    const double ms = m.mass(i), cx = m.mc(i, 0), cy = m.mc(i, 1), cz = m.mc(i, 2);
                    I.A[0] += ms; I.A[3] += ms; I.A[5] += ms;
                    I.B[1] += cz;  I.B[2] += -cy;
                    I.B[3] += -cz; I.B[5] += cx;
                    I.B[6] += cy;  I.B[7] += -cx;
#pragma unroll
                    for (int k = 0; k < 6; ++k) I.C[k] += m.Io(i, k);
                    T h[6], pb[6];
                    inertia_mul(m, i, v, h);
                    crossf(v, h, pb);
#pragma unroll
                    for (int k = 0; k < 6; ++k) p[k] += pb[k];
                }
                T U[6], D;
                if (!pr) {
                    U[0] = I.B[2]; U[1] = I.B[5]; U[2] = I.B[8];
                    U[3] = I.C[2]; U[4] = I.C[4]; U[5] = I.C[5];
                    D = I.C[5] + m.arm(i);
                } else {
                    U[0] = I.A[2]; U[1] = I.A[4]; U[2] = I.A[5];
                    U[3] = I.B[6]; U[4] = I.B[7]; U[5] = I.B[8];
                    D = I.A[5] + m.arm(i);
                }
                if (!(value_of(D) > 0.0)) { ok = false; D = T(nan_value()); }  // singular: NaN outputs, never a plausible wrong number
                const T Dinv = recip(D);
                const T u = tau[i] - p[pr ? 2 : 5];
#pragma unroll
                for (int k = 0; k < 6; ++k) L[i].U[k] = U[k];
                L[i].Dinv = Dinv;
                L[i].u = u;
                if (par >= 0) {
                    T UD[6];
#pragma unroll
                    for (int k = 0; k < 6; ++k) UD[k] = U[k] * Dinv;
                    const int rr[6] = {0, 0, 0, 1, 1, 2}, cc[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
                    for (int k = 0; k < 6; ++k) {
                        I.A[k] -= UD[rr[k]] * U[cc[k]];
                        I.C[k] -= UD[3 + rr[k]] * U[3 + cc[k]];
                    }
#pragma unroll
                    for (int r = 0; r < 3; ++r)
#pragma unroll
                        for (int c = 0; c < 3; ++c) I.B[3 * r + c] -= UD[r] * U[3 + c];
                    T cb[6], pa[6];
                    bias_c(m, i, v, qd[i], cb);
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        pa[r] = p[r] + UD[r] * u + symget(I.A, r, 0) * cb[0] + symget(I.A, r, 1) * cb[1] + symget(I.A, r, 2) * cb[2] +
                                I.B[3 * r] * cb[3] + I.B[3 * r + 1] * cb[4] + I.B[3 * r + 2] * cb[5];
                        pa[3 + r] = p[3 + r] + UD[3 + r] * u + I.B[r] * cb[0] + I.B[3 + r] * cb[1] + I.B[6 + r] * cb[2] +
                                    symget(I.C, r, 0) * cb[3] + symget(I.C, r, 1) * cb[4] + symget(I.C, r, 2) * cb[5];
                    }
                    const JointVar<T> jv = L[i].jv;
                    if (!pr) {
                        T c2 = jv.c * jv.c - jv.s * jv.s, s2 = 2.0 * (jv.c * jv.s);
                        rotz_sym(I.A, jv.c, jv.s, c2, s2);
                        rotz_sym(I.C, jv.c, jv.s, c2, s2);
                        rotz_full(I.B, jv.c, jv.s);
                    } else {
                        T pz[3] = {T(0.0), T(0.0), jv.c};
                        translate(I.A, I.B, I.C, pz);
                    }
                    Art O;
                    rot_sym(m, i, I.A, O.A);
                    rot_sym(m, i, I.C, O.C);
                    rot_full(m, i, I.B, O.B);
                    double pp[3] = {m.pp(i, 0), m.pp(i, 1), m.pp(i, 2)};
                    translate(O.A, O.B, O.C, pp);
                    T fp[6];
                    force_to_parent(m, i, jv, pa, fp);
                    if (par == i - 1) {
                        cI = O;
#pragma unroll
                        for (int k = 0; k < 6; ++k) cp[k] = fp[k];
                        have = true;
                    } else {
                        Art &Ip = IA[par];
#pragma unroll
                        for (int k = 0; k < 6; ++k) { Ip.A[k] += O.A[k]; Ip.C[k] += O.C[k]; pA[par][k] += fp[k]; }
#pragma unroll
                        for (int k = 0; k < 9; ++k) Ip.B[k] += O.B[k];
                    }
                }
            }
        }
        {
            T ac[6];  // acceleration of the previous link; pA[i] is reused to hold a_i of the links others branch off
#pragma unroll 1
            for (int i = 0; i < n; ++i) {
                const int par = m.parent(i), s = sidx(m, i);
                T ap[6], a[6], cb[6];
                if (par < 0) {
                    ap[0] = T(-m.grav(0)); ap[1] = T(-m.grav(1)); ap[2] = T(-m.grav(2));
                    ap[3] = T(0.0); ap[4] = T(0.0); ap[5] = T(0.0);
                } else if (par == i - 1) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) ap[k] = ac[k];
                } else {
#pragma unroll
                    for (int k = 0; k < 6; ++k) ap[k] = pA[par][k];
                }
                motion_to_child(m, i, L[i].jv, ap, a);
                bias_c(m, i, L[i].v, qd[i], cb);
                T acc = L[i].u;
#pragma unroll
                for (int k = 0; k < 6; ++k) { a[k] += cb[k]; acc -= L[i].U[k] * a[k]; }
                const T qa = L[i].Dinv * acc;
                qdd[i] = qa;
                a[s] += qa;
#pragma unroll
                for (int k = 0; k < 6; ++k) ac[k] = a[k];
                if (m.keep(i)) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) pA[i][k] = a[k];
                }
            }
        }
        return ok;
    }

    // =========================================================================================
    // fatigue compartment ODE and its exact zero-order-hold map
    // =========================================================================================
    static MPCF_DI T fatigue_rhs(const MP &m, int i, T f, T tau, T qd)
    {
        return m.fat(i, 1) * (m.fat(i, 2) * (tau * tau) + m.fat(i, 3) * (qd * qd)) - m.fat(i, 0) * f;
    }

    // =========================================================================================
    // Forward dynamics through the joint-space inertia matrix: qdd = M^-1 (tau - h).
    // One fused sweep pair computes the RNEA bias h = ID(q, qd, 0) and, from the composite rigid-body inertias,
    // the columns of M (CRBA); M is factorised M = L D L^T in place.  For short chains (n <~ 9) this is cheaper than ABA
    // (no 6x6 articulated inertias to carry and transform).  Static forests of revolute chains only (parent = i - 1).
    // =========================================================================================
    // MINV: also return C = M^-1 per chain as a packed lower triangle, Minv[chain * L (L + 1) / 2 + r (r + 1) / 2 + c], c <= r
    // (from the factors: C = Lm^-T D^-1 Lm^-1) — the Jacobian pipeline's derivative kernel consumes it.
    // (Per-link scheduling fences, StaticModel::skip, were tried here: fewer spills, but the RK4 step kernel ran 4 % slower.)
    template <int L, bool MINV = false>
    static MPCF_DI bool fd_crba(const MP &m, const T *q, const T *qd, const T *tau, T *qdd, T *Minv = nullptr)
    {
        static_assert(MP::kStatic, "fd_crba needs a compile-time forest of chains");
        constexpr int N = MAXN;
        JointVar<T> jv[N];
        T f[N][6];
        T Mx[N][L];  // M[i][j] stored as Mx[i][j - c0], same chain only
        T h[N];
        {   // pass 1: velocities, bias accelerations (qdd = 0), link forces
            T v[6], a[6];
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const bool root = m.parent(i) < 0;
                joint_var(m, i, q[i], jv[i]);
                T vp[6], ap[6];
#pragma unroll
                for (int k = 0; k < 6; ++k) { vp[k] = root ? T(0.0) : v[k]; ap[k] = root ? T(0.0) : a[k]; }
                if (root) { ap[0] = T(-m.grav(0)); ap[1] = T(-m.grav(1)); ap[2] = T(-m.grav(2)); }
                motion_to_child(m, i, jv[i], vp, v);
                v[5] += qd[i];
                motion_to_child(m, i, jv[i], ap, a);
                T c[6];
                bias_c(m, i, v, qd[i], c);
#pragma unroll
                for (int k = 0; k < 6; ++k) a[k] += c[k];
                T hv[6], fa[6], fb[6];
                inertia_mul(m, i, v, hv);
                inertia_mul(m, i, a, fa);
                crossf(v, hv, fb);
#pragma unroll
                for (int k = 0; k < 6; ++k) f[i][k] = fa[k] + fb[k];
            }
        }
        {   // pass 2: bias torques, composite inertias (mass, mass*com, inertia about the joint origin), columns of M
            T cm, cmc[3], cI[6];
#pragma unroll
            for (int i = N - 1; i >= 0; --i) {
                const bool leaf = ((i + 1) % L) == 0;
                const int c0 = (i / L) * L;
                if (leaf) {
                    cm = T(m.mass(i));
#pragma unroll
                    for (int k = 0; k < 3; ++k) cmc[k] = T(m.mc(i, k));
#pragma unroll
                    for (int k = 0; k < 6; ++k) cI[k] = T(m.Io(i, k));
                } else {
                    cm += m.mass(i);
#pragma unroll
                    for (int k = 0; k < 3; ++k) cmc[k] += m.mc(i, k);
#pragma unroll
                    for (int k = 0; k < 6; ++k) cI[k] += m.Io(i, k);
                }
                h[i] = f[i][5];
                // column i of M: F = Yc_i S (S = e5) = [-(mc x z); Io[:, 2]], then carried up the chain
                T F[6] = {-cmc[1], cmc[0], T(0.0), cI[2], cI[4], cI[5]};
                Mx[i][i - c0] = F[5] + m.arm(i);
#pragma unroll
                for (int j = i; j > c0; --j) {
                    T Fp[6];
                    force_to_parent(m, j, jv[j], F, Fp);
#pragma unroll
                    for (int k = 0; k < 6; ++k) F[k] = Fp[k];
                    Mx[i][j - 1 - c0] = F[5];
                }
                if (i > c0) {
                    // bias force and composite inertia of the sub-chain move to the parent frame
                    T fp[6];
                    force_to_parent(m, i, jv[i], f[i], fp);
#pragma unroll
                    for (int k = 0; k < 6; ++k) f[i - 1][k] += fp[k];
                    // variable stage: rotate by Rz(q)
                    const T c = jv[i].c, s = jv[i].s;
                    const T c2 = c * c - s * s, s2 = 2.0 * (c * s);
                    rotz_sym(cI, c, s, c2, s2);
                    const T mx = c * cmc[0] - s * cmc[1], my = s * cmc[0] + c * cmc[1];
                    cmc[0] = mx; cmc[1] = my;
                    // constant stage: rotate by Rp, shift by pp:  Io' = R Io R^T + (2 a.p + m p.p) 1 - (a p^T + p a^T + m p p^T)
                    T RI[6], a3[3];
                    rot_sym(m, i, cI, RI);
#pragma unroll
                    for (int r = 0; r < 3; ++r) a3[r] = m.Rp(i, 3 * r) * cmc[0] + m.Rp(i, 3 * r + 1) * cmc[1] + m.Rp(i, 3 * r + 2) * cmc[2];
                    const double p0 = m.pp(i, 0), p1 = m.pp(i, 1), p2 = m.pp(i, 2);
                    const T ap = a3[0] * p0 + a3[1] * p1 + a3[2] * p2;
                    const T dg = 2.0 * ap + cm * (p0 * p0 + p1 * p1 + p2 * p2);
                    const double pv[3] = {p0, p1, p2};
                    const int rr[6] = {0, 0, 0, 1, 1, 2}, cc[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
                    for (int k = 0; k < 6; ++k) {
                        T e = RI[k] - (a3[rr[k]] * pv[cc[k]] + a3[cc[k]] * pv[rr[k]] + cm * (pv[rr[k]] * pv[cc[k]]));
                        if (rr[k] == cc[k]) e += dg;
                        cI[k] = e;
                    }
#pragma unroll
                    for (int r = 0; r < 3; ++r) cmc[r] = a3[r] + cm * pv[r];
                }
            }
        }
        // per chain: M = Lm D Lm^T, then solve for qdd
        bool ok = true;
#pragma unroll
        for (int c0 = 0; c0 < N; c0 += L) {
            T Lm[L][L], LD[L][L], Dinv[L], x[L];
#pragma unroll
            for (int j = 0; j < L; ++j) {
                T d = Mx[c0 + j][j];
#pragma unroll
                for (int k = 0; k < j; ++k) d -= Lm[j][k] * LD[j][k];
                if (!(value_of(d) > 0.0)) { ok = false; d = T(nan_value()); }  // non-positive pivot of M: NaN outputs
                Dinv[j] = recip(d);
#pragma unroll
                for (int i = j + 1; i < L; ++i) {
                    T e = Mx[c0 + i][j];
#pragma unroll
                    for (int k = 0; k < j; ++k) e -= Lm[i][k] * LD[j][k];
                    LD[i][j] = e;
                    Lm[i][j] = e * Dinv[j];
                }
            }
#pragma unroll
            for (int i = 0; i < L; ++i) {
                x[i] = tau[c0 + i] - h[c0 + i];
#pragma unroll
                for (int k = 0; k < i; ++k) x[i] -= Lm[i][k] * x[k];
            }
#pragma unroll
            for (int i = 0; i < L; ++i) x[i] = x[i] * Dinv[i];
#pragma unroll
            for (int i = L - 1; i >= 0; --i) {
#pragma unroll
                for (int k = i + 1; k < L; ++k) x[i] -= Lm[k][i] * x[k];
                qdd[c0 + i] = x[i];
            }
            if constexpr (MINV) {
                T Li[L][L];  // Lm^-1 (unit lower triangular), strictly-lower entries
#pragma unroll
                for (int j = 0; j < L; ++j)
#pragma unroll
                    for (int i = j + 1; i < L; ++i) {
                        T e = -Lm[i][j];
#pragma unroll
                        for (int k = j + 1; k < i; ++k) e -= Lm[i][k] * Li[k][j];
                        Li[i][j] = e;
                    }
                T *Cp = Minv + (c0 / L) * (L * (L + 1) / 2);
#pragma unroll
                for (int i = 0; i < L; ++i)
#pragma unroll
                    for (int j = 0; j <= i; ++j) {
                        T e = (i == j) ? Dinv[i] : Li[i][j] * Dinv[i];  // k = i term: Li[i][i] = 1
#pragma unroll
                        for (int k = i + 1; k < L; ++k) e += (Li[k][i] * Dinv[k]) * Li[k][j];
                        Cp[i * (i + 1) / 2 + j] = e;
                    }
            }
        }
        return ok;
    }

    // forward dynamics: through M for short static chains, ABA otherwise
    static MPCF_DI bool fd(const MP &m, const T *q, const T *qd, const T *tau, T *qdd)
    {
        if constexpr (MP::kStatic && MP::kChain > 0 && MP::kChain <= 8) return fd_crba<MP::kChain>(m, q, qd, tau, qdd);
        else return aba(m, q, qd, tau, qdd);
    }

    // xdot = (qd, FD(q, qd, tau), fatigue_rhs); x = [q | qd | f]
    // theat: the torque that heats the windings; tau unless the arms' fatigue is coupled through a shared load (kernels_couple.cu)
    static MPCF_DI bool xdot(const MP &m, const T *x, const T *tau, const T *theat, T *k)
    {
        const int n = m.n();
        constexpr int UNR = MP::kStatic ? MAXN : 1;
        bool ok = fd(m, x, x + n, tau, k + n);
#pragma unroll UNR
        for (int i = 0; i < n; ++i) {
            k[i] = x[n + i];
            k[2 * n + i] = fatigue_rhs(m, i, x[2 * n + i], theat[i], x[n + i]);
        }
        return ok;
    }

    // classical RK4, tau held over the step.  The four stages run as a rolled loop: fully unrolled, the step kernel of a
    // 6-joint chain is 190 KB of straight-line code and spends half its time waiting for instruction fetch
    // (profiles/r01_jvp_pipeline.md); rolled, one stage body (48 KB) stays in the instruction cache.
    static MPCF_DI bool step_rk4(const MP &m, const T *x, const T *tau, T dt, T *xn) { return step_rk4(m, x, tau, tau, dt, xn); }
    static MPCF_DI bool step_rk4(const MP &m, const T *x, const T *tau, const T *theat, T dt, T *xn)
    {
        const int n3 = 3 * m.n();
        constexpr int UNR3 = MP::kStatic ? 3 * MAXN : 1;
        T k[3 * MAXN], xs[3 * MAXN];
#pragma unroll UNR3
        for (int i = 0; i < n3; ++i) { xn[i] = x[i]; xs[i] = x[i]; }
        bool ok = true;
#pragma unroll 1
        for (int s = 0; s < 4; ++s) {
            ok &= xdot(m, xs, tau, theat, k);
            const T w = dt * ((s == 0 || s == 3) ? (1.0 / 6.0) : (1.0 / 3.0));
            const T c = dt * (s < 2 ? 0.5 : (s == 2 ? 1.0 : 0.0));
#pragma unroll UNR3
            for (int i = 0; i < n3; ++i) {
                xn[i] += w * k[i];
                xs[i] = x[i] + c * k[i];
            }
        }
        return ok;
    }
};

}  // namespace mpcf
