// kernels.cuh — model policies + launcher declarations shared by kernels.cu and capi.cpp
#pragma once

#include <cuda_runtime.h>

#include "../../include/mpcf.h"

namespace mpcf {

// ---- compile-time topology: a forest of N/L serial revolute chains of length L ----
// The constants travel as a __grid_constant__ kernel parameter, i.e. they sit in the constant bank and
// are consumed directly as DFMA/DMUL operands (no load instruction, no register) once the link loops
// are fully unrolled.
template <int N>
struct StaticParams {
    double Rp[N][9], pp[N][3], mass[N], mc[N][3], Io[N][6], arm[N], fat[N][4], grav[3];
    int fence0;  // always 0; see StaticModel::skip
};

// ---- run-time topology: model blob staged into shared memory by every block ----
// blob layout (doubles): Rp 9n | pp 3n | mass n | mc 3n | Io 6n | arm n | fat 4n | grav 3
// followed by ints: parent n | jtype n | keep n | depth n | rowptr n + 1  (keep[i] = 1 when some link other than i + 1 has
// parent i, i.e. link i's kinematic state must outlive the next link of the sweep; depth / rowptr: packed ancestor storage of
// the tree Jacobian pipeline, rowptr[i] = sum of (depth[k] + 1) over k < i)
struct GenericBlob {
    const double *dbl;  // device
    const int *ints;    // device
    int n;
};
inline size_t blob_doubles(int n) { return (size_t)27 * n + 3; }
inline __host__ __device__ int blob_ints(int n) { return 5 * n + 1; }
inline size_t blob_smem_bytes(int n) { return blob_doubles(n) * sizeof(double) + (size_t)blob_ints(n) * sizeof(int); }

struct FrameArg {
    int joint;  // parent joint, -1 = world
    double R[9], p[3];
};
struct EeArgs {
    int nee;
    FrameArg f[MPCF_MAX_EE];
};
struct ZohArg {
    double a[MPCF_MAX_DOF];  // exp(-lambda_i h), computed once on the host
    double g[MPCF_MAX_DOF];  // gain -expm1(-lambda_i h) kappa_i / lambda_i (lambda_i != 0): 1 - a_i cancels as lambda_i h -> 0
};

enum Family { FAM_GENERIC16 = 0, FAM_GENERIC64, FAM_CHAIN3, FAM_CHAIN6, FAM_FOREST12x6, FAM_CHAIN7, FAM_FOREST14x7, FAM_COUNT };
// serial-chain length of a static family (0 for run-time-topology families) and number of chains
inline int family_chain_len(Family f) { return f == FAM_CHAIN3 ? 3 : (f == FAM_CHAIN6 || f == FAM_FOREST12x6) ? 6 : (f == FAM_CHAIN7 || f == FAM_FOREST14x7) ? 7 : 0; }
inline int family_chains(Family f) { return (f == FAM_FOREST12x6 || f == FAM_FOREST14x7) ? 2 : (family_chain_len(f) ? 1 : 0); }

struct LaunchModel {
    Family fam;
    int n;
    GenericBlob blob;
    const void *static_params;  // host pointer to StaticParams<N> for static families
    const void *chain_params;   // static families: host array of StaticParams<L>, one per serial chain
};

struct CostArgs {
    double dt, w_qd, w_tau, tau0, alpha, tau_floor, f_max;
};

// launchers (kernels.cu). All return cudaError_t of the launch.
cudaError_t launch_rnea(const LaunchModel &m, long U, const double *q, const double *qd, const double *qdd, double *tau, cudaStream_t s);
cudaError_t launch_fk(const LaunchModel &m, const FrameArg &f, long U, const double *q, double *pos, double *rot, cudaStream_t s);
cudaError_t launch_jac(const LaunchModel &m, const FrameArg &f, long U, const double *q, double *J, cudaStream_t s);
cudaError_t launch_node_eval(const LaunchModel &m, const EeArgs &ee, double wsign, long U, const double *q, const double *qd,
                             const double *qdd, const double *W, const double *T, double h, const ZohArg &zoh, double *tau,
                             double *qnext, double *Tnext, bool jtw_only, cudaStream_t s);
cudaError_t launch_node_eval_jvp_dual(const LaunchModel &m, const EeArgs &ee, double wsign, long U, const double *q, const double *qd,
                                      const double *qdd, const double *W, double *dtau_dq, double *dtau_dqd, cudaStream_t s);
cudaError_t launch_node_eval_jvp(const LaunchModel &m, const EeArgs &ee, double wsign, long U, const double *q, const double *qd,
                                 const double *qdd, const double *W, double *dtau_dq, double *dtau_dqd, cudaStream_t s);
cudaError_t launch_aba(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, double *qdd, cudaStream_t s);
cudaError_t launch_step(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, const double *f,
                        double dt, const double *dt_u, double *qn, double *qdn, double *fn, cudaStream_t s, const double *theat = nullptr);
// coupled fatigue of a two-arm model (kernels_couple.cu): host-side description and the pre / post kernel
struct CoupleHost {
    bool on = false;
    double weight = 0.0;
    int ee_joint[2] = {0, 0};      // end-effector joint, local to its arm
    double ee_p[2][3] = {{0, 0, 0}, {0, 0, 0}};
};
cudaError_t launch_couple(const LaunchModel &m, const CoupleHost &ch, long cnt, long ld, const double *q, const double *f, const double *tau,
                          double *theat, long ld_t, int mode, double dt, const double *dt_u, double *jac, long UJ, cudaStream_t s);
cudaError_t launch_rollout(const LaunchModel &m, long B, int N, const double *q0, const double *qd0, const double *f0, const double *tau,
                           double dt, double *qt, double *qdt, double *ft, cudaStream_t s);
cudaError_t launch_step_jvp(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, const double *f,
                            double dt, const double *dt_u, double *qn, double *qdn, double *fn, double *jac, cudaStream_t s,
                            long cnt = -1, long UJ = 0);
cudaError_t launch_cost_residual(int n, long B, int N, const double *q, const double *qd, const double *f, const double *tau,
                                 const double *qn, const double *qdn, const double *fn, const CostArgs &c, double *out,
                                 cudaStream_t s);
cudaError_t launch_cost_residual_table(int n, long B, int N, const double *q, const double *qd, const double *f, const double *tau,
                                       const double *qn, const double *qdn, const double *fn, double w_qd, double w_tau, double f_max,
                                       const double *table, double *out, long ld_out, cudaStream_t s);
cudaError_t launch_gather_planes(const double *src, double *dst, const int *map, int nplanes, long U, long ld_src, cudaStream_t s);
// analytic Jacobian pipeline (kernels_jvp2.cu): static chain families, caller-provided workspace
bool jvp2_supported(const LaunchModel &m);
size_t jvp_ws_bytes_per_unit(const LaunchModel &m);  // forests run one chain at a time: the chain length sizes it
cudaError_t launch_step_jvp_ws(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, const double *f,
                               double dt, const double *dt_u, double *qn, double *qdn, double *fn, double *jac, double *ws,
                               size_t ws_bytes, cudaStream_t s, long cnt = -1, long UJ = 0, const double *theat = nullptr, long UT = 0);
cudaError_t launch_rnea_derivs(const LaunchModel &m, long U, const double *q, const double *qd, const double *qdd, double *Dq, double *Dv,
                               double *M, cudaStream_t s);
cudaError_t launch_fd_derivs(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, double *A, double *B,
                             double *C, cudaStream_t s);
// fused reference-mode OCP node rows (kernels_rows.cu)
struct RowsHost {
    int narm = 1, N = 0;
    long B = 0;
    int ee_joint[2] = {0, 0};  // end-effector joint: global index, -1 = world-fixed frame
    double ee_p[2][3] = {{0, 0, 0}, {0, 0, 0}}, ee_R[2][9] = {{1, 0, 0, 0, 1, 0, 0, 0, 1}, {1, 0, 0, 0, 1, 0, 0, 0, 1}};
    double wsign = -1.0, fdes[3] = {0, 0, 0}, dist2_ref = 0.0, mu = 0.0, p_ref[3] = {0, 0, 0}, w_box = 0.0, w_qd = 0.0, w_F = 0.0, h = 0.0;
};
cudaError_t launch_ocp_rows(const LaunchModel &m, const RowsHost &h, const double *q, const double *qd, const double *F, const double *T,
                            const double *q_last, const double *T_last, const double *rel_pos0, const double *rel_ori0, double *rows,
                            double *cost, double *dtau_dF, double *dT_dtau, double *kin_jac, cudaStream_t s);
// analytic Jacobian pipeline for run-time trees (kernels_tree.cu): n <= 40; npat = size of the ancestor pattern
bool tree_jvp_supported(const LaunchModel &m);
size_t tree_jvp_workspace_bytes(int n, int npat, long U);
cudaError_t launch_step_jvp_tree(const LaunchModel &m, int npat, long U, long cnt, const double *q, const double *qd, const double *tau,
                                 const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn, double *jac, long UJ,
                                 double *ws, size_t ws_bytes, cudaStream_t s);
// Vector-Jacobian product of the RK4 step (reverse mode): the adjoint lambda = (lq, lqd, lf) and the addend (aq, aqd, af) of g_x
// (both NULL = 0) come in, g_x = lambda^T d x+/d x + addend, g_tau and g_dt go out.  Every plane group has its own stride, so the
// rollout adjoint can read a trajectory slice (stride N B) and write an O(B) buffer in one call.
struct VjpArgs {
    const double *lq = nullptr, *lqd = nullptr, *lf = nullptr;
    long ldl = 0;
    const double *aq = nullptr, *aqd = nullptr, *af = nullptr;
    long lda = 0;
    double *gq = nullptr, *gqd = nullptr, *gf = nullptr;
    long ldg = 0;
    double *gtau = nullptr;
    long ldgt = 0;
    double *gdt = nullptr;  // [units] or NULL
    // the same planes from joint j0 on (forests: one chain per launch)
    __host__ VjpArgs rows(int j0) const
    {
        auto sh = [](auto *p, long ld, int j) { return p ? p + (size_t)j * ld : p; };
        VjpArgs r = *this;
        r.lq = sh(lq, ldl, j0); r.lqd = sh(lqd, ldl, j0); r.lf = sh(lf, ldl, j0);
        r.aq = sh(aq, lda, j0); r.aqd = sh(aqd, lda, j0); r.af = sh(af, lda, j0);
        r.gq = sh(gq, ldg, j0); r.gqd = sh(gqd, ldg, j0); r.gf = sh(gf, ldg, j0);
        r.gtau = sh(gtau, ldgt, j0);
        return r;
    }
};
// static families (kernels_jvp2.cu): K1 + K2 of the Jacobian pipeline, then the reverse sweep; caller workspace as for the JVP
cudaError_t launch_step_vjp_ws(const LaunchModel &m, long U, long cnt, const double *q, const double *qd, const double *tau, const double *f,
                               double dt, const double *dt_u, const VjpArgs &a, double *qn, double *qdn, double *fn, double *ws,
                               size_t ws_bytes, cudaStream_t s);
// run-time trees with n <= 40 (kernels_tree.cu): T1, T2, the factor with L^-1, then the reverse sweep
cudaError_t launch_step_vjp_tree(const LaunchModel &m, int npat, long U, long cnt, const double *q, const double *qd, const double *tau,
                                 const double *f, double dt, const double *dt_u, const VjpArgs &a, double *qn, double *qdn, double *fn,
                                 double *ws, size_t ws_bytes, cudaStream_t s);
// run-time models with n > 40 (kernels_jvp.cu): one dual-number sweep per input direction, contracted with lambda
cudaError_t launch_step_vjp_dual(const LaunchModel &m, long U, long cnt, const double *q, const double *qd, const double *tau, const double *f,
                                 double dt, const double *dt_u, const VjpArgs &a, double *qn, double *qdn, double *fn, cudaStream_t s);
// second derivatives of the RK4 step (kernels_hess.cu): hyper-dual sweeps, every family, no workspace; HessArgs holds the adjoint,
// the HVP direction and the outputs, all [n][U] planes (vdt, hdt: [U]), NULL inputs = 0
struct HessArgs {
    const double *lq = nullptr, *lqd = nullptr, *lf = nullptr;
    const double *vq = nullptr, *vqd = nullptr, *vtau = nullptr, *vf = nullptr, *vdt = nullptr;
    double *H = nullptr;  // [4n+1][4n+1][U]
    double *hq = nullptr, *hqd = nullptr, *htau = nullptr, *hf = nullptr, *hdt = nullptr;
    double *jq = nullptr, *jqd = nullptr, *jf = nullptr;  // J v, all or none
};
cudaError_t launch_step_hess(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, const double *f,
                             double dt, const double *dt_u, const HessArgs &h, cudaStream_t s);
cudaError_t launch_step_hvp(const LaunchModel &m, long U, const double *q, const double *qd, const double *tau, const double *f,
                            double dt, const double *dt_u, const HessArgs &h, cudaStream_t s);
// Riccati solve of the multiple-shooting LQ subproblem (kernels_riccati.cu): one warp per scenario, n <= 16.  Every pointer is a
// device plane set as in include/mpcf.h (mpcf_riccati_batch); NULL optional inputs are zero.  ws: K_k and k_k of the chunk's
// scenarios, riccati_ws_bytes_per_scenario(n, N) each, scenario b0 + i at offset i.
struct RiccatiArgs {
    int n = 0, N = 0;
    long B = 0;
    const double *jac = nullptr, *H = nullptr, *wx = nullptr, *wu = nullptr, *gx = nullptr, *gu = nullptr, *d = nullptr;
    const double *HN = nullptr, *wN = nullptr, *gN = nullptr, *dx0 = nullptr;
    double *dx = nullptr, *du = nullptr, *lam = nullptr, *ws = nullptr;
};
int riccati_warps_per_cta(int n);  // scenarios per CTA: chunk sizes are multiples of it
size_t riccati_ws_bytes_per_scenario(int n, int N);
cudaError_t launch_riccati(const RiccatiArgs &a, long b0, long cnt, cudaStream_t s);
// mpcf_riccati_gains_batch: every scenario in one launch, the gains written to the planes a.ws = K [n][3n+1][N B] (dx, du, lam optional)
cudaError_t launch_riccati_gains(const RiccatiArgs &a, cudaStream_t s);
// iLQR rollouts (kernels_ilqr.cu): the tracking cost of include/mpcf.h (mpcf_track_cost; NULL pointers = 0 or absent) and the
// arguments of both passes.  Every [.][N B] plane has units k B + b, x / xbar are [3n][(N+1) B], x0 [3n][B].
constexpr int kIlqrMaxAlphas = 16;
struct TrackCost {
    const double *x_ref = nullptr, *tau_ref = nullptr, *wx = nullptr, *wu = nullptr, *wN = nullptr, *bound = nullptr;
    double rho_tau = 0.0, f_max = 0.0, rho_f = 0.0;
};
struct IlqrArgs {
    int N = 0;
    long B = 0;
    double dt = 0.0;
    TrackCost cost;
    const double *x0 = nullptr, *xbar = nullptr, *taubar = nullptr, *K = nullptr;  // K [n][3n+1][N B] or NULL (open loop)
    double *J = nullptr;                                                            // [na][B] (costs) or [B] (accept)
    int na = 0;                                                                     // costs pass: the step lengths
    double alphas[kIlqrMaxAlphas] = {};
    const double *alpha = nullptr;                                                  // accept pass: alpha [B]
    double *x = nullptr, *tau = nullptr;
    double *gx = nullptr, *gu = nullptr, *wxo = nullptr, *wuo = nullptr, *gN = nullptr, *wNo = nullptr;  // all or none
};
cudaError_t launch_ilqr_costs(const LaunchModel &m, const IlqrArgs &a, cudaStream_t s);
cudaError_t launch_feedback_rollout(const LaunchModel &m, const IlqrArgs &a, cudaStream_t s);
void jvp_profile_enable(bool on);
int jvp_profile_read(double *ms3, long *launches);
cudaError_t launch_fp64_probe(long iters, int blocks, double *out, cudaStream_t s);
long launch_count();

}  // namespace mpcf
