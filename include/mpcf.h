/*
 * mpcf.h — C-ABI of the B200-native batched dynamics + fatigue evaluator (libmpcf.so).
 *
 * Drop-in boundary for the hot path of ADVRHumanoids/mpc_fatigue.  The reference exposes three
 * generator functions through pybind11 (bindings/python/pynocchio_casadi.cpp:11-16) that return
 * serialized CasADi Functions traced from Pinocchio (src/casadi_pinocchio_bridge.hpp:57,87,119).
 * This library replaces what those Functions *evaluate*, batched over U independent
 * (scenario, shooting-node) units on one GPU:
 *
 *   mpcf_rnea_batch               <- Function "inverse_dynamics"(q,qdot,qddot)->tau   bridge.hpp:57-85
 *   mpcf_fk_batch                 <- Function "forward_kinematics"(q)->ee_pos,ee_rot   bridge.hpp:87-117
 *   mpcf_frame_jac_batch          <- Function "jacobian"(q)->J (LOCAL_WORLD_ALIGNED)   bridge.hpp:119-153
 *   mpcf_node_eval_ref_batch      <- the per-node composition the callers build around them:
 *                                    tau = ID -/+ J^T W, q+ = q + h qd, T+ = a T + (1-a) Rth P
 *                                    (python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:290-293,463;
 *                                     python/Centauro_script/mpc_principal.py:267-301)
 *   mpcf_aba_batch, mpcf_step_rk4_batch, mpcf_step_rk4_jvp_batch, mpcf_cost_residual_batch
 *                                 <- north-star additions (forward dynamics, RK4 over (q,qd,f) with
 *                                    the fatigue compartment ODE, forward-mode Jacobians, per-scenario
 *                                    cost/residual reduction); no reference code exists for these.
 *   mpcf_model_create_from_urdf   <- urdf::parseURDF + pinocchio::urdf::buildModel     bridge.hpp:60-63
 *   mpcf_frame_id                 <- model.getFrameId(body_name)                       bridge.hpp:103
 *
 * Conventions
 *   - every batch array is a raw DEVICE pointer to fp64 data in SoA layout `[component][U]`
 *     (component-major planes, U contiguous); the library allocates nothing per call;
 *   - kernels are enqueued on `stream` (a cudaStream_t passed as void*); no hidden synchronisation;
 *   - every function returns 0 on success or a negative MPCF_E* code and never throws across the ABI;
 *     mpcf_last_error() returns a thread-local message for the last failure;
 *   - a model handle is immutable after creation apart from the two explicit setters, is owned by the
 *     caller (create/destroy), and may be shared between streams and host threads.  The setters are the exception:
 *     the caller must not run them concurrently with launches on the same handle (they re-upload the constants after a
 *     cudaDeviceSynchronize, so work already queued finishes with the old values).  One handle per device.
 */
#ifndef MPCF_H
#define MPCF_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPCF_OK 0
#define MPCF_EINVAL (-1)     /* bad argument (null pointer, negative size, ...) */
#define MPCF_EPARSE (-2)     /* malformed URDF */
#define MPCF_EJOINT (-3)     /* unsupported joint type */
#define MPCF_EFRAME (-4)     /* unknown frame */
#define MPCF_ESINGULAR (-5)  /* zero joint-space inertia D_i without armature (forward dynamics) */
#define MPCF_ECUDA (-6)      /* CUDA runtime error */
#define MPCF_ELIMIT (-7)     /* model too large for this build (n > MPCF_MAX_DOF) */

#define MPCF_MAX_DOF 64
#define MPCF_MAX_EE 4

typedef struct mpcf_model mpcf_model;

typedef struct {
    double armature;    /* rotor inertia added to every joint (reference: 0; config C2: 1e-2) */
    double gravity[3];  /* default (0, 0, -9.81) */
    /* fatigue compartment ODE per joint: fdot = -lambda f + kappa (ctau tau^2 + cv qd^2).
       Defaults are the motor-winding thermal model of python/Libraries/Tmodel_library.py:9-32:
       lambda = 1/tau_th, kappa = R_th/tau_th, ctau = Ra/ktau^2 (ktau = 40), cv = 1/Rh. */
    double lambda, kappa, ctau, cv;
} mpcf_opts;

/* synthetic model kinds */
#define MPCF_SYNTH_CHAIN 0      /* serial revolute chain of ndof joints */
#define MPCF_SYNTH_HUMANOID 1   /* floating-base-like branched tree: 3 prismatic + 3 revolute root chain,
                                   1 torso joint, 2 arms x 7, 4 legs x 4 (37 DOF when ndof = 37) */

#define MPCF_SYNTH_DUAL_ARM 2    /* two serial revolute arms of ndof/2 joints on a fixed torso (Centauro layout: 2 x 7) */

void mpcf_opts_default(mpcf_opts *opts);

int mpcf_model_create_from_urdf(const char *xml, size_t len, const mpcf_opts *opts, mpcf_model **out);
int mpcf_model_create_synthetic(int kind, int ndof, unsigned long long seed, const mpcf_opts *opts,
                                mpcf_model **out);
int mpcf_model_destroy(mpcf_model *model);
int mpcf_model_info(const mpcf_model *model, int *nq, int *nv, int *nbody, int *nframe);
int mpcf_frame_id(const mpcf_model *model, const char *name);          /* >= 0, or MPCF_EFRAME */
const char *mpcf_joint_name(const mpcf_model *model, int joint);       /* NULL if out of range */
const char *mpcf_frame_name(const mpcf_model *model, int frame);
/* Copy a model array to host memory (tests, input generation).  field is one of:
   "parent" "jtype" "fparent" "jcontinuous" (int32; jcontinuous[i] = 1 for URDF `continuous` joints, which this library
   parametrises by the plain angle, nq = nv = 1, where Pinocchio uses (cos, sin), nq = 2) | "Rp" "pp" "mass" "mc" "Io" "arm" "fat" "fR" "fp"
   "q_lo" "q_hi" "v_max" "tau_max" "grav" (fp64).  Returns bytes written or a negative code. */
long mpcf_model_export(const mpcf_model *model, const char *field, void *out, size_t cap_bytes);
int mpcf_model_set_armature(mpcf_model *model, const double *arm /* [n] host */);
int mpcf_model_set_fatigue(mpcf_model *model, const double *rows /* [n][4] host: lambda kappa ctau cv */);
/* Coupled fatigue of a two-arm model carrying one box (config C3 "dual-arm with coupled fatigue states"; builder-defined, the
   reference only has the box equilibrium F_L,z + F_R,z = m g, python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:197,272-274).  Zero-order
   hold over the step: arm c carries the share s_c = Phi_other / (Phi_0 + Phi_1) of the box weight (Phi_c = sum of the arm's
   fatigue states at the start of the step), and its windings heat with theat_i = tau_i + s_c [J_ee,c(q)^T (0,0,weight,0,0,0)]_i
   while the dynamics keep tau.  mpcf_step_rk4_batch and the three analytic mpcf_step_rk4_jvp*_batch entries then evaluate the
   coupled step and its Jacobian (d f+/d f becomes a dense cross-arm block, d f+/d q gains the load term).  Two-arm families
   only (forest12x6, forest14x7); ee_frame[c] must be carried by arm c.  NULL removes the coupling. */
typedef struct {
    int ee_frame[2];
    double weight; /* m g of the box, e.g. 30 * 9.81 (Box_Pilz_6DOF2.py:197) */
} mpcf_coupling;
int mpcf_model_set_coupling(mpcf_model *model, const mpcf_coupling *coupling);
/* name of the kernel family a model dispatches to: "chain3", "chain6", "chain7", "forest12x6", "forest14x7" (compile-time
 * topologies: serial revolute chains and forests of two of them) or "generic16" / "generic64" (run-time topology) */
const char *mpcf_model_kernel_family(const mpcf_model *model);

/* tau[n][U] = RNEA(q, qd, qdd); qdd may be NULL (= 0, as every reference caller passes) */
int mpcf_rnea_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *qdd,
                    double *tau, void *stream);
/* pos[3][U], rot[9][U] (row-major element planes) of frame `frame` */
int mpcf_fk_batch(const mpcf_model *model, int frame, long U, const double *q, double *pos, double *rot,
                  void *stream);
/* J[6*n][U], plane index r*n + i, rows 0-2 linear / 3-5 angular, LOCAL_WORLD_ALIGNED */
int mpcf_frame_jac_batch(const mpcf_model *model, int frame, long U, const double *q, double *J, void *stream);
/* out[n][U] = J_frame(q)^T W, W[6][U]  (the fused form every caller actually uses) */
int mpcf_frame_jac_t_wrench_batch(const mpcf_model *model, int frame, long U, const double *q,
                                  const double *W, double *out, void *stream);
/* Reference-mode node evaluation (one launch):
     tau   = RNEA(q, qd, qdd) + wsign * sum_e J_e^T W_e      W[6*nee][U]
     qnext = q + h qd                                        (optional, may be NULL)
     Tnext = exact zero-order-hold fatigue/thermal map       (optional; needs T)            */
int mpcf_node_eval_ref_batch(const mpcf_model *model, int nee, const int *ee_frames, double wsign, long U,
                             const double *q, const double *qd, const double *qdd, const double *W,
                             const double *T, double h, double *tau, double *qnext, double *Tnext,
                             void *stream);
/* First derivatives of the reference-mode torque rows tau = RNEA(q, qd, qdd) + wsign * sum_e J_e^T W_e:
   dtau_dq, dtau_dqd as [n*n][U] (plane row*n + col).  d tau / d W_e = wsign * J_e^T: use mpcf_frame_jac_batch. */
int mpcf_node_eval_ref_jvp_batch(const mpcf_model *model, int nee, const int *ee_frames, double wsign, long U,
                                 const double *q, const double *qd, const double *qdd, const double *W,
                                 double *dtau_dq, double *dtau_dqd, void *stream);
/* qdd[n][U] = forward dynamics(q, qd, tau) */
int mpcf_aba_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                   double *qdd, void *stream);
/* One RK4 step of x = (q, qd, f) under xdot = (qd, FD(q,qd,tau), fatigue(f,tau,qd)), tau held.
   dt_u (per-unit step, [U]) overrides the scalar dt when non-NULL. */
int mpcf_step_rk4_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                        const double *f, double dt, const double *dt_u, double *qn, double *qdn, double *fn,
                        void *stream);
/* Sequential rollout (single shooting) of B scenarios over N steps: x_{k+1} = RK4(x_k, tau_k, dt), x_0 = (q0, qd0, f0)
   given as [n][B].  tau and the trajectory outputs qt/qdt/ft are [n][N*B] node-major (unit k*B + b); entry k of the
   outputs is x_{k+1}.  One thread per scenario keeps the state in registers across the steps. */
int mpcf_rollout_rk4_batch(const mpcf_model *model, long B, int N, const double *q0, const double *qd0,
                           const double *f0, const double *tau, double dt, double *qt, double *qdt, double *ft,
                           void *stream);
/* Same plus the dense forward-mode Jacobian jac[3n][4n+1][U]:
   rows (q+, qd+, f+), columns (q, qd, tau, f, dt).  qn/qdn/fn may be NULL.
   Compile-time families ("chain3", "chain6", "chain7", "forest12x6", "forest14x7") run the analytic pipeline (forward-dynamics
   derivatives per RK4 stage + a chain rule through the stages) staged through a device workspace that this entry takes from
   the device's stream-ordered memory pool (cudaMallocAsync / cudaFreeAsync on `stream`: no synchronisation, and the pool
   keeps the block between calls).  Run-time-topology models with n <= 40 (branched trees, prismatic joints: config C4) run the
   tree form of the same pipeline (ancestor-pattern derivatives, M = L^T D L, one CTA per unit for the chain rule); larger
   run-time-topology models run 3n + 1 dual-number sweeps. */
int mpcf_step_rk4_jvp_batch(const mpcf_model *model, long U, const double *q, const double *qd,
                            const double *tau, const double *f, double dt, const double *dt_u, double *qn,
                            double *qdn, double *fn, double *jac, void *stream);
/* Same with a caller-owned DEVICE workspace (one per stream): mpcf_step_rk4_jvp_workspace_bytes() returns the size to
   allocate (bounded: units are processed in chunks of 2^20), or 0 when the model has no workspace path (then `workspace`
   is ignored).  `workspace` must be 128-byte aligned (it is read with cp.async.bulk) and at least 32 units large; a
   misaligned or too small non-NULL workspace is MPCF_EINVAL.  workspace == NULL behaves like mpcf_step_rk4_jvp_batch. */
size_t mpcf_step_rk4_jvp_workspace_bytes(const mpcf_model *model, long U);
int mpcf_step_rk4_jvp_ws_batch(const mpcf_model *model, long U, const double *q, const double *qd,
                               const double *tau, const double *f, double dt, const double *dt_u, double *qn,
                               double *qdn, double *fn, double *jac, void *workspace, size_t workspace_bytes,
                               void *stream);
/* Unit-range form of the same call: evaluates `cnt` units whose input / state planes have stride `ld` (pass base pointers
   shifted to the first unit of the range) and writes the Jacobian into a buffer of plane stride `ld_jac` >= cnt,
   jac[3n][4n+1][ld_jac].  A caller sweeps a batch larger than the Jacobian memory it owns by reusing one chunk-sized
   Jacobian buffer (config C5).  Needs a caller workspace for the compile-time families. */
int mpcf_step_rk4_jvp_strided_batch(const mpcf_model *model, long cnt, long ld, const double *q, const double *qd,
                                    const double *tau, const double *f, double dt, const double *dt_u, double *qn,
                                    double *qdn, double *fn, double *jac, long ld_jac, void *workspace,
                                    size_t workspace_bytes, void *stream);
/* The same result by 3n + 1 dual-number sweeps of the RK4 step for EVERY family: an independent cross-check of the analytic
   pipeline (results agree to rounding; ~15x slower on the compile-time families). */
int mpcf_step_rk4_jvp_dual_batch(const mpcf_model *model, long U, const double *q, const double *qd,
                                 const double *tau, const double *f, double dt, const double *dt_u, double *qn,
                                 double *qdn, double *fn, double *jac, void *stream);
/* Reverse mode.  Vector-Jacobian product of one RK4 step (the step and families of mpcf_step_rk4_jvp_batch): with
   J = d(q+, qd+, f+)/d(q, qd, tau, f, h) and the adjoint lambda = (lq, lqd, lf), [n][U] each (any may be NULL = 0):
     gq, gqd, gtau, gf [n][U] = lambda^T J (blocks q, qd, tau, f);  gdt [U] = lambda^T dx+/dh (optional, NULL to skip).
   qn/qdn/fn: the step itself, all or none.  workspace: as for mpcf_step_rk4_jvp_ws_batch (size from
   mpcf_step_rk4_jvp_workspace_bytes, 128-byte aligned; NULL = stream-ordered pool).  Coupled models: MPCF_EINVAL.
   Compile-time families run the Jacobian pipeline's stage and derivative kernels and then one reverse sweep per unit that
   contracts the stored stage matrices with one vector (no dense Jacobian); run-time trees with n <= 40 the same with the tree
   kernels; larger run-time models 3n + 1 dual-number sweeps contracted with lambda.  dt = 0 is allowed (nothing divides by h). */
int mpcf_step_rk4_vjp_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                            const double *f, double dt, const double *dt_u, const double *lq, const double *lqd,
                            const double *lf, double *gq, double *gqd, double *gtau, double *gf, double *gdt,
                            double *qn, double *qdn, double *fn, void *workspace, size_t workspace_bytes, void *stream);
/* Adjoint of mpcf_rollout_rk4_batch.  Loss L(x_1..x_N); gqt/gqdt/gft [n][N*B] = dL/d(trajectory entry k) in the rollout's
   node-major layout (entry k = x_{k+1}; any may be NULL = 0); qt/qdt/ft = the trajectory that mpcf_rollout_rk4_batch
   returned for (q0, qd0, f0, tau, dt).  Outputs: gtau [n][N*B] = dL/dtau, gq0/gqd0/gf0 [n][B] = dL/dx_0.
   Workspace: mpcf_step_rk4_jvp_workspace_bytes(model, B) or NULL.  Coupled models: MPCF_EINVAL.  One step VJP per node,
   k = N-1 .. 0, in stream order; besides the workspace it takes 4 n B doubles of stream-ordered scratch (nothing of size N B). */
int mpcf_rollout_rk4_vjp_batch(const mpcf_model *model, long B, int N, const double *q0, const double *qd0,
                               const double *f0, const double *tau, double dt, const double *qt, const double *qdt,
                               const double *ft, const double *gqt, const double *gqdt, const double *gft, double *gtau,
                               double *gq0, double *gqd0, double *gf0, void *workspace, size_t workspace_bytes, void *stream);
/* Second order.  With z = (q, qd, tau, f, dt) (P = 4n + 1 components) and the adjoint lambda = (lq, lqd, lf) as for
   mpcf_step_rk4_vjp_batch (any may be NULL = 0):
   H[4n+1][4n+1][U] (plane r*(4n+1)+c, both triangles written) = d2(lambda^T x+)/dz dz, z = (q, qd, tau, f, dt).
   The two mirrored planes hold the same double.  One hyper-dual sweep per pair of the 3n + 1 directions (q, qd, tau, dt); the f rows
   and columns are closed form (zero except H[f_i][dt] = lf_i Lambda_i amp'(Lambda_i dt)).  No workspace.  dt_u: per-unit step or NULL.
   Every kernel family; coupled models: MPCF_EINVAL.  A singular model gives NaN. */
int mpcf_step_rk4_hess_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                             const double *f, double dt, const double *dt_u, const double *lq, const double *lqd,
                             const double *lf, double *H, void *stream);
/* Hessian-vector product of the same H with v = (vq, vqd, vtau, vf [n][U], vdt [U]; any may be NULL = 0):
   hq, hqd, htau, hf [n][U], hdt [U] (optional) = H v;  jq, jqd, jf [n][U] = J v (all or none), J = d(q+, qd+, f+)/dz.
   One hyper-dual sweep per direction (3n + 1); no dense Hessian or Jacobian is formed.  Coupled models: MPCF_EINVAL. */
int mpcf_step_rk4_hvp_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                            const double *f, double dt, const double *dt_u, const double *lq, const double *lqd,
                            const double *lf, const double *vq, const double *vqd, const double *vtau, const double *vf,
                            const double *vdt, double *hq, double *hqd, double *htau, double *hf, double *hdt,
                            double *jq, double *jqd, double *jf, void *stream);
/* Riccati solve of the multiple-shooting linear-quadratic subproblem of B scenarios over N nodes (units u = k*B + b), with the state
   x = (q, qd, f) (3n components, the row order of the step Jacobian) and the input u = tau (n components):
     minimise  sum_{k<N} 1/2 z_k^T W_k z_k + g_k^T z_k + 1/2 dx_N^T W_N dx_N + g_N^T dx_N,   z_k = (dx_k, du_k)
     s.t.      dx_0 = dx0,   dx_{k+1} = A_k dx_k + B_k du_k + d_k.
   A_k = the q, qd and f columns of jac[3n][4n+1][N*B] (mpcf_step_rk4_jvp_batch: columns 0..2n and 3n..4n), B_k = its tau columns
   2n..3n; the dt column is not read.  W_k = the (x, tau) rows and columns of H[4n+1][4n+1][N*B] in the layout of
   mpcf_step_rk4_hess_batch (its output can be passed as is; the upper triangle in the order (tau, q, qd, f) is read, so H must be
   symmetric) + diag(wx [3n][N*B], wu [n][N*B]) (e.g. interior-point barrier diagonals).  W_N = HN [3n*3n][B] (plane r*3n + c,
   symmetric) + diag(wN [3n][B]).  g_k = (gx [3n][N*B], gu [n][N*B]), g_N [3n][B], the defect d_k = x+_k - x_{k+1} [3n][N*B] (the sign
   of mpcf_cost_residual_batch) and dx0 [3n][B]: every one of H, wx, wu, gx, gu, d, HN, wN, gN, dx0 may be NULL (= 0).
   Outputs, node-major: dx [3n][(N+1)*B], du [n][N*B] and, when lam is not NULL, the costates lam [3n][(N+1)*B]:
     lambda_N = W_N dx_N + g_N,   lambda_k = Q_k dx_k + S_k^T du_k + gx_k + A_k^T lambda_{k+1}
   (W_k = [Q_k S_k^T; S_k R_k]), the multipliers of the dynamics in
     L = obj - lambda_0^T (dx_0 - dx0) - sum_k lambda_{k+1}^T (dx_{k+1} - A_k dx_k - B_k du_k - d_k),
   i.e. the adjoint that the next mpcf_step_rk4_hess_batch call takes.  No regularisation: a scenario whose R + B^T P B is not
   positive definite at some node gets NaN in all its outputs; the other scenarios are unaffected.  Models with n <= 16 (every
   family but generic64, coupled models included: only jac is read); n > 16 is MPCF_ELIMIT.  B = 0 launches nothing.
   Workspace (one per stream): mpcf_riccati_workspace_bytes() gives the size for B scenarios (bounded: scenarios run in chunks);
   it must be 128-byte aligned and hold at least one chunk of one CTA's scenarios (a smaller size gives more, smaller chunks);
   NULL takes it from the stream-ordered pool.  One warp per scenario, the nodes serially. */
size_t mpcf_riccati_workspace_bytes(const mpcf_model *model, long B, int N);
int mpcf_riccati_batch(const mpcf_model *model, long B, int N, const double *jac, const double *H, const double *wx, const double *wu,
                       const double *gx, const double *gu, const double *d, const double *HN, const double *wN, const double *gN,
                       const double *dx0, double *dx, double *du, double *lam, void *workspace, size_t workspace_bytes, void *stream);
/* The same backward pass with the feedback gains as an output and no workspace: K [n][3n+1][N*B], plane t*(3n+1) + j, unit k*B + b,
   holds row t of [K_k | k_k] (columns j < 3n: K_k, column 3n: the feedforward k_k), so that du_k = K_k dx_k + k_k in the solve.
   Inputs as for mpcf_riccati_batch.  dx and du are optional, both or neither: when both are NULL only the backward pass runs (all
   that iLQR needs); lam needs dx.  When dx is given, dx, du and lam are bit-identical to mpcf_riccati_batch's.  A scenario whose
   R + B^T P B is not positive definite at some node gets NaN in all its K planes (and in dx, du, lam); the others are unaffected.
   n > 16 is MPCF_ELIMIT. */
int mpcf_riccati_gains_batch(const mpcf_model *model, long B, int N, const double *jac, const double *H, const double *wx,
                             const double *wu, const double *gx, const double *gu, const double *d, const double *HN, const double *wN,
                             const double *gN, const double *dx0, double *K, double *dx, double *du, double *lam, void *stream);

/* iLQR on the device (DESIGN.md §4g).  State x = (q, qd, f) [3n], input u = tau [n]; units node-major u = k*B + b; trajectories
   x / xbar [3n][(N+1)*B] (nodes 0..N), torques [n][N*B], x0 [3n][B].  The tracking cost of one scenario, with every pointer of
   mpcf_track_cost a DEVICE array or NULL (= 0, or absent for bound_table):
     J = sum_{k<N} [ 1/2 sum_i wx_i (x_ki - x_ref_ki)^2 + 1/2 sum_j wu_j (tau_kj - tau_ref_kj)^2
                     + 1/2 rho_tau sum_j ((lb_kj - tau_kj)+^2 + (tau_kj - ub_kj)+^2) + 1/2 rho_f sum_j (f_kj - f_max)+^2 ]
         + 1/2 sum_i wN_i (x_Ni - x_ref_Ni)^2 + 1/2 rho_f sum_j (f_Nj - f_max)+^2
   x_ref [3n][(N+1)*B], tau_ref [n][N*B], wx, wN [3n], wu [n], bound_table [N][n][2] = (lb, ub) (the table of
   mpcf_cost_residual_table_batch).  A NaN in any state, torque or reference makes J NaN.  Under the feedback law
     tau_k = taubar_k + alpha k_k + K_k (x_k - xbar_k),   x_{k+1} = RK4(x_k, tau_k, dt),   x_0 = x0,
   with K the gains of mpcf_riccati_gains_batch.  alpha == 0 reads neither K nor xbar: tau_k = taubar_k exactly, so a rejected step
   reproduces the trajectory it started from bit for bit, even where the gains are NaN.  Every kernel family; coupled models:
   MPCF_EINVAL. */
typedef struct {
    const double *x_ref, *tau_ref, *wx, *wu, *wN, *bound_table;
    double rho_tau, f_max, rho_f;
} mpcf_track_cost;
/* Line-search pass: J [na][B] = the cost of the closed-loop rollout for each of the na step lengths alphas[0..na) (host array,
   1 <= na <= 16, finite, >= 0), one thread per (step length, scenario).  K == NULL: the open-loop cost of taubar for every entry
   (xbar may then be NULL).  No trajectory is stored.  J of step length a has the same bits as mpcf_feedback_rollout_batch's J with
   alpha = a. */
int mpcf_ilqr_costs_batch(const mpcf_model *model, const mpcf_track_cost *cost, long B, int N, const double *x0, const double *xbar,
                          const double *taubar, const double *K, const double *alphas, int na, double dt, double *J, void *stream);
/* Accept pass: the closed-loop rollout with the per-scenario step length alpha [B] (DEVICE); K == NULL (alpha and xbar may then be
   NULL) rolls taubar out open loop from x0, bit-identical to mpcf_rollout_rk4_batch.  Writes x [3n][(N+1)*B] (node 0 = x0),
   tau [n][N*B] and J [B].  Optionally (all or none) the Riccati inputs of the cost at the new trajectory, to pass straight to
   mpcf_riccati_gains_batch: the gradient gx [3n][N*B], gu [n][N*B], gN [3n][B] and the Gauss-Newton curvature wx_out [3n][N*B] =
   wx + rho_f [f > f_max] on the f rows, wu_out [n][N*B] = wu + rho_tau [tau outside (lb, ub)], wN_out [3n][B]. */
int mpcf_feedback_rollout_batch(const mpcf_model *model, const mpcf_track_cost *cost, long B, int N, const double *x0,
                                const double *xbar, const double *taubar, const double *K, const double *alpha, double dt, double *x,
                                double *tau, double *J, double *gx, double *gu, double *wx_out, double *wu_out, double *gN,
                                double *wN_out, void *stream);

/* Forward-dynamics derivatives at (q, qd, tau): A = d qdd/d q, B = d qdd/d qd, C = M^-1 = d qdd/d tau,
   each [n*n][U] with plane index row*n + col. */
int mpcf_fd_derivs_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *tau,
                         double *A, double *B, double *C, void *stream);

/* Inverse-dynamics derivatives at (q, qd, qdd) — what an NLP solver needs for the reference-mode torque rows
   tau = ID(q, qd, 0) -/+ J^T W (python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:134): dtau_dq = d ID/d q,
   dtau_dqd = d ID/d qd, M = d ID/d qdd (joint-space inertia incl. armature), each [n*n][U], plane row*n + col.
   qdd may be NULL (= 0). */
int mpcf_rnea_derivs_batch(const mpcf_model *model, long U, const double *q, const double *qd, const double *qdd,
                           double *dtau_dq, double *dtau_dqd, double *M, void *stream);

/* Per-scenario reduction over the N nodes of each of B scenarios (unit index u = k*B + b):
     cost[b]      = sum_k  w_qd |qd_k|^2 + w_tau |tau_k|^2
     resid[0][b]  = max_k |x+_k - x_{k+1}|_inf          multiple-shooting defect (k < N-1)
     resid[1][b]  = max_k max_i (|tau_ki| - bound_k)+   F0 decaying torque bound
                    bound_k = max(tau0 exp(-alpha k dt), tau_floor)
                                                        (python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:136-148)
     resid[2][b]  = max_k max_i (f+_ki - f_max)+        fatigue / temperature bound
   out[4][B] = (cost, resid0, resid1, resid2): written directly into the caller's (all-gather send) buffer.
   A row is NaN when any entry it reads is NaN (a failed step's NaN is never dropped from a maximum). */
int mpcf_cost_residual_batch(const mpcf_model *model, long B, int N, const double *q, const double *qd,
                             const double *f, const double *tau, const double *qn, const double *qdn,
                             const double *fn, double dt, double w_qd, double w_tau, double tau0,
                             double alpha, double tau_floor, double f_max, double *out, void *stream);

/* Same reduction with the torque limits given as a DEVICE table bound_table[N][n][2] = (lb, ub) per node and joint, which
   covers the reference's three torque-limit mechanisms: F0 decaying bound (force_optimization_pilz_6DOF.py:136-148), F2
   stepwise bounds over segments of the horizon (both_robots_torque_limited_2_pilz.py:129-147, Box_Pilz_6DOF2.py:303-433) and
   F3 joint switch-off |tau_i| <= C_i after the first third for the joints selected by S (Centauro_dynamics.py:327-348).
     resid[1][b] = max_k max_i max(lb_ki - tau_ki, tau_ki - ub_ki, 0)
   out has row stride ld_out >= B (0 = B): a scenario chunk can write its columns of a larger [4][B_total] send buffer.
   2 n N doubles must fit 200 KB of shared memory (MPCF_ELIMIT otherwise).  As above, a row is NaN when any entry it reads
   (the bound table's included) is NaN. */
int mpcf_cost_residual_table_batch(const mpcf_model *model, long B, int N, const double *q, const double *qd,
                                   const double *f, const double *tau, const double *qn, const double *qdn,
                                   const double *fn, double w_qd, double w_tau, const double *bound_table,
                                   double f_max, double *out, long ld_out, void *stream);

/* Fused reference-mode OCP node rows: every constraint row and the running cost the reference's scripts build per shooting
   node, one launch for B scenarios x N nodes (node-major units u = k*B + b).  The same kernel serves every family; the
   families differ only in how the arm count is set and which frames they accept:
     compile-time families: chain3/6/7 have one arm, forest12x6 / forest14x7 two (opts->ee_frame[1] is ignored on the
       one-arm chains); ee_frame[c] must be carried by arm c (MPCF_EFRAME otherwise, world-fixed frames included).
     run-time trees (generic16 / generic64: branched trees, prismatic and continuous joints, up to 64 DOF): one arm when
       opts->ee_frame[1] < 0, two otherwise; the frames may sit anywhere in the tree.  On a tree both end-effectors may share
       ancestors (e.g. a torso joint): tau = ID(q,qd,0) + wsign (J_L^T [F_L;0] + J_R^T [F_R;0]) sums both terms there, and
       dtau_dF is non-zero in both arm blocks on those joints (on the forests the cross-arm blocks are structural zeros).  A
       prismatic joint contributes z_j to J_lin and nothing to the rotation.  A frame whose parent is the world (fparent -1)
       has a constant pose and a zero Jacobian.
   A frame index out of range is MPCF_EFRAME.  mpcf_ocp_rows_count_arms gives the row count for either arm count.
   One arm (python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:130-177), 3 + 3n rows:
     [0,3) ee_pos - p_ref | n: tau = ID(q,qd,0) + wsign J^T [F;0] | n: q + h qd - q_next | n: T+ - T_next (thermal ZOH)
     cost = w_F F.F + w_qd qd.qd                                                   (w_F = -1: the script's -F^T F)
   Two arms (Box_Pilz_6DOF2.py:244-293,454-475, mpc_principal.py:229-327,
   RepeatedMPCwithThermal_confriction.py:251-273), 26 + 3n rows:
     [0,3) F_L + F_R - fdes | [3,6) (pL-pR) x F_L + (pR-pL) x F_R | [6] |pL-pR|^2 - dist2_ref |
     [7,10) R_L^T (pR-pL) - (the same at the previous node | rel_pos0 at node 0) | [10,13) e(R_L R_R^T) - rel_ori0 |
     [13,23) friction cones A1 (-R_L^T F_L), A2 (-R_R^T F_R) (<= 0) | [23,26) (pL+pR)/2 - p_ref | tau | q defect | T defect
     cost = w_box |p_box - p_ref|^2 + w_qd qd.qd + w_F (F_L.F_L + F_R.F_R)
   Arrays: q, qd [n][U]; F [3 arms][U]; T [n][U] or NULL (thermal rows = 0); q_last / T_last [n][B]: the trailing state the
   last node's defects compare with (NULL: zero defect there); rel_pos0 / rel_ori0 [3][B] (two arms; NULL = 0);
   rows [rows][U], cost [U].  Optional derivative outputs (NULL to skip): dtau_dF [n][3 arms][U] = wsign J_c,lin^T (arm c's
   block; J_c,lin = linear rows of the frame Jacobian of arm c's end-effector),
   dT_dtau [n][U] = d T+ / d tau (chain it with mpcf_node_eval_ref_jvp_batch for the thermal rows), kin_jac
   [26 | 3][n + 3 arms][U] = d (kinematic rows) / d (q, F) of the node's own variables (the relative-position row's block
   with respect to the previous node's q is minus the same block evaluated there). */
typedef struct {
    int ee_frame[2];
    double wsign;      /* -1: force exerted ON the robot (Pilz scripts), +1: force the robot exerts (Centauro scripts) */
    double fdes[3];    /* e.g. (0, 0, m g) */
    double dist2_ref, mu, p_ref[3], w_box, w_qd, w_F, h;
} mpcf_rows_opts;
/* rows of mpcf_ocp_rows_batch for a compile-time family (26 + 3n with two arms, 3 + 3n with one); MPCF_EINVAL on run-time trees */
int mpcf_ocp_rows_count(const mpcf_model *model);
/* (narm == 2 ? 26 : 3) + 3n for any family; MPCF_EINVAL when narm is not 1 or 2, or differs from a compile-time family's
   arm count.  Host only. */
int mpcf_ocp_rows_count_arms(const mpcf_model *model, int narm);
int mpcf_ocp_rows_batch(const mpcf_model *model, const mpcf_rows_opts *opts, long B, int N, const double *q,
                        const double *qd, const double *F, const double *T, const double *q_last, const double *T_last,
                        const double *rel_pos0, const double *rel_ori0, double *rows, double *cost, double *dtau_dF,
                        double *dT_dtau, double *kin_jac, void *stream);

/* FP64-pipe probe for the roofline denominator: every thread of `blocks` x 256 runs 8 independent DFMA
   chains for `iters` iterations and writes one double to out[blocks*256] (device).
   flops = blocks * 256 * iters * 16.  Time it with events on `stream`. */
int mpcf_probe_fp64(long iters, int blocks, double *out, void *stream);

/* Pitched copy of `height` rows of `width_bytes` between pinned host memory and the device, enqueued on
   `stream` (kind 1 = host->device, 2 = device->host).  Used by the host-facing pipeline to move the
   scenario-chunk slice of every SoA plane in one DMA. */
int mpcf_memcpy2d_async(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width_bytes,
                        size_t height, int kind, void *stream);

/* dst[k][u] = src[plane_map[k]][u] for k < nplanes, u < U (src planes have stride ld_src >= U; plane_map is a DEVICE int32
   array; src and dst 16-byte aligned): packs the planes a host consumer wants (states + the structurally non-zero Jacobian
   planes) into one contiguous device buffer, so that a scenario chunk goes back to the host in ONE copy.  Every plane_map
   entry must be a valid plane index of src: the entry cannot check a device array without a synchronising copy. */
int mpcf_gather_planes(const double *src, long ld_src, const int *plane_map, int nplanes, long U, double *dst,
                       void *stream);

/* Diagnostics: bracket each kernel of the workspace Jacobian pipeline with CUDA events on its launch stream.
   mpcf_profile_read synchronises and returns accumulated ms of (step_stages, stage_derivs, chain_rule) and the
   number of timed launches since the last read.  Off by default; single-threaded use only. */
int mpcf_profile_enable(int on);
int mpcf_profile_read(double *ms3, long *launches);

const char *mpcf_last_error(void);
/* number of kernel launches issued by this library in the calling process since load (bench.py) */
long mpcf_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
