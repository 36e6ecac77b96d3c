"""BatchEvaluator: the batched node evaluation that replaces the per-node CasADi calls of the reference
(python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:259-274 calls `Idyn(q=..,qdot=..,qddot=..)['tau']` once
per node; here one launch evaluates U = B*N nodes).

All tensors are torch CUDA float64 in the SoA layout of the C-ABI: `[component, U]`, contiguous.
PyTorch is only the owner of device memory and streams; every operation is a hand-written kernel in
libmpcf.so launched on `torch.cuda.current_stream()`.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _capi
from .model import Model


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class BatchEvaluator:
    def __init__(self, model: Model, device: torch.device | str | int | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError("mpc_fatigue_b200 needs a CUDA device (there is no CPU fallback)")
        self.model = model
        self.n = model.n
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("BatchEvaluator runs on CUDA devices only")

    # ---- argument checking ----
    def _in(self, t: torch.Tensor | None, rows: int, U: int, name: str, optional: bool = False):
        if t is None:
            if optional:
                return None
            raise ValueError("%s is required" % name)
        if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
            raise ValueError("%s must be a contiguous CUDA float64 tensor" % name)
        if t.device != self.device:
            raise ValueError("%s is on %s, evaluator is on %s" % (name, t.device, self.device))
        if tuple(t.shape) != (rows, U):
            raise ValueError("%s has shape %s, expected (%d, %d)" % (name, tuple(t.shape), rows, U))
        return C.c_void_p(t.data_ptr())

    def _out(self, t: torch.Tensor | None, rows, U: int, name: str) -> torch.Tensor:
        shape = tuple(rows) + (U,) if isinstance(rows, tuple) else (rows, U)
        if t is None:
            return torch.empty(shape, dtype=torch.float64, device=self.device)
        if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and tuple(t.shape) == shape and t.device == self.device):
            raise ValueError("output %s must be a contiguous CUDA float64 tensor of shape %s" % (name, shape))
        return t

    @staticmethod
    def _U(q: torch.Tensor) -> int:
        if q.dim() != 2:
            raise ValueError("expected [component, U] tensors")
        return q.shape[1]

    # ---- the reference's three Functions, batched ----
    def rnea(self, q, qd, qdd=None, out=None):
        """tau = inverse_dynamics(q, qdot, qddot)   (bridge.hpp:76-78); qdd=None means zeros."""
        U, n = self._U(q), self.n
        tau = self._out(out, n, U, "tau")
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_rnea_batch(self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"),
                                                  self._in(qdd, n, U, "qdd", True), C.c_void_p(tau.data_ptr()), _stream()))
        return tau

    def fk(self, frame: int, q, out_pos=None, out_rot=None):
        """ee_pos[3,U], ee_rot[9,U] (row-major) = forward_kinematics(q)   (bridge.hpp:106-111)."""
        U, n = self._U(q), self.n
        pos, rot = self._out(out_pos, 3, U, "pos"), self._out(out_rot, 9, U, "rot")
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_fk_batch(self.model.handle, int(frame), U, self._in(q, n, U, "q"),
                                                C.c_void_p(pos.data_ptr()), C.c_void_p(rot.data_ptr()), _stream()))
        return pos, rot

    def jacobian(self, frame: int, q, out=None):
        """J[6*n,U] (plane r*n+i) = jacobian(q), LOCAL_WORLD_ALIGNED   (bridge.hpp:141-146)."""
        U, n = self._U(q), self.n
        J = self._out(out, 6 * n, U, "J")
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_frame_jac_batch(self.model.handle, int(frame), U, self._in(q, n, U, "q"),
                                                       C.c_void_p(J.data_ptr()), _stream()))
        return J

    def jac_t_wrench(self, frame: int, q, W, out=None):
        """J(q)^T W without materialising J (what every caller does with the Jacobian)."""
        U, n = self._U(q), self.n
        o = self._out(out, n, U, "out")
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_frame_jac_t_wrench_batch(self.model.handle, int(frame), U, self._in(q, n, U, "q"),
                                                                self._in(W, 6, U, "W"), C.c_void_p(o.data_ptr()), _stream()))
        return o

    def node_eval_ref(self, ee_frames, wsign: float, q, qd, W=None, T=None, h: float = 0.0, qdd=None,
                      want_qnext=True, want_Tnext=True):
        """Reference-mode node: tau = RNEA + wsign*sum J^T W, qnext = q + h qd, Tnext = thermal ZOH."""
        U, n = self._U(q), self.n
        nee = len(ee_frames)
        fr = (C.c_int * max(nee, 1))(*[int(f) for f in ee_frames])
        tau = self._out(None, n, U, "tau")
        qn = self._out(None, n, U, "qnext") if want_qnext else None
        Tn = self._out(None, n, U, "Tnext") if (want_Tnext and T is not None) else None
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_node_eval_ref_batch(
                self.model.handle, nee, fr, float(wsign), U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"),
                self._in(qdd, n, U, "qdd", True), self._in(W, 6 * nee, U, "W", nee == 0), self._in(T, n, U, "T", True),
                float(h), p(tau), p(qn), p(Tn), _stream()))
        return tau, qn, Tn

    def node_eval_ref_jvp(self, ee_frames, wsign: float, q, qd, W=None, qdd=None):
        """d tau/d q, d tau/d qd ([n*n, U], plane row*n + col) of the reference-mode torque
        tau = RNEA(q, qd, qdd) + wsign * sum_e J_e^T W_e;  d tau/d W_e = wsign * J_e^T (see `jacobian`)."""
        U, n = self._U(q), self.n
        nee = len(ee_frames)
        fr = (C.c_int * max(nee, 1))(*[int(f) for f in ee_frames])
        Dq, Dv = self._out(None, n * n, U, "dtau_dq"), self._out(None, n * n, U, "dtau_dqd")
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_node_eval_ref_jvp_batch(
                self.model.handle, nee, fr, float(wsign), U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"),
                self._in(qdd, n, U, "qdd", True), self._in(W, 6 * nee, U, "W", nee == 0), C.c_void_p(Dq.data_ptr()),
                C.c_void_p(Dv.data_ptr()), _stream()))
        return Dq, Dv

    # ---- north-star additions ----
    def aba(self, q, qd, tau, out=None):
        U, n = self._U(q), self.n
        qdd = self._out(out, n, U, "qdd")
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_aba_batch(self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"),
                                                 self._in(tau, n, U, "tau"), C.c_void_p(qdd.data_ptr()), _stream()))
        return qdd

    def _dt(self, dt, U):
        if isinstance(dt, torch.Tensor):
            if not (dt.is_cuda and dt.dtype == torch.float64 and dt.is_contiguous() and tuple(dt.shape) == (U,)):
                raise ValueError("per-unit dt must be a contiguous CUDA float64 tensor of shape (U,)")
            return 0.0, C.c_void_p(dt.data_ptr())
        return float(dt), None

    def step_rk4(self, q, qd, tau, f, dt, out=None):
        """(q+, qd+, f+) = one RK4 step of (q, qd, f), tau held; dt scalar or per-unit tensor [U]."""
        U, n = self._U(q), self.n
        qn, qdn, fn = out if out is not None else (None, None, None)
        qn, qdn, fn = self._out(qn, n, U, "qn"), self._out(qdn, n, U, "qdn"), self._out(fn, n, U, "fn")
        dts, dtu = self._dt(dt, U)
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_step_rk4_batch(
                self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"), self._in(tau, n, U, "tau"),
                self._in(f, n, U, "f"), dts, dtu, C.c_void_p(qn.data_ptr()), C.c_void_p(qdn.data_ptr()),
                C.c_void_p(fn.data_ptr()), _stream()))
        return qn, qdn, fn

    def rollout_rk4(self, q0, qd0, f0, tau, N: int, dt: float):
        """Single-shooting rollout of B scenarios over N steps: x0 tensors are [n, B], tau is [n, N*B] node-major
        (unit k*B + b); returns (q, qd, f) trajectories [n, N*B] with entry k = x_{k+1}."""
        if q0.dim() != 2:
            raise ValueError("expected [n, B] initial states")
        n, B = self.n, q0.shape[1]
        U = B * int(N)
        qt, qdt, ft = (self._out(None, n, U, nm) for nm in ("qt", "qdt", "ft"))
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_rollout_rk4_batch(
                self.model.handle, B, int(N), self._in(q0, n, B, "q0"), self._in(qd0, n, B, "qd0"), self._in(f0, n, B, "f0"),
                self._in(tau, n, U, "tau"), float(dt), C.c_void_p(qt.data_ptr()), C.c_void_p(qdt.data_ptr()),
                C.c_void_p(ft.data_ptr()), _stream()))
        return qt, qdt, ft

    def fd_derivs(self, q, qd, tau):
        """A = d qdd/d q, B = d qdd/d qd, C = M^-1 as [n*n, U] planes (row*n + col)."""
        U, n = self._U(q), self.n
        A, B, Cm = (self._out(None, n * n, U, nm) for nm in "ABC")
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_fd_derivs_batch(self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"),
                                                       self._in(tau, n, U, "tau"), C.c_void_p(A.data_ptr()),
                                                       C.c_void_p(B.data_ptr()), C.c_void_p(Cm.data_ptr()), _stream()))
        return A, B, Cm

    def rnea_derivs(self, q, qd, qdd=None):
        """d tau/d q, d tau/d qd, M = d tau/d qdd of tau = inverse_dynamics(q, qd, qdd) as [n*n, U] planes (row*n + col):
        the Jacobian blocks of the reference-mode torque rows (force_optimization_pilz_6DOF.py:134)."""
        U, n = self._U(q), self.n
        Dq, Dv, M = (self._out(None, n * n, U, nm) for nm in ("dtau_dq", "dtau_dqd", "M"))
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_rnea_derivs_batch(self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"),
                                                         self._in(qdd, n, U, "qdd", True), C.c_void_p(Dq.data_ptr()),
                                                         C.c_void_p(Dv.data_ptr()), C.c_void_p(M.data_ptr()), _stream()))
        return Dq, Dv, M

    def _workspace(self, U: int):
        """Device workspace of the analytic Jacobian pipeline (cached; bounded by the library's chunking)."""
        need = int(_capi.lib.mpcf_step_rk4_jvp_workspace_bytes(self.model.handle, U))
        if need == 0:
            return None, 0
        ws = getattr(self, "_ws", None)
        if ws is None or ws.numel() * 8 < need:
            self._ws = ws = torch.empty(need // 8, dtype=torch.float64, device=self.device)
        return C.c_void_p(ws.data_ptr()), ws.numel() * 8

    def step_rk4_jvp(self, q, qd, tau, f, dt, out=None, jac=None, direct: bool = False):
        """Step plus dense forward-mode Jacobian jac[3n, 4n+1, U]: rows (q+,qd+,f+), cols (q,qd,tau,f,dt).
        Chain models use the analytic workspace pipeline (the evaluator keeps one workspace per instance, i.e. per stream
        of use); `direct=True` runs the 3n + 1 dual-number sweeps instead (cross-check)."""
        U, n = self._U(q), self.n
        qn, qdn, fn = out if out is not None else (None, None, None)
        qn, qdn, fn = self._out(qn, n, U, "qn"), self._out(qdn, n, U, "qdn"), self._out(fn, n, U, "fn")
        jac = self._out(jac, (3 * n, 4 * n + 1), U, "jac")
        dts, dtu = self._dt(dt, U)
        with torch.cuda.device(self.device):
            if direct:
                _capi.check(_capi.lib.mpcf_step_rk4_jvp_dual_batch(
                    self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"), self._in(tau, n, U, "tau"),
                    self._in(f, n, U, "f"), dts, dtu, C.c_void_p(qn.data_ptr()), C.c_void_p(qdn.data_ptr()),
                    C.c_void_p(fn.data_ptr()), C.c_void_p(jac.data_ptr()), _stream()))
                return qn, qdn, fn, jac
            ws, ws_bytes = self._workspace(U)
            _capi.check(_capi.lib.mpcf_step_rk4_jvp_ws_batch(
                self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"), self._in(tau, n, U, "tau"),
                self._in(f, n, U, "f"), dts, dtu, C.c_void_p(qn.data_ptr()), C.c_void_p(qdn.data_ptr()),
                C.c_void_p(fn.data_ptr()), C.c_void_p(jac.data_ptr()), ws, ws_bytes, _stream()))
        return qn, qdn, fn, jac

    def step_rk4_vjp(self, q, qd, tau, f, dt, lq=None, lqd=None, lf=None, want_dt=False):
        """Reverse mode of `step_rk4`: with the adjoint lambda = (lq, lqd, lf) ([n, U] each; None = 0) returns
        (gq, gqd, gtau, gf) = lambda^T d(q+, qd+, f+)/d(q, qd, tau, f), and gdt [U] = lambda^T d x+/d dt as a fifth element with
        want_dt=True.  dt is a scalar or a per-unit tensor [U], as in `step_rk4`.  No dense Jacobian is formed."""
        U, n = self._U(q), self.n
        g = [self._out(None, n, U, nm) for nm in ("gq", "gqd", "gtau", "gf")]
        gdt = self._out(None, 1, U, "gdt").view(U) if want_dt else None
        dts, dtu = self._dt(dt, U)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            ws, ws_bytes = self._workspace(U)
            _capi.check(_capi.lib.mpcf_step_rk4_vjp_batch(
                self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"), self._in(tau, n, U, "tau"),
                self._in(f, n, U, "f"), dts, dtu, self._in(lq, n, U, "lq", True), self._in(lqd, n, U, "lqd", True),
                self._in(lf, n, U, "lf", True), *[p(t) for t in g], p(gdt), None, None, None, ws, ws_bytes, _stream()))
        return (*g, gdt) if want_dt else tuple(g)

    def step_rk4_hess(self, q, qd, tau, f, dt, lq=None, lqd=None, lf=None):
        """Second derivatives of `step_rk4`: H [4n+1, 4n+1, U] = d2(lambda^T x+)/dz dz with z = (q, qd, tau, f, dt) and the adjoint
        lambda = (lq, lqd, lf) ([n, U] each; None = 0).  dt is a scalar or a per-unit tensor [U], as in `step_rk4`."""
        U, n = self._U(q), self.n
        P = 4 * n + 1
        H = self._out(None, (P, P), U, "H")
        dts, dtu = self._dt(dt, U)
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_step_rk4_hess_batch(
                self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"), self._in(tau, n, U, "tau"),
                self._in(f, n, U, "f"), dts, dtu, self._in(lq, n, U, "lq", True), self._in(lqd, n, U, "lqd", True),
                self._in(lf, n, U, "lf", True), C.c_void_p(H.data_ptr()), _stream()))
        return H

    def step_rk4_hvp(self, q, qd, tau, f, dt, lam, v, want_dt=False, want_jv=False):
        """Hessian-vector product of `step_rk4_hess` without forming H: lam = (lq, lqd, lf), v = (vq, vqd, vtau, vf, vdt) ([n, U] each,
        vdt [U]; None entries = 0).  Returns (hq, hqd, htau, hf) = H v, then hdt [U] with want_dt=True, then (jq, jqd, jf) = J v of the
        step Jacobian J = d(q+, qd+, f+)/dz with want_jv=True."""
        U, n = self._U(q), self.n
        lq, lqd, lf = lam
        vq, vqd, vtau, vf, vdt = v
        h = [self._out(None, n, U, nm) for nm in ("hq", "hqd", "htau", "hf")]
        hdt = self._out(None, 1, U, "hdt").view(U) if want_dt else None
        jv = [self._out(None, n, U, nm) for nm in ("jq", "jqd", "jf")] if want_jv else [None] * 3
        dts, dtu = self._dt(dt, U)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_step_rk4_hvp_batch(
                self.model.handle, U, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"), self._in(tau, n, U, "tau"),
                self._in(f, n, U, "f"), dts, dtu, self._in(lq, n, U, "lq", True), self._in(lqd, n, U, "lqd", True),
                self._in(lf, n, U, "lf", True), self._in(vq, n, U, "vq", True), self._in(vqd, n, U, "vqd", True),
                self._in(vtau, n, U, "vtau", True), self._in(vf, n, U, "vf", True),
                None if vdt is None else self._in(vdt.view(1, -1), 1, U, "vdt"), *[p(t) for t in h], p(hdt), *[p(t) for t in jv],
                _stream()))
        return (*h, *((hdt,) if want_dt else ()), *((tuple(jv),) if want_jv else ()))

    def rollout_rk4_vjp(self, q0, qd0, f0, tau, N: int, dt: float, traj, gqt=None, gqdt=None, gft=None):
        """Adjoint of `rollout_rk4`: `traj` = the (qt, qdt, ft) it returned for the same inputs, gqt/gqdt/gft [n, N*B] = dL/d(trajectory)
        (None = 0).  Returns (gtau [n, N*B], gq0, gqd0, gf0 [n, B]) = dL/d(tau, x0).  One step VJP per node in reverse order; nothing
        of size N*B is allocated besides gtau."""
        if q0.dim() != 2:
            raise ValueError("expected [n, B] initial states")
        n, B = self.n, q0.shape[1]
        U = B * int(N)
        qt, qdt, ft = traj
        gtau = self._out(None, n, U, "gtau")
        g0 = [self._out(None, n, B, nm) for nm in ("gq0", "gqd0", "gf0")]
        with torch.cuda.device(self.device):
            ws, ws_bytes = self._workspace(B)
            _capi.check(_capi.lib.mpcf_rollout_rk4_vjp_batch(
                self.model.handle, B, int(N), self._in(q0, n, B, "q0"), self._in(qd0, n, B, "qd0"), self._in(f0, n, B, "f0"),
                self._in(tau, n, U, "tau"), float(dt), self._in(qt, n, U, "qt"), self._in(qdt, n, U, "qdt"), self._in(ft, n, U, "ft"),
                self._in(gqt, n, U, "gqt", True), self._in(gqdt, n, U, "gqdt", True), self._in(gft, n, U, "gft", True),
                C.c_void_p(gtau.data_ptr()), *[C.c_void_p(t.data_ptr()) for t in g0], ws, ws_bytes, _stream()))
        return (gtau, *g0)

    def step_rk4_jvp_range(self, q, qd, tau, f, dt: float, u0: int, cnt: int, out, jac):
        """Units [u0, u0 + cnt) of a larger batch: states go to columns [u0, u0 + cnt) of the full-size `out` = (qn, qdn, fn),
        the Jacobian to the chunk-local buffer jac[3n, 4n+1, cap] (cap >= cnt) — one Jacobian buffer is reused over the
        chunks of a batch whose dense Jacobian would not fit the device (configs C3, C4, C5)."""
        U, n = self._U(q), self.n
        if not (0 <= u0 and cnt >= 0 and u0 + cnt <= U):
            raise ValueError("unit range out of bounds")
        qn, qdn, fn = out
        for t, nm in ((q, "q"), (qd, "qd"), (tau, "tau"), (f, "f"), (qn, "qn"), (qdn, "qdn"), (fn, "fn")):
            self._in(t, n, U, nm)
        if not (jac.is_cuda and jac.dtype == torch.float64 and jac.is_contiguous() and jac.dim() == 3
                and tuple(jac.shape[:2]) == (3 * n, 4 * n + 1) and jac.shape[2] >= cnt and jac.device == self.device):
            raise ValueError("jac must be a contiguous CUDA float64 tensor [3n, 4n+1, cap >= cnt]")
        off = lambda t: C.c_void_p(t.data_ptr() + 8 * u0)
        with torch.cuda.device(self.device):
            ws, ws_bytes = self._workspace(cnt)
            _capi.check(_capi.lib.mpcf_step_rk4_jvp_strided_batch(
                self.model.handle, cnt, U, off(q), off(qd), off(tau), off(f), float(dt), None, off(qn), off(qdn), off(fn),
                C.c_void_p(jac.data_ptr()), jac.shape[2], ws, ws_bytes, _stream()))
        return jac

    def cost_residual(self, B: int, N: int, q, qd, f, tau, qn, qdn, fn, dt: float, w_qd=1.0, w_tau=1e-2, tau0=50.0,
                      alpha=2.0, tau_floor=15.0, f_max=80.0, out=None):
        """Per-scenario (cost, defect, torque-bound, fatigue-bound) -> out[4, B]; units are node-major u = k*B + b."""
        n, U = self.n, B * N
        o = self._out(out, 4, B, "out")
        args = [self._in(t, n, U, nm) for t, nm in ((q, "q"), (qd, "qd"), (f, "f"), (tau, "tau"), (qn, "qn"), (qdn, "qdn"), (fn, "fn"))]
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_cost_residual_batch(self.model.handle, B, N, *args, float(dt), float(w_qd), float(w_tau),
                                                           float(tau0), float(alpha), float(tau_floor), float(f_max),
                                                           C.c_void_p(o.data_ptr()), _stream()))
        return o

    def cost_residual_table(self, B: int, N: int, q, qd, f, tau, qn, qdn, fn, bound_table, w_qd=1.0, w_tau=1e-2, f_max=80.0, out=None,
                            out_col0: int = 0):
        """Same reduction with a per-node, per-joint torque-bound table `bound_table` [N, n, 2] = (lb, ub) (device tensor; build it
        with ocp.f0_bound_table / ocp.step_bound_table / ocp.switch_off_bound_table).  With `out` = a [4, B_total] buffer and
        `out_col0`, the B scenarios of this call fill columns [out_col0, out_col0 + B) (scenario chunks of one send buffer)."""
        n, U = self.n, B * N
        if out is None:
            out = torch.empty((4, B), dtype=torch.float64, device=self.device)
        if not (out.is_cuda and out.dtype == torch.float64 and out.is_contiguous() and out.dim() == 2 and out.shape[0] == 4
                and 0 <= out_col0 and out_col0 + B <= out.shape[1] and out.device == self.device):
            raise ValueError("out must be a contiguous CUDA float64 tensor [4, >= out_col0 + B]")
        tb = bound_table
        if not (tb.is_cuda and tb.dtype == torch.float64 and tb.is_contiguous() and tuple(tb.shape) == (N, n, 2) and tb.device == self.device):
            raise ValueError("bound_table must be a contiguous CUDA float64 tensor of shape (N, n, 2)")
        args = [self._in(t, n, U, nm) for t, nm in ((q, "q"), (qd, "qd"), (f, "f"), (tau, "tau"), (qn, "qn"), (qdn, "qdn"), (fn, "fn"))]
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_cost_residual_table_batch(self.model.handle, B, N, *args, float(w_qd), float(w_tau),
                                                                 C.c_void_p(tb.data_ptr()), float(f_max),
                                                                 C.c_void_p(out.data_ptr() + 8 * out_col0), out.shape[1], _stream()))
        return out if out.shape[1] != B else out

    def ocp_rows(self, B: int, N: int, ee_frames, q, qd, F, T=None, q_last=None, T_last=None, rel_pos0=None, rel_ori0=None, *, wsign=-1.0,
                 fdes=(0.0, 0.0, 0.0), dist2_ref=0.0, mu=0.0, p_ref=(0.0, 0.0, 0.0), w_box=0.0, w_qd=0.0, w_F=0.0, h=0.0, derivatives=False):
        """Fused reference-mode OCP node rows (include/mpcf.h: mpcf_ocp_rows_batch): every constraint row + the running cost of
        the reference's per-node loops in one launch.  Returns (rows [nrows, U], cost [U]) and, with derivatives=True, also
        (dtau_dF [n, 3 arms, U], dT_dtau [n, U], kin_jac [26 | 3, n + 3 arms, U]).
        Compile-time families fix the arm count (chain3/6/7: one frame, forest12x6/14x7: two); on run-time trees (branched
        trees, prismatic joints) the arm count is len(ee_frames), one or two, and the frames may share ancestors."""
        n, U = self.n, B * N
        if self.model.kernel_family.startswith("generic"):
            narm = len(ee_frames)
            if narm not in (1, 2):
                raise ValueError("the OCP rows need one or two end-effector frames, got %d" % narm)
        else:
            nrows = int(_capi.lib.mpcf_ocp_rows_count(self.model.handle))
            _capi.check(nrows)
            narm = 2 if nrows == 26 + 3 * n else 1
            if len(ee_frames) != narm:
                raise ValueError("this model needs %d end-effector frame(s)" % narm)
        nrows = int(_capi.lib.mpcf_ocp_rows_count_arms(self.model.handle, narm))
        _capi.check(nrows)
        fr = [self.model.frame_id(f) if isinstance(f, str) else int(f) for f in ee_frames]
        if any(f < 0 for f in fr):  # a negative second frame would mean "one arm" to the library
            raise IndexError("end-effector frame index out of range: %s" % fr)
        fr += [-1] * (2 - narm)
        o = _capi.RowsOpts((C.c_int * 2)(*fr), float(wsign), (C.c_double * 3)(*[float(v) for v in fdes]), float(dist2_ref), float(mu),
                           (C.c_double * 3)(*[float(v) for v in p_ref]), float(w_box), float(w_qd), float(w_F), float(h))
        f64 = dict(dtype=torch.float64, device=self.device)
        rows, cost = torch.empty((nrows, U), **f64), torch.empty(U, **f64)
        kin = nrows - 3 * n
        dF = torch.empty((n, 3 * narm, U), **f64) if derivatives else None
        dT = torch.empty((n, U), **f64) if derivatives else None
        kj = torch.empty((kin, n + 3 * narm, U), **f64) if derivatives else None
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib.mpcf_ocp_rows_batch(
                self.model.handle, C.byref(o), B, N, self._in(q, n, U, "q"), self._in(qd, n, U, "qd"), self._in(F, 3 * narm, U, "F"),
                self._in(T, n, U, "T", True), self._in(q_last, n, B, "q_last", True), self._in(T_last, n, B, "T_last", True),
                self._in(rel_pos0, 3, B, "rel_pos0", True), self._in(rel_ori0, 3, B, "rel_ori0", True), p(rows), p(cost), p(dF), p(dT), p(kj),
                _stream()))
        return (rows, cost, dF, dT, kj) if derivatives else (rows, cost)
