"""Batched OCP node evaluation — the python/Libraries layer of the reference, re-cut for the GPU evaluator.

The reference builds its NLPs node by node and, after the solve, replays the solution with one CasADi call per
node and per arm (python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:259-274,
python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:534-546).  Here one launch evaluates every node of every scenario:
trajectories are `[B, N, n]` (scenario, node, joint) tensors on the GPU and come back the same way.

  RobotFunctions      InvDyn / ForwKin / Jac wrappers (python/Libraries/Centauro_functions.py:51-78), batched
  f0_bound_schedule   decaying torque bound  b_k = max(tau0 exp(-alpha k h), floor)
                      (python/Pilz_6_DOF/force_optimization_pilz_6DOF.py:136-148)
  step_bound_table    piecewise-constant torque bounds over thirds of the horizon
                      (python/2_pilz_6_DOF/both_robots_torque_limited_2_pilz.py:129-147)
  PilzForceOCP        g-rows and cost of the 6-DOF force OCP (force_optimization_pilz_6DOF.py:103-178)
  DualArmBoxOCP       g-rows of the dual-arm box OCP (Box_Pilz_6DOF2.py:217-475) and the solution.csv layout
  ThermalMPCNodes     tau / Euler / thermal-ZOH rows of the Centauro thermal MPC (mpc_principal.py:267-327)
  FusedBoxOCP         every row + cost of the two-arm box-carrying nodes (equilibrium, relative pose, friction cones, torque,
                      defects) from ONE fused kernel launch, with derivative blocks (mpcf_ocp_rows_batch)
"""
from __future__ import annotations

import math

import numpy as np
import torch

from .evaluator import BatchEvaluator
from .model import Model


def _soa(x: torch.Tensor) -> torch.Tensor:
    """[..., c] -> contiguous [c, U]"""
    return x.reshape(-1, x.shape[-1]).t().contiguous()


def _aos(x: torch.Tensor, batch) -> torch.Tensor:
    """[c, U] -> [*batch, c]"""
    return x.t().reshape(*batch, x.shape[0])


class RobotFunctions:
    """Batched equivalents of the L3 wrappers InvDyn / ForwKin* / Jac_* (Centauro_functions.py:51-78)."""

    def __init__(self, urdf: str, device=None, armature: float = 0.0, **model_kw):
        self.model = Model.from_urdf(urdf, armature=armature, **model_kw)
        self.ev = BatchEvaluator(self.model, device)
        self.n = self.model.n

    def InvDyn(self, q, qd, qdd=None):
        b = q.shape[:-1]
        return _aos(self.ev.rnea(_soa(q), _soa(qd), None if qdd is None else _soa(qdd)), b)

    def ForwKin(self, frame: str, q):
        b = q.shape[:-1]
        pos, rot = self.ev.fk(self.model.frame_id(frame), _soa(q))
        return _aos(pos, b), _aos(rot, b).reshape(*b, 3, 3)

    def Jac(self, frame: str, q):
        b = q.shape[:-1]
        return _aos(self.ev.jacobian(self.model.frame_id(frame), _soa(q)), b).reshape(*b, 6, self.n)

    def joint_torque(self, frame: str, q, qd, W, wsign: float = -1.0, qdd=None):
        """tau = InvDyn(q, qd, qdd) + wsign * J^T W in one launch (Pilz scripts: wsign=-1, Centauro: +1)."""
        b = q.shape[:-1]
        tau, _, _ = self.ev.node_eval_ref([self.model.frame_id(frame)], wsign, _soa(q), _soa(qd), _soa(W), None, 0.0,
                                          qdd=None if qdd is None else _soa(qdd), want_qnext=False, want_Tnext=False)
        return _aos(tau, b)


def f0_bound_schedule(N: int, h: float, tau0: float = 50.0, alpha: float = 2.0, floor: float = 15.0) -> np.ndarray:
    """b_k, k = 0..N-1 (force_optimization_pilz_6DOF.py:136-148: exponential decay, floored)."""
    k = np.arange(N)
    b = tau0 * np.exp(-alpha * k * h)
    return np.where(b > floor, b, floor)


def step_bound_table(N: int, segments: list[tuple[np.ndarray, np.ndarray]]) -> tuple[np.ndarray, np.ndarray]:
    """Piecewise-constant [lb, ub] per joint over equal segments of the horizon -> arrays [N, n]
    (both_robots_torque_limited_2_pilz.py:129-147; Box_Pilz_6DOF2.py:303-433 uses thirds)."""
    S = len(segments)
    lb = np.stack([np.asarray(segments[min(S - 1, (k * S) // N)][0], dtype=np.float64) for k in range(N)])
    ub = np.stack([np.asarray(segments[min(S - 1, (k * S) // N)][1], dtype=np.float64) for k in range(N)])
    return lb, ub


def f0_bound_table(N: int, n: int, h: float, tau0: float = 50.0, alpha: float = 2.0, floor: float = 15.0) -> np.ndarray:
    """F0 as a [N, n, 2] (lb, ub) table for mpcf_cost_residual_table_batch: -b_k <= tau <= b_k on every joint."""
    b = f0_bound_schedule(N, h, tau0, alpha, floor)
    return np.ascontiguousarray(np.stack([-b[:, None].repeat(n, 1), b[:, None].repeat(n, 1)], axis=-1))


def bound_table_from(lb: np.ndarray, ub: np.ndarray) -> np.ndarray:
    """[N, n] lower / upper arrays (e.g. from step_bound_table) -> [N, n, 2] table."""
    return np.ascontiguousarray(np.stack([np.asarray(lb, dtype=np.float64), np.asarray(ub, dtype=np.float64)], axis=-1))


def switch_off_bound_table(N: int, lbtorque, ubtorque, S, C) -> np.ndarray:
    """F3 joint switch-off (python/Centauro_script/Centauro_dynamics.py:327-348, strings S / C of CentaurOCP.py:64-71): joints
    with S[i] = 1 keep their torque limits for k < int(N / 3) and are clamped to |tau_i| <= C[i] afterwards; the others keep
    [lbtorque_i, ubtorque_i] over the whole horizon.  Returns the [N, n, 2] (lb, ub) table."""
    lbt, ubt = np.asarray(lbtorque, dtype=np.float64), np.asarray(ubtorque, dtype=np.float64)
    S, C = np.asarray(S).astype(bool), np.asarray(C, dtype=np.float64)
    n = len(lbt)
    tb = np.empty((N, n, 2))
    for k in range(N):
        late = S & (k >= int(N / 3))
        tb[k, :, 0] = np.where(late, -C, lbt)
        tb[k, :, 1] = np.where(late, C, ubt)
    return tb


class PilzForceOCP:
    """Node rows of python/Pilz_6_DOF/force_optimization_pilz_6DOF.py for B scenarios at once.

    decision variables per node: q_k(6), qd_k(6), Fx_k(1); trailing q_N(6)
    g per node: tau_k(6) in +-b_k ; ee_pos_xy - ref (2) = 0 ; Euler defect (6) = 0 ; cost -= Fx^2

    The fused row kernel takes any model, one kernel for every family: a bare revolute chain, or any other URDF (prismatic or
    continuous joints, a branched tree with the frame anywhere in it); n is then the model's DOF.
    """

    def __init__(self, urdf: str, frame: str = "prbt_link_5", N: int = 60, T: float = 2.0, tau0: float = 50.0, alpha: float = 2.0,
                 floor: float = 15.0, device=None):
        self.rf = RobotFunctions(urdf, device)
        self.frame = self.rf.model.frame_id(frame)
        self.N, self.h = N, T / N
        self.bound = f0_bound_schedule(N, self.h, tau0, alpha, floor)

    def evaluate(self, q: torch.Tensor, qd: torch.Tensor, Fx: torch.Tensor, ref_xy) -> dict:
        """q [B, N+1, 6], qd [B, N, 6], Fx [B, N] -> dict of rows.  ONE launch of the fused row kernel (mpcf_ocp_rows_batch):
        torque rows, end-effector position error, Euler defects and the node cost -F^T F."""
        B, N, n = qd.shape
        ev = self.rf.ev
        U = B * N
        # node-major units u = k*B + b
        nm = lambda x: x.permute(2, 1, 0).reshape(x.shape[2], -1).contiguous()
        F = torch.zeros((3, U), dtype=torch.float64, device=q.device)
        F[0] = Fx.t().reshape(-1)
        rows, cost = ev.ocp_rows(B, N, [self.frame], nm(q[:, :N]), nm(qd), F, None, q[:, N].t().contiguous(), wsign=-1.0,
                                 p_ref=(float(ref_xy[0]), float(ref_xy[1]), 0.0), w_F=-1.0, h=self.h)
        back = lambda r: r.reshape(r.shape[0], N, B).permute(2, 1, 0)
        tau = back(rows[3:3 + n])
        bound = torch.as_tensor(self.bound, dtype=torch.float64, device=q.device).reshape(1, N, 1)
        return {
            "tau": tau,
            "tau_bound": bound.reshape(N),
            "tau_violation": (tau.abs() - bound).clamp_min(0.0).amax(dim=(1, 2)),
            "line": back(rows[0:2]),
            "defect": back(rows[3 + n:3 + 2 * n]),
            "cost": cost.reshape(N, B).sum(0),
        }

    def jacobian(self, q: torch.Tensor, qd: torch.Tensor, Fx: torch.Tensor) -> dict:
        """First derivatives of the g-rows of `evaluate` with respect to the node's own decision variables
        (what IPOPT's `jac_g` needs; CasADi derives them from the SX graph in the reference):
          dtau_dq, dtau_dqd [B, N, 6, 6];  dtau_dFx [B, N, 6] = -J[0, :];  dline_dq [B, N, 2, 6] = J[0:2, :];
          the Euler defect q_k + h qd_k - q_{k+1} has constant blocks (I, h I, -I)."""
        B, N, n = qd.shape
        ev = self.rf.ev
        qk = q[:, :N]
        W = torch.zeros((B, N, 6), dtype=torch.float64, device=q.device)
        W[..., 0] = Fx
        Dq, Dv = ev.node_eval_ref_jvp([self.frame], -1.0, _soa(qk), _soa(qd), _soa(W))
        J = _aos(ev.jacobian(self.frame, _soa(qk)), (B, N)).reshape(B, N, 6, n)
        return {"dtau_dq": _aos(Dq, (B, N)).reshape(B, N, n, n), "dtau_dqd": _aos(Dv, (B, N)).reshape(B, N, n, n),
                "dtau_dFx": -J[:, :, 0, :], "dline_dq": J[:, :, 0:2, :], "defect_dq": 1.0, "defect_dqd": self.h, "defect_dqnext": -1.0}


class DualArmBoxOCP:
    """Dual-arm box OCP (python/2_pilz_6_DOF/Box_Pilz_6DOF2.py): two separate 6-DOF models.

    solution.csv layout (Box_Pilz_6DOF2.py:520-537): per node [q(12), qd(12), F_LR(3), F_RR(3)], then q_N(12).
    """

    NQ, NF = 12, 3

    def __init__(self, urdf_first: str, urdf_second: str, frame: str = "end_effector", device=None, mass: float = 30.0):
        self.left = RobotFunctions(urdf_first, device)
        self.right = RobotFunctions(urdf_second, device)
        self.fl = self.left.model.frame_id(frame)
        self.fr = self.right.model.frame_id(frame)
        self.Fdes = 9.81 * mass  # Box_Pilz_6DOF2.py:197

    @classmethod
    def parse_solution(cls, vec) -> dict:
        """solution.csv vector -> q [N+1, 12], qd [N, 12], F_LR [N, 3], F_RR [N, 3]."""
        v = np.asarray(vec, dtype=np.float64).reshape(-1)
        stride = 2 * cls.NQ + 2 * cls.NF
        N, rem = divmod(len(v) - cls.NQ, stride)
        if rem:
            raise ValueError("vector length %d is not N*%d+%d" % (len(v), stride, cls.NQ))
        nodes = v[:N * stride].reshape(N, stride)
        return {"N": N, "q": np.vstack([nodes[:, :12], v[N * stride:][None]]), "qd": nodes[:, 12:24],
                "F_LR": nodes[:, 24:27], "F_RR": nodes[:, 27:30]}

    def evaluate(self, q: torch.Tensor, qd: torch.Tensor, F_LR: torch.Tensor, F_RR: torch.Tensor, T: float = 2.0) -> dict:
        """q [B, N+1, 12], qd [B, N, 12], F_* [B, N, 3] -> constraint rows of Box_Pilz_6DOF2.py:244-293,463-475."""
        B, N, _ = qd.shape
        h = T / N
        z3 = torch.zeros((B, N, 3), dtype=torch.float64, device=q.device)
        out = {}
        for side, rf, fr, sl, F in (("L", self.left, self.fl, slice(0, 6), F_LR), ("R", self.right, self.fr, slice(6, 12), F_RR)):
            qs, qds = q[:, :N, sl], qd[:, :, sl]
            W = torch.cat([F, z3], dim=-1)
            tau, qn, _ = rf.ev.node_eval_ref([fr], -1.0, _soa(qs), _soa(qds), _soa(W), None, h, want_Tnext=False)
            pos, rot = rf.ev.fk(fr, _soa(q[:, :, sl]))
            out["tau_" + side] = _aos(tau, (B, N))
            out["defect_" + side] = _aos(qn, (B, N)) - q[:, 1:, sl]
            out["E_" + side] = _aos(pos, (B, N + 1))
            out["R_" + side] = _aos(rot, (B, N + 1)).reshape(B, N + 1, 3, 3)
        E1, E2 = out["E_L"][:, :N], out["E_R"][:, :N]
        out["force_eq"] = torch.stack([F_LR[..., 2] + F_RR[..., 2] - self.Fdes, F_LR[..., 0] + F_RR[..., 0], F_LR[..., 1] + F_RR[..., 1]], dim=-1)
        out["moment_eq"] = torch.linalg.cross(E1 - E2, F_LR) + torch.linalg.cross(E2 - E1, F_RR)
        out["dist2"] = ((E1 - E2) ** 2).sum(-1)
        return out


class ThermalMPCNodes:
    """tau / Euler / thermal rows of the Centauro thermal MPC node (python/Centauro_script/mpc_principal.py:267-327):
    tau = InvDyn(q, qd, 0) + sum_e J_e^T W_e ; q_next = q + h qd ; T_next = a T + (1 - a) R_theta P_loss."""

    def __init__(self, model: Model, ee_frames: list[str], T: float = 20.0, N: int = 40, device=None, temperature_bound: float = 80.0):
        self.model = model
        self.ev = BatchEvaluator(model, device)
        self.frames = [model.frame_id(f) for f in ee_frames]
        self.h = T / N
        self.N = N
        self.temperature_bound = temperature_bound  # python/Libraries/MPC_parameters.py:49

    def evaluate(self, q, qd, W, Temp) -> dict:
        """q [B, N+1, n], qd [B, N, n], W [B, N, 6*nee] (force the robot exerts), Temp [B, N+1, n]."""
        B, N, n = qd.shape
        tau, qn, Tn = self.ev.node_eval_ref(self.frames, +1.0, _soa(q[:, :N]), _soa(qd), _soa(W), _soa(Temp[:, :N]), self.h)
        Tn = _aos(Tn, (B, N))
        return {"tau": _aos(tau, (B, N)), "q_defect": _aos(qn, (B, N)) - q[:, 1:], "T_defect": Tn - Temp[:, 1:],
                "T_violation": (Tn - self.temperature_bound).clamp_min(0.0).amax(dim=(1, 2))}

    def box_rows(self, q, qd, F_L, F_R, mass: float, rel_pos0, rel_ori0, box_ini) -> dict:
        """Rows of the dual-arm box-carrying OCP that involve both end-effectors (mpc_principal.py:229-260) and its running
        cost (:281-284); needs exactly two end-effector frames (left, right).

        q [B, N+1, n], qd [B, N, n], F_L / F_R [B, N, 3] world-frame forces the arms exert, rel_pos0 / rel_ori0 [B, 3]
        (relative pose at the initial condition), box_ini [3].  Returns force_eq, moment_eq, rel_pos, rel_ori (each
        [B, N, 3], residuals that the NLP pins to zero) and cost [B]."""
        if len(self.frames) != 2:
            raise ValueError("box rows need a left and a right end-effector frame")
        B, N, n = qd.shape
        qs = _soa(q[:, :N])
        pL, RL = self.ev.fk(self.frames[0], qs)
        pR, RR = self.ev.fk(self.frames[1], qs)
        pL, pR = _aos(pL, (B, N)), _aos(pR, (B, N))
        RL, RR = _aos(RL, (B, N)).reshape(B, N, 3, 3), _aos(RR, (B, N)).reshape(B, N, 3, 3)
        Fdes = torch.tensor([0.0, 0.0, 9.81 * mass], dtype=torch.float64, device=q.device)  # :156
        rel = torch.einsum("bnji,bnj->bni", RL, pR - pL)  # R01^T (pR - pL), :241
        prev = torch.cat([torch.as_tensor(rel_pos0, dtype=torch.float64, device=q.device).reshape(B, 1, 3), rel[:, :-1]], dim=1)
        Ro = RL @ RR.transpose(-1, -2)  # :248
        sk = 0.5 * (Ro - Ro.transpose(-1, -2))
        e = torch.stack([sk[..., 2, 1], sk[..., 2, 0], sk[..., 1, 0]], dim=-1)  # :252-255
        pbox = 0.5 * (pL + pR)
        dbox = pbox - torch.as_tensor(box_ini, dtype=torch.float64, device=q.device)
        cost = (1000.0 * (dbox * dbox).sum(-1) + 100.0 * (qd * qd).sum(-1) + 10.0 * (F_L * F_L).sum(-1) + 10.0 * (F_R * F_R).sum(-1)).sum(-1)
        return {"force_eq": F_L + F_R - Fdes,
                "moment_eq": torch.linalg.cross(pL - pR, F_L) + torch.linalg.cross(pR - pL, F_R),
                "rel_pos": rel - prev,
                "rel_ori": e - torch.as_tensor(rel_ori0, dtype=torch.float64, device=q.device).reshape(B, 1, 3),
                "cost": cost, "pL": pL, "pR": pR}


class FusedBoxOCP:
    """Box-carrying node rows of the two-arm OCPs through the fused row kernel (include/mpcf.h: mpcf_ocp_rows_batch): the
    dual Pilz box OCP on the single-tree URDF (python/2_pilz_6_DOF/Box_Pilz_6DOF2.py:244-293,454-475) and the Centauro thermal
    MPC node (python/Centauro_script/mpc_principal.py:229-327, friction cones of RepeatedMPCwithThermal_confriction.py:251-273):
    force / moment equilibrium, end-effector distance, relative pose, friction cones, torque rows, Euler and thermal defects
    and the running cost — ONE launch for all B scenarios x N nodes, plus the derivative blocks on request.

    Any model with the two end-effector frames works, through the same kernel: the two-arm forests (forest12x6 / forest14x7),
    where each frame must sit on its own arm, and every other tree — two arms on a torso joint (the Centauro upper body), a
    humanoid holding the box with both hands, arms with prismatic joints.  On shared ancestors the torque rows carry both forces and
    dtau_dF has both arm blocks."""

    ROWS = {"force_eq": (0, 3), "moment_eq": (3, 6), "dist2": (6, 7), "rel_pos": (7, 10), "rel_ori": (10, 13), "friction": (13, 23),
            "box_err": (23, 26)}

    def __init__(self, model: Model, ee_frames, device=None, *, wsign: float = +1.0, mass: float = 30.0, dist2_ref: float = 0.0, mu: float = 0.5,
                 p_ref=(0.0, 0.0, 0.0), w_box: float = 1000.0, w_qd: float = 100.0, w_F: float = 10.0, T: float = 20.0, N: int = 40):
        self.model, self.ev = model, BatchEvaluator(model, device)
        self.frames = [model.frame_id(f) if isinstance(f, str) else int(f) for f in ee_frames]
        self.N, self.h = N, T / N
        self.kw = dict(wsign=wsign, fdes=(0.0, 0.0, 9.81 * mass), dist2_ref=dist2_ref, mu=mu, p_ref=tuple(p_ref), w_box=w_box, w_qd=w_qd, w_F=w_F,
                       h=self.h)

    def evaluate(self, q, qd, F_L, F_R, Temp=None, rel_pos0=None, rel_ori0=None, derivatives: bool = False) -> dict:
        """q [B, N+1, n], qd [B, N, n], F_L / F_R [B, N, 3], Temp [B, N+1, n] or None, rel_pos0 / rel_ori0 [B, 3] or None."""
        B, N, n = qd.shape
        nm = lambda x: x.permute(2, 1, 0).reshape(x.shape[2], -1).contiguous()
        tb = lambda x: None if x is None else torch.as_tensor(x, dtype=torch.float64, device=q.device).reshape(B, 3).t().contiguous()
        F = torch.cat([nm(F_L), nm(F_R)], dim=0)
        res = self.ev.ocp_rows(B, N, self.frames, nm(q[:, :N]), nm(qd), F, None if Temp is None else nm(Temp[:, :N]), q[:, N].t().contiguous(),
                               None if Temp is None else Temp[:, N].t().contiguous(), tb(rel_pos0), tb(rel_ori0), derivatives=derivatives, **self.kw)
        rows, cost = res[0], res[1]
        back = lambda r: r.reshape(r.shape[0], N, B).permute(2, 1, 0)
        out = {k: back(rows[a:b]) for k, (a, b) in self.ROWS.items()}
        out.update({"tau": back(rows[26:26 + n]), "q_defect": back(rows[26 + n:26 + 2 * n]), "T_defect": back(rows[26 + 2 * n:26 + 3 * n]),
                    "cost": cost.reshape(N, B).sum(0)})
        if derivatives:
            out.update({"dtau_dF": res[2], "dT_dtau": res[3], "kin_jac": res[4]})
        return out


def temp_simulation(Ic: float, Tin: float, T: float = 120.0, N: int = 200, Tbound: float = 70.0, ktau: float = 1.0):
    """Closed-form twin of python/Libraries/TemperatureModel.py:TempSimulation (constant current, zero speed):
    returns (violated, list of winding temperatures up to the first violation)."""
    Ra, Rth = 10.0, 300.0 * 9.0 / 309.0
    tth = Rth * 15.0
    a = math.e ** (-T / N / tth)
    Tw = [Tin]
    for i in range(N):
        if Tw[i] > Tbound:
            return True, Tw
        Tw.append(a * Tw[i] + Ra * Ic * Ic * Rth * (1 - a))
    return False, Tw[:N]
