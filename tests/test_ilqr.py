"""Batched iLQR (mpcf_riccati_gains_batch, mpcf_ilqr_costs_batch, mpcf_feedback_rollout_batch, mpc_fatigue_b200.ilqr).

This file holds its own references: the tracking cost and its Gauss-Newton derivatives restated in numpy (checked against the
complex-step derivative), both rollout entries restated on the oracle's RK4 step (checked against a literal (k, b, alpha) loop), and
a numpy iLQR built on the oracle step, its Jacobian and test_riccati.riccati_ref.  The GPU tests pin the kernels to these references,
check the exactness rules (alpha = 0, open loop, pass 1 against pass 2), the gains against mpcf_riccati_batch, and the solver on
planted and unreachable problems."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from conftest import ROOT, oracle_model_from_export, rel_err_rows
from mpc_fatigue_b200.model import Model, data_urdf
from test_riccati import OPT, _synthetic_device, nodes, planes, riccati_ref, ucols, xcols

MODELS = {
    "pilz3": lambda: Model.from_urdf(data_urdf("pilz3"), armature=1e-2),
    "pilz6": lambda: Model.from_urdf(data_urdf("pilz6"), armature=1e-2),
    "chain7": lambda: Model.synthetic("chain", 7, seed=2, armature=1e-2),
    "pilz6x2": lambda: Model.from_urdf(data_urdf("pilz6x2"), armature=1e-2),
    "dual_arm14": lambda: Model.synthetic("dual_arm", 14, seed=3, armature=1e-2),
    "pilz6x2_torso": lambda: Model.from_urdf(open(os.path.join(ROOT, "tests", "golden", "pilz6x2_torso.urdf")).read(), armature=1e-2),
    "humanoid37": lambda: Model.synthetic("humanoid", 37, seed=7, armature=1e-2),
}
FAMILY = {"pilz3": "chain3", "pilz6": "chain6", "chain7": "chain7", "pilz6x2": "forest12x6", "dual_arm14": "forest14x7",
          "pilz6x2_torso": "generic16", "humanoid37": "generic64"}


# ------------------------------------------------------------------------------------------------ references
def node_cost_ref(n, k, N, x, t, c, want=False):
    """One node's term of the tracking cost for S scenarios: x [3n, S], t [n, S] (k < N), complex allowed.  c: dict with xr [3n, S]
    or None, tr [n, S] or None, wx, wu, wN (vectors or None), lb, ub [n] or None, rho_tau, f_max, rho_f.  Returns (term [S],
    sum of |individual terms| [S]) and with want=True also (gx, gu, hx, hu): gradient and Gauss-Newton curvature."""
    term = k == N
    w = c["wN"] if term else c["wx"]
    w = np.zeros(3 * n) if w is None else w
    e = x - (0.0 if c["xr"] is None else c["xr"])
    pos = lambda d: np.where(d.real > 0, d, 0.0)
    parts = [0.5 * w[:, None] * e * e]
    pf = pos(x[2 * n:] - c["f_max"])
    parts.append(0.5 * c["rho_f"] * pf * pf)
    gx = w[:, None] * e
    gx[2 * n:] += c["rho_f"] * pf
    hx = np.repeat(w[:, None], x.shape[1], axis=1).astype(float)
    hx[2 * n:] += c["rho_f"] * (pf.real > 0)
    gu = hu = None
    if not term:
        wu = np.zeros(n) if c["wu"] is None else c["wu"]
        eu = t - (0.0 if c["tr"] is None else c["tr"])
        parts.append(0.5 * wu[:, None] * eu * eu)
        gu = wu[:, None] * eu
        hu = np.repeat(wu[:, None], x.shape[1], axis=1).astype(float)
        if c["lb"] is not None:
            pl, pu = pos(c["lb"][:, None] - t), pos(t - c["ub"][:, None])
            parts += [0.5 * c["rho_tau"] * pl * pl, 0.5 * c["rho_tau"] * pu * pu]
            gu = gu + c["rho_tau"] * (pu - pl)
            hu = hu + c["rho_tau"] * ((pl.real > 0) | (pu.real > 0))
    val = sum(p.sum(axis=0) for p in parts)
    mag = sum(np.abs(p).sum(axis=0) for p in parts)
    return (val, mag, gx, gu, hx, hu) if want else (val, mag)


def _node_c(cost, n, k, N, B, cols=None):
    """The node-k slice of a host cost dict (the device layouts: x_ref [3n, (N+1) B], tau_ref [n, N B], bound [N, n, 2])."""
    cols = np.arange(B) if cols is None else cols
    xr = None if cost.get("x_ref") is None else cost["x_ref"][:, k * B + cols]
    tr = None if (cost.get("tau_ref") is None or k == N) else cost["tau_ref"][:, k * B + cols]
    bt = cost.get("bound_table")
    lb, ub = (None, None) if (bt is None or k == N) else (bt[k, :, 0], bt[k, :, 1])
    return dict(xr=xr, tr=tr, wx=cost.get("wx"), wu=cost.get("wu"), wN=cost.get("wN"), lb=lb, ub=ub, rho_tau=cost.get("rho_tau", 0.0),
                f_max=cost.get("f_max", math.inf), rho_f=cost.get("rho_f", 0.0))


def rollout_ref(orc, n, cost, x0, taubar, N, B, dt, xbar=None, K=None, alpha=None, derivs=False):
    """Closed-loop rollout of B scenarios with per-scenario alpha [B] on the oracle step (vectorised over b).  Returns x [3n, (N+1)B],
    tau [n, N B], J [B], Jmag [B] (sum of |terms|) and with derivs the planes of mpcf_feedback_rollout_batch."""
    U = N * B
    x = np.empty((3 * n, (N + 1) * B))
    tau = np.empty((n, U))
    xk = x0.copy()
    x[:, :B] = xk
    J, mag = np.zeros(B), np.zeros(B)
    dv = dict(gx=np.empty((3 * n, U)), gu=np.empty((n, U)), wx=np.empty((3 * n, U)), wu=np.empty((n, U)))
    for k in range(N):
        sl = slice(k * B, (k + 1) * B)
        t = taubar[:, sl].copy()
        if K is not None:
            a = np.asarray(alpha, dtype=float)
            Kk = K[:, :, sl]  # [n, 3n+1, B]
            fb = np.einsum("jib,ib->jb", Kk[:, :3 * n], xk - xbar[:, sl]) + a[None] * Kk[:, 3 * n]
            t = np.where(a[None] != 0.0, t + fb, t)
        tau[:, sl] = t
        val, m, gx, gu, hx, hu = node_cost_ref(n, k, N, xk, t, _node_c(cost, n, k, N, B), want=True)
        J += val
        mag += m
        dv["gx"][:, sl], dv["gu"][:, sl], dv["wx"][:, sl], dv["wu"][:, sl] = gx, gu, hx, hu
        q, qd, f = orc.step_rk4(*[np.ascontiguousarray(v) for v in (xk[:n], xk[n:2 * n], t, xk[2 * n:])], dt)
        xk = np.concatenate([q, qd, f])
        x[:, (k + 1) * B:(k + 2) * B] = xk
    val, m, gN, _, hN, _ = node_cost_ref(n, N, N, xk, None, _node_c(cost, n, N, N, B), want=True)
    J += val
    mag += m
    dv["gN"], dv["wN"] = gN, hN
    return (x, tau, J, mag, dv) if derivs else (x, tau, J, mag)


def costs_ref(orc, n, cost, x0, xbar, taubar, K, alphas, N, B, dt):
    """J [na, B] and the magnitudes [na, B] of the line-search pass"""
    out = [rollout_ref(orc, n, cost, x0, taubar, N, B, dt, xbar=xbar, K=K, alpha=np.full(B, a)) for a in alphas]
    return np.stack([o[2] for o in out]), np.stack([o[3] for o in out])


def random_cost(n, N, B, rng, x_ref=True, tau_ref=True, bounds=True, fmax=True, xs=None, ts=None):
    """A host cost dict with the penalties active on some nodes (bounds and f_max placed inside the range of xs / ts)."""
    c = dict(wx=rng.uniform(0.5, 2.0, 3 * n), wu=rng.uniform(0.01, 0.1, n), wN=rng.uniform(1.0, 3.0, 3 * n))
    if x_ref:
        c["x_ref"] = (xs if xs is not None else 0.0) + 0.1 * rng.standard_normal((3 * n, (N + 1) * B))
    if tau_ref:
        c["tau_ref"] = (ts if ts is not None else 0.0) + rng.standard_normal((n, N * B))
    if bounds:
        mid = np.zeros(n) if ts is None else np.median(ts, axis=1)
        half = 0.2 + (0.0 if ts is None else 0.3 * np.abs(ts).mean(axis=1))
        bt = np.empty((N, n, 2))
        bt[:, :, 0] = mid - half * rng.uniform(0.5, 1.5, (N, n))
        bt[:, :, 1] = mid + half * rng.uniform(0.5, 1.5, (N, n))
        c["bound_table"], c["rho_tau"] = bt, 3.0
    if fmax:
        c["f_max"] = 50.0 if xs is None else float(np.median(xs[2 * n:])) if xs is not None else 50.0
        c["rho_f"] = 0.5
    return c


def _pilz3_oracle():
    from oracle.pyoracle import Oracle
    m = MODELS["pilz3"]()
    return m, Oracle(oracle_model_from_export(m))


def _x0_tau(om, B, N, rng):
    from conftest import random_inputs
    q, qd, tau, f, _ = random_inputs(om, B * N, seed=int(rng.integers(1 << 30)))
    x0 = np.concatenate([q[:, :B], 0.2 * qd[:, :B], f[:, :B]])
    return np.ascontiguousarray(x0), np.ascontiguousarray(0.2 * tau)


# ------------------------------------------------------------------------------------------------ CPU
def test_rollout_reference_matches_a_literal_loop():
    m, orc = _pilz3_oracle()
    n, B, N, dt = 3, 3, 4, 0.01
    rng = np.random.default_rng(1)
    x0, tb = _x0_tau(orc.model, B, N, rng)
    xbar, _, _, _ = rollout_ref(orc, n, {}, x0, tb, N, B, dt)
    cost = random_cost(n, N, B, rng, xs=xbar, ts=tb)
    K = 0.3 * rng.standard_normal((n, 3 * n + 1, N * B))
    alpha = np.array([0.0, 0.5, 1.0])
    x0p = x0 + 1e-3 * rng.standard_normal(x0.shape)
    x, tau, J, _ = rollout_ref(orc, n, cost, x0p, tb, N, B, dt, xbar=xbar, K=K, alpha=alpha)
    for b in range(B):
        xk = x0p[:, b].copy()
        Jb = 0.0
        for k in range(N):
            u = k * B + b
            t = tb[:, u].copy()
            if alpha[b] != 0.0:
                for j in range(n):
                    t[j] += alpha[b] * K[j, 3 * n, u] + sum(K[j, i, u] * (xk[i] - xbar[i, u]) for i in range(3 * n))
            assert np.allclose(tau[:, u], t, rtol=1e-14, atol=1e-14)
            for i in range(3 * n):
                Jb += 0.5 * cost["wx"][i] * (xk[i] - cost["x_ref"][i, u]) ** 2
            for j in range(n):
                Jb += 0.5 * cost["wu"][j] * (t[j] - cost["tau_ref"][j, u]) ** 2
                lb, ub = cost["bound_table"][k, j]
                Jb += 0.5 * cost["rho_tau"] * (max(lb - t[j], 0.0) ** 2 + max(t[j] - ub, 0.0) ** 2)
                Jb += 0.5 * cost["rho_f"] * max(xk[2 * n + j] - cost["f_max"], 0.0) ** 2
            q, qd, f = orc.step_rk4(*[np.ascontiguousarray(v.reshape(n, 1)) for v in (xk[:n], xk[n:2 * n], t, xk[2 * n:])], dt)
            xk = np.concatenate([q, qd, f]).ravel()
            assert np.allclose(x[:, (k + 1) * B + b], xk, rtol=1e-13, atol=1e-13)
        for i in range(3 * n):
            Jb += 0.5 * cost["wN"][i] * (xk[i] - cost["x_ref"][i, N * B + b]) ** 2
        for j in range(n):
            Jb += 0.5 * cost["rho_f"] * max(xk[2 * n + j] - cost["f_max"], 0.0) ** 2
        assert abs(J[b] - Jb) <= 1e-13 * max(abs(Jb), 1.0)
    # the line-search pass is the same rollout per candidate
    Jc, _ = costs_ref(orc, n, cost, x0p, xbar, tb, K, [0.0, 0.5], N, B, dt)
    assert np.array_equal(Jc[1, 1], J[1]) and np.array_equal(Jc[0, 0], J[0])


def test_cost_derivatives_match_the_complex_step():
    n, S, N = 4, 50, 3
    rng = np.random.default_rng(2)
    x = rng.standard_normal((3 * n, S)) + np.r_[np.zeros(2 * n), np.full(n, 50.0)][:, None]
    x[2 * n:] += 3.0 * rng.standard_normal((n, S))
    t = 2.0 * rng.standard_normal((n, S))
    cost = dict(wx=rng.uniform(0.5, 2, 3 * n), wu=rng.uniform(0.1, 1, n), wN=rng.uniform(0.5, 2, 3 * n), rho_tau=3.0, f_max=50.0, rho_f=0.7,
                x_ref=rng.standard_normal((3 * n, (N + 1) * S)), tau_ref=rng.standard_normal((n, N * S)),
                bound_table=np.stack([-np.ones((N, n)), np.ones((N, n))], axis=2))
    h = 1e-30
    for k in (1, N):
        c = _node_c(cost, n, k, N, S)
        _, _, gx, gu, hx, hu = node_cost_ref(n, k, N, x, t, c, want=True)
        for i in range(3 * n):
            xp = x.astype(complex)
            xp[i] += 1j * h
            d = node_cost_ref(n, k, N, xp, None if t is None else t.astype(complex), c)[0].imag / h
            assert np.abs(d - gx[i]).max() <= 1e-12 * max(np.abs(gx[i]).max(), 1.0)
            # curvature: the complex-step derivative of the gradient, away from the kink f = f_max
            g2 = node_cost_ref(n, k, N, xp, t.astype(complex), c, want=True)[2][i].imag / h
            away = np.abs(x[i] - 50.0) > 1e-6 if i >= 2 * n else np.ones(S, bool)
            assert np.abs(g2 - hx[i])[away].max() <= 1e-12 * max(np.abs(hx[i]).max(), 1.0)
        if k < N:
            for j in range(n):
                tp = t.astype(complex)
                tp[j] += 1j * h
                d = node_cost_ref(n, k, N, x.astype(complex), tp, c)[0].imag / h
                assert np.abs(d - gu[j]).max() <= 1e-12 * max(np.abs(gu[j]).max(), 1.0)
                g2 = node_cost_ref(n, k, N, x.astype(complex), tp, c, want=True)[3][j].imag / h
                away = (np.abs(t[j] - 1.0) > 1e-6) & (np.abs(t[j] + 1.0) > 1e-6)
                assert np.abs(g2 - hu[j])[away].max() <= 1e-12 * max(np.abs(hu[j]).max(), 1.0)
            assert (hu > c["wu"][:, None]).any() and (hu == c["wu"][:, None]).any()  # the penalty is active on some entries only
    # a NaN anywhere makes the term NaN
    xn = x.copy()
    xn[2 * n, 3] = np.nan
    assert np.isnan(node_cost_ref(n, 1, N, xn, t, _node_c(cost, n, 1, N, S))[0][3])


def numpy_ilqr(orc, n, cost, x0, tau0, N, B, dt, alphas=(1.0, 0.5, 0.25, 0.125), iters=40, mu=1e-8):
    """The solver of mpc_fatigue_b200.ilqr restated on the oracle: Gauss-Newton model, gains from test_riccati.riccati_ref's
    recursion, the same step-length rule and Levenberg update (no freezing: the iteration count is fixed)."""
    x, tau, J, _, dv = rollout_ref(orc, n, cost, x0, tau0, N, B, dt, derivs=True)
    mu = np.full(B, mu)
    for _ in range(iters):
        jac = orc.step_rk4_jvp(*[np.ascontiguousarray(x[r * n:(r + 1) * n, :N * B]) for r in (0, 1)], np.ascontiguousarray(tau),
                               np.ascontiguousarray(x[2 * n:, :N * B]), dt)[3]
        J4 = jac.reshape(3 * n, 4 * n + 1, N, B).transpose(3, 2, 0, 1)
        pr = dict(A=J4[..., xcols(n)], Bm=J4[..., ucols(n)], Q=np.einsum("bki,ij->bkij", nodes(dv["wx"], B, N), np.eye(3 * n)),
                  Sm=np.zeros((B, N, n, 3 * n)), R=np.einsum("bki,ij->bkij", nodes(dv["wu"], B, N) + mu[:, None, None], np.eye(n)),
                  gx=nodes(dv["gx"], B, N), gu=nodes(dv["gu"], B, N), d=np.zeros((B, N, 3 * n)),
                  WN=np.einsum("bi,ij->bij", dv["wN"].T, np.eye(3 * n)), gN=dv["gN"].T, dx0=np.zeros((B, 3 * n)))
        Kp = np.empty((n, 3 * n + 1, N * B))
        Kp[:, :3 * n] = _gains_ref(pr)
        Kp[:, 3 * n] = _ff_ref(pr)
        Jc = costs_ref(orc, n, cost, x0, x, tau, Kp, alphas, N, B, dt)[0]
        ok = Jc < J[None]
        Jm = np.where(ok, Jc, np.inf)
        idx = np.argmin(Jm, axis=0)
        acc = ok.any(axis=0)
        alpha = np.where(acc, np.asarray(alphas)[idx], 0.0)
        x, tau, J, _, dv = rollout_ref(orc, n, cost, x0, tau, N, B, dt, xbar=x, K=Kp, alpha=alpha, derivs=True)
        mu = np.where(acc, np.maximum(mu / 10, 1e-12), mu * 10)
    return x, tau, J


def _gains_ref(pr):
    """K_k of the textbook recursion as planes [n, 3n, N B]"""
    A, Bm, Q, Sm, R = pr["A"], pr["Bm"], pr["Q"], pr["Sm"], pr["R"]
    S, N, nx, nu = Bm.shape
    T = lambda M: np.swapaxes(M, -1, -2)
    P = pr["WN"]
    Ks = [None] * N
    for k in range(N - 1, -1, -1):
        Quu = R[:, k] + T(Bm[:, k]) @ P @ Bm[:, k]
        Qux = Sm[:, k] + T(Bm[:, k]) @ P @ A[:, k]
        Ks[k] = -np.linalg.solve(Quu, Qux)
        Pn = Q[:, k] + T(A[:, k]) @ P @ A[:, k] + T(Qux) @ Ks[k]
        P = 0.5 * (Pn + T(Pn))
    K = np.stack(Ks, axis=1)  # [S, N, nu, nx]
    return np.ascontiguousarray(K.transpose(2, 3, 1, 0).reshape(nu, nx, N * S))


def _ff_ref(pr):
    """k_k as planes [n, N B]: du_k - K_k dx_k of the reference solve"""
    dx, du, _ = riccati_ref(pr)
    S, N, nx, nu = pr["Bm"].shape
    K = _gains_ref(pr).reshape(nu, nx, N, S).transpose(3, 2, 0, 1)
    ff = du - np.einsum("skij,skj->ski", K, dx[:, :N])
    return planes(ff)


def test_numpy_ilqr_recovers_a_planted_solution():
    m, orc = _pilz3_oracle()
    n, B, N, dt = 3, 2, 6, 0.01
    rng = np.random.default_rng(3)
    x0, _ = _x0_tau(orc.model, B, N, rng)
    ts = np.repeat(rng.uniform(-2, 2, (n, 1, B)), N, axis=1).reshape(n, N * B) + 0.2 * rng.standard_normal((n, N * B))
    xs, _, _, _ = rollout_ref(orc, n, {}, x0, ts, N, B, dt)
    cost = dict(x_ref=xs, tau_ref=ts, wx=np.ones(3 * n), wu=np.full(n, 1e-2), wN=np.ones(3 * n))
    tau0 = ts + 0.3 * rng.standard_normal(ts.shape)
    J0 = rollout_ref(orc, n, cost, x0, tau0, N, B, dt)[2]
    _, tau, J = numpy_ilqr(orc, n, cost, x0, tau0, N, B, dt)
    assert (J <= 1e-14 * J0).all(), (J, J0)
    assert np.abs(tau - ts).max() <= 1e-7 * np.abs(ts).max()


def test_alpha_selection_rule():
    import torch
    from mpc_fatigue_b200.ilqr import select_alpha
    nan = float("nan")
    al = (1.0, 0.5, 0.25)
    Jc = torch.tensor([[1.0, 5.0, nan, 2.0, 3.0],
                       [1.0, 6.0, 0.5, 2.5, nan],
                       [0.5, 7.0, nan, 2.0, nan]], dtype=torch.float64)
    Jbar = torch.tensor([2.0, 4.0, 1.0, 3.0, nan], dtype=torch.float64)
    a, acc = select_alpha(Jc, Jbar, al)
    # 0: smallest wins (0.25); 1: all worse -> 0; 2: NaN never wins -> 0.5; 3: tie at 2.0 -> the earlier (1.0); 4: NaN Jbar -> 0
    assert a.tolist() == [0.25, 0.0, 0.5, 1.0, 0.0]
    assert acc.tolist() == [True, False, True, True, False]
    a1, acc1 = select_alpha(Jc[:1], Jbar, (0.75,))
    assert a1.tolist() == [0.75, 0.0, 0.0, 0.75, 0.0] and acc1.tolist() == [True, False, False, True, False]
    # a candidate equal to Jbar is not strictly below it
    a2, acc2 = select_alpha(torch.tensor([[2.0]], dtype=torch.float64), torch.tensor([2.0], dtype=torch.float64), (1.0,))
    assert a2.tolist() == [0.0] and acc2.tolist() == [False]


# ------------------------------------------------------------------------------------------------ GPU helpers
def _dev(a):
    import torch
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _tc(cost):
    from mpc_fatigue_b200.ilqr import TrackingCost
    return TrackingCost(x_ref=_dev(cost.get("x_ref")), tau_ref=_dev(cost.get("tau_ref")), wx=_dev(cost.get("wx")), wu=_dev(cost.get("wu")),
                        wN=_dev(cost.get("wN")), bound_table=_dev(cost.get("bound_table")), rho_tau=cost.get("rho_tau", 0.0),
                        f_max=cost.get("f_max", math.inf), rho_f=cost.get("rho_f", 0.0))


def _setup(name, B, N, seed, dt=0.01, variant="all", offset=True):
    """model, oracle, x0, xbar (open-loop rollout of taubar), taubar, K (random, scaled), host cost"""
    from oracle.pyoracle import Oracle
    m = MODELS[name]()
    assert m.kernel_family == FAMILY[name]
    om = oracle_model_from_export(m)
    orc = Oracle(om, fast=True)
    n = m.n
    rng = np.random.default_rng(seed)
    x0, tb = _x0_tau(om, B, N, rng)
    xbar = rollout_ref(orc, n, {}, x0, tb, N, B, dt)[0]
    on = dict(all=(True, True, True, True), none=(False, False, False, False), refs=(True, True, False, False),
              pen=(False, False, True, True))[variant]
    cost = random_cost(n, N, B, rng, *on, xs=xbar, ts=tb)
    K = 0.05 * rng.standard_normal((n, 3 * n + 1, N * B)) / np.sqrt(3 * n)
    x0p = x0 + (1e-4 * rng.standard_normal(x0.shape) if offset else 0.0)
    return m, orc, x0p, xbar, tb, K, cost


def _check_rollout(name, B, N, na, variant, seed):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m, orc, x0, xbar, tb, K, cost = _setup(name, B, N, seed, variant=variant)
    n = m.n
    ev = BatchEvaluator(m)
    alphas = [1.0, 0.0, 0.5, 0.25, 0.7, 0.125, 2.0, 0.3, 0.1, 0.05, 0.9, 0.6, 0.4, 0.01, 1.5, 0.2][:na]
    Jc = ev.ilqr_costs(_tc(cost), _dev(x0), _dev(xbar), _dev(tb), _dev(K), alphas, N, 0.01)
    Jr, mag = costs_ref(orc, n, cost, x0, xbar, tb, K, alphas, N, B, 0.01)
    torch.cuda.synchronize()
    assert (np.abs(Jc.cpu().numpy() - Jr) <= 1e-9 * mag).all(), (name, float((np.abs(Jc.cpu().numpy() - Jr) / mag).max()))
    alpha = np.array(alphas * (B // na + 1))[:B]
    x, tau, J, dv = ev.feedback_rollout(_tc(cost), _dev(x0), _dev(tb), N, 0.01, xbar=_dev(xbar), K=_dev(K), alpha=_dev(alpha),
                                        derivatives=True)
    xr, taur, Jr1, mag1, dvr = rollout_ref(orc, n, cost, x0, tb, N, B, 0.01, xbar=xbar, K=K, alpha=alpha, derivs=True)
    torch.cuda.synchronize()
    assert rel_err_rows(x.cpu().numpy(), xr) <= 1e-9, (name, rel_err_rows(x.cpu().numpy(), xr))
    assert rel_err_rows(tau.cpu().numpy(), taur) <= 1e-9
    assert (np.abs(J.cpu().numpy() - Jr1) <= 1e-9 * mag1).all()
    for k in ("gx", "gu", "wx", "wu", "gN", "wN"):
        assert rel_err_rows(dv[k].cpu().numpy(), dvr[k]) <= 1e-9, (name, k, rel_err_rows(dv[k].cpu().numpy(), dvr[k]))
    # pass 1 and pass 2 give the same bits for the same step length
    Jcn = Jc.cpu().numpy()
    Jn = J.cpu().numpy()
    for b in range(B):
        assert Jn[b].tobytes() == Jcn[alphas.index(alpha[b]), b].tobytes(), (name, b)
    return dvr


# ------------------------------------------------------------------------------------------------ GPU: gains
@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6, 7, 12, 14, 16])
@pytest.mark.parametrize("N,B", [(1, 33), (7, 257), (40, 1)])
def test_gains_on_synthetic_problems(n, N, B):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from test_riccati import _chain
    m = _chain(n)
    pr, ins = _synthetic_device(n, N, B, seed=100 * n + N)
    ev = BatchEvaluator(m)
    kw = {k: ins[k] for k in OPT}
    ref = ev.riccati(ins["jac"], B, N, **kw, want_lam=True)
    K, dx, du, lam = ev.riccati_gains(ins["jac"], B, N, **kw, want_lam=True)
    K2 = ev.riccati_gains(ins["jac"], B, N, **kw)
    torch.cuda.synchronize()
    for a, b in zip((dx, du, lam), ref):
        assert torch.equal(a, b)
    assert torch.equal(K, K2)  # the backward pass alone writes the same gains
    # du_k = K_k dx_k + k_k
    nx = 3 * n
    Kh, dxh, duh = K.cpu().numpy(), dx.cpu().numpy()[:, :N * B], du.cpu().numpy()
    rec = np.einsum("jiu,iu->ju", Kh[:, :nx], dxh) + Kh[:, nx]
    assert np.abs(rec - duh).max() <= 1e-12 * max(np.abs(duh).max(), 1.0)
    # against the reference recursion, per plane
    from test_riccati import problem_from_layout
    host = problem_from_layout(n, B, N, **{k: (None if v is None else v.cpu().numpy()) for k, v in ins.items()})
    assert rel_err_rows(Kh[:, :nx].reshape(n * nx, -1), _gains_ref(host).reshape(n * nx, -1)) <= 1e-9
    assert rel_err_rows(Kh[:, nx], _ff_ref(host)) <= 1e-9
    del pr


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz3", "pilz6", "pilz6x2", "dual_arm14", "pilz6x2_torso"])
def test_gains_on_the_librarys_own_jacobians(name):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from test_riccati import problem_from_layout
    m, orc, x0, xbar, tb, _, cost = _setup(name, 33, 7, seed=5)
    n, B, N = m.n, 33, 7
    ev = BatchEvaluator(m)
    xs = [_dev(np.ascontiguousarray(xbar[r * n:(r + 1) * n, :N * B])) for r in range(3)]
    jac = ev.step_rk4_jvp(xs[0], xs[1], _dev(tb), xs[2], 0.01)[3]
    _, _, _, dv = ev.feedback_rollout(_tc(cost), _dev(x0), _dev(tb), N, 0.01, derivatives=True)
    kw = dict(wx=dv["wx"], wu=dv["wu"] + 1e-3, gx=dv["gx"], gu=dv["gu"], wN=dv["wN"], gN=dv["gN"])
    K, dx, du = ev.riccati_gains(jac, B, N, **kw, want_solution=True)
    dxr, dur = ev.riccati(jac, B, N, **kw)
    torch.cuda.synchronize()
    assert torch.equal(dx, dxr) and torch.equal(du, dur)
    host = problem_from_layout(n, B, N, jac.cpu().numpy(), **{k: v.cpu().numpy() for k, v in kw.items()})
    Kh = K.cpu().numpy()
    assert rel_err_rows(Kh[:, :3 * n].reshape(n * 3 * n, -1), _gains_ref(host).reshape(n * 3 * n, -1)) <= 1e-9
    assert rel_err_rows(Kh[:, 3 * n], _ff_ref(host)) <= 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 13])
def test_gains_indefinite_scenario_canaries_and_rejection(n):
    import torch
    from mpc_fatigue_b200 import _capi
    from test_riccati import _chain, _p, _stream
    lib = _capi.lib
    m = _chain(n)
    N, B, bad, GAP = 5, 33, 17, 2048
    _, ins = _synthetic_device(n, N, B, seed=61)
    nk = n * (3 * n + 1) * N * B
    pool = torch.full((nk + 2 * GAP,), -7.25e300, dtype=torch.float64, device="cuda")
    K = pool[GAP:GAP + nk]
    rc = lib.mpcf_riccati_gains_batch(m.handle, B, N, _p(ins["jac"]), *[_p(ins[k]) for k in OPT], _p(K), None, None, None, _stream())
    assert rc == 0
    wu = ins["wu"].clone()
    wu[0, 3 * B + bad] = -1e6
    K2 = torch.empty_like(K)
    rc = lib.mpcf_riccati_gains_batch(m.handle, B, N, _p(ins["jac"]), *[_p(wu if k == "wu" else ins[k]) for k in OPT], _p(K2), None, None,
                                      None, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    assert bool((pool[:GAP] == -7.25e300).all()) and bool((pool[GAP + nk:] == -7.25e300).all())
    assert bool(torch.isfinite(K).all())
    Kv, K2v = K.view(-1, N * B), K2.view(-1, N * B)
    cols = torch.arange(N, device="cuda") * B + bad
    assert bool(torch.isnan(K2v[:, cols]).all())
    keep = torch.ones(N * B, dtype=torch.bool, device="cuda")
    keep[cols] = False
    assert torch.equal(K2v[:, keep], Kv[:, keep])
    st = _stream()
    call = lambda **kw: lib.mpcf_riccati_gains_batch(kw.get("model", m).handle, kw.get("B", B), kw.get("N", N), _p(kw.get("jac", ins["jac"])),
                                                     *[None] * 10, _p(kw.get("K", K)), _p(kw.get("dx")), _p(kw.get("du")), _p(kw.get("lam")), st)
    dx = torch.empty((3 * n, (N + 1) * B), dtype=torch.float64, device="cuda")
    assert call(jac=None) == _capi.EINVAL and call(K=None) == _capi.EINVAL
    assert call(N=0) == _capi.EINVAL and call(B=-1) == _capi.EINVAL
    assert call(dx=dx) == _capi.EINVAL  # du missing
    assert call(lam=dx) == _capi.EINVAL  # lam without dx
    mh = MODELS["humanoid37"]()
    assert call(model=mh) == _capi.ELIMIT and "n <= 16" in _capi.last_error()
    n0 = lib.mpcf_launch_count()
    assert call(B=0) == _capi.OK and lib.mpcf_launch_count() == n0


# ------------------------------------------------------------------------------------------------ GPU: rollouts against the reference
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODELS))
@pytest.mark.parametrize("B,N,na,variant", [(1, 1, 1, "all"), (33, 7, 3, "refs"), (257, 40, 16, "all"), (33, 7, 16, "none"),
                                            (257, 7, 3, "pen")])
def test_rollouts_match_the_oracle_reference(name, B, N, na, variant):
    if name == "humanoid37" and B * N > 2000:
        B = 33  # the oracle reference of the 37-joint tree is slow; the kernel path is the same for every B
    dvr = _check_rollout(name, B, N, na, variant, seed=hash((name, B, N)) % 1000)
    if variant in ("all", "pen") and N > 1:  # the penalties are active on some nodes and not on others
        assert (dvr["wu"] > 0.1).any() and (dvr["wu"] < 0.2).any()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz3", "pilz6", "pilz6x2", "dual_arm14", "pilz6x2_torso", "humanoid37"])
def test_exactness_rules(name):
    """K = NULL is rollout_rk4 bit for bit; alpha = 0 reproduces (xbar, taubar) bit for bit even with NaN gains; the line-search
    J of alpha equals the accept pass's J of the same alpha."""
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m, orc, x0, _, tb, K, cost = _setup(name, 65, 9, seed=9, offset=False)
    n, B, N = m.n, 65, 9
    ev = BatchEvaluator(m)
    tc = _tc(cost)
    x, tau, J = ev.feedback_rollout(tc, _dev(x0), _dev(tb), N, 0.01)
    qt, qdt, ft = ev.rollout_rk4(*[_dev(np.ascontiguousarray(x0[r * n:(r + 1) * n])) for r in range(3)], _dev(tb), N, 0.01)
    torch.cuda.synchronize()
    assert torch.equal(x[:, B:], torch.cat([qt, qdt, ft])) and torch.equal(tau, _dev(tb))
    Kn = _dev(K)
    Kn[:, :, ::3] = float("nan")
    x2, tau2, J2 = ev.feedback_rollout(tc, _dev(x0), tau, N, 0.01, xbar=x, K=Kn, alpha=torch.zeros(B, dtype=torch.float64, device="cuda"))
    Jc = ev.ilqr_costs(tc, _dev(x0), x, tau, Kn, [0.0, 0.5], N, 0.01)
    Jo = ev.ilqr_costs(tc, _dev(x0), None, tau, None, [0.0], N, 0.01)
    torch.cuda.synchronize()
    assert torch.equal(x2, x) and torch.equal(tau2, tau) and torch.equal(J2, J)
    assert torch.equal(Jc[0], J) and torch.equal(Jo[0], J)
    a = torch.full((B,), 0.5, dtype=torch.float64, device="cuda")
    _, _, J3 = ev.feedback_rollout(tc, _dev(x0), tau, N, 0.01, xbar=x, K=_dev(K), alpha=a)
    Jc3 = ev.ilqr_costs(tc, _dev(x0), x, tau, _dev(K), [0.25, 0.5], N, 0.01)
    torch.cuda.synchronize()
    assert torch.equal(J3, Jc3[1])


@pytest.mark.gpu
def test_rollout_argument_rejection():
    import torch
    from mpc_fatigue_b200 import _capi
    from mpc_fatigue_b200.coupling import box_load_coupling
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m, _, x0, xbar, tb, K, cost = _setup("pilz3", 4, 3, seed=1)
    ev = BatchEvaluator(m)
    tc = _tc(cost)
    d = [_dev(v) for v in (x0, xbar, tb, K)]
    for bad in ([], [0.5] * 17, [float("nan")], [-0.5], [float("inf")]):
        with pytest.raises(ValueError):
            ev.ilqr_costs(tc, *d, bad, 3, 0.01)
    lib = _capi.lib
    c = ev._track_cost(tc, 4, 3)
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    J = torch.empty(16 * 4, dtype=torch.float64, device="cuda")
    al = (C.c_double * 2)(0.5, 1.0)
    call = lambda **kw: lib.mpcf_ilqr_costs_batch(m.handle, C.byref(c), kw.get("B", 4), kw.get("N", 3), p(kw.get("x0", d[0])), p(kw.get("xbar", d[1])),
                                                  p(d[2]), p(kw.get("K", d[3])), al, kw.get("na", 2), 0.01, p(J), None)
    assert call() == _capi.OK
    assert call(N=0) == _capi.EINVAL and call(B=-1) == _capi.EINVAL and call(na=0) == _capi.EINVAL and call(na=17) == _capi.EINVAL
    assert call(x0=None) == _capi.EINVAL and call(xbar=None) == _capi.EINVAL
    assert call(xbar=None, K=None) == _capi.OK
    assert lib.mpcf_ilqr_costs_batch(m.handle, None, 4, 3, p(d[0]), p(d[1]), p(d[2]), p(d[3]), al, 2, 0.01, p(J), None) == _capi.EINVAL
    x = torch.empty((9, 16), dtype=torch.float64, device="cuda")
    g = torch.empty(64, dtype=torch.float64, device="cuda")
    a = torch.ones(4, dtype=torch.float64, device="cuda")
    fr = lambda **kw: lib.mpcf_feedback_rollout_batch(m.handle, C.byref(c), 4, 3, p(d[0]), p(kw.get("xbar", d[1])), p(d[2]), p(kw.get("K", d[3])),
                                                      p(kw.get("alpha", a)), 0.01, p(x), p(kw.get("tau", g)), p(J), *[p(t) for t in kw.get("dv", [None] * 6)],
                                                      None)
    assert fr() == _capi.OK
    assert fr(alpha=None) == _capi.EINVAL and fr(xbar=None) == _capi.EINVAL and fr(tau=None) == _capi.EINVAL
    assert fr(alpha=None, xbar=None, K=None) == _capi.OK
    assert fr(dv=[g, None, None, None, None, None]) == _capi.EINVAL
    mc = Model.from_urdf(data_urdf("pilz6x2"), armature=1e-2)
    mc.set_coupling(box_load_coupling(mc, mass=30.0))
    assert lib.mpcf_feedback_rollout_batch(mc.handle, C.byref(c), 4, 3, p(d[0]), None, p(d[2]), None, None, 0.01, p(x), p(g), p(J),
                                           *[None] * 6, None) == _capi.EINVAL


# ------------------------------------------------------------------------------------------------ GPU: gradient
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz3", "pilz6", "pilz6x2_torso"])
def test_gradient_from_the_rollout_adjoint_matches_central_differences(name):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m, orc, x0, _, tb, _, cost = _setup(name, 5, 6, seed=21, variant="all")
    n, B, N, dt = m.n, 5, 6, 0.01
    ev = BatchEvaluator(m)
    tc = _tc(cost)
    x, tau, J, dv = ev.feedback_rollout(tc, _dev(x0), _dev(tb), N, dt, derivatives=True)
    U = N * B
    G = torch.cat([dv["gx"][:, B:], dv["gN"]], dim=1)  # cotangent of trajectory entries 0..N-1 = x_1..x_N
    x0s = [_dev(np.ascontiguousarray(x0[r * n:(r + 1) * n])) for r in range(3)]
    traj = ev.rollout_rk4(*x0s, _dev(tb), N, dt)
    gtau = ev.rollout_rk4_vjp(*x0s, _dev(tb), N, dt, traj, G[:n].contiguous(), G[n:2 * n].contiguous(), G[2 * n:].contiguous())[0]
    grad = (gtau + dv["gu"]).cpu().numpy()
    h = 1e-6
    fd = np.empty((n, U))
    for j in range(n):
        for k in range(N):
            tp, tm = tb.copy(), tb.copy()
            tp[j, k * B:(k + 1) * B] += h
            tm[j, k * B:(k + 1) * B] -= h
            Jp = ev.ilqr_costs(tc, _dev(x0), None, _dev(tp), None, [0.0], N, dt)[0].cpu().numpy()
            Jm = ev.ilqr_costs(tc, _dev(x0), None, _dev(tm), None, [0.0], N, dt)[0].cpu().numpy()
            fd[j, k * B:(k + 1) * B] = (Jp - Jm) / (2 * h)
    # away from the kinks: torques and fatigue states not within a step of a bound
    scale = np.abs(fd).max()
    assert np.abs(grad - fd).max() <= 1e-6 * max(scale, 1.0), (name, float(np.abs(grad - fd).max()), scale)


# ------------------------------------------------------------------------------------------------ GPU: the solver
def _planted(name, B, N, seed, dt=0.01, pert=0.3):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from mpc_fatigue_b200.ilqr import TrackingCost
    from oracle.pyoracle import Oracle  # noqa: F401
    m = MODELS[name]()
    om = oracle_model_from_export(m)
    n = m.n
    rng = np.random.default_rng(seed)
    x0, _ = _x0_tau(om, B, N, rng)
    # a smooth random torque signal per scenario: a few low-frequency sines around gravity-compensating levels
    s = np.linspace(0.0, 1.0, N)[:, None, None]
    amp = np.array(om.tau_max)[None, :, None] * 0.05
    ts = amp * (rng.uniform(-1, 1, (1, n, B)) + sum(rng.uniform(-1, 1, (1, n, B)) * np.sin((i + 1) * np.pi * s + rng.uniform(0, 6, (1, n, B)))
                                                    for i in range(3)))
    ts = np.ascontiguousarray(ts.transpose(1, 0, 2).reshape(n, N * B))
    ev = BatchEvaluator(m)
    zero = TrackingCost()
    xs = ev.feedback_rollout(zero, _dev(x0), _dev(ts), N, dt)[0]
    cost = TrackingCost(x_ref=xs, tau_ref=_dev(ts), wx=torch.ones(3 * n, dtype=torch.float64, device="cuda"),
                        wu=torch.full((n,), 1e-2, dtype=torch.float64, device="cuda"), wN=torch.ones(3 * n, dtype=torch.float64, device="cuda"))
    tau0 = ts + pert * amp.reshape(n, 1) * rng.standard_normal((n, N * B))
    return m, ev, _dev(x0), ts, _dev(np.ascontiguousarray(tau0)), cost


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz3", "pilz6", "pilz6x2", "pilz6x2_torso"])
def test_solver_recovers_a_planted_solution(name):
    import torch
    from mpc_fatigue_b200.ilqr import CONVERGED, solve_ilqr
    B, N, dt = 17, 20, 0.01
    m, ev, x0, ts, tau0, cost = _planted(name, B, N, seed=31)
    r = solve_ilqr(ev, x0, tau0, N, dt, cost, iters=60)
    torch.cuda.synchronize()
    assert bool((r.status == CONVERGED).all()), (name, r.status.tolist(), r.iters.tolist())
    J0 = r.history[0]
    assert bool((r.J <= 1e-14 * J0).all()), (name, (r.J / J0).max().item())
    err = np.abs(r.tau.cpu().numpy() - ts).max() / np.abs(ts).max()
    assert err <= 1e-7, (name, err)
    assert bool((r.history[1:] <= r.history[:-1]).all())


def _unreachable(name, B, N, seed, rho_tau=3.0, penalties=True):
    import torch
    from mpc_fatigue_b200.ilqr import TrackingCost
    m, ev, x0, ts, tau0, cost = _planted(name, B, N, seed, pert=0.2)
    n = m.n
    rng = np.random.default_rng(seed + 1)
    xr = cost.x_ref + _dev(0.05 * rng.standard_normal(tuple(cost.x_ref.shape)))
    kw = {}
    if penalties:
        amp = np.abs(ts).max(axis=1)
        bt = np.stack([np.broadcast_to(-0.6 * amp, (N, n)), np.broadcast_to(0.6 * amp, (N, n))], axis=2)
        fx = np.median(xr[2 * n:].cpu().numpy())
        kw = dict(bound_table=_dev(np.ascontiguousarray(bt)), rho_tau=rho_tau, f_max=float(fx), rho_f=0.5)
    return m, ev, x0, tau0, TrackingCost(x_ref=xr, tau_ref=cost.tau_ref + 0.5, wx=cost.wx, wu=cost.wu, wN=cost.wN, **kw)


def _grad(ev, cost, x0, tau, N, dt):
    n = ev.n
    B = x0.shape[1]
    import torch
    x, _, _, dv = ev.feedback_rollout(cost, x0, tau, N, dt, derivatives=True)
    G = torch.cat([dv["gx"][:, B:], dv["gN"]], dim=1)
    x0s = [x0[r * n:(r + 1) * n].contiguous() for r in range(3)]
    traj = [x[r * n:(r + 1) * n, B:].contiguous() for r in range(3)]
    gtau = ev.rollout_rk4_vjp(*x0s, tau, N, dt, traj, *[G[r * n:(r + 1) * n].contiguous() for r in range(3)])[0]
    return gtau + dv["gu"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz3", "pilz6"])
def test_solver_on_an_unreachable_reference_with_active_penalties(name):
    import torch
    from mpc_fatigue_b200.ilqr import CONVERGED, solve_ilqr
    B, N, dt = 9, 20, 0.01
    m, ev, x0, tau0, cost = _unreachable(name, B, N, seed=41)
    r = solve_ilqr(ev, x0, tau0, N, dt, cost, iters=100, tol=1e-13)
    torch.cuda.synchronize()
    assert bool((r.history[1:] <= r.history[:-1]).all())
    g0 = _grad(ev, cost, x0, tau0, N, dt).view(m.n * N, B).abs().amax(dim=0)
    g1 = _grad(ev, cost, x0, r.tau, N, dt).view(m.n * N, B).abs().amax(dim=0)
    assert bool((r.status == CONVERGED).all()), r.status.tolist()
    assert bool((g1 <= 1e-6 * g0).all()), (g1 / g0).max().item()
    # a larger rho_tau strictly reduces the torque-bound violation of cost_residual_table
    _, _, _, _, cost2 = _unreachable(name, B, N, seed=41, rho_tau=300.0)
    r2 = solve_ilqr(ev, x0, tau0, N, dt, cost2, iters=100, tol=1e-13)
    n = m.n
    viol = []
    for rr in (r, r2):
        q, qd, f = [rr.x[i * n:(i + 1) * n, :N * B].contiguous() for i in range(3)]
        qn, qdn, fn = [rr.x[i * n:(i + 1) * n, B:].contiguous() for i in range(3)]
        viol.append(ev.cost_residual_table(B, N, q, qd, f, rr.tau, qn, qdn, fn, cost.bound_table)[2])
    torch.cuda.synchronize()
    act = viol[0] > 0  # the bounds bind in (almost) every scenario; where they do, the violation shrinks strictly
    assert int(act.sum()) >= B - 2, viol[0].tolist()
    assert bool((viol[1][act] < viol[0][act]).all()) and bool((viol[1] <= viol[0]).all()), (viol[0].tolist(), viol[1].tolist())


@pytest.mark.gpu
def test_solver_matches_scipy_lbfgsb_on_pilz3():
    import scipy.optimize as so
    import torch
    from mpc_fatigue_b200.ilqr import solve_ilqr
    from oracle.pyoracle import Oracle
    B, N, dt = 1, 10, 0.01  # 30 variables
    m, ev, x0, tau0, cost = _unreachable("pilz3", B, N, seed=51, penalties=False)
    r = solve_ilqr(ev, x0, tau0, N, dt, cost, iters=100, tol=1e-14)
    orc = Oracle(oracle_model_from_export(m))
    hc = dict(x_ref=cost.x_ref.cpu().numpy(), tau_ref=cost.tau_ref.cpu().numpy(), wx=cost.wx.cpu().numpy(), wu=cost.wu.cpu().numpy(),
              wN=cost.wN.cpu().numpy())
    x0h = x0.cpu().numpy()
    f = lambda v: rollout_ref(orc, 3, hc, x0h, v.reshape(3, N), N, 1, dt)[2][0]

    def fg(v):
        Jv = f(v)
        g = np.empty_like(v)
        for i in range(v.size):
            e = np.zeros_like(v)
            e[i] = 1e-6
            g[i] = (f(v + e) - f(v - e)) / 2e-6
        return Jv, g
    res = so.minimize(fg, tau0.cpu().numpy().ravel(), jac=True, method="L-BFGS-B", options=dict(maxiter=5000, ftol=1e-16, gtol=1e-10))
    torch.cuda.synchronize()
    Jg = float(r.J[0])
    assert Jg <= res.fun * (1 + 1e-8), (Jg, res.fun)
    assert np.abs(r.tau.cpu().numpy().ravel() - res.x).max() <= 1e-5 * max(np.abs(res.x).max(), 1.0)


@pytest.mark.gpu
def test_batch_independence_of_the_solver():
    import torch
    from mpc_fatigue_b200.ilqr import NONFINITE, solve_ilqr
    B, N, dt = 257, 15, 0.01
    m, ev, x0, ts, tau0, cost = _planted("pilz6", B, N, seed=61)
    # scenarios that need many more iterations (large perturbations) and one NaN start
    tau0 = tau0.view(m.n, N, B).clone()
    tau0[:, :, 100:140] *= 3.0
    tau0[2, 4, 200] = float("nan")
    tau0 = tau0.view(m.n, N * B).contiguous()
    r = solve_ilqr(ev, x0, tau0, N, dt, cost, iters=60)
    b = 7
    iu = torch.arange(N, device="cuda") * B + b
    ix = torch.arange(N + 1, device="cuda") * B + b
    from mpc_fatigue_b200.ilqr import TrackingCost
    c1 = TrackingCost(x_ref=cost.x_ref[:, ix].contiguous(), tau_ref=cost.tau_ref[:, iu].contiguous(), wx=cost.wx, wu=cost.wu, wN=cost.wN)
    r1 = solve_ilqr(ev, x0[:, b:b + 1].contiguous(), tau0[:, iu].contiguous(), N, dt, c1, iters=60)
    torch.cuda.synchronize()
    assert int(r.status[200]) == NONFINITE
    assert int(r1.iters[0]) == int(r.iters[b]) and int(r.iters.max()) > int(r.iters[b])
    assert torch.equal(r1.tau, r.tau[:, iu]) and torch.equal(r1.x, r.x[:, ix]) and torch.equal(r1.J, r.J[b:b + 1])


# ------------------------------------------------------------------------------------------------ GPU: full size
@pytest.mark.gpu
def test_full_size_pilz6_rollouts_on_a_sample():
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from oracle.pyoracle import Oracle
    m = MODELS["pilz6"]()
    om = oracle_model_from_export(m)
    n, B, N, dt = m.n, 65536, 100, 0.0125
    ev = BatchEvaluator(m)
    rng = np.random.default_rng(71)
    x0, tb = _x0_tau(om, B, N, rng)
    from mpc_fatigue_b200.ilqr import TrackingCost
    xbar = ev.feedback_rollout(TrackingCost(), _dev(x0), _dev(tb), N, dt)[0]
    g = torch.Generator(device="cuda").manual_seed(72)
    K = 0.01 * torch.randn((n, 3 * n + 1, N * B), generator=g, dtype=torch.float64, device="cuda")
    wx, wu, wN = rng.uniform(0.5, 2, 3 * n), rng.uniform(0.01, 0.1, n), rng.uniform(1, 3, 3 * n)
    cost = TrackingCost(x_ref=xbar, wx=_dev(wx), wu=_dev(wu), wN=_dev(wN), f_max=50.0, rho_f=0.5)
    x0p = _dev(x0 + 1e-4 * rng.standard_normal(x0.shape))
    alphas = [1.0, 0.5, 0.25, 0.125]
    Jc = ev.ilqr_costs(cost, x0p, xbar, _dev(tb), K, alphas, N, dt)
    alpha = torch.tensor(alphas, dtype=torch.float64, device="cuda").repeat(B // 4)
    x, tau, J = ev.feedback_rollout(cost, x0p, _dev(tb), N, dt, xbar=xbar, K=K, alpha=alpha)
    torch.cuda.synchronize()
    sel = np.sort(rng.choice(B, 512, replace=False))
    bs = torch.from_numpy(sel).cuda()
    iu = (torch.arange(N, device="cuda")[:, None] * B + bs[None]).reshape(-1)
    ix = (torch.arange(N + 1, device="cuda")[:, None] * B + bs[None]).reshape(-1)
    S = len(sel)
    hc = dict(x_ref=xbar[:, ix].cpu().numpy(), wx=wx, wu=wu, wN=wN, f_max=50.0, rho_f=0.5)
    orc = Oracle(om, fast=True)
    Kh = K[:, :, iu].cpu().numpy()
    xbh = xbar[:, ix].cpu().numpy()
    ah = alpha[bs].cpu().numpy()
    xr, tr, Jr, mag = rollout_ref(orc, n, hc, x0p[:, bs].cpu().numpy(), tb[:, :].reshape(n, N, B)[:, :, sel].reshape(n, N * S), N, S, dt,
                                  xbar=xbh, K=Kh, alpha=ah)
    assert rel_err_rows(x[:, ix].cpu().numpy(), xr) <= 1e-9
    assert rel_err_rows(tau[:, iu].cpu().numpy(), tr) <= 1e-9
    assert (np.abs(J[bs].cpu().numpy() - Jr) <= 1e-9 * mag).all()
    Jcr, magc = costs_ref(orc, n, hc, x0p[:, bs].cpu().numpy(), xbh, tb.reshape(n, N, B)[:, :, sel].reshape(n, N * S), Kh, alphas, N, S, dt)
    assert (np.abs(Jc[:, bs].cpu().numpy() - Jcr) <= 1e-9 * magc).all()
