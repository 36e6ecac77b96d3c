"""Per-joint model parameters (Model.set_fatigue, Model.set_armature) through every kernel family.

Every other test builds its models with one fatigue row copied to all joints (lambda = 1 / (R_th C_th) ~ 7.6e-3 1/s) and one scalar
armature.  There a kernel that reads joint 0's row, the other arm's row or a chain-local index where the row is global gives the
same numbers as a correct one, and at lambda dt ~ 1.5e-4 the cubic and quartic terms of the closed-form RK4 amplification
amp(z) = 1 - z + z^2/2 - z^3/6 + z^4/24 sit below the 1e-9 tolerance.  Here every model runs under seeded parameter sets:

  het     distinct rows on every joint: lambda log-uniform in [0.05, 60] 1/s, kappa in [0.02, 0.5], c_tau in [1e-3, 2e-2],
          c_v in [0.1, 1], armature in [1e-3, 5e-2]; the two arms of a forest draw from disjoint halves of every range
  stiff   the het rows with lambda_i dt in [0.5, 2.5] (inside RK4's stability limit 2.785): every term of amp is >= 1e-3
  F0      the reference's capacity-decay instance: lambda = 2, kappa = 0 on every joint
  mixed0  lambda = 0 (kappa > 0) on the even joints, stiff rows on the others: the per-joint lambda = 0 branch
  tiny    lambda in {1e-6, 1e-9, 1e-12}: the thermal zero-order hold only, whose gain must stay continuous into lambda = 0

CPU tests show that the GPU tests can fail: a rolled or swapped parameter row, and a sign flip of the z^3 or z^4 coefficient of
amp, move the oracle by far more than the tolerance; the complex-step and hyper-dual references agree with central differences
in the new regimes; the zero-order hold matches an expm1 restatement from lambda = 0 to 1e-3.  GPU tests compare every entry with
the oracle built from the model's export (which carries the per-joint rows), per state row and per Jacobian plane at 1e-9."""
import copy
import os

import numpy as np
import pytest

from conftest import ROOT, oracle_model_from_export, random_inputs, rel_err_rows
from mpc_fatigue_b200.model import Model, data_urdf
from oracle.pyoracle import Oracle
from test_hess import _assert_scaled, _hv, oracle_hess, oracle_hvp
from test_vjp import assert_vjp_close, rollout_adjoint_ref, vjp_ref, vjp_scale

TOL = 1e-9
DT = 0.02  # step of the stiff set: lambda_i = z_i / DT

MODELS = {
    "pilz3": (lambda: Model.from_urdf(data_urdf("pilz3"), armature=1e-2), "chain3"),
    "pilz6": (lambda: Model.from_urdf(data_urdf("pilz6"), armature=1e-2), "chain6"),
    "chain7": (lambda: Model.synthetic("chain", 7, seed=2, armature=1e-2), "chain7"),
    "pilz6x2": (lambda: Model.from_urdf(data_urdf("pilz6x2"), armature=1e-2), "forest12x6"),
    "dual_arm14": (lambda: Model.synthetic("dual_arm", 14, seed=3, armature=1e-2), "forest14x7"),
    "chain10": (lambda: Model.synthetic("chain", 10, seed=3, armature=1e-3), "generic16"),
    "mixed": (lambda: Model.from_urdf(open(os.path.join(ROOT, "tests", "golden", "mixed_joints.urdf")).read(), armature=1e-3), "generic16"),
    "humanoid37": (lambda: Model.synthetic("humanoid", 37, seed=7, armature=1e-2), "generic64"),
    "chain48": (lambda: Model.synthetic("chain", 48, seed=5, armature=1e-2), "generic64"),  # n > 40: the dual-number sweeps
}
STEP_SETS = ["het", "stiff", "F0", "mixed0"]
SEED = {"het": 1, "stiff": 2, "F0": 3, "mixed0": 4, "tiny": 5}


def _units(name):
    """ragged against the 128-thread block; the large trees run smaller batches (the oracle sweeps every column per unit)"""
    return {"chain10": 65, "mixed": 65, "humanoid37": 33, "chain48": 33}.get(name, 130)


def _arms(m):
    """joint index ranges drawn from disjoint parameter ranges: the two chains of a forest family, else the whole model"""
    if m.kernel_family.startswith("forest"):
        L = m.n // 2
        return [np.arange(L), np.arange(L, m.n)]
    return [np.arange(m.n)]


def param_rows(m, pset):
    """(fat [n, 4], arm [n]) of parameter set `pset` for model m, seeded by the set and the model size"""
    n = m.n
    rng = np.random.default_rng(1000 * SEED[pset] + n)
    fat, arm = np.empty((n, 4)), np.empty(n)
    arms = _arms(m)

    def draw(lo, hi, idx, c, log=False):
        f = (lambda x: np.log(x), np.exp) if log else (lambda x: x, lambda x: x)
        a, b = f[0](lo), f[0](hi)
        k = len(arms)
        return f[1](rng.uniform(a + (b - a) * c / k, a + (b - a) * (c + 1) / k, len(idx)))

    for c, idx in enumerate(arms):
        fat[idx, 0] = draw(0.05, 60.0, idx, c, log=True)
        fat[idx, 1] = draw(0.02, 0.5, idx, c)
        fat[idx, 2] = draw(1e-3, 2e-2, idx, c)
        fat[idx, 3] = draw(0.1, 1.0, idx, c)
        arm[idx] = draw(1e-3, 5e-2, idx, c)
        if pset in ("stiff", "mixed0"):
            fat[idx, 0] = draw(0.5, 2.5, idx, c) / DT
    if pset == "F0":
        fat[:, 0], fat[:, 1] = 2.0, 0.0
    elif pset == "mixed0":
        fat[0::2, 0] = 0.0
    elif pset == "tiny":
        fat[:, 0] = np.array([1e-6, 1e-9, 1e-12])[np.arange(n) % 3]
    return fat, arm


def build(name, pset=None):
    """(model, oracle model) with parameter set `pset` applied through the setters; the oracle model is built from the export"""
    make, fam = MODELS[name]
    m = make()
    assert m.kernel_family == fam, (name, m.kernel_family)
    if pset is not None:
        fat, arm = param_rows(m, pset)
        m.set_fatigue(fat)
        m.set_armature(arm)
        assert np.array_equal(m.export("fat"), fat) and np.array_equal(m.export("arm"), arm)
    return m, oracle_model_from_export(m)


def _oracle_with(om, fat=None, arm=None):
    """oracle of `om` with its fatigue rows and / or armature replaced"""
    om2 = copy.copy(om)
    if fat is not None:
        om2.fat = [list(r) for r in fat]
    if arm is not None:
        om2.arm = list(arm)
    return Oracle(om2)


def amp(z, c3=-1.0 / 6.0, c4=1.0 / 24.0):
    """RK4 amplification of fdot = -lambda f over one step, z = lambda dt"""
    return 1.0 - z + z * z / 2.0 + c3 * z ** 3 + c4 * z ** 4


def zoh_ref(fat, T, tau, qd, h):
    """numpy restatement of the thermal zero-order hold: a T + g P with a = exp(-lambda h), g = -expm1(-lambda h) kappa / lambda
    (h kappa at lambda = 0), P = c_tau tau^2 + c_v qd^2; returns (T+, a, g, P)"""
    lam, kap, ct, cv = (fat[:, k][:, None] for k in range(4))
    a = np.exp(-lam * h)
    g = np.where(lam == 0.0, h * kap, -np.expm1(-lam * h) * kap / np.where(lam == 0.0, 1.0, lam))
    P = ct * tau * tau + cv * qd * qd
    return a * T + g * P, a, g, P


# ================================================================================================================ CPU
def test_parameter_sets_are_what_they_claim():
    for name in MODELS:
        m = MODELS[name][0]()
        for pset in ("het", "stiff", "F0", "mixed0", "tiny"):
            fat, arm = param_rows(m, pset)
            assert (arm >= 1e-3).all() and (arm <= 5e-2).all() and len(np.unique(arm)) == m.n
            lam = fat[:, 0]
            if pset == "het":
                assert len(np.unique(fat, axis=0)) == m.n and (lam >= 0.05).all() and (lam <= 60).all()
                assert (lam * 0.03 < 2.785).all()  # the largest per-unit dt of the GPU tests stays inside RK4's stability limit
            if pset == "stiff":
                assert (lam * DT >= 0.5).all() and (lam * DT <= 2.5).all()
                z = lam * DT
                assert (np.minimum(z ** 3 / 6, z ** 4 / 24) >= 1e-3 * np.abs(amp(z))).all()
            if pset == "F0":
                assert (lam == 2.0).all() and (fat[:, 1] == 0.0).all()
            if pset == "mixed0":
                assert (lam[0::2] == 0).all() and (lam[1::2] * DT >= 0.5).all() and (fat[0::2, 1] > 0).all()
            for a, b in zip(_arms(m), _arms(m)[1:]):  # forests: every range of arm 0 lies below that of arm 1
                cols = [fat[:, 2], fat[:, 3], arm] + ([fat[:, 1]] if pset != "F0" else []) + ([lam] if pset in ("het", "stiff") else [])
                for col in cols:
                    assert col[a].max() < col[b].min(), (name, pset)


def _step_and_jac(orc, x, dt=DT):
    q, qd, tau, f = x
    return orc.step_rk4_jvp(q, qd, tau, f, dt)


@pytest.mark.parametrize("pset", ["het", "stiff", "mixed0"])
@pytest.mark.parametrize("name", list(MODELS))
def test_index_errors_move_the_reference_far_beyond_the_tolerance(name, pset):
    """An indexing error in a kernel reads another joint's (or arm's) row.  Rolled fatigue rows, swapped arms and a rolled armature
    must move the oracle's step and Jacobian by > 1e3 TOL in the rows the GPU tests check: the fatigue rows of EVERY joint for the
    fatigue parameters, the dynamics rows for the armature.  (F0 is left out: its rows are the same on every joint.)"""
    m, om = build(name, pset)
    n = m.n
    x = random_inputs(om, 3, seed=7)[:4]
    base = _step_and_jac(Oracle(om), x)
    fat, arm = np.array(om.fat), np.array(om.arm)
    fr = slice(2 * n, 3 * n)

    def moved(orc):
        got = _step_and_jac(orc, x)
        return got, [rel_err_rows(got[2][i:i + 1], base[2][i:i + 1]) for i in range(n)], \
            [rel_err_rows(got[3][2 * n + i], base[3][2 * n + i]) for i in range(n)]

    variants = [("fat rolled", np.roll(fat, 1, axis=0))]
    if len(_arms(m)) == 2:
        L = n // 2
        variants.append(("arms swapped", np.concatenate([fat[L:], fat[:L]])))
    for what, f2 in variants:
        _, ef, ej = moved(_oracle_with(om, fat=f2))
        assert min(ef) > 1e3 * TOL and min(ej) > 1e3 * TOL, (name, pset, what, min(ef), min(ej))
    got = _step_and_jac(_oracle_with(om, arm=np.roll(arm, 1)), x)
    assert rel_err_rows(got[1], base[1]) > 1e3 * TOL and rel_err_rows(got[3][n:2 * n], base[3][n:2 * n]) > 1e3 * TOL
    assert np.array_equal(got[3][fr, 3 * n:4 * n], base[3][fr, 3 * n:4 * n])  # d f+ / d f does not see the armature


@pytest.mark.parametrize("name", ["pilz6", "pilz6x2", "humanoid37"])
def test_amplification_coefficients_are_visible_under_stiff(name):
    """d f+_i / d f_i = amp(lambda_i dt) exactly; under `stiff` a sign flip of its z^3 or z^4 coefficient moves every diagonal entry
    by > 1e3 TOL (at the default lambda dt ~ 1.5e-4 the same flips move it by 6e-13 and 2e-17)."""
    m, om = build(name, "stiff")
    n = m.n
    x = random_inputs(om, 2, seed=9)[:4]
    J = _step_and_jac(Oracle(om), x)[3]
    diag = np.stack([J[2 * n + i, 3 * n + i] for i in range(n)])
    z = np.array(om.fat)[:, 0:1] * DT
    assert np.abs(diag - amp(z)).max() <= 1e-14
    for c3, c4 in ((1.0 / 6.0, 1.0 / 24.0), (-1.0 / 6.0, -1.0 / 24.0)):
        assert (np.abs(amp(z, c3, c4) - diag) / np.abs(diag) > 1e3 * TOL).all(), (c3, c4)
    zd = 0.00762963 * DT
    assert 2 * zd ** 3 / 6 < TOL and 2 * zd ** 4 / 24 < TOL  # what the default rows cannot see


@pytest.mark.parametrize("pset", ["het", "stiff"])
@pytest.mark.parametrize("name", ["pilz6", "pilz6x2"])
def test_complex_step_jacobian_matches_central_differences(name, pset):
    m, om = build(name, pset)
    orc = Oracle(om)
    n, U = m.n, 2
    x = random_inputs(om, U, seed=13)[:4]
    J = orc.step_rk4_jvp(*x, DT)[3]
    for c in range(4 * n + 1):
        blk, j = divmod(c, n)
        eps = 1e-6 * (1.0 if blk == 4 else max(1.0, float(np.abs(x[blk][j]).max())))
        if blk == 4:
            fp, fm = (np.concatenate(orc.step_rk4(*x, DT + s * eps)) for s in (1, -1))
        else:
            xp, xm = [a.copy() for a in x], [a.copy() for a in x]
            xp[blk][j] += eps
            xm[blk][j] -= eps
            fp, fm = np.concatenate(orc.step_rk4(*xp, DT)), np.concatenate(orc.step_rk4(*xm, DT))
        fd = (fp - fm) / (2 * eps)
        assert np.abs(J[:, c] - fd).max() < 2e-6 * max(1.0, np.abs(fd).max()), (name, pset, c)


@pytest.mark.parametrize("pset", ["het", "stiff"])
def test_hyper_dual_hessian_matches_central_differences_of_the_complex_step_vjp(pset):
    m, om = build("pilz3", pset)
    orc = Oracle(om)
    n, U = m.n, 2
    P = 4 * n + 1
    x = random_inputs(om, U, seed=17)[:4]
    lam = np.random.default_rng(18).standard_normal((3 * n, U))
    dt_u = np.ascontiguousarray([DT, 0.6 * DT])
    H = oracle_hess(orc, *x, 0.0, *[np.ascontiguousarray(lam[i * n:(i + 1) * n]) for i in range(3)], dt_u=dt_u)
    zz = np.vstack(list(x) + [dt_u[None]])

    def vjp(zv):
        parts = [np.ascontiguousarray(zv[i * n:(i + 1) * n]) for i in range(4)]
        return np.einsum("ru,rcu->cu", lam, orc.step_rk4_jvp(*parts, 0.0, dt_u=np.ascontiguousarray(zv[4 * n]))[3])

    scale = np.abs(H).max(axis=(0, 1))
    for c in range(P):
        eps = 1e-5 if c < 4 * n else 1e-7
        zp, zm = zz.copy(), zz.copy()
        zp[c] += eps
        zm[c] -= eps
        fd = (vjp(zp) - vjp(zm)) / (2 * eps)
        assert (np.abs(H[:, c] - fd) <= 1e-6 * scale).all(), (pset, c, float((np.abs(H[:, c] - fd) / scale).max()))
    # the fatigue entries at z of order 1: H[f_i][dt] = lf_i lambda_i amp'(lambda_i h), amp' = -1 + z - z^2/2 + z^3/6
    lamb = np.array(om.fat)[:, 0:1]
    z = lamb * dt_u[None]
    ref = lam[2 * n:] * lamb * (-1.0 + z - z * z / 2 + z ** 3 / 6)
    assert np.abs(H[3 * n:4 * n, 4 * n] - ref).max() <= 1e-12 * np.abs(H).max()


LAMS = np.array([0.0, 1e-14, 1e-12, 1e-9, 1e-6, 1e-3])


@pytest.mark.parametrize("h", [2.0 / 60.0, 0.5])
def test_zero_order_hold_is_continuous_as_lambda_goes_to_zero(h):
    """The oracle's thermal ZOH (decay factor and gain, one lambda per joint of pilz6) against -expm1(-lambda h) kappa / lambda,
    to 1e-12 relative: 1 - exp(-lambda h) would lose ~8e-4 of the gain at lambda = 1e-12."""
    m, _ = build("pilz6")
    fat = np.array(param_rows(m, "het")[0])
    fat[:, 0] = LAMS
    m.set_fatigue(fat)
    orc = Oracle(oracle_model_from_export(m))
    U = 4
    rng = np.random.default_rng(3)
    tau, qd = rng.uniform(-20, 20, (6, U)), rng.uniform(-2, 2, (6, U))
    T = np.ascontiguousarray(rng.uniform(20, 80, (6, U)))
    ref, a, g, P = zoh_ref(fat, T, tau, qd, h)
    gain = orc.fatigue_zoh(np.zeros((6, U)), tau, qd, h) / P
    assert (np.abs(gain - g) <= 1e-12 * np.abs(g)).all(), np.abs(gain / g - 1).max(axis=1)
    decay = orc.fatigue_zoh(T, np.zeros((6, U)), np.zeros((6, U)), h) / T
    assert (np.abs(decay - a) <= 1e-15).all()
    assert (np.abs(orc.fatigue_zoh(T, tau, qd, h) - ref) <= 1e-12 * np.abs(ref)).all()
    # continuity into the lambda = 0 branch: the gain approaches h kappa
    assert (np.abs(g[1:4] / (h * fat[1:4, 1:2]) - 1) < 1e-8).all()


# ================================================================================================================ GPU helpers
def _dev(a):
    import torch
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(ts):
    return [None if t is None else t.cpu().numpy() for t in ts]


def _case(name, pset, U, seed):
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m, om = build(name, pset)
    x = random_inputs(om, U, seed=seed)
    return m, om, BatchEvaluator(m), x, [_dev(a) for a in x]


def _check_step_jac(gj, rj, n, what):
    for r0 in (0, n, 2 * n):
        e = rel_err_rows(gj[r0:r0 + n], rj[r0:r0 + n])
        assert e < TOL, (what, r0, e)
    # structure: d(q+, qd+)/df == 0 exactly, d f+/d f diagonal
    assert not gj[:2 * n, 3 * n:4 * n].any(), what
    assert not (gj[2 * n:, 3 * n:4 * n] * (1 - np.eye(n))[:, :, None]).any(), what


# ================================================================================================================ GPU: the step
@pytest.mark.gpu
@pytest.mark.parametrize("pset", STEP_SETS)
@pytest.mark.parametrize("name", list(MODELS))
def test_step_and_rollout(name, pset):
    import torch
    U = _units(name)
    m, om, ev, x, d = _case(name, pset, U, seed=31)
    q, qd, tau, f, _ = x
    orc = Oracle(om, fast=True)
    for got, ref in zip(_host(ev.step_rk4(*d[:4], DT)), orc.step_rk4(q, qd, tau, f, DT)):
        assert rel_err_rows(got, ref) < TOL, (name, pset)
    dt_u = np.ascontiguousarray(np.random.default_rng(32).uniform(0.25 * DT, DT, U))
    for got, ref in zip(_host(ev.step_rk4(*d[:4], _dev(dt_u))), orc.step_rk4(q, qd, tau, f, 0.0, dt_u=dt_u)):
        assert rel_err_rows(got, ref) < TOL, (name, pset, "per-unit dt")
    # rollout over N = 5 nodes == 5 chained oracle steps
    n, B, N = m.n, 9, 5
    rng = np.random.default_rng(33)
    x0 = [np.ascontiguousarray(a[:, :B]) for a in (q, 0.3 * qd, f)]
    taus = np.ascontiguousarray(np.tile(tau[:, :B], (1, N)) * rng.uniform(0.5, 1.0, (n, N * B)))
    traj = _host(ev.rollout_rk4(*[_dev(a) for a in x0], _dev(taus), N, DT))
    xr = tuple(x0)
    for k in range(N):
        xr = orc.step_rk4(xr[0], xr[1], np.ascontiguousarray(taus[:, k * B:(k + 1) * B]), xr[2], DT)
        for got, ref in zip(traj, xr):
            assert rel_err_rows(got[:, k * B:(k + 1) * B], ref) < 1e-8, (name, pset, k)  # N steps of error growth
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("pset", STEP_SETS)
@pytest.mark.parametrize("name", list(MODELS))
def test_step_jacobian_and_vjp(name, pset, monkeypatch):
    """step_rk4_jvp through the workspace pipeline, the dual-number sweeps and (run-time trees) the DFMA chain kernel, every plane
    including the fatigue and dt columns; step_rk4_vjp against lambda^T J of the oracle, with a per-unit dt."""
    U = _units(name)
    m, om, ev, x, d = _case(name, pset, U, seed=41)
    n = m.n
    orc = Oracle(om, fast=True)
    rq, rqd, rf, rj = orc.step_rk4_jvp(*x[:4], DT)
    paths = [("workspace", False, None), ("direct", True, None)]
    if m.kernel_family.startswith("generic"):
        paths.append(("scalar tree chain", False, "scalar"))
    for what, direct, env in paths:
        if env:
            monkeypatch.setenv("MPCF_TREE_CHAIN", env)
        gq, gqd, gf, gj = _host(ev.step_rk4_jvp(*d[:4], DT, direct=direct))
        monkeypatch.delenv("MPCF_TREE_CHAIN", raising=False)
        assert rel_err_rows(gq, rq) < TOL and rel_err_rows(gqd, rqd) < TOL and rel_err_rows(gf, rf) < TOL, (name, pset, what)
        _check_step_jac(gj, rj, n, (name, pset, what))
    # reverse mode, per-unit dt
    dt_u = np.ascontiguousarray(np.random.default_rng(42).uniform(0.25 * DT, DT, U))
    J = orc.step_rk4_jvp(*x[:4], 0.0, dt_u=dt_u)[3]
    _check_step_jac(_host(ev.step_rk4_jvp(*d[:4], _dev(dt_u)))[3], J, n, (name, pset, "per-unit dt"))
    lam = np.random.default_rng(43).standard_normal((3 * n, U))
    dl = [_dev(lam[i * n:(i + 1) * n]) for i in range(3)]
    g = _host(ev.step_rk4_vjp(*d[:4], _dev(dt_u), *dl, want_dt=True))
    got = np.vstack(g[:4] + [g[4][None]])
    assert_vjp_close(got, vjp_ref(J, lam), vjp_scale(J, lam), TOL, (name, pset, "vjp"))


@pytest.mark.gpu
@pytest.mark.parametrize("pset", ["het", "stiff"])
@pytest.mark.parametrize("name", list(MODELS))
def test_rollout_vjp(name, pset):
    m, om, ev, x, d = _case(name, pset, 4 * 5, seed=51)
    n, B, N = m.n, 4, 5
    q, qd, tau, f, _ = x
    x0 = [np.ascontiguousarray(a[:, :B]) for a in (q, 0.3 * qd, f)]
    dev = [_dev(a) for a in x0] + [d[2]]
    traj = ev.rollout_rk4(*dev, N, DT)
    G = np.random.default_rng(52).standard_normal((3 * n, N * B))
    got = _host(ev.rollout_rk4_vjp(*dev, N, DT, traj, *[_dev(G[i * n:(i + 1) * n]) for i in range(3)]))
    T = np.vstack(_host(traj))
    X = np.hstack([np.vstack(x0), T[:, :(N - 1) * B]])
    gtau, gx0 = rollout_adjoint_ref(Oracle(om, fast=True), X, tau, N, B, DT, G)
    assert rel_err_rows(got[0], gtau) < TOL, (name, pset)
    for i in range(3):
        assert rel_err_rows(got[1 + i], gx0[i * n:(i + 1) * n]) < TOL, (name, pset, i)


# ================================================================================================================ GPU: second order
HESS_MODELS = ["pilz3", "pilz6", "chain7", "pilz6x2", "dual_arm14", "chain10", "mixed", "humanoid37", "chain48"]


@pytest.mark.gpu
@pytest.mark.parametrize("pset", ["het", "stiff"])
@pytest.mark.parametrize("name", HESS_MODELS)
def test_hessian_and_hvp(name, pset):
    """H[f][dt] = lf lambda amp'(lambda h) at z of order 1, and every other entry, against the hyper-dual oracle"""
    from test_hess import _raw_hess, _raw_hvp
    big = name in ("humanoid37", "chain48")
    U = 3 if big else 33
    m, om, ev, x, d = _case(name, pset, U, seed=61)
    n, P = m.n, 4 * m.n + 1
    orc = Oracle(om, fast=True)
    rng = np.random.default_rng(62)
    lam, v = rng.standard_normal((3 * n, U)), rng.standard_normal((P, U))
    ls = [np.ascontiguousarray(lam[i * n:(i + 1) * n]) for i in range(3)]
    dl = [_dev(a) for a in ls]
    dt_u = np.ascontiguousarray(rng.uniform(0.25 * DT, DT, U))
    if name != "chain48":  # the dense oracle sweeps P (P + 1) / 2 pairs per unit
        for dt, du in ((DT, None), (0.0, dt_u)):
            H = _raw_hess(m, d[:4], dt, _dev(du), dl).cpu().numpy()
            ref = oracle_hess(orc, *x[:4], dt, *ls, dt_u=du)
            assert rel_err_rows(H.reshape(P * P, U), ref.reshape(P * P, U)) < TOL, (name, pset, du is not None)
    vs = [np.ascontiguousarray(v[i * n:(i + 1) * n]) for i in range(4)] + [np.ascontiguousarray(v[4 * n])]
    out = _host(_raw_hvp(m, d[:4], 0.0, _dev(dt_u), dl, [_dev(a) for a in vs]))
    rh, rj = oracle_hvp(orc, *x[:4], 0.0, ls, vs, dt_u=dt_u)
    assert rel_err_rows(np.vstack(out[:4] + [out[4][None]]), np.vstack(list(rh[:4]) + [rh[4][None]])) < TOL, (name, pset, "hvp")
    assert rel_err_rows(np.vstack(out[5:]), np.vstack(rj)) < TOL, (name, pset, "jv")
    if name != "chain48":
        H = _raw_hess(m, d[:4], 0.0, _dev(dt_u), dl).cpu().numpy()
        _assert_scaled(np.vstack(out[:4] + [out[4][None]]), *_hv(H, v), 1e-12, (name, pset, "H v"))


# ================================================================================================================ GPU: coupled fatigue
@pytest.mark.gpu
@pytest.mark.parametrize("pset", ["het", "stiff"])
@pytest.mark.parametrize("name", ["pilz6x2", "dual_arm14"])
def test_coupled_step_and_jacobian(name, pset):
    from mpc_fatigue_b200.coupling import box_load_coupling
    U = 97
    m, om, ev, x, d = _case(name, pset, U, seed=71)
    n, P = m.n, 4 * m.n + 1
    cpl = box_load_coupling(m)
    m.set_coupling(cpl)
    orc = Oracle(om, fast=True)
    for dt, du in ((DT, None), (0.0, np.ascontiguousarray(np.random.default_rng(72).uniform(0.25 * DT, DT, U)))):
        dtg = dt if du is None else _dev(du)
        rq, rqd, rf, rj = orc.step_rk4_coupled(cpl[:2], cpl[2], *x[:4], dt, dt_u=du, jac=True)
        for got, ref in zip(_host(ev.step_rk4(*d[:4], dtg)), (rq, rqd, rf)):
            assert rel_err_rows(got, ref) < TOL, (name, pset)
        got = _host(ev.step_rk4_jvp(*d[:4], dtg))
        for g, r in zip(got[:3], (rq, rqd, rf)):
            assert rel_err_rows(g, r) < TOL, (name, pset)
        assert rel_err_rows(got[3].reshape(3 * n * P, U), rj.reshape(3 * n * P, U)) < TOL, (name, pset, du is not None)


# ================================================================================================================ GPU: node rows
# (case, model, end-effector frames): static one- and two-arm families and run-time trees
ROW_CASES = [("pilz6", "pilz6", None), ("pilz6x2", "pilz6x2", ["end_effector", "sec_end_effector"]),
             ("humanoid37_one", "humanoid37", ["larm_ee"]), ("humanoid37_two", "humanoid37", ["larm_ee", "rarm_ee"]),
             ("mixed", "mixed", ["tip"])]


def _frames(m, frames):
    if frames is None:
        fpar = m.export("fparent").tolist()
        return [max(i for i, p in enumerate(fpar) if p == m.n - 1)]
    return [m.frame_id(f) for f in frames]


@pytest.mark.gpu
@pytest.mark.parametrize("pset", ["het", "F0", "mixed0", "tiny"])
@pytest.mark.parametrize("case,name,frames", ROW_CASES, ids=[c[0] for c in ROW_CASES])
def test_node_eval_and_ocp_rows(case, name, frames, pset):
    """node_eval_ref (T+ by the host's ZOH factors) and ocp_rows (T rows, dF and dT blocks) against the oracle and, for the
    zero-order hold, against the numpy expm1 restatement: the increment T+ - a T and dT+/dtau = g 2 c_tau tau carry the gain's
    relative error undiluted by T."""
    from test_ocp_rows_tree import KW, OPTS1, OPTS2
    from test_ocp_rows_tree import _inputs as rows_inputs
    B, N = 33, 3
    U = B * N
    m, om, ev, x, d = _case(name, pset, U, seed=81)
    n = m.n
    fat = np.array(om.fat)
    orc = Oracle(om, fast=True)
    ee = _frames(m, frames)
    narm = len(ee)
    q, qd, _, T, qdd = x
    W = np.ascontiguousarray(np.random.default_rng(82).uniform(-50, 50, (6 * narm, U)))
    for h in (2.0 / 60.0, 0.5):
        for Tin in (T, np.zeros_like(T)):
            for wsign in (-1.0, 1.0):
                rt, rq, rT = orc.node_eval_ref(ee, wsign, q, qd, W, Tin, h, qdd=qdd)
                gt, gq, gT = _host(ev.node_eval_ref(ee, wsign, d[0], d[1], _dev(W), _dev(Tin), h, qdd=d[4]))
                assert rel_err_rows(gt, rt) < TOL and rel_err_rows(gq, rq) < TOL and rel_err_rows(gT, rT) < TOL, (case, pset, h)
                ref, a, g, P = zoh_ref(fat, Tin, rt, qd, h)
                assert rel_err_rows(gT - a * Tin, g * P) < TOL, (case, pset, h, "ZOH increment")
    # fused OCP rows with the thermal rows and their derivative blocks
    q, qd, F, T, q_last, T_last, rp0, ro0 = rows_inputs(om, B, N, narm, seed=83)
    two = narm == 2
    opts = dict(OPTS2 if two else OPTS1, narm=narm, ee_frame=ee, h=2.0 / 60.0)
    rrows, rcost, rJ = orc.ocp_rows(opts, B, N, q, qd, F, T, q_last, T_last, rp0 if two else None, ro0 if two else None, kin_jac=True)
    rows, cost, dF, dT, kj = _host(ev.ocp_rows(B, N, ee, _dev(q), _dev(qd), _dev(F), _dev(T), _dev(q_last), _dev(T_last),
                                               _dev(rp0) if two else None, _dev(ro0) if two else None, derivatives=True,
                                               **{k: opts[k] for k in KW}))
    kin = 26 if two else 3
    assert rel_err_rows(rows, rrows) < TOL, (case, pset)
    assert np.abs(cost - rcost).max() <= TOL * max(1.0, np.abs(rcost).max())
    assert rel_err_rows(kj.reshape(-1, U), rJ.reshape(-1, U)) < TOL
    for c in range(narm):
        J = orc.jacobian(ee[c], q).reshape(6, n, U)
        assert rel_err_rows(dF[:, 3 * c:3 * c + 3].reshape(-1, U), (opts["wsign"] * J[:3].transpose(1, 0, 2)).reshape(-1, U)) < TOL, c
    tau = rrows[kin:kin + n]
    _, _, g, _ = zoh_ref(fat, T, tau, qd, opts["h"])
    assert rel_err_rows(dT, g * 2.0 * fat[:, 2:3] * tau) < TOL, (case, pset, "dT+/dtau")


# ================================================================================================================ GPU: dynamics
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_dynamics_under_per_joint_armature(name):
    """rnea, aba, rnea_derivs (the diagonal of M carries the armature) and fd_derivs"""
    m, om, ev, x, d = _case(name, "het", _units(name), seed=91)
    orc = Oracle(om, fast=True)
    q, qd, tau, f, qdd = x
    assert rel_err_rows(ev.rnea(d[0], d[1], d[4]).cpu().numpy(), orc.rnea(q, qd, qdd)) < TOL
    assert rel_err_rows(ev.aba(d[0], d[1], d[2]).cpu().numpy(), orc.aba(q, qd, tau)) < TOL
    U = 40
    sl = [np.ascontiguousarray(a[:, :U]) for a in x]
    ds = [t[:, :U].contiguous() for t in d]
    # M = d tau / d qdd carries the armature on its diagonal: every plane to TOL.  d tau / d (q, qd) do not depend on the armature;
    # their structurally zero planes hold rounding noise of O(max) terms in both implementations, hence the floor of fd_derivs
    (gDq, gDv, gM), (rDq, rDv, rM) = _host(ev.rnea_derivs(ds[0], ds[1], ds[4])), orc.rnea_derivs(sl[0], sl[1], sl[4])
    assert rel_err_rows(gM, rM) < TOL, name
    n = m.n
    crba = orc.crba(sl[0][:, 0].copy())  # the joint-space inertia, armature on the diagonal
    assert np.abs(gM[:, 0].reshape(n, n) - crba).max() <= TOL * np.abs(crba).max(), name
    assert rel_err_rows(gDq, rDq, floor=1e-4) < TOL and rel_err_rows(gDv, rDv, floor=1e-4) < TOL, name
    # A, B, C = d qdd / d (q, qd, tau) scaled together: a decoupled joint's structurally zero planes of B hold ~1e-15 rounding noise
    # in both implementations, which an absolute floor would compare at 1e-9.  As test_gpu_parity.test_fd_derivs, cross-limb planes
    # of the large trees are conditioning-limited.
    fl = 1e-4 if m.n > 16 else 1e-6
    got, ref = np.vstack(_host(ev.fd_derivs(ds[0], ds[1], ds[2]))), np.vstack(orc.fd_derivs(sl[0], sl[1], sl[2]))
    assert rel_err_rows(got, ref, floor=fl) < TOL, name


# ================================================================================================================ GPU: changed after use
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz6", "dual_arm14", "humanoid37"])
def test_parameters_changed_after_first_use(name):
    """A model already used must see new rows on the next call through the same evaluator (static families rebuild their
    grid-constant parameters, run-time trees re-upload their blob), and restoring the old rows must restore the old results bit
    for bit."""
    import torch
    U = _units(name)
    m, om0, ev, x, d = _case(name, None, U, seed=101)
    first = [t.clone() for t in ev.step_rk4_jvp(*d[:4], DT)]
    torch.cuda.synchronize()
    old_fat, old_arm = m.export("fat"), m.export("arm")
    fat, arm = param_rows(m, "stiff")
    m.set_fatigue(fat)
    m.set_armature(arm)
    orc = Oracle(oracle_model_from_export(m), fast=True)
    rq, rqd, rf, rj = orc.step_rk4_jvp(*x[:4], DT)
    for direct in (False, True):
        gq, gqd, gf, gj = _host(ev.step_rk4_jvp(*d[:4], DT, direct=direct))
        assert rel_err_rows(gq, rq) < TOL and rel_err_rows(gqd, rqd) < TOL and rel_err_rows(gf, rf) < TOL, (name, direct)
        _check_step_jac(gj, rj, m.n, (name, direct))
    assert rel_err_rows(ev.aba(d[0], d[1], d[2]).cpu().numpy(), orc.aba(*[x[i] for i in (0, 1, 2)])) < TOL
    m.set_fatigue(old_fat)
    m.set_armature(old_arm)
    again = ev.step_rk4_jvp(*d[:4], DT)
    torch.cuda.synchronize()
    for a, b in zip(again, first):
        assert torch.equal(a, b), name
