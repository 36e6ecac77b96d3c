"""Reverse mode: the vector-Jacobian product of the RK4 step (mpcf_step_rk4_vjp_batch), the adjoint of the single-shooting rollout
(mpcf_rollout_rk4_vjp_batch) and their PyTorch autograd wrappers (mpc_fatigue_b200/autograd.py).

The CPU test pins the reverse sweep of DESIGN.md §4d in numpy, built from oracle pieces (ABA, fatigue right-hand side, forward-
dynamics derivatives), against lambda^T J of the oracle's complex-step Jacobian, and the rollout recursion against central
differences.  The GPU tests check every kernel path against the oracle, the library's own dense pipelines, argument handling,
workspace chunking and buffer bounds."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT, oracle_model_from_export, random_inputs, rel_err_rows
from mpc_fatigue_b200.model import Model, data_urdf
from oracle.pyoracle import Oracle

TOL = 1e-9
CW = (0.5, 0.5, 1.0)
WW = (1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0)

MODELS = {
    "pilz3": lambda: Model.from_urdf(data_urdf("pilz3"), armature=1e-2),
    "pilz6": lambda: Model.from_urdf(data_urdf("pilz6"), armature=1e-2),
    "chain7": lambda: Model.synthetic("chain", 7, seed=2, armature=1e-2),
    "pilz6x2": lambda: Model.from_urdf(data_urdf("pilz6x2"), armature=1e-2),
    "dual_arm14": lambda: Model.synthetic("dual_arm", 14, seed=3, armature=1e-2),
    "mixed": lambda: Model.from_urdf(open(os.path.join(ROOT, "tests", "golden", "mixed_joints.urdf")).read(), armature=1e-3),
    "dual_arm10": lambda: Model.synthetic("dual_arm", 10, seed=3, armature=1e-2),
    "chain9": lambda: Model.synthetic("chain", 9, seed=4, armature=1e-2),
    "humanoid37": lambda: Model.synthetic("humanoid", 37, seed=7, armature=1e-2),
    "chain48": lambda: Model.synthetic("chain", 48, seed=5, armature=1e-2),
}
FAMILY = {"pilz3": "chain3", "pilz6": "chain6", "chain7": "chain7", "pilz6x2": "forest12x6", "dual_arm14": "forest14x7",
          "mixed": "generic16", "dual_arm10": "generic16", "chain9": "generic16", "humanoid37": "generic64", "chain48": "generic64"}


# ---------------------------------------------------------------------------------------------------------------- references
def vjp_ref(jac, lam):
    """lambda^T J per unit: jac [3n, 4n+1, U], lam [3n, U] -> [4n+1, U]."""
    return np.einsum("ru,rcu->cu", lam, jac)


def vjp_scale(jac, lam):
    """S = sum_r |lambda_r| |J_rc|: the condition scale of the sum lambda^T J, per output entry."""
    return np.einsum("ru,rcu->cu", np.abs(lam), np.abs(jac))


def assert_vjp_close(g, ref, S, tol=TOL, what=""):
    """|g - ref| <= tol * max(S, 1e-6 max S) for every entry."""
    bound = tol * np.maximum(S, 1e-6 * max(S.max(), 1e-300))
    err = np.abs(g - ref)
    assert (err <= bound).all(), (what, float((err / np.maximum(bound, 1e-300)).max()))


def numpy_step_vjp(orc, om, q, qd, tau, f, h, lam):
    """The reverse sweep of DESIGN.md §4d from oracle pieces: stage states by ABA and the fatigue rows, A_s, B_s, C_s by the
    oracle's forward-dynamics derivatives.  h: [U] array.  Returns (g_x [3n, U], g_tau [n, U], g_h [U])."""
    n, U = q.shape
    fat = np.array(om.fat)
    lamb, kap, ctau, cv = (fat[:, k][:, None] for k in range(4))
    x = np.vstack([q, qd, f])
    xs, st = x.copy(), []
    for s in range(4):
        qs, vs, fs = xs[:n], xs[n:2 * n], xs[2 * n:]
        qdd = orc.aba(np.ascontiguousarray(qs), np.ascontiguousarray(vs), tau)
        fd = orc.fatigue_rhs(np.ascontiguousarray(fs), tau, np.ascontiguousarray(vs))
        A, B, Cm = (M.reshape(n, n, U) for M in orc.fd_derivs(np.ascontiguousarray(qs), np.ascontiguousarray(vs), tau))
        k = np.vstack([vs, qdd, fd])
        st.append((vs, k, A, B, Cm))
        if s < 3:
            xs = x + CW[s] * h * k
    gx, gt, gh = lam.copy(), np.zeros((n, U)), np.zeros(U)
    a = np.zeros((3 * n, U))
    for s in range(3, -1, -1):
        vs, k, A, B, Cm = st[s]
        rho = WW[s] * lam + (CW[s] * a if s < 3 else 0.0)
        gh += (rho * k).sum(0)
        r = h * rho
        rq, rv, rf = r[:n], r[n:2 * n], r[2 * n:]
        a = np.vstack([np.einsum("rcu,ru->cu", A, rv), rq + np.einsum("rcu,ru->cu", B, rv) + 2 * kap * cv * vs * rf, -lamb * rf])
        gt += np.einsum("cru,ru->cu", Cm, rv) + 2 * kap * ctau * tau * rf
        gx += a
    return gx, gt, gh


def xcols(n):
    return np.r_[0:2 * n, 3 * n:4 * n]


def rollout_adjoint_ref(orc, X, tau, N, B, dt, G):
    """The rollout recursion over oracle step Jacobians evaluated at the given states.  X: [3n, N*B] = (x_0; trajectory entries
    0 .. N-2), tau [n, N*B], G [3n, N*B] = dL/d(trajectory).  Returns (g_tau [n, N*B], g_x0 [3n, B])."""
    n = tau.shape[0]
    gtau = np.zeros((n, N * B))
    lam = G[:, (N - 1) * B:].copy()
    for k in range(N - 1, -1, -1):
        sl = slice(k * B, (k + 1) * B)
        J = orc.step_rk4_jvp(*(np.ascontiguousarray(X[i * n:(i + 1) * n, sl]) for i in (0, 1)), np.ascontiguousarray(tau[:, sl]),
                             np.ascontiguousarray(X[2 * n:, sl]), dt)[3]
        g = vjp_ref(J, lam)
        gtau[:, sl] = g[2 * n:3 * n]
        lam = g[xcols(n)] + (G[:, (k - 1) * B:k * B] if k > 0 else 0.0)
    return gtau, lam


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", ["pilz6", "mixed"])
def test_numpy_reverse_sweep_matches_the_complex_step_jacobian(name):
    m = MODELS[name]()
    om = oracle_model_from_export(m)
    orc = Oracle(om)
    n, U = m.n, 12
    q, qd, tau, f, _ = random_inputs(om, U, seed=11)
    rng = np.random.default_rng(12)
    lam = rng.standard_normal((3 * n, U))
    dt_u = np.ascontiguousarray(rng.uniform(0.0, 0.03, U))
    dt_u[0] = 0.0
    J = orc.step_rk4_jvp(q, qd, tau, f, 0.0, dt_u=dt_u)[3]
    ref, S = vjp_ref(J, lam), vjp_scale(J, lam)
    gx, gt, gh = numpy_step_vjp(orc, om, q, qd, tau, f, dt_u, lam)
    assert_vjp_close(gx, ref[xcols(n)], S[xcols(n)], 1e-12, "g_x")
    assert_vjp_close(gt, ref[2 * n:3 * n], S[2 * n:3 * n], 1e-12, "g_tau")
    assert_vjp_close(gh[None], ref[4 * n:], S[4 * n:], 1e-12, "g_dt")

    # the rollout recursion against central differences of L = sum_k W_k . x_{k+1}
    B, N, dt = 2, 4, 0.02
    q0, qd0, f0 = q[:, :B].copy(), qd[:, :B].copy(), f[:, :B].copy()
    taus = np.ascontiguousarray(random_inputs(om, N * B, seed=13)[2])
    W = rng.standard_normal((3 * n, N * B))

    def roll(q0, qd0, f0, taus):
        x, traj = (q0, qd0, f0), []
        for k in range(N):
            q, qd, f = (np.ascontiguousarray(v) for v in x)
            x = orc.step_rk4(q, qd, np.ascontiguousarray(taus[:, k * B:(k + 1) * B]), f, dt)
            traj.append(np.vstack(x))
        return np.hstack(traj)

    T = roll(q0, qd0, f0, taus)
    X = np.hstack([np.vstack([q0, qd0, f0]), T[:, :(N - 1) * B]])
    gtau, gx0 = rollout_adjoint_ref(orc, X, taus, N, B, dt, W)
    loss = lambda *a: float((roll(*a) * W).sum())
    eps = 1e-6
    for (i, u) in [(0, 0), (n - 1, 1 + (N - 2) * B), (2, N * B - 1)]:
        tp, tm = taus.copy(), taus.copy()
        tp[i, u] += eps
        tm[i, u] -= eps
        fdv = (loss(q0, qd0, f0, tp) - loss(q0, qd0, f0, tm)) / (2 * eps)
        assert abs(fdv - gtau[i, u]) <= 1e-6 * max(1.0, abs(fdv)), (i, u, fdv, gtau[i, u])
    x0 = np.vstack([q0, qd0, f0])
    for r in (0, n + 1, 2 * n + n - 1):
        for b in range(B):
            xp, xm = x0.copy(), x0.copy()
            xp[r, b] += eps
            xm[r, b] -= eps
            fdv = (loss(xp[:n], xp[n:2 * n], xp[2 * n:], taus) - loss(xm[:n], xm[n:2 * n], xm[2 * n:], taus)) / (2 * eps)
            assert abs(fdv - gx0[r, b]) <= 1e-6 * max(1.0, abs(fdv)), (r, b, fdv, gx0[r, b])


# ---------------------------------------------------------------------------------------------------------------- GPU helpers
def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _raw_vjp(m, d, dt, dt_u, lam, states=True, gdt=True, ws=None, ws_bytes=0, out=None):
    """mpcf_step_rk4_vjp_batch with every option; d = (q, qd, tau, f) device tensors, lam = (lq, lqd, lf) (None entries allowed).
    Returns (gq, gqd, gtau, gf, gdt, qn, qdn, fn) as device tensors (None where not requested)."""
    import torch
    from mpc_fatigue_b200 import _capi
    n, U = d[0].shape
    if out is None:
        out = [torch.empty((n, U), dtype=torch.float64, device="cuda") for _ in range(4)]
        out.append(torch.empty(U, dtype=torch.float64, device="cuda") if gdt else None)
        out += [torch.empty((n, U), dtype=torch.float64, device="cuda") if states else None for _ in range(3)]
    _capi.check(_capi.lib.mpcf_step_rk4_vjp_batch(m.handle, U, *[_p(t) for t in d], float(dt), _p(dt_u), *[_p(t) for t in lam],
                                                  *[_p(t) for t in out], _p(ws) if ws is not None else None, ws_bytes, _stream()))
    return out


def _case(name, U, seed, dt=0.0125, dt_u=None):
    import torch
    m = MODELS[name]()
    om = oracle_model_from_export(m)
    q, qd, tau, f, _ = random_inputs(om, U, seed=seed)
    lam = np.random.default_rng(seed + 1).standard_normal((3 * m.n, U))
    d = [torch.from_numpy(a).cuda() for a in (q, qd, tau, f)]
    dl = [torch.from_numpy(np.ascontiguousarray(lam[i * m.n:(i + 1) * m.n])).cuda() for i in range(3)]
    return m, om, (q, qd, tau, f), d, lam, dl


def _check_against_oracle(name, U, seed, dt=0.0125, dt_u=None):
    import torch
    m, om, h, d, lam, dl = _case(name, U, seed)
    assert m.kernel_family == FAMILY[name]
    n = m.n
    rq, rqd, rf, J = Oracle(om, fast=True).step_rk4_jvp(*h, dt, dt_u=dt_u)
    out = _raw_vjp(m, d, dt, None if dt_u is None else torch.from_numpy(dt_u).cuda(), dl)
    torch.cuda.synchronize()
    gq, gqd, gtau, gf, gdt, qn, qdn, fn = [t.cpu().numpy() for t in out]
    ref, S = vjp_ref(J, lam), vjp_scale(J, lam)
    for g, sl, nm in ((gq, slice(0, n), "gq"), (gqd, slice(n, 2 * n), "gqd"), (gtau, slice(2 * n, 3 * n), "gtau"),
                      (gf, slice(3 * n, 4 * n), "gf"), (gdt[None], slice(4 * n, 4 * n + 1), "gdt")):
        assert_vjp_close(g, ref[sl], S[sl], TOL, (name, U, nm))
    assert rel_err_rows(qn, rq) < TOL and rel_err_rows(qdn, rqd) < TOL and rel_err_rows(fn, rf) < TOL
    return m, d, dl, out


# ---------------------------------------------------------------------------------------------------------------- GPU: step
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_step_vjp_matches_the_oracle(name):
    U = 33
    dt_u = np.ascontiguousarray(np.random.default_rng(5).uniform(0.002, 0.02, U))
    _check_against_oracle(name, U, seed=21, dt_u=dt_u)
    _check_against_oracle(name, 31, seed=22, dt=0.0)  # dt = 0: g_x = lambda, g_dt = lambda^T k_avg


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz6", "pilz6x2", "humanoid37", "chain48"])
@pytest.mark.parametrize("U", [1, 257])
def test_step_vjp_ragged_batches(name, U):
    _check_against_oracle(name, U, seed=23 + U)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz3", "pilz6x2", "dual_arm14", "dual_arm10", "humanoid37", "chain48"])
def test_step_vjp_equals_the_contracted_dense_jacobians(name):
    """lambda^T jac of the library's dense analytic pipeline and of its dual-number sweeps, to 1e-11."""
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m, om, h, d, lam, dl = _case(name, 65, seed=31)
    n = m.n
    ev = BatchEvaluator(m)
    g = [t.cpu().numpy() for t in ev.step_rk4_vjp(*d, 0.0125, *dl, want_dt=True)]
    got = np.vstack([g[0], g[1], g[2], g[3], g[4][None]])
    for direct in (False, True):
        J = ev.step_rk4_jvp(*d, 0.0125, direct=direct)[3].cpu().numpy()
        assert_vjp_close(got, vjp_ref(J, lam), vjp_scale(J, lam), 1e-11, (name, "dual" if direct else "analytic"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz6", "pilz6x2", "humanoid37", "chain48"])
def test_null_adjoints_act_as_zeros(name):
    import torch
    m, om, h, d, lam, dl = _case(name, 40, seed=41)
    for k in range(3):
        part = [t if i == k else None for i, t in enumerate(dl)]
        zeros = [t if i == k else torch.zeros_like(t) for i, t in enumerate(dl)]
        a = _raw_vjp(m, d, 0.0125, None, part)
        b = _raw_vjp(m, d, 0.0125, None, zeros)
        torch.cuda.synchronize()
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    # every adjoint NULL: all gradients zero (g_x = 0 + nothing)
    out = _raw_vjp(m, d, 0.0125, None, [None, None, None])
    torch.cuda.synchronize()
    for t in out[:5]:
        assert not bool(t.any())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz6", "pilz6x2"])
def test_small_caller_workspace_chunks_bit_identically(name):
    import torch
    from mpc_fatigue_b200 import _capi
    m, om, h, d, lam, dl = _case(name, 257, seed=51)
    need = int(_capi.lib.mpcf_step_rk4_jvp_workspace_bytes(m.handle, 40))
    full = int(_capi.lib.mpcf_step_rk4_jvp_workspace_bytes(m.handle, 257))
    assert need * 3 < full
    ws = torch.empty(need // 8, dtype=torch.float64, device="cuda")
    wsf = torch.empty(full // 8, dtype=torch.float64, device="cuda")
    a = _raw_vjp(m, d, 0.0125, None, dl, ws=ws, ws_bytes=need)
    b = _raw_vjp(m, d, 0.0125, None, dl, ws=wsf, ws_bytes=full)
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        assert torch.equal(x, y)


CANARY = -7.25e300


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz6", "pilz6x2", "humanoid37", "chain9"])
@pytest.mark.parametrize("U", [1, 33, 131])
def test_canary_gaps_around_outputs_and_workspace(name, U):
    import torch
    from mpc_fatigue_b200 import _capi
    m, om, h, d, lam, dl = _case(name, U, seed=61)
    n, GAP = m.n, 64
    ws_bytes = int(_capi.lib.mpcf_step_rk4_jvp_workspace_bytes(m.handle, U))
    sizes = [n * U] * 4 + [U] + [n * U] * 3 + [ws_bytes // 8]
    total = GAP + sum(s + GAP for s in sizes) + 16
    pool = torch.full((total,), CANARY, dtype=torch.float64, device="cuda")
    views, gaps, off = [], [slice(0, GAP)], GAP
    for i, s in enumerate(sizes):
        if i == len(sizes) - 1:  # the workspace must be 128-byte aligned
            off += (-(pool.data_ptr() + 8 * off)) % 128 // 8
            gaps[-1] = slice(gaps[-1].start, off)
        views.append(pool[off:off + s])
        gaps.append(slice(off + s, off + s + GAP))
        off += s + GAP
    outs = [v.view(n, U) for v in views[:4]] + [views[4]] + [v.view(n, U) for v in views[5:8]]
    _raw_vjp(m, d, 0.0125, None, dl, out=outs, ws=views[8] if ws_bytes else None, ws_bytes=ws_bytes)
    torch.cuda.synchronize()
    for i, g in enumerate(gaps):
        assert bool((pool[g] == CANARY).all()), (name, U, "canary gap %d was written" % i)
    for i, v in enumerate(views[:8]):
        assert not bool((v == CANARY).any()), (name, U, i, "has unwritten elements")


@pytest.mark.gpu
def test_invalid_arguments():
    import torch
    from mpc_fatigue_b200 import _capi
    m, om, h, d, lam, dl = _case("pilz6", 40, seed=71)
    out = _raw_vjp(m, d, 0.0125, None, dl)
    torch.cuda.synchronize()
    st = _stream()

    def call(model=m, q=d[0], gq=out[0], ws=None, ws_bytes=0):
        return _capi.lib.mpcf_step_rk4_vjp_batch(model.handle, 40, _p(q), *[_p(t) for t in d[1:]], 0.0125, None, *[_p(t) for t in dl],
                                                 _p(gq), *[_p(t) for t in out[1:]], ws, ws_bytes, st)
    assert call(q=None) == _capi.EINVAL
    assert call(gq=None) == _capi.EINVAL
    need = int(_capi.lib.mpcf_step_rk4_jvp_workspace_bytes(m.handle, 40))
    ws = torch.empty(need // 8 + 16, dtype=torch.float64, device="cuda")
    assert call(ws=C.c_void_p(ws.data_ptr() + 8), ws_bytes=need) == _capi.EINVAL
    assert call(ws=C.c_void_p(ws.data_ptr()), ws_bytes=1024) == _capi.EINVAL
    assert _capi.lib.mpcf_step_rk4_vjp_batch(m.handle, -1, *[None] * 4, 0.0, None, *[None] * 11, None, 0, st) == _capi.EINVAL
    # coupled fatigue is refused by both entries
    mc = MODELS["pilz6x2"]()
    fpar = mc.export("fparent")
    mc.set_coupling((int(np.flatnonzero((fpar >= 0) & (fpar < 6))[-1]), int(np.flatnonzero(fpar >= 6)[-1]), 30 * 9.81))
    z = torch.zeros((12, 8), dtype=torch.float64, device="cuda")
    zz = [torch.zeros_like(z) for _ in range(9)]
    assert _capi.lib.mpcf_step_rk4_vjp_batch(mc.handle, 8, *[_p(z)] * 4, 0.01, None, *[_p(z)] * 3, *[_p(t) for t in zz[:4]], None,
                                             None, None, None, None, 0, st) == _capi.EINVAL
    assert _capi.lib.mpcf_rollout_rk4_vjp_batch(mc.handle, 8, 1, *[_p(z)] * 4, 0.01, *[_p(z)] * 3, None, None, None, _p(zz[4]),
                                                *[_p(t) for t in zz[5:8]], None, 0, st) == _capi.EINVAL
    # N <= 0
    zt = torch.zeros((6, 40), dtype=torch.float64, device="cuda")
    for N in (0, -1):
        assert _capi.lib.mpcf_rollout_rk4_vjp_batch(m.handle, 40, N, *[_p(zt)] * 4, 0.01, *[_p(zt)] * 3, None, None, None, _p(zt),
                                                    *[_p(zt)] * 3, None, 0, st) == _capi.EINVAL
    assert _capi.lib.mpcf_rollout_rk4_vjp_batch(m.handle, 40, 1, *[_p(zt)] * 4, 0.01, *[_p(zt)] * 3, None, None, None, None,
                                                *[_p(zt)] * 3, None, 0, st) == _capi.EINVAL


# ---------------------------------------------------------------------------------------------------------------- GPU: rollout
def _rollout_case(name, B, N, seed, which=None, dt=0.005):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m = MODELS[name]()
    om = oracle_model_from_export(m)
    n = m.n
    q0, qd0, _, f0, _ = random_inputs(om, B, seed=seed)
    tau = random_inputs(om, N * B, seed=seed + 1)[2]
    G = np.random.default_rng(seed + 2).standard_normal((3 * n, N * B))
    if which is not None:  # a loss on only one of q, qd, f
        G[np.r_[0:3 * n] // n != which] = 0.0
    ev = BatchEvaluator(m)
    dev = [torch.from_numpy(a).cuda() for a in (q0, qd0, f0, tau)]
    traj = ev.rollout_rk4(*dev, N, dt)
    gd = [None if which is not None and i != which else torch.from_numpy(np.ascontiguousarray(G[i * n:(i + 1) * n])).cuda()
          for i in range(3)]
    got = [t.cpu().numpy() for t in ev.rollout_rk4_vjp(*dev, N, dt, traj, *gd)]
    T = np.vstack([t.cpu().numpy() for t in traj])
    X = np.hstack([np.vstack([q0, qd0, f0]), T[:, :(N - 1) * B]])
    ref = rollout_adjoint_ref(Oracle(om, fast=True), X, tau, N, B, dt, G)
    return m, got, ref


@pytest.mark.gpu
@pytest.mark.parametrize("name,B,N,which", [("pilz6", 64, 20, None), ("pilz6", 33, 7, 2), ("pilz6x2", 17, 12, None), ("pilz6x2", 9, 5, 1),
                                            ("humanoid37", 16, 8, None), ("humanoid37", 5, 6, 0), ("chain48", 8, 4, None), ("pilz3", 3, 1, None)])
def test_rollout_adjoint_matches_the_oracle_recursion(name, B, N, which):
    m, got, (gtau, gx0) = _rollout_case(name, B, N, seed=81 + B, which=which)
    n = m.n
    assert all(np.isfinite(g).all() for g in got)
    assert rel_err_rows(got[0], gtau) < TOL
    for i in range(3):
        assert rel_err_rows(got[1 + i], gx0[i * n:(i + 1) * n]) < TOL, i


@pytest.mark.gpu
def test_rollout_adjoint_full_size_samples():
    """B = 65,536 scenarios x N = 100 nodes on pilz6; 64 sampled scenarios against the oracle recursion at the GPU states."""
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m = MODELS["pilz6"]()
    om = oracle_model_from_export(m)
    n, B, N, dt = 6, 65536, 100, 0.005
    q0, qd0, _, f0, _ = random_inputs(om, B, seed=91)
    tau = random_inputs(om, N * B, seed=92)[2]
    ev = BatchEvaluator(m)
    dev = [torch.from_numpy(a).cuda() for a in (q0, qd0, f0, tau)]
    traj = ev.rollout_rk4(*dev, N, dt)
    gen = torch.Generator(device="cuda").manual_seed(93)
    gd = [torch.randn((n, N * B), dtype=torch.float64, device="cuda", generator=gen) for _ in range(3)]
    gtau, gq0, gqd0, gf0 = ev.rollout_rk4_vjp(*dev, N, dt, traj, *gd)
    torch.cuda.synchronize()
    sc = np.sort(np.random.default_rng(94).choice(B, 64, replace=False))
    cols = (np.arange(N)[:, None] * B + sc[None, :]).reshape(-1)  # node-major columns of the sample
    colst = torch.from_numpy(cols).cuda()
    pick = lambda t: t[:, colst].cpu().numpy()
    T = np.vstack([pick(t) for t in traj])
    x0 = np.vstack([a[:, sc] for a in (q0, qd0, f0)])
    X = np.hstack([x0, T[:, :(N - 1) * 64]])
    G = np.vstack([pick(t) for t in gd])
    rg, rx = rollout_adjoint_ref(Oracle(om, fast=True), X, np.ascontiguousarray(tau[:, cols]), N, 64, dt, G)
    assert rel_err_rows(pick(gtau), rg) < TOL
    scc = torch.from_numpy(sc).cuda()
    for i, g in enumerate((gq0, gqd0, gf0)):
        assert rel_err_rows(g[:, scc].cpu().numpy(), rx[i * n:(i + 1) * n]) < TOL, i


# ---------------------------------------------------------------------------------------------------------------- GPU: autograd
@pytest.mark.gpu
def test_autograd_gradcheck():
    import torch
    from mpc_fatigue_b200 import autograd as mad
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m = MODELS["pilz3"]()
    om = oracle_model_from_export(m)
    ev = BatchEvaluator(m)
    q, qd, tau, f, _ = random_inputs(om, 4, seed=101)
    leaf = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda().requires_grad_()
    dt = leaf(np.random.default_rng(102).uniform(0.005, 0.02, 4))
    args = [leaf(a) for a in (q, qd, tau, f)]
    assert torch.autograd.gradcheck(lambda *x: mad.step_rk4(ev, *x), (*args, dt), eps=1e-6, atol=1e-7, rtol=1e-6)
    q0, qd0, _, f0, _ = random_inputs(om, 2, seed=103)
    taus = random_inputs(om, 6, seed=104)[2]
    rargs = [leaf(a) for a in (q0, qd0, f0, taus)]
    assert torch.autograd.gradcheck(lambda *x: mad.rollout_rk4(ev, *x, 3, 0.02), tuple(rargs), eps=1e-6, atol=1e-7, rtol=1e-6)


@pytest.mark.gpu
def test_autograd_backward_equals_the_rollout_adjoint():
    import torch
    from mpc_fatigue_b200 import autograd as mad
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m = MODELS["pilz6"]()
    om = oracle_model_from_export(m)
    ev = BatchEvaluator(m)
    B, N, dt = 32, 10, 0.02
    q0, qd0, _, f0, _ = random_inputs(om, B, seed=111)
    tau = random_inputs(om, N * B, seed=112)[2]
    leaves = [torch.from_numpy(a).cuda().requires_grad_() for a in (q0, qd0, f0, tau)]
    qt, qdt, ft = mad.rollout_rk4(ev, *leaves, N, dt)
    loss = (qt[:, -B:] ** 2).sum() + 0.5 * (ft ** 2).sum()  # qdt unused: its gradient reaches the backward as zeros or None
    loss.backward()
    traj = tuple(t.detach() for t in (qt, qdt, ft))
    gtau, gq0, gqd0, gf0 = ev.rollout_rk4_vjp(*[t.detach() for t in leaves], N, dt, traj,
                                              torch.cat([torch.zeros_like(qt[:, :-B]), 2 * qt[:, -B:]], 1).detach().contiguous(),
                                              None, ft.detach().clone())
    for a, b in zip((leaves[0].grad, leaves[1].grad, leaves[2].grad, leaves[3].grad), (gq0, gqd0, gf0, gtau)):
        assert torch.allclose(a, b, rtol=1e-12, atol=1e-12 * float(b.abs().max()))
