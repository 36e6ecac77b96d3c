"""Riccati solve of the multiple-shooting LQ subproblem (mpcf_riccati_batch, BatchEvaluator.riccati).

Per scenario: min sum_k 1/2 z_k^T W_k z_k + g_k^T z_k + 1/2 dx_N^T W_N dx_N + g_N^T dx_N, z_k = (dx_k, du_k), subject to dx_0 = dx0 and
dx_{k+1} = A_k dx_k + B_k du_k + d_k; lambda are the multipliers of L = obj - lambda_0^T (dx_0 - dx0) - sum lambda_{k+1}^T (dx_{k+1} - A_k dx_k
- B_k du_k - d_k).  This file holds its own references: a numpy Riccati recursion (costates from P_k dx_k + p_k) and the KKT system
of the whole horizon, assembled block by block and solved directly.  The CPU tests pin the first to the second; the GPU tests
check the kernel against the direct solve, the KKT residual of the kernel's own solution, NULL handling, chunking, buffer bounds,
the NaN rule and argument rejection."""
import ctypes as C
import os

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from conftest import ROOT, rel_err_rows
from mpc_fatigue_b200.model import Model, data_urdf

# ------------------------------------------------------------------------------------------------ problem, layouts, references
# A problem is a dict of per-scenario arrays: A [S,N,nx,nx], Bm [S,N,nx,nu], Q [S,N,nx,nx], Sm [S,N,nu,nx], R [S,N,nu,nu], gx [S,N,nx],
# gu [S,N,nu], d [S,N,nx], WN [S,nx,nx], gN [S,nx], dx0 [S,nx].  Solutions: dx [S,N+1,nx], du [S,N,nu], lam [S,N+1,nx].


def xcols(n):
    """columns of the state x = (q, qd, f) in z = (q, qd, tau, f, dt)"""
    return np.r_[0:2 * n, 3 * n:4 * n]


def ucols(n):
    return np.arange(2 * n, 3 * n)


def random_problem(n, N, S, seed, eps=0.1):
    """Well-posed data: every [Q S^T; S R] and W_N is a Gram matrix plus eps I; S != 0, nonzero d, dx0 and gradients."""
    rng = np.random.default_rng(seed)
    nx, nu = 3 * n, n
    nz = nx + nu
    G = rng.standard_normal((S, N, nz, nz)) / np.sqrt(nz)
    W = np.einsum("sknz,sknw->skzw", G, G) + eps * np.eye(nz)
    GN = rng.standard_normal((S, nx, nx)) / np.sqrt(nx)
    return dict(A=0.5 * np.eye(nx) + 0.5 * rng.standard_normal((S, N, nx, nx)) / np.sqrt(nx),
                Bm=rng.standard_normal((S, N, nx, nu)) / np.sqrt(nx),
                Q=W[:, :, :nx, :nx], Sm=W[:, :, nx:, :nx], R=W[:, :, nx:, nx:],
                gx=rng.standard_normal((S, N, nx)), gu=rng.standard_normal((S, N, nu)), d=0.1 * rng.standard_normal((S, N, nx)),
                WN=np.einsum("szx,szy->sxy", GN, GN) + eps * np.eye(nx), gN=rng.standard_normal((S, nx)), dx0=rng.standard_normal((S, nx)))


def riccati_ref(pr):
    """Textbook Riccati recursion (standard x, u order, np.linalg.solve), costates as lambda_k = P_k dx_k + p_k."""
    A, Bm, Q, Sm, R = pr["A"], pr["Bm"], pr["Q"], pr["Sm"], pr["R"]
    S, N, nx, nu = Bm.shape
    T = lambda M: np.swapaxes(M, -1, -2)
    mv = lambda M, v: np.einsum("sij,sj->si", M, v)
    Ps, ps = [None] * (N + 1), [None] * (N + 1)
    Ks, ks = [None] * N, [None] * N
    Ps[N], ps[N] = pr["WN"], pr["gN"]
    for k in range(N - 1, -1, -1):
        P, p, Ak, Bk = Ps[k + 1], ps[k + 1], A[:, k], Bm[:, k]
        v = p + mv(P, pr["d"][:, k])
        Qxx = Q[:, k] + T(Ak) @ P @ Ak
        Quu = R[:, k] + T(Bk) @ P @ Bk
        Qux = Sm[:, k] + T(Bk) @ P @ Ak
        qx = pr["gx"][:, k] + mv(T(Ak), v)
        qu = pr["gu"][:, k] + mv(T(Bk), v)
        Ks[k] = -np.linalg.solve(Quu, Qux)
        ks[k] = -np.linalg.solve(Quu, qu[..., None])[..., 0]
        Pn = Qxx + T(Qux) @ Ks[k]
        Ps[k], ps[k] = 0.5 * (Pn + T(Pn)), qx + mv(T(Qux), ks[k])
    dx, du, lam = np.empty((S, N + 1, nx)), np.empty((S, N, nu)), np.empty((S, N + 1, nx))
    dx[:, 0] = pr["dx0"]
    for k in range(N):
        du[:, k] = mv(Ks[k], dx[:, k]) + ks[k]
        dx[:, k + 1] = mv(A[:, k], dx[:, k]) + mv(Bm[:, k], du[:, k]) + pr["d"][:, k]
    for k in range(N + 1):
        lam[:, k] = mv(Ps[k], dx[:, k]) + ps[k]
    return dx, du, lam


def kkt_system(pr):
    """The KKT system of all S scenarios (block diagonal, one block per scenario) as a sparse matrix and its right-hand side.
    Per scenario the unknowns are (dx_0, du_0, ..., dx_{N-1}, du_{N-1}, dx_N, lambda_0, ..., lambda_N); rows: stationarity
    W z + g - C^T lambda = 0 of every primal block, then C z = e (dx_0 = dx0, dx_{k+1} - A_k dx_k - B_k du_k = d_k)."""
    S, N, nx, nu = pr["Bm"].shape
    nw = N * (nx + nu) + nx
    nt = nw + (N + 1) * nx
    xo = lambda k: k * (nx + nu)
    uo = lambda k: k * (nx + nu) + nx
    lo = lambda k: nw + k * nx
    rows, cols, vals = [], [], []

    def put(r0, c0, M):  # M [S, a, b] at (r0, c0) of every scenario's block
        a, b = M.shape[1:]
        rr = (np.arange(S)[:, None, None] * nt + r0 + np.arange(a)[None, :, None]) + 0 * np.arange(b)[None, None, :]
        cc = (np.arange(S)[:, None, None] * nt + c0 + np.arange(b)[None, None, :]) + 0 * np.arange(a)[None, :, None]
        rows.append(rr.ravel())
        cols.append(cc.ravel())
        vals.append(M.ravel())

    I = np.broadcast_to(np.eye(nx), (S, nx, nx))
    for k in range(N):
        put(xo(k), xo(k), pr["Q"][:, k])
        put(xo(k), uo(k), np.swapaxes(pr["Sm"][:, k], 1, 2))
        put(uo(k), xo(k), pr["Sm"][:, k])
        put(uo(k), uo(k), pr["R"][:, k])
        put(xo(k), lo(k + 1), np.swapaxes(pr["A"][:, k], 1, 2))
        put(uo(k), lo(k + 1), np.swapaxes(pr["Bm"][:, k], 1, 2))
        put(xo(k + 1), lo(k + 1), -I)
        put(lo(k + 1), xo(k + 1), I)
        put(lo(k + 1), xo(k), -pr["A"][:, k])
        put(lo(k + 1), uo(k), -pr["Bm"][:, k])
    put(xo(N), xo(N), pr["WN"])
    put(xo(0), lo(0), -I)
    put(lo(0), xo(0), I)
    K = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(S * nt, S * nt))
    rhs = np.zeros((S, nt))
    for k in range(N):
        rhs[:, xo(k):xo(k) + nx] = -pr["gx"][:, k]
        rhs[:, uo(k):uo(k) + nu] = -pr["gu"][:, k]
        rhs[:, lo(k + 1):lo(k + 1) + nx] = pr["d"][:, k]
    rhs[:, xo(N):xo(N) + nx] = -pr["gN"]
    rhs[:, lo(0):lo(0) + nx] = pr["dx0"]
    return K, rhs.ravel(), nt


def pack(sol_dx, sol_du, sol_lam):
    """(dx, du, lam) -> the unknown vector of kkt_system, [S, nt]"""
    S, N1, nx = sol_dx.shape
    N = N1 - 1
    w = np.concatenate([np.concatenate([sol_dx[:, :N], sol_du], axis=2).reshape(S, -1), sol_dx[:, N], sol_lam.reshape(S, -1)], axis=1)
    return w


def unpack(z, S, N, nx, nu):
    z = z.reshape(S, -1)
    nw = N * (nx + nu) + nx
    body = z[:, :N * (nx + nu)].reshape(S, N, nx + nu)
    dx = np.concatenate([body[:, :, :nx], z[:, None, N * (nx + nu):nw]], axis=1)
    return dx, body[:, :, nx:], z[:, nw:].reshape(S, N + 1, nx)


def kkt_solve(pr, dense=False):
    S, N, nx, nu = pr["Bm"].shape
    K, rhs, nt = kkt_system(pr)
    blk = lambda s: K[s * nt:(s + 1) * nt, s * nt:(s + 1) * nt]
    if dense:
        z = [np.linalg.solve(blk(s).toarray(), rhs[s * nt:(s + 1) * nt]) for s in range(S)]
    else:  # one sparse LU per scenario, fill-reducing order for the symmetric pattern
        z = [spla.spsolve(blk(s).tocsc(), rhs[s * nt:(s + 1) * nt], permc_spec="MMD_AT_PLUS_A") for s in range(S)]
    return unpack(np.concatenate(z), S, N, nx, nu)


def kkt_residual(pr, dx, du, lam):
    """per scenario |K sol - rhs|_inf / (|K|_inf |sol|_inf + |rhs|_inf)"""
    S = dx.shape[0]
    K, rhs, nt = kkt_system(pr)
    z = pack(dx, du, lam).ravel()
    r = np.abs(K @ z - rhs).reshape(S, nt).max(axis=1)
    knorm = np.asarray(abs(K).sum(axis=1)).reshape(S, nt).max(axis=1)
    return r / (knorm * np.abs(z.reshape(S, nt)).max(axis=1) + np.abs(rhs.reshape(S, nt)).max(axis=1))


# ---- the library's plane layouts (units u = k B + b) and this file's own index mapping back to the problem ----
def nodes(a, B, N):
    """[planes, N*B] -> [B, N, planes]"""
    return a.reshape(a.shape[0], N, B).transpose(2, 1, 0)


def planes(a):
    """[B, N, planes] -> [planes, N*B]"""
    return np.ascontiguousarray(a.transpose(2, 1, 0).reshape(a.shape[2], -1))


def problem_from_layout(n, B, N, jac, H=None, wx=None, wu=None, gx=None, gu=None, d=None, HN=None, wN=None, gN=None, dx0=None):
    nx, nu, P = 3 * n, n, 4 * n + 1
    xc, uc = xcols(n), ucols(n)
    J = jac.reshape(nx, P, N, B).transpose(3, 2, 0, 1)  # [B, N, row, col]
    Hh = H.reshape(P, P, N, B).transpose(3, 2, 0, 1) if H is not None else np.zeros((B, N, P, P))
    z = lambda rws, shp: np.zeros(shp) if rws is None else nodes(rws, B, N)
    Q = Hh[:, :, xc][:, :, :, xc] + np.einsum("bki,ij->bkij", z(wx, (B, N, nx)), np.eye(nx))
    R = Hh[:, :, uc][:, :, :, uc] + np.einsum("bki,ij->bkij", z(wu, (B, N, nu)), np.eye(nu))
    WN = (np.zeros((B, nx, nx)) if HN is None else HN.T.reshape(B, nx, nx)) + \
        np.einsum("bi,ij->bij", np.zeros((B, nx)) if wN is None else wN.T, np.eye(nx))
    return dict(A=J[..., xc], Bm=J[..., uc], Q=Q, Sm=Hh[:, :, uc][:, :, :, xc], R=R, gx=z(gx, (B, N, nx)), gu=z(gu, (B, N, nu)),
                d=z(d, (B, N, nx)), WN=WN, gN=np.zeros((B, nx)) if gN is None else gN.T, dx0=np.zeros((B, nx)) if dx0 is None else dx0.T)


def layout_from_problem(pr, seed):
    """The device planes of a random problem: W_k split into H (Gram part, merged into the Hessian layout) and the diagonal
    planes; the dt row / column of jac and H is filled with noise the solve must not read."""
    rng = np.random.default_rng(seed)
    B, N, nx, nu = pr["Bm"].shape
    n = nu
    P = 4 * n + 1
    xc, uc = xcols(n), ucols(n)
    wx = rng.uniform(0.0, 0.05, (B, N, nx))
    wu = rng.uniform(0.0, 0.05, (B, N, nu))
    wN = rng.uniform(0.0, 0.05, (B, nx))
    J = np.zeros((B, N, nx, P))
    J[..., xc] = pr["A"]
    J[..., uc] = pr["Bm"]
    J[..., 4 * n] = rng.standard_normal((B, N, nx))
    Hh = np.zeros((B, N, P, P))
    Hh[:, :, xc[:, None], xc[None, :]] = pr["Q"] - np.einsum("bki,ij->bkij", wx, np.eye(nx))
    Hh[:, :, uc[:, None], uc[None, :]] = pr["R"] - np.einsum("bki,ij->bkij", wu, np.eye(nu))
    Hh[:, :, uc[:, None], xc[None, :]] = pr["Sm"]
    Hh[:, :, xc[:, None], uc[None, :]] = np.swapaxes(pr["Sm"], 2, 3)
    noise = rng.standard_normal((B, N, P))
    Hh[:, :, 4 * n, :] = noise
    Hh[:, :, :, 4 * n] = noise
    Hh = 0.5 * (Hh + np.swapaxes(Hh, 2, 3))  # exactly symmetric
    HN = pr["WN"] - np.einsum("bi,ij->bij", wN, np.eye(nx))
    HN = 0.5 * (HN + np.swapaxes(HN, 1, 2))
    return dict(jac=np.ascontiguousarray(J.transpose(2, 3, 1, 0).reshape(nx, P, N * B)),
                H=np.ascontiguousarray(Hh.transpose(2, 3, 1, 0).reshape(P, P, N * B)),
                wx=planes(wx), wu=planes(wu), gx=planes(pr["gx"]), gu=planes(pr["gu"]), d=planes(pr["d"]),
                HN=np.ascontiguousarray(HN.reshape(B, nx * nx).T), wN=np.ascontiguousarray(wN.T), gN=np.ascontiguousarray(pr["gN"].T),
                dx0=np.ascontiguousarray(pr["dx0"].T))


OPT = ("H", "wx", "wu", "gx", "gu", "d", "HN", "wN", "gN", "dx0")


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("n", [1, 3, 6])
@pytest.mark.parametrize("N", [1, 2, 7])
def test_reference_riccati_matches_the_dense_kkt_solve(n, N):
    pr = random_problem(n, N, 3, seed=10 * n + N)
    assert np.abs(pr["Sm"]).max() > 0.1 and np.abs(pr["d"]).max() > 0 and np.abs(pr["dx0"]).max() > 0
    ref = kkt_solve(pr, dense=True)
    got = riccati_ref(pr)
    for a, b, nm in zip(got, ref, ("dx", "du", "lam")):
        assert np.abs(a - b).max() <= 1e-10 * max(np.abs(b).max(), 1.0), (nm, float(np.abs(a - b).max()))
    assert kkt_residual(pr, *got).max() < 1e-14


@pytest.mark.parametrize("n", [1, 3, 6, 16])
def test_random_problems_are_well_posed(n):
    eps = 0.1
    pr = random_problem(n, 4, 5, seed=n, eps=eps)
    W = np.concatenate([np.concatenate([pr["Q"], np.swapaxes(pr["Sm"], 2, 3)], axis=3), np.concatenate([pr["Sm"], pr["R"]], axis=3)], axis=2)
    assert np.abs(W - np.swapaxes(W, 2, 3)).max() == 0.0
    assert np.linalg.eigvalsh(W).min() >= eps * (1 - 1e-9)
    assert np.linalg.eigvalsh(pr["WN"]).min() >= eps * (1 - 1e-9)


def test_layout_round_trip_and_the_sign_of_the_costates():
    """The device layout maps back to the same problem; the costates are the multipliers of L as documented: lambda_N = W_N dx_N + g_N
    and stationarity in du_k reads R du + S dx + gu + B^T lambda_{k+1} = 0."""
    n, N, B = 2, 3, 4
    pr = random_problem(n, N, B, seed=5)
    lay = layout_from_problem(pr, seed=6)
    back = problem_from_layout(n, B, N, **lay)
    for k in pr:
        assert np.abs(back[k] - pr[k]).max() <= 1e-15 * max(np.abs(pr[k]).max(), 1.0), k
    dx, du, lam = riccati_ref(pr)
    assert np.abs(lam[:, N] - (np.einsum("sij,sj->si", pr["WN"], dx[:, N]) + pr["gN"])).max() < 1e-12
    st = np.einsum("skij,skj->ski", pr["R"], du) + np.einsum("skij,skj->ski", pr["Sm"], dx[:, :N]) + pr["gu"] + \
        np.einsum("skji,skj->ski", pr["Bm"], lam[:, 1:])
    assert np.abs(st).max() < 1e-12


# ------------------------------------------------------------------------------------------------ GPU helpers
def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(a):
    import torch
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _raw(m, B, N, ins, lam=True, out=None, ws=None, ws_bytes=0):
    """mpcf_riccati_batch with the device inputs `ins` (dict: jac + any of OPT); returns (rc, dx, du, lam)."""
    import torch
    from mpc_fatigue_b200 import _capi
    nx, nu = 3 * m.n, m.n
    if out is None:
        f = dict(dtype=torch.float64, device="cuda")
        out = (torch.empty((nx, (N + 1) * B), **f), torch.empty((nu, N * B), **f), torch.empty((nx, (N + 1) * B), **f) if lam else None)
    rc = _capi.lib.mpcf_riccati_batch(m.handle, B, N, _p(ins["jac"]), *[_p(ins.get(k)) for k in OPT], *[_p(t) for t in out], _p(ws),
                                      ws_bytes, _stream())
    return (rc, *out)


def _sol(out, B, N):
    """device (dx, du, lam) -> [B, N(+1), planes] host arrays"""
    dx, du, lam = [t.cpu().numpy() for t in out]
    return nodes(dx, B, N + 1), nodes(du, B, N), nodes(lam, B, N + 1)


def _chain(n):
    return Model.synthetic("chain", n, seed=n, armature=1e-2)


# ------------------------------------------------------------------------------------------------ GPU: synthetic LQ data
@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6, 7, 12, 14, 16])
@pytest.mark.parametrize("N", [1, 2, 7, 40])
@pytest.mark.parametrize("B", [1, 33, 257])
def test_synthetic_lq_matches_the_kkt_solve_with_a_small_kkt_residual(n, N, B):
    import torch
    from mpc_fatigue_b200 import _capi
    m = _chain(n)
    pr = random_problem(n, N, B, seed=1000 * n + 10 * N + B)
    lay = layout_from_problem(pr, seed=7)
    rc, *out = _raw(m, B, N, {k: _dev(v) for k, v in lay.items()})
    _capi.check(rc)
    torch.cuda.synchronize()
    got = _sol(out, B, N)
    # the direct KKT solve and the residual on every 8th scenario (the last included), the numpy Riccati on all of them
    sel = np.unique(np.r_[0:B:8, B - 1])
    part = {k: v[sel] for k, v in pr.items()}
    for g, r, rr, nm in zip(got, kkt_solve(part), riccati_ref(pr), ("dx", "du", "lam")):
        assert np.isfinite(g).all(), nm
        assert rel_err_rows(planes(g[sel]), planes(r)) <= 1e-9, (nm, rel_err_rows(planes(g[sel]), planes(r)))
        assert rel_err_rows(planes(g), planes(rr)) <= 1e-9, (nm, rel_err_rows(planes(g), planes(rr)))
    res = kkt_residual(part, *[g[sel] for g in got])
    assert res.max() <= 1e-12, float(res.max())


# ------------------------------------------------------------------------------------------------ GPU: the library's own producers
def _producer_model(name):
    from mpc_fatigue_b200.coupling import box_load_coupling
    if name == "pilz6x2_torso":
        return Model.from_urdf(open(os.path.join(ROOT, "tests", "golden", "pilz6x2_torso.urdf")).read(), armature=1e-2)
    if name == "dual_arm14":
        return Model.synthetic("dual_arm", 14, seed=3, armature=1e-2)
    m = Model.from_urdf(data_urdf(name.replace("_coupled", "")), armature=1e-2)
    if name.endswith("_coupled"):
        m.set_coupling(box_load_coupling(m, mass=30.0))
    return m


PRODUCERS = {"pilz3": "chain3", "pilz6": "chain6", "pilz6x2": "forest12x6", "pilz6x2_coupled": "forest12x6", "dual_arm14": "forest14x7",
             "pilz6x2_torso": "generic16"}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PRODUCERS))
def test_solve_on_the_librarys_own_jacobian_and_hessian(name):
    """States from a rollout (perturbed, so the defects are not zero), jac from step_rk4_jvp, H from step_rk4_hess with a random
    adjoint (for the coupled model, whose rollout and Hessian entries refuse the coupling: both from the same arms uncoupled), diagonally dominant weights, d from the step
    outputs.  The reference reads A, B, Q, S, R from the same host copies with this file's own index mapping."""
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from mpc_fatigue_b200.synth import synth_batch
    m = _producer_model(name)
    assert m.kernel_family == PRODUCERS[name]
    n, B, N, dt = m.n, 33, 7, 0.0125
    nx = 3 * n
    ev = BatchEvaluator(m)
    mh = _producer_model(name.replace("_coupled", "")) if name.endswith("_coupled") else m
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    q0, qd0, tau, f0 = synth_batch(lim, 0, B, N, seed=11, device="cuda")
    x0 = [t[:, :B].contiguous() for t in (q0, qd0, f0)]
    traj = BatchEvaluator(mh).rollout_rk4(*x0, tau, N, dt)  # the rollout entry has no coupled form: the uncoupled twin's
    rng = np.random.default_rng(12)
    # x_k for k = 0..N: rollout states with a small perturbation
    xs = [torch.cat([x0[i]] + [traj[i][:, k * B:(k + 1) * B] for k in range(N)], dim=1) for i in range(3)]
    xs = [x + _dev(1e-3 * rng.standard_normal(tuple(x.shape))) for x in xs]
    q, qd, f = [x[:, :N * B].contiguous() for x in xs]
    qn, qdn, fn, jac = ev.step_rk4_jvp(q, qd, tau, f, dt)
    lam_in = [_dev(rng.standard_normal((n, N * B))) for _ in range(3)]
    H = BatchEvaluator(mh).step_rk4_hess(q, qd, tau, f, dt, *lam_in)
    Hh = H.cpu().numpy()
    xc, uc = xcols(n), ucols(n)
    rows = np.abs(Hh[np.r_[xc, uc]][:, np.r_[xc, uc]]).sum(axis=1)  # Gershgorin: diagonal weights that make every W_k positive definite
    wx, wu = rows[:nx] + 1.0, rows[nx:] + 1.0
    d = torch.cat([qn, qdn, fn]) - torch.cat([x[:, B:].contiguous() for x in xs])
    ins = dict(jac=jac, H=H, wx=_dev(wx), wu=_dev(wu), gx=_dev(rng.standard_normal((nx, N * B))), gu=_dev(rng.standard_normal((n, N * B))),
               d=d.contiguous(), HN=None, wN=_dev(rng.uniform(1.0, 2.0, (nx, B))), gN=_dev(rng.standard_normal((nx, B))),
               dx0=_dev(rng.standard_normal((nx, B))))
    dxg, dug, lamg = ev.riccati(ins["jac"], B, N, **{k: v for k, v in ins.items() if k != "jac"}, want_lam=True)
    torch.cuda.synchronize()
    host = {k: (None if v is None else v.cpu().numpy()) for k, v in ins.items()}
    pr = problem_from_layout(n, B, N, **host)
    if name.endswith("_coupled"):  # the dense cross-arm f block goes through unchanged
        A = pr["A"]
        assert np.abs(A[:, :, 2 * n:2 * n + 6, 2 * n + 6:]).max() > 0
    ref = kkt_solve(pr)
    got = (nodes(dxg.cpu().numpy(), B, N + 1), nodes(dug.cpu().numpy(), B, N), nodes(lamg.cpu().numpy(), B, N + 1))
    for g, r, nm in zip(got, ref, ("dx", "du", "lam")):
        assert rel_err_rows(planes(g), planes(r)) <= 1e-9, (name, nm, rel_err_rows(planes(g), planes(r)))
    assert kkt_residual(pr, *got).max() <= 1e-12


# ------------------------------------------------------------------------------------------------ GPU: NULL, chunks, batch position
def _synthetic_device(n, N, B, seed):
    pr = random_problem(n, N, B, seed=seed)
    return pr, {k: _dev(v) for k, v in layout_from_problem(pr, seed=seed + 1).items()}


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6, 13])
def test_null_inputs_are_bit_identical_to_explicit_zeros(n):
    import torch
    m = _chain(n)
    N, B = 7, 33
    _, ins = _synthetic_device(n, N, B, seed=31)
    for k in OPT:
        a = _raw(m, B, N, {**ins, k: None})
        b = _raw(m, B, N, {**ins, k: torch.zeros_like(ins[k])})
        assert a[0] == 0 and b[0] == 0
        torch.cuda.synchronize()
        for x, y in zip(a[1:], b[1:]):
            assert torch.equal(x, y), k
            assert bool(torch.isfinite(x).all()), k
    # every optional input NULL: dx = 0, du = 0, lam = 0
    zero = _raw(m, B, N, {"jac": ins["jac"], "wx": ins["wx"], "wu": ins["wu"]})
    torch.cuda.synchronize()
    assert all(float(t.abs().max()) == 0.0 for t in zero[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6, 13])
def test_each_scenario_is_independent_of_its_batch_and_of_the_chunking(n):
    import torch
    from mpc_fatigue_b200 import _capi
    m = _chain(n)
    N, B = 5, 257
    _, ins = _synthetic_device(n, N, B, seed=41)
    full = _raw(m, B, N, ins)
    assert full[0] == 0
    # the minimum workspace (one CTA's scenarios per chunk): many chunks
    wmin = int(_capi.lib.mpcf_riccati_workspace_bytes(m.handle, 1, N))
    assert wmin > 0 and int(_capi.lib.mpcf_riccati_workspace_bytes(m.handle, B, N)) > wmin
    ws = torch.empty(wmin // 8, dtype=torch.float64, device="cuda")
    small = _raw(m, B, N, ins, ws=ws, ws_bytes=wmin)
    assert small[0] == 0
    torch.cuda.synchronize()
    for x, y in zip(full[1:], small[1:]):
        assert torch.equal(x, y)
    # one scenario alone
    for b in (0, 100, 256):
        one = {}
        for k, v in ins.items():
            per_node = v.shape[-1] == N * B
            idx = torch.arange(N, device="cuda") * B + b if per_node else torch.tensor([b], device="cuda")
            one[k] = v[..., idx].contiguous()
        alone = _raw(m, 1, N, one)
        assert alone[0] == 0
        torch.cuda.synchronize()
        ix = torch.arange(N + 1, device="cuda") * B + b
        iu = torch.arange(N, device="cuda") * B + b
        assert torch.equal(alone[1], full[1][:, ix]) and torch.equal(alone[2], full[2][:, iu]) and torch.equal(alone[3], full[3][:, ix]), b


CANARY = -7.25e300


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6, 14])
@pytest.mark.parametrize("B", [1, 33, 131])
def test_canary_gaps_around_the_outputs_and_the_workspace(n, B):
    import torch
    from mpc_fatigue_b200 import _capi
    m = _chain(n)
    N, nx, GAP = 4, 3 * n, 4096
    _, ins = _synthetic_device(n, N, B, seed=51)
    wmin = int(_capi.lib.mpcf_riccati_workspace_bytes(m.handle, 1, N))
    sizes = [nx * (N + 1) * B, n * N * B, nx * (N + 1) * B, wmin // 8]
    views, gaps, off = [], [slice(0, GAP)], GAP
    for s in sizes:
        off = (off + 15) // 16 * 16  # 128-byte aligned buffers
        views.append((off, s))
        gaps.append(slice(off + s, off + s + GAP))
        off += s + GAP
    pool = torch.full((off,), CANARY, dtype=torch.float64, device="cuda")
    dx, du, lam, ws = [pool[o:o + s] for o, s in views]
    rc = _raw(m, B, N, ins, out=(dx.view(nx, -1), du.view(n, -1), lam.view(nx, -1)), ws=ws, ws_bytes=wmin)[0]
    assert rc == 0
    torch.cuda.synchronize()
    for i, g in enumerate(gaps):
        assert bool((pool[g] == CANARY).all()), (n, B, "canary gap %d was written" % i)
    for t, nm in ((dx, "dx"), (du, "du"), (lam, "lam")):
        assert not bool((t == CANARY).any()) and bool(torch.isfinite(t).all()), (n, B, nm)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6, 13])
def test_an_indefinite_scenario_is_nan_and_leaves_its_neighbours_bit_identical(n):
    import torch
    m = _chain(n)
    N, B, bad = 7, 33, 17
    _, ins = _synthetic_device(n, N, B, seed=61)
    ref = _raw(m, B, N, ins)
    wu = ins["wu"].clone()
    wu[0, 3 * B + bad] = -1e6  # R indefinite at node 3 of scenario `bad`
    out = _raw(m, B, N, {**ins, "wu": wu})
    assert ref[0] == 0 and out[0] == 0
    torch.cuda.synchronize()
    for x, y, N1 in zip(out[1:], ref[1:], (N + 1, N, N + 1)):
        cols = torch.arange(N1, device="cuda") * B + bad
        assert bool(torch.isnan(x[:, cols]).all())
        keep = torch.ones(x.shape[1], dtype=torch.bool, device="cuda")
        keep[cols] = False
        assert torch.equal(x[:, keep], y[:, keep])


@pytest.mark.gpu
def test_argument_rejection():
    import torch
    from mpc_fatigue_b200 import _capi
    lib = _capi.lib
    m = _chain(6)
    N, B = 3, 8
    _, ins = _synthetic_device(6, N, B, seed=71)
    rc, dx, du, lam = _raw(m, B, N, ins)
    assert rc == 0
    torch.cuda.synchronize()
    st = _stream()

    def call(model=m, B=B, N=N, jac=ins["jac"], dx=dx, du=du, ws=None, wsb=0):
        return lib.mpcf_riccati_batch(model.handle, B, N, _p(jac), *[_p(ins[k]) for k in OPT], _p(dx), _p(du), _p(lam), _p(ws) if ws is not None else None,
                                      wsb, st)
    assert call(jac=None) == _capi.EINVAL
    assert call(dx=None) == _capi.EINVAL
    assert call(du=None) == _capi.EINVAL
    assert call(N=0) == _capi.EINVAL
    assert call(B=-1) == _capi.EINVAL
    wmin = int(lib.mpcf_riccati_workspace_bytes(m.handle, 1, N))
    ws = torch.empty(wmin // 8 + 32, dtype=torch.float64, device="cuda")
    assert call(ws=ws, wsb=wmin - 8) == _capi.EINVAL and "too small" in _capi.last_error()
    mis = C.c_void_p(ws.data_ptr() + 8)
    assert lib.mpcf_riccati_batch(m.handle, B, N, _p(ins["jac"]), *[_p(ins[k]) for k in OPT], _p(dx), _p(du), _p(lam), mis, wmin, st) == _capi.EINVAL
    assert "aligned" in _capi.last_error()
    # B = 0: OK and no launch
    n0 = lib.mpcf_launch_count()
    assert call(B=0) == _capi.OK
    assert lib.mpcf_launch_count() == n0
    # n = 37 is over the one-warp design's limit
    mh = Model.synthetic("humanoid", 37, seed=7, armature=1e-2)
    assert lib.mpcf_riccati_batch(mh.handle, B, N, _p(ins["jac"]), *[None] * 10, _p(dx), _p(du), None, None, 0, st) == _capi.ELIMIT
    assert "n <= 16" in _capi.last_error()
    assert int(lib.mpcf_riccati_workspace_bytes(mh.handle, B, N)) == 0
    # the evaluator maps the codes to exceptions
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    with pytest.raises(ValueError):
        BatchEvaluator(mh).riccati(torch.zeros((111, 149, N * B), dtype=torch.float64, device="cuda"), B, N)


# ------------------------------------------------------------------------------------------------ GPU: full size
@pytest.mark.gpu
def test_full_size_pilz6_kkt_residual_on_a_sample():
    """pilz6 at the C2 shape (65,536 scenarios x 100 nodes): jac from step_rk4_jvp on synthetic states, diagonal weights and random
    gradients / defects / initial offsets; the KKT residual of 512 random scenarios, copied to the host, is <= 1e-12."""
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from mpc_fatigue_b200.synth import synth_batch
    m = Model.from_urdf(data_urdf("pilz6"), armature=1e-2)
    ev = BatchEvaluator(m)
    n, B, N = m.n, 65536, 100
    nx, U = 3 * n, N * B
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    q, qd, tau, f = synth_batch(lim, 0, B, N, seed=81, device="cuda")
    jac = ev.step_rk4_jvp(q, qd, tau, f, 0.0125)[3]
    del q, qd, tau, f
    g = torch.Generator(device="cuda").manual_seed(82)
    rnd = lambda r, c, lo=-1.0, hi=1.0: torch.rand((r, c), generator=g, dtype=torch.float64, device="cuda") * (hi - lo) + lo
    ins = dict(wx=rnd(nx, U, 0.1, 1.0), wu=rnd(n, U, 0.1, 1.0), gx=rnd(nx, U), gu=rnd(n, U), d=rnd(nx, U, -1e-3, 1e-3), wN=rnd(nx, B, 0.1, 1.0),
               gN=rnd(nx, B), dx0=rnd(nx, B, -1e-2, 1e-2))
    dx, du, lam = ev.riccati(jac, B, N, **ins, want_lam=True)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(dx).all() and torch.isfinite(du).all() and torch.isfinite(lam).all())
    sel = np.sort(np.random.default_rng(83).choice(B, 512, replace=False))
    bsel = torch.from_numpy(sel).cuda()
    iu = (torch.arange(N, device="cuda")[:, None] * B + bsel[None]).reshape(-1)
    ix = (torch.arange(N + 1, device="cuda")[:, None] * B + bsel[None]).reshape(-1)
    S = len(sel)
    host = dict(jac=jac[:, :, iu].cpu().numpy(), **{k: ins[k][:, iu].cpu().numpy() for k in ("wx", "wu", "gx", "gu", "d")},
                **{k: ins[k][:, bsel].cpu().numpy() for k in ("wN", "gN", "dx0")})
    pr = problem_from_layout(n, S, N, **host)
    got = (nodes(dx[:, ix].cpu().numpy(), S, N + 1), nodes(du[:, iu].cpu().numpy(), S, N), nodes(lam[:, ix].cpu().numpy(), S, N + 1))
    worst = 0.0
    for c in range(0, S, 64):
        part = {k: v[c:c + 64] for k, v in pr.items()}
        worst = max(worst, float(kkt_residual(part, *[a[c:c + 64] for a in got]).max()))
    assert worst <= 1e-12, worst
