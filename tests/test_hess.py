"""Second order: the adjoint-weighted Hessian of the RK4 step (mpcf_step_rk4_hess_batch), its Hessian-vector product
(mpcf_step_rk4_hvp_batch) and the twice-differentiable autograd wrapper (mpc_fatigue_b200/autograd.py: step_rk4_2).

H = d2(lambda^T x+)/dz dz with z = (q, qd, tau, f, dt).  The CPU tests pin the hyper-dual oracle (oracle/second_order.cpp) against
central differences of lambda^T J of the complex-step Jacobian, its symmetry across independent sweeps and the closed-form fatigue
entries.  The GPU tests check every kernel family against the oracle, the library's own Jacobian and VJP entries, argument handling
and buffer bounds."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT, oracle_model_from_export, random_inputs, rel_err_rows
from mpc_fatigue_b200.model import Model, data_urdf
from oracle.pyoracle import Oracle

TOL = 1e-9

MODELS = {
    "pilz3": lambda: Model.from_urdf(data_urdf("pilz3"), armature=1e-2),
    "pilz6": lambda: Model.from_urdf(data_urdf("pilz6"), armature=1e-2),
    "chain7": lambda: Model.synthetic("chain", 7, seed=2, armature=1e-2),
    "pilz6x2": lambda: Model.from_urdf(data_urdf("pilz6x2"), armature=1e-2),
    "dual_arm14": lambda: Model.synthetic("dual_arm", 14, seed=3, armature=1e-2),
    "mixed": lambda: Model.from_urdf(open(os.path.join(ROOT, "tests", "golden", "mixed_joints.urdf")).read(), armature=1e-3),
    "humanoid37": lambda: Model.synthetic("humanoid", 37, seed=7, armature=1e-2),
}
FAMILY = {"pilz3": "chain3", "pilz6": "chain6", "chain7": "chain7", "pilz6x2": "forest12x6", "dual_arm14": "forest14x7",
          "mixed": "generic16", "humanoid37": "generic64"}


# ---------------------------------------------------------------------------------------------------------------- hyper-dual oracle
_HD = {}


def _hd_lib():
    """oracle/second_order.cpp (core.inc.h instantiated with a hyper-dual scalar), compiled once per process into a temporary
    directory with the flags of the reproducible checker build (-O2, no FMA contraction)."""
    if "lib" not in _HD:
        _HD["dir"] = d = tempfile.TemporaryDirectory(prefix="mpcf_oracle_hd_")
        out = os.path.join(d.name, "libmpcf_oracle_hd.so")
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
        subprocess.run([cxx, "-std=c++17", "-fPIC", "-shared", "-fopenmp", "-O2", "-ffp-contract=off", "-Wall", "-Wno-unused-function",
                        "-Wno-unknown-pragmas", "-o", out, os.path.join(ROOT, "oracle", "second_order.cpp"), "-lm"], check=True)
        _HD["lib"] = C.CDLL(out)
    return _HD["lib"]


def _np(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(C.POINTER(C.c_double))


def oracle_hess(orc, q, qd, tau, f, dt, lq=None, lqd=None, lf=None, dt_u=None):
    """H [4n+1, 4n+1, U] = d2(lambda^T x+)/dz dz, z = (q, qd, tau, f, dt), by hyper-dual sweeps over EVERY pair of inputs (the
    fatigue inputs included) on the oracle model of `orc`; lambda = (lq, lqd, lf), None = 0."""
    n, U = q.shape
    P = 4 * n + 1
    H = np.empty((P, P, U))
    keep = [np.ascontiguousarray(a, dtype=np.float64) if a is not None else None for a in (q, qd, tau, f, dt_u, lq, lqd, lf)]
    rc = _hd_lib().mpcfo_step_rk4_hess_batch(orc._ref(), C.c_long(U), *[_np(a) for a in keep[:4]], C.c_double(dt), _np(keep[4]),
                                             *[_np(a) for a in keep[5:]], _np(H))
    assert rc == 0, rc
    return H


def oracle_hvp(orc, q, qd, tau, f, dt, lam, v, dt_u=None):
    """((hq, hqd, htau, hf [n, U], hdt [U]) = H v, (jq, jqd, jf) = J v) by one hyper-dual sweep per input; lam = (lq, lqd, lf),
    v = (vq, vqd, vtau, vf, vdt [U]), None entries = 0."""
    n, U = q.shape
    h = [np.empty((n, U)) for _ in range(4)] + [np.empty(U)]
    j = [np.empty((n, U)) for _ in range(3)]
    keep = [np.ascontiguousarray(a, dtype=np.float64) if a is not None else None for a in (q, qd, tau, f, dt_u, *lam, *v)]
    rc = _hd_lib().mpcfo_step_rk4_hvp_batch(orc._ref(), C.c_long(U), *[_np(a) for a in keep[:4]], C.c_double(dt), _np(keep[4]),
                                            *[_np(a) for a in keep[5:]], *[_np(a) for a in h], *[_np(a) for a in j])
    assert rc == 0, rc
    return tuple(h), tuple(j)


def amp_prime(z):
    return -1.0 + z - z * z / 2.0 + z ** 3 / 6.0


def _inputs(name, U, seed):
    m = MODELS[name]()
    om = oracle_model_from_export(m)
    q, qd, tau, f, _ = random_inputs(om, U, seed=seed)
    rng = np.random.default_rng(seed + 1)
    lam = rng.standard_normal((3 * m.n, U))
    v = rng.standard_normal((4 * m.n + 1, U))
    return m, om, [q, qd, tau, f], lam, v


def _split(a, n, k):
    return [np.ascontiguousarray(a[i * n:(i + 1) * n]) for i in range(k)]


def _hv(H, v):
    """H v per unit: H [P, P, U], v [P, U] -> [P, U], and its condition scale sum_c |H_rc| |v_c|."""
    return np.einsum("rcu,cu->ru", H, v), np.einsum("rcu,cu->ru", np.abs(H), np.abs(v))


def _assert_scaled(got, ref, S, tol, what):
    bound = tol * np.maximum(S, 1e-6 * max(S.max(), 1e-300))
    err = np.abs(got - ref)
    assert (err <= bound).all(), (what, float((err / np.maximum(bound, 1e-300)).max()))


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", ["pilz6", "pilz6x2", "mixed"])
def test_oracle_hessian_matches_central_differences_of_the_complex_step_vjp(name):
    m, om, z, lam, _ = _inputs(name, 3, seed=201)
    n, U = m.n, 3
    P = 4 * n + 1
    orc = Oracle(om)
    dt_u = np.ascontiguousarray([0.0125, 0.004, 0.02])
    H = oracle_hess(orc, *z, 0.0, *_split(lam, n, 3), dt_u=dt_u)
    zz = np.vstack(z + [dt_u[None]])

    def vjp(zv):
        J = orc.step_rk4_jvp(*_split(zv, n, 4), 0.0, dt_u=np.ascontiguousarray(zv[4 * n]))[3]
        return np.einsum("ru,rcu->cu", lam, J)

    eps = 1e-5
    for c in range(P):
        zp, zm = zz.copy(), zz.copy()
        zp[c] += eps
        zm[c] -= eps
        fd = (vjp(zp) - vjp(zm)) / (2 * eps)
        scale = np.abs(H).max(axis=(0, 1))
        assert (np.abs(H[:, c] - fd) <= 1e-6 * scale).all(), (name, c, float((np.abs(H[:, c] - fd) / scale).max()))


@pytest.mark.parametrize("name", ["pilz6", "pilz6x2", "mixed"])
def test_oracle_hessian_is_symmetric_with_closed_form_fatigue_entries_and_its_hvp_is_h_times_v(name):
    m, om, z, lam, v = _inputs(name, 4, seed=211)
    n, U = m.n, 4
    P = 4 * n + 1
    orc = Oracle(om)
    dt_u = np.ascontiguousarray([0.0125, 0.0, 0.02, 0.007])
    ls = _split(lam, n, 3)
    H = oracle_hess(orc, *z, 0.0, *ls, dt_u=dt_u)
    scale = np.abs(H).max()
    # column c by the HVP sweeps (direction a on the first tangent, e_c on the second): the transpose of what the dense entry swept
    Hc = np.empty_like(H)
    for c in range(P):
        e = np.zeros((P, U))
        e[c] = 1.0
        h, _ = oracle_hvp(orc, *z, 0.0, ls, _split(e, n, 4) + [e[4 * n]], dt_u=dt_u)
        Hc[:, c] = np.vstack(list(h[:4]) + [h[4][None]])
    assert np.abs(Hc - Hc.transpose(1, 0, 2)).max() <= 1e-12 * scale
    assert np.abs(Hc - H).max() <= 1e-12 * scale
    # fatigue rows and columns: zero except H[f_i][dt] = lf_i Lambda_i amp'(Lambda_i h)
    fat = np.array(om.fat)
    fi = np.arange(3 * n, 4 * n)
    ref = np.zeros((n, P, U))
    ref[:, 4 * n] = lam[2 * n:] * fat[:, 0:1] * amp_prime(fat[:, 0:1] * dt_u[None])
    assert np.abs(H[fi] - ref).max() <= 1e-12 * scale
    assert np.abs(H[:, fi] - ref.transpose(1, 0, 2)).max() <= 1e-12 * scale
    # H v, and J v against the complex-step Jacobian
    h, j = oracle_hvp(orc, *z, 0.0, ls, _split(v, n, 4) + [v[4 * n]], dt_u=dt_u)
    ref, S = _hv(H, v)
    _assert_scaled(np.vstack(list(h[:4]) + [h[4][None]]), ref, S, 1e-12, "hvp")
    J = orc.step_rk4_jvp(*z, 0.0, dt_u=dt_u)[3]
    _assert_scaled(np.vstack(j), np.einsum("rcu,cu->ru", J, v), np.einsum("rcu,cu->ru", np.abs(J), np.abs(v)), 1e-12, "jv")


# ---------------------------------------------------------------------------------------------------------------- GPU helpers
def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(a):
    import torch
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _raw_hess(m, d, dt, dt_u, dl, H=None):
    import torch
    from mpc_fatigue_b200 import _capi
    n, U = d[0].shape
    if H is None:
        H = torch.empty((4 * n + 1, 4 * n + 1, U), dtype=torch.float64, device="cuda")
    _capi.check(_capi.lib.mpcf_step_rk4_hess_batch(m.handle, U, *[_p(t) for t in d], float(dt), _p(dt_u), *[_p(t) for t in dl], _p(H),
                                                   _stream()))
    return H


def _raw_hvp(m, d, dt, dt_u, dl, dv, out=None, hdt=True, jv=True):
    """mpcf_step_rk4_hvp_batch; returns [hq, hqd, htau, hf, hdt, jq, jqd, jf] (None where not requested)."""
    import torch
    from mpc_fatigue_b200 import _capi
    n, U = d[0].shape
    if out is None:
        out = [torch.empty((n, U), dtype=torch.float64, device="cuda") for _ in range(4)]
        out.append(torch.empty(U, dtype=torch.float64, device="cuda") if hdt else None)
        out += [torch.empty((n, U), dtype=torch.float64, device="cuda") if jv else None for _ in range(3)]
    _capi.check(_capi.lib.mpcf_step_rk4_hvp_batch(m.handle, U, *[_p(t) for t in d], float(dt), _p(dt_u), *[_p(t) for t in dl],
                                                  *[_p(t) for t in dv], *[_p(t) for t in out], _stream()))
    return out


def _gpu_case(name, U, seed):
    m, om, z, lam, v = _inputs(name, U, seed)
    n = m.n
    d = [_dev(a) for a in z]
    dl = [_dev(a) for a in _split(lam, n, 3)]
    dv = [_dev(a) for a in _split(v, n, 4)] + [_dev(v[4 * n])]
    return m, om, z, lam, v, d, dl, dv


# (model, U) pairs of the dense checks: the oracle sweeps all P (P + 1) / 2 pairs per unit, so the 37-joint tree runs small batches
DENSE = [(nm, U) for nm in ("pilz3", "pilz6", "chain7", "pilz6x2", "dual_arm14", "mixed") for U in (1, 33, 257)] + \
        [("humanoid37", 1), ("humanoid37", 3)]


# ---------------------------------------------------------------------------------------------------------------- GPU: dense H
@pytest.mark.gpu
@pytest.mark.parametrize("name,U", DENSE)
def test_dense_hessian_matches_the_oracle(name, U):
    import torch
    m, om, z, lam, v, d, dl, dv = _gpu_case(name, U, seed=301 + U)
    assert m.kernel_family == FAMILY[name]
    n, P = m.n, 4 * m.n + 1
    orc = Oracle(om, fast=True)
    dt_u = np.ascontiguousarray(np.random.default_rng(302).uniform(0.002, 0.02, U))
    cases = [(0.0125, None, dl), (0.0, dt_u, dl), (0.0, None, dl)]  # scalar dt, per-unit dt, dt = 0
    if U == 33:
        cases += [(0.0125, None, [dl[0], None, None]), (0.0125, None, [None, dl[1], dl[2]]), (0.0125, None, [None, None, dl[2]])]
    for dt, du, lp in cases:
        H = _raw_hess(m, d, dt, _dev(du), lp)
        torch.cuda.synchronize()
        assert torch.equal(H, H.transpose(0, 1)), (name, U, "mirrored planes differ")
        ref = oracle_hess(orc, *z, dt, *[None if t is None else t.cpu().numpy() for t in lp], dt_u=du)
        got = H.cpu().numpy()
        assert np.isfinite(got).all()
        assert rel_err_rows(got.reshape(P * P, U), ref.reshape(P * P, U)) < TOL, (name, U, dt, du is not None)


# ---------------------------------------------------------------------------------------------------------------- GPU: H v and J v
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_hvp_matches_the_oracle_the_dense_hessian_and_the_jacobian(name):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    U = 5 if name == "humanoid37" else 33
    m, om, z, lam, v, d, dl, dv = _gpu_case(name, U, seed=401)
    n = m.n
    dt_u = np.ascontiguousarray(np.random.default_rng(402).uniform(0.002, 0.02, U))
    dt_u[0] = 0.0
    du = _dev(dt_u)
    out = [t.cpu().numpy() for t in _raw_hvp(m, d, 0.0, du, dl, dv)]
    hv = np.vstack(out[:4] + [out[4][None]])
    jv = np.vstack(out[5:])
    (rh, rj) = oracle_hvp(Oracle(om, fast=True), *z, 0.0, _split(lam, n, 3), _split(v, n, 4) + [v[4 * n]], dt_u=dt_u)
    assert rel_err_rows(hv, np.vstack(list(rh[:4]) + [rh[4][None]])) < TOL
    assert rel_err_rows(jv, np.vstack(rj)) < TOL
    H = _raw_hess(m, d, 0.0, du, dl).cpu().numpy()
    _assert_scaled(hv, *_hv(H, v), 1e-12, (name, "H v"))
    J = BatchEvaluator(m).step_rk4_jvp(*d, du)[3].cpu().numpy()
    _assert_scaled(jv, np.einsum("rcu,cu->ru", J, v), np.einsum("rcu,cu->ru", np.abs(J), np.abs(v)), 1e-12, (name, "J v"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz3", "pilz6", "pilz6x2", "dual_arm14", "mixed", "humanoid37"])
def test_hvp_equals_finite_differences_of_the_library_vjp(name):
    """(VJP(z + eps v) - VJP(z - eps v)) / 2 eps of mpcf_step_rk4_vjp_batch, dt as a per-unit tensor."""
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    U = 17
    m, om, z, lam, v, d, dl, dv = _gpu_case(name, U, seed=501)
    n = m.n
    ev = BatchEvaluator(m)
    dt_u = np.ascontiguousarray(np.random.default_rng(502).uniform(0.005, 0.02, U))
    zz = np.vstack(z + [dt_u[None]])
    hv = np.vstack([t.cpu().numpy() if t.dim() == 2 else t.cpu().numpy()[None]
                    for t in ev.step_rk4_hvp(*d, _dev(dt_u), dl, dv, want_dt=True)])

    def vjp(zv):
        g = ev.step_rk4_vjp(*[_dev(a) for a in _split(zv, n, 4)], _dev(zv[4 * n]), *dl, want_dt=True)
        return np.vstack([g[i].cpu().numpy() for i in range(4)] + [g[4].cpu().numpy()[None]])

    eps = 1e-6
    fd = (vjp(zz + eps * v) - vjp(zz - eps * v)) / (2 * eps)
    scale = np.abs(hv).max()
    assert np.abs(hv - fd).max() <= 1e-6 * scale, (name, float(np.abs(hv - fd).max() / scale))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz6", "pilz6x2", "mixed"])
def test_null_hvp_parts_act_as_zeros_and_outputs_are_optional(name):
    import torch
    m, om, z, lam, v, d, dl, dv = _gpu_case(name, 40, seed=601)
    full = _raw_hvp(m, d, 0.0125, None, dl, dv)
    for k in range(5):
        part = [None if i == k else t for i, t in enumerate(dv)]
        zeros = [torch.zeros_like(t) if i == k else t for i, t in enumerate(dv)]
        a, b = _raw_hvp(m, d, 0.0125, None, dl, part), _raw_hvp(m, d, 0.0125, None, dl, zeros)
        torch.cuda.synchronize()
        for x, y in zip(a, b):
            assert torch.equal(x, y), k
    # hdt and J v are optional and leave the other outputs unchanged
    short = _raw_hvp(m, d, 0.0125, None, dl, dv, hdt=False, jv=False)
    torch.cuda.synchronize()
    for x, y in zip(short[:4], full[:4]):
        assert torch.equal(x, y)


CANARY = -7.25e300


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz6", "pilz6x2", "mixed", "humanoid37"])
@pytest.mark.parametrize("U", [1, 33, 131])
def test_canary_gaps_around_h_and_every_hvp_output(name, U):
    import torch
    m, om, z, lam, v, d, dl, dv = _gpu_case(name, U, seed=701)
    n, P, GAP = m.n, 4 * m.n + 1, 64
    sizes = [P * P * U] + [n * U] * 4 + [U] + [n * U] * 3
    pool = torch.full((GAP + sum(s + GAP for s in sizes),), CANARY, dtype=torch.float64, device="cuda")
    views, gaps, off = [], [slice(0, GAP)], GAP
    for s in sizes:
        views.append(pool[off:off + s])
        gaps.append(slice(off + s, off + s + GAP))
        off += s + GAP
    _raw_hess(m, d, 0.0125, None, dl, H=views[0].view(P, P, U))
    _raw_hvp(m, d, 0.0125, None, dl, dv, out=[t.view(n, U) for t in views[1:5]] + [views[5]] + [t.view(n, U) for t in views[6:]])
    torch.cuda.synchronize()
    for i, g in enumerate(gaps):
        assert bool((pool[g] == CANARY).all()), (name, U, "canary gap %d was written" % i)
    for i, t in enumerate(views):
        assert not bool((t == CANARY).any()), (name, U, i, "has unwritten elements")


@pytest.mark.gpu
def test_invalid_arguments():
    import torch
    from mpc_fatigue_b200 import _capi
    m, om, z, lam, v, d, dl, dv = _gpu_case("pilz6", 40, seed=801)
    H = _raw_hess(m, d, 0.0125, None, dl)
    out = _raw_hvp(m, d, 0.0125, None, dl, dv)
    torch.cuda.synchronize()
    st = _stream()
    lib = _capi.lib

    def hess(model=m, U=40, x=d, H=H):
        return lib.mpcf_step_rk4_hess_batch(model.handle, U, *[_p(t) for t in x], 0.0125, None, *[_p(t) for t in dl], _p(H), st)

    def hvp(model=m, U=40, x=d, o=out):
        return lib.mpcf_step_rk4_hvp_batch(model.handle, U, *[_p(t) for t in x], 0.0125, None, *[_p(t) for t in dl], *[_p(t) for t in dv],
                                           *[_p(t) for t in o], st)
    for k in range(4):
        assert hess(x=[None if i == k else t for i, t in enumerate(d)]) == _capi.EINVAL, k
        assert hvp(x=[None if i == k else t for i, t in enumerate(d)]) == _capi.EINVAL, k
        assert hvp(o=[None if i == k else t for i, t in enumerate(out)]) == _capi.EINVAL, k
    assert hess(H=None) == _capi.EINVAL
    assert hess(U=-1) == _capi.EINVAL and hvp(U=-1) == _capi.EINVAL
    for k in range(5, 8):  # a partial set of J v outputs
        assert hvp(o=[None if i == k else t for i, t in enumerate(out)]) == _capi.EINVAL, k
    # U = 0 launches nothing
    n0 = lib.mpcf_launch_count()
    assert hess(U=0) == _capi.OK and hvp(U=0) == _capi.OK
    assert lib.mpcf_launch_count() == n0
    # coupled models are refused
    mc = MODELS["pilz6x2"]()
    fpar = mc.export("fparent")
    mc.set_coupling((int(np.flatnonzero((fpar >= 0) & (fpar < 6))[-1]), int(np.flatnonzero(fpar >= 6)[-1]), 30 * 9.81))
    zc = torch.zeros((12, 8), dtype=torch.float64, device="cuda")
    Hc = torch.zeros((49, 49, 8), dtype=torch.float64, device="cuda")
    assert lib.mpcf_step_rk4_hess_batch(mc.handle, 8, *[_p(zc)] * 4, 0.01, None, None, None, None, _p(Hc), st) == _capi.EINVAL
    assert lib.mpcf_step_rk4_hvp_batch(mc.handle, 8, *[_p(zc)] * 4, 0.01, None, *[None] * 8, *[_p(zc)] * 4, *[None] * 4, st) == _capi.EINVAL


# ---------------------------------------------------------------------------------------------------------------- GPU: autograd
def _leaves(name, U, seed):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m, om, z, lam, v = _inputs(name, U, seed)
    leaf = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda().requires_grad_()
    dt = leaf(np.random.default_rng(seed + 2).uniform(0.005, 0.02, U))
    return BatchEvaluator(m), m, [leaf(a) for a in z] + [dt], lam, v


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pilz3", "mixed"])
def test_autograd_gradcheck_and_gradgradcheck(name):
    import torch
    from mpc_fatigue_b200 import autograd as mad
    ev, m, args, _, _ = _leaves(name, 3, seed=901)
    fn = lambda *x: mad.step_rk4_2(ev, *x)
    assert torch.autograd.gradcheck(fn, tuple(args), eps=1e-6, atol=1e-7, rtol=1e-6)
    assert torch.autograd.gradgradcheck(fn, tuple(args), eps=1e-6, atol=1e-6, rtol=1e-5)


@pytest.mark.gpu
def test_double_backward_equals_the_hvp_entry():
    import torch
    from mpc_fatigue_b200 import autograd as mad
    ev, m, args, lam, v = _leaves("pilz6", 16, seed=911)
    n = m.n
    lt = [_dev(a) for a in _split(lam, n, 3)]
    vt = [_dev(a) for a in _split(v, n, 4)] + [_dev(v[4 * n])]
    out = mad.step_rk4_2(ev, *args)
    # the first backward with create_graph: g = lambda^T J, then d (g . v) / d z = H v
    g = torch.autograd.grad(out, args, grad_outputs=lt, create_graph=True)
    ref_g = ev.step_rk4_vjp(*[a.detach() for a in args[:4]], args[4].detach(), *lt, want_dt=True)
    for a, b in zip(g, ref_g):
        assert torch.equal(a.detach(), b)
    hv = torch.autograd.grad(sum((gi * vi).sum() for gi, vi in zip(g, vt)), args)
    ref = ev.step_rk4_hvp(*[a.detach() for a in args[:4]], args[4].detach(), lt, vt, want_dt=True)
    for a, b in zip(hv, ref):
        assert torch.allclose(a, b, rtol=1e-12, atol=1e-12 * float(b.abs().max()))
