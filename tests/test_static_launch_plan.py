"""Launch plan of the compile-time families (chain3 / chain6 / chain7, forest12x6 / forest14x7).

These families run most entries once per serial chain.  Each test counts the kernels an entry launches
(`mpcf_launch_count`) at a size that fits one workspace chunk, so a chain loop that skips or repeats a chain changes the count
even where the outputs of the skipped chain would go unnoticed."""
import ctypes as C

import numpy as np
import pytest

from conftest import oracle_model_from_export, random_inputs
from mpc_fatigue_b200.model import Model, data_urdf

pytestmark = pytest.mark.gpu

U = 257  # ragged against the 128-thread block; one workspace chunk
MODELS = {
    "pilz3": (lambda: Model.from_urdf(data_urdf("pilz3"), armature=1e-2), "chain3", 1),
    "pilz6": (lambda: Model.from_urdf(data_urdf("pilz6"), armature=1e-2), "chain6", 1),
    "chain7": (lambda: Model.synthetic("chain", 7, seed=2, armature=1e-2), "chain7", 1),
    "pilz6x2": (lambda: Model.from_urdf(data_urdf("pilz6x2"), armature=1e-2), "forest12x6", 2),
    "dual_arm14": (lambda: Model.synthetic("dual_arm", 14, seed=3, armature=1e-2), "forest14x7", 2),
}


def _launches(fn):
    from mpc_fatigue_b200 import _capi
    n0 = _capi.lib.mpcf_launch_count()
    fn()
    return _capi.lib.mpcf_launch_count() - n0


def _setup(name):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    make, family, nchains = MODELS[name]
    m = make()
    assert m.kernel_family == family
    q, qd, tau, f, qdd = (torch.from_numpy(a).cuda() for a in random_inputs(oracle_model_from_export(m), U, seed=3))
    return m, BatchEvaluator(m), nchains, (q, qd, tau, f, qdd)


def _step_jvp_pool(m, q, qd, tau, f):
    """mpcf_step_rk4_jvp_batch: the pipeline on a workspace from the stream-ordered pool."""
    import torch
    from mpc_fatigue_b200 import _capi
    n = m.n
    out = [torch.empty_like(q) for _ in range(3)]
    jac = torch.empty((3 * n, 4 * n + 1, U), dtype=torch.float64, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    _capi.check(_capi.lib.mpcf_step_rk4_jvp_batch(m.handle, U, p(q), p(qd), p(tau), p(f), 0.02, None, *[p(t) for t in out], p(jac),
                                                  C.c_void_p(torch.cuda.current_stream().cuda_stream)))


@pytest.mark.parametrize("name", list(MODELS))
def test_launch_plan(name):
    import torch
    m, ev, nchains, (q, qd, tau, f, qdd) = _setup(name)
    L = m.n // nchains
    fparent = m.export("fparent")
    # the last frame carried by each arm (a frame on arm c picks chain c)
    arm_frames = [int(max(i for i, j in enumerate(fparent) if c * L <= j < (c + 1) * L)) for c in range(nchains)]
    W = torch.from_numpy(np.random.default_rng(4).uniform(-50, 50, (6 * nchains, U))).cuda()
    got, want = {}, {}
    for c, fr in enumerate(arm_frames):
        got["fk arm %d" % c] = _launches(lambda: ev.fk(fr, q))
        got["jacobian arm %d" % c] = _launches(lambda: ev.jacobian(fr, q))
        got["jac_t_wrench arm %d" % c] = _launches(lambda: ev.jac_t_wrench(fr, q, W[:6].contiguous()))
        want.update({"fk arm %d" % c: 1, "jacobian arm %d" % c: 1, "jac_t_wrench arm %d" % c: 1})
    got["node_eval_ref"] = _launches(lambda: ev.node_eval_ref(arm_frames, -1.0, q, qd, W, f, 0.02, qdd=qdd))
    got["node_eval_ref_jvp"] = _launches(lambda: ev.node_eval_ref_jvp(arm_frames, -1.0, q, qd, W, qdd=qdd))
    got["rnea_derivs"] = _launches(lambda: ev.rnea_derivs(q, qd, qdd))
    got["fd_derivs"] = _launches(lambda: ev.fd_derivs(q, qd, tau))
    got["step_rk4_jvp"] = _launches(lambda: _step_jvp_pool(m, q, qd, tau, f))
    got["step_rk4_vjp"] = _launches(lambda: ev.step_rk4_vjp(q, qd, tau, f, 0.02, lq=q, lqd=qd, lf=f, want_dt=True))
    want.update({"node_eval_ref": nchains, "node_eval_ref_jvp": nchains, "rnea_derivs": nchains, "fd_derivs": nchains,
                 # K1, K2, K3 per chain; forests add one pass that zeroes the Jacobian entries between chains
                 "step_rk4_jvp": 3 * nchains + (nchains > 1),
                 # K1, K2 and the reverse sweep per chain
                 "step_rk4_vjp": 3 * nchains})
    torch.cuda.synchronize()
    assert got == want


def test_launch_plan_coupled_forest():
    """With coupled fatigue the forest pipeline is bracketed by the heating-torque kernel and the Jacobian patch."""
    import torch
    from mpc_fatigue_b200.coupling import box_load_coupling
    m, _, nchains, (q, qd, tau, f, _) = _setup("pilz6x2")
    m.set_coupling(box_load_coupling(m))
    assert _launches(lambda: _step_jvp_pool(m, q, qd, tau, f)) == 3 * nchains + 1 + 2
    torch.cuda.synchronize()
