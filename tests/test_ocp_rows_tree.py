"""Fused reference-mode OCP node rows on run-time-topology models (include/mpcf.h: mpcf_ocp_rows_batch / mpcf_ocp_rows_count_arms,
csrc/kernels_rows.cu: RowsBody / RowsJacBody; oracle/core.inc.h: ocp_rows): branched trees with a torso joint shared by
both arms, a humanoid holding a box with both hands, prismatic and continuous joints, a world-fixed second frame.

CPU: the row counts of every family.  GPU: rows, cost and every derivative output against the oracle on ragged sizes; optional
inputs absent; the run-time-tree and compile-time instantiations on the same two Pilz arms (torso held at zero); FusedBoxOCP
against the per-function composition; canary gaps around every output, compile-time families included; argument rejection,
and the frame checks of the compile-time families."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT, oracle_model_from_export, random_inputs, rel_err_rows
from mpc_fatigue_b200 import _capi
from mpc_fatigue_b200.model import Model, data_urdf
from oracle.pyoracle import Oracle

GOLD = os.path.join(ROOT, "tests", "golden")


def _golden(name):
    with open(os.path.join(GOLD, name + ".urdf")) as fh:
        return fh.read()


def _model(name):
    if name == "pilz6x2_torso":
        return Model.from_urdf(_golden("pilz6x2_torso"), armature=1e-2)
    if name == "mixed_joints":
        return Model.from_urdf(_golden("mixed_joints"), armature=1e-2)
    if name == "dual_arm10":
        return Model.synthetic("dual_arm", 10, seed=3, armature=1e-2)
    if name == "humanoid37":
        return Model.synthetic("humanoid", 37, seed=7, armature=1e-2)
    if name in ("pilz6", "pilz6x2"):
        return Model.from_urdf(data_urdf(name), armature=1e-2)
    if name == "dual_arm14":
        return Model.synthetic("dual_arm", 14, seed=3, armature=1e-2)
    raise KeyError(name)


def _inputs(om, B, N, narm, seed):
    """q, qd, F, T, q_last, T_last, rel_pos0, rel_ori0 in the value ranges of the other row tests"""
    U = B * N
    q, qd, _, T, _ = random_inputs(om, U, seed=seed)
    rng = np.random.default_rng(seed + 1)
    c = lambda a: np.ascontiguousarray(a)
    return (q, qd, c(rng.uniform(-60, 60, (3 * narm, U))), T, c(rng.uniform(-1, 1, (om.n, B))), c(rng.uniform(20, 80, (om.n, B))),
            c(rng.uniform(-0.5, 0.5, (3, B))), c(rng.uniform(-0.5, 0.5, (3, B))))


OPTS2 = dict(wsign=+1.0, fdes=(0.0, 0.0, 9.81 * 30), dist2_ref=0.04, mu=0.5, p_ref=(0.3, 0.6, 0.4), w_box=1000.0, w_qd=100.0, w_F=10.0, h=0.5)
OPTS1 = dict(OPTS2, wsign=-1.0, w_F=-1.0)
KW = ("wsign", "fdes", "dist2_ref", "mu", "p_ref", "w_box", "w_qd", "w_F", "h")

# (case id, model, end-effector frames)
CASES = [
    ("pilz6x2_torso", "pilz6x2_torso", ["end_effector", "sec_end_effector"]),   # both arms on a torso joint (generic16)
    ("dual_arm10", "dual_arm10", ["left_ee", "right_ee"]),                     # two separate chains, not a forest family
    ("humanoid37_hands", "humanoid37", ["larm_ee", "rarm_ee"]),                 # generic64: shared root chain, prismatic roots
    ("humanoid37_one", "humanoid37", ["larm_ee"]),
    ("mixed_joints_one", "mixed_joints", ["tip"]),                              # prismatic + continuous joints
    ("torso_world_fixed", "pilz6x2_torso", ["end_effector", "world"]),         # second frame has no parent joint
]
SIZES = [(1, 1), (33, 1), (1, 5), (37, 5), (257, 5)]


def test_ocp_rows_count_arms_on_every_family():
    models = {"pilz3": (Model.from_urdf(data_urdf("pilz3")), "chain3", 1), "pilz6": (Model.from_urdf(data_urdf("pilz6")), "chain6", 1),
              "chain7": (Model.synthetic("chain", 7, seed=4), "chain7", 1), "pilz6x2": (_model("pilz6x2"), "forest12x6", 2),
              "dual_arm14": (Model.synthetic("dual_arm", 14, seed=3), "forest14x7", 2),
              "pilz6x2_torso": (_model("pilz6x2_torso"), "generic16", 0), "mixed_joints": (_model("mixed_joints"), "generic16", 0),
              "humanoid37": (_model("humanoid37"), "generic64", 0)}
    for name, (m, fam, arms) in models.items():
        assert m.kernel_family == fam, name
        for narm in (0, 3, -1):
            assert _capi.lib.mpcf_ocp_rows_count_arms(m.handle, narm) == _capi.EINVAL, (name, narm)
        for narm in (1, 2):
            want = (26 if narm == 2 else 3) + 3 * m.n
            got = _capi.lib.mpcf_ocp_rows_count_arms(m.handle, narm)
            assert got == (want if arms in (0, narm) else _capi.EINVAL), (name, narm, got)
        # the compile-time count is unchanged, and still refuses run-time trees
        assert _capi.lib.mpcf_ocp_rows_count(m.handle) == (_capi.lib.mpcf_ocp_rows_count_arms(m.handle, arms) if arms else _capi.EINVAL), name
    assert _capi.lib.mpcf_ocp_rows_count_arms(None, 1) == _capi.EINVAL


def test_torso_model_layout():
    m = _model("pilz6x2_torso")
    assert m.n == 13 and m.kernel_family == "generic16"
    par = m.export("parent").tolist()
    assert m.joint_names[0] == "torso_yaw" and par[0] == -1
    assert par[m.joint_names.index("prbt_joint_1")] == 0 and par[m.joint_names.index("sec_prbt_joint_1")] == 0
    assert m.export("fparent")[m.frame_id("world")] == -1


def _run(name, frames, B, N, seed, derivatives=True):
    """oracle and GPU rows of one case: (model, oracle, evaluator, frame ids, inputs, opts, oracle (rows, cost, kin_jac), GPU outputs)"""
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m = _model(name)
    om = oracle_model_from_export(m)
    orc, ev = Oracle(om), BatchEvaluator(m)
    narm = len(frames)
    ee = [m.frame_id(f) for f in frames]
    x = _inputs(om, B, N, narm, seed)
    q, qd, F, T, q_last, T_last, rp0, ro0 = x
    opts = dict(OPTS2 if narm == 2 else OPTS1, narm=narm, ee_frame=ee)
    two = narm == 2
    ref = orc.ocp_rows(opts, B, N, q, qd, F, T, q_last, T_last, rp0 if two else None, ro0 if two else None, kin_jac=True)
    g = lambda a: None if a is None else torch.from_numpy(a).cuda()
    kw = {k: opts[k] for k in KW}
    out = ev.ocp_rows(B, N, ee, g(q), g(qd), g(F), g(T), g(q_last), g(T_last), g(rp0) if two else None, g(ro0) if two else None,
                      derivatives=derivatives, **kw)
    torch.cuda.synchronize()
    return m, orc, ev, ee, x, opts, ref, [None if t is None else t.cpu().numpy() for t in out]


@pytest.mark.gpu
@pytest.mark.parametrize("B,N", SIZES)
@pytest.mark.parametrize("case,name,frames", CASES, ids=[c[0] for c in CASES])
def test_gpu_tree_ocp_rows_against_the_oracle(case, name, frames, B, N):
    m, orc, ev, ee, x, opts, (rrows, rcost, rJ), (rows, cost, dF, dT, kj) = _run(name, frames, B, N, seed=60 + B + N)
    q, qd, F, T = x[:4]
    n, U, narm = m.n, B * N, len(frames)
    kin = 26 if narm == 2 else 3
    assert rows.shape == (kin + 3 * n, U) and dF.shape == (n, 3 * narm, U) and dT.shape == (n, U) and kj.shape == (kin, n + 3 * narm, U)
    assert rel_err_rows(rows, rrows) <= 1e-9
    assert np.abs(cost - rcost).max() <= 1e-9 * max(1.0, np.abs(rcost).max())
    assert rel_err_rows(kj.reshape(-1, U), rJ.reshape(-1, U)) <= 1e-9
    # d tau / d F = wsign J_c,lin^T of every arm's end-effector (oracle frame Jacobian rows 0-2): both arm blocks on shared ancestors
    for c in range(narm):
        J = orc.jacobian(ee[c], q).reshape(6, n, U)
        assert rel_err_rows(dF[:, 3 * c:3 * c + 3].reshape(-1, U), (opts["wsign"] * J[:3].transpose(1, 0, 2)).reshape(-1, U)) <= 1e-9, c
    # d T+ / d tau by central differences of the oracle's ZOH map at the computed torque
    tau = rrows[kin:kin + n]
    eps = 1e-4
    fd = (orc.fatigue_zoh(T, tau + eps, qd, opts["h"]) - orc.fatigue_zoh(T, tau - eps, qd, opts["h"])) / (2 * eps)
    assert np.abs(dT - fd).max() < 1e-7 * max(1.0, np.abs(fd).max())


def test_shared_ancestor_cases_have_cross_arm_blocks():
    """the oracle's frame Jacobians of the torso and humanoid cases overlap on the shared joints (what the GPU test then checks)"""
    for name, frames, shared in (("pilz6x2_torso", ["end_effector", "sec_end_effector"], ["torso_yaw"]),
                                 ("humanoid37", ["larm_ee", "rarm_ee"], ["root_px", "root_rz", "torso"])):
        m = _model(name)
        om = oracle_model_from_export(m)
        q = random_inputs(om, 3, seed=1)[0]
        JL, JR = (Oracle(om).jacobian(m.frame_id(f), q).reshape(6, m.n, 3) for f in frames)
        for j in (m.joint_names.index(s) for s in shared):
            assert np.abs(JL[:3, j]).max() > 1e-3 and np.abs(JR[:3, j]).max() > 1e-3, (name, j)


@pytest.mark.gpu
@pytest.mark.parametrize("case,name,frames", CASES, ids=[c[0] for c in CASES])
def test_gpu_tree_ocp_rows_optional_inputs_absent(case, name, frames):
    import torch
    B, N = 37, 5
    m, orc, ev, ee, x, opts, _, (rows, cost) = _run(name, frames, B, N, seed=70, derivatives=False)
    q, qd, F, T, q_last, T_last, rp0, ro0 = x
    n, narm = m.n, len(frames)
    kin = 26 if narm == 2 else 3
    g = lambda a: torch.from_numpy(a).cuda()
    rows2, cost2 = ev.ocp_rows(B, N, ee, g(q), g(qd), g(F), **{k: opts[k] for k in KW})
    r2 = rows2.cpu().numpy()
    assert not r2[kin + 2 * n:].any()                                       # thermal rows
    assert not r2[kin + n:kin + 2 * n, (N - 1) * B:].any()                  # last node's Euler defects
    assert np.array_equal(r2[kin + n:kin + 2 * n, :(N - 1) * B], rows[kin + n:kin + 2 * n, :(N - 1) * B])
    assert np.array_equal(r2[kin:kin + n], rows[kin:kin + n])                # torque rows
    assert np.array_equal(cost2.cpu().numpy(), cost)
    if narm == 2:  # rel_pos0 / rel_ori0 = 0: the relative-pose rows shift by exactly those inputs, every other row is unchanged
        keep = [r for r in range(26) if not 7 <= r < 13]
        assert np.array_equal(r2[keep], rows[keep])
        assert np.array_equal(r2[7:10, B:], rows[7:10, B:])
        assert np.abs(r2[7:10, :B] - (rows[7:10, :B] + rp0)).max() < 1e-12
        assert np.abs(r2[10:13] - (rows[10:13] + np.tile(ro0, (1, N)))).max() < 1e-12
    else:
        assert np.array_equal(r2[:3], rows[:3])


@pytest.mark.gpu
def test_gpu_tree_kernels_agree_with_the_compile_time_kernels():
    """pilz6x2_torso (run-time tree: the GenericModel instantiation of the row bodies, torso angle / velocity / temperature held
    at 0) against pilz6x2 (forest12x6: their StaticModel instantiation) on the same arm inputs.  At zero angle the torso rotation
    is exactly the identity: only the order of summation differs, so every compared plane agrees to 1e-11 of its own scale
    (rel_err_rows).  Planes whose exact value is zero (joint 6 of each arm: the end-effector frame lies on its axis and the
    flange carries no mass, so its torque and Jacobian column vanish) hold only rounding noise — about 1e-15, from the forces'
    moments about joint origins a flange length apart and the Jacobian columns' cross products, which the 1e-6 floor of
    rel_err_rows would count as 3e-11 — and must be zero to 1e-12 of their block's scale in both instantiations."""
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    mt, ms = _model("pilz6x2_torso"), _model("pilz6x2")
    assert ms.kernel_family == "forest12x6" and mt.kernel_family == "generic16"
    idx = [mt.joint_names.index(nm) for nm in ms.joint_names]
    nt, ns = mt.n, ms.n
    B, N = 37, 5
    U = B * N
    q, qd, F, T, q_last, T_last, rp0, ro0 = _inputs(oracle_model_from_export(ms), B, N, 2, seed=80)

    def lift(a):
        out = np.zeros((nt, a.shape[1]))
        out[idx] = a
        return out
    g = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    kw = {k: OPTS2[k] for k in KW}
    res = {}
    for tag, m, lf in (("tree", mt, lift), ("static", ms, lambda a: a)):
        ee = [m.frame_id("end_effector"), m.frame_id("sec_end_effector")]
        out = BatchEvaluator(m).ocp_rows(B, N, ee, g(lf(q)), g(lf(qd)), g(F), g(lf(T)), g(lf(q_last)), g(lf(T_last)), g(rp0), g(ro0),
                                          derivatives=True, **kw)
        res[tag] = [t.cpu().numpy() for t in out]
    (rt, ct, dFt, dTt, kjt), (rs, cs, dFs, dTs, kjs) = res["tree"], res["static"]
    idx = np.array(idx)

    def agree(a, ref, tol=1e-11, noise=1e-12):
        a, ref = a.reshape(-1, U), ref.reshape(-1, U)
        big = np.abs(ref).max()
        # exact zeros held as rounding noise (and structural zeros: d force-rows / d q, F-free rows, cross-arm blocks)
        zero = np.abs(ref).max(axis=1) <= noise * big
        assert (~zero).any()
        return max(rel_err_rows(a[~zero], ref[~zero]) / tol, np.abs(a[zero]).max(initial=0.0) / (noise * big))
    assert agree(rt[:26], rs[:26]) <= 1                                            # kinematic rows
    for blk in range(3):                                                           # arm torque rows, Euler and thermal defects
        assert agree(rt[26 + blk * nt + idx], rs[26 + blk * ns:26 + (blk + 1) * ns]) <= 1, blk
    assert agree(ct[None], cs[None]) <= 1
    assert agree(dTt[idx], dTs) <= 1
    cols = np.concatenate([idx, nt + np.arange(6)])                                # arm joints and the two forces
    assert agree(kjt[:, cols], kjs) <= 1
    assert agree(dFt[idx], dFs) <= 1
    # the torso column is there on the tree (both arms move with it), and the forest's cross-arm blocks are zeros
    assert np.abs(kjt[:, 0]).max() > 1e-3 and np.abs(dFt[0]).max() > 1e-3
    assert not dFs[:6, 3:].any() and not dFs[6:, :3].any()


@pytest.mark.gpu
def test_gpu_fused_box_ocp_on_a_humanoid_agrees_with_the_per_function_composition():
    """FusedBoxOCP (tree kernels) against ThermalMPCNodes.evaluate + box_rows (node_eval_ref / fk launches composed in torch)
    on the 37-joint humanoid carrying the box with both hands."""
    import torch
    from mpc_fatigue_b200.ocp import FusedBoxOCP, ThermalMPCNodes
    m = _model("humanoid37")
    n, B, N = m.n, 9, 6
    names = ["larm_ee", "rarm_ee"]
    g = torch.Generator(device="cuda").manual_seed(5)
    r = lambda *s: torch.rand(*s, dtype=torch.float64, device="cuda", generator=g)
    q, qd = 2 * r(B, N + 1, n) - 1, r(B, N, n) - 0.5
    FL, FR = 40 * (r(B, N, 3) - 0.5), 40 * (r(B, N, 3) - 0.5)
    Temp = 20 + 40 * r(B, N + 1, n)
    rp0, ro0, box0 = r(B, 3) - 0.5, r(B, 3) - 0.5, (0.2, 0.1, 0.5)
    fused = FusedBoxOCP(m, names, p_ref=box0, T=20.0, N=N).evaluate(q, qd, FL, FR, Temp, rp0, ro0)
    old = ThermalMPCNodes(m, names, T=20.0, N=N)
    W = torch.cat([FL, torch.zeros_like(FL), FR, torch.zeros_like(FR)], dim=-1)
    a = old.evaluate(q, qd, W, Temp)
    b = old.box_rows(q, qd, FL, FR, 30.0, rp0, ro0, box0)
    close = lambda x, y: float((x - y).abs().max()) < 1e-9 * max(1.0, float(y.abs().max()))
    assert close(fused["tau"], a["tau"]) and close(fused["q_defect"], a["q_defect"]) and close(fused["T_defect"], a["T_defect"])
    assert close(fused["force_eq"], b["force_eq"]) and close(fused["moment_eq"], b["moment_eq"])
    assert close(fused["rel_pos"], b["rel_pos"]) and close(fused["rel_ori"], b["rel_ori"]) and close(fused["cost"], b["cost"])
    assert close(fused["box_err"], 0.5 * (b["pL"] + b["pR"]) - torch.tensor(box0, dtype=torch.float64, device="cuda"))


GAP = 4096  # doubles on each side of every carved buffer
CANARY = -7.25e300


def _carve(pool, sizes):
    """views of `pool` separated by GAP canary doubles; returns (views, gap slices, total length)"""
    views, gaps, off = [], [], 0
    for sz in sizes:
        gaps.append(slice(off, off + GAP))
        off = (off + GAP + 15) // 16 * 16
        views.append(pool[off:off + sz])
        off += sz
    gaps.append(slice(off, off + GAP))
    return views, gaps, off + GAP


@pytest.mark.gpu
@pytest.mark.parametrize("U", [1, 33, 131])
@pytest.mark.parametrize("name,frames", [("humanoid37", ["larm_ee", "rarm_ee"]), ("pilz6x2_torso", ["end_effector", "sec_end_effector"]),
                                         ("pilz6x2", ["end_effector", "sec_end_effector"]), ("dual_arm14", ["left_ee", "right_ee"]),
                                         ("pilz6", ["prbt_flange"])])
def test_gpu_tree_ocp_rows_outputs_stay_inside_their_buffers(name, frames, U):
    """rows, cost, dtau_dF, dT_dtau and kin_jac carved out of one allocation with canary gaps: no gap written, no element left
    unwritten (structural zeros included).  Buffer sizes follow the arm count."""
    import torch
    B, N = {1: (1, 1), 33: (11, 3), 131: (131, 1)}[U]
    m = _model(name)
    n, narm = m.n, len(frames)
    kin = 26 if narm == 2 else 3
    q, qd, F, T, q_last, T_last, rp0, ro0 = (torch.from_numpy(a).cuda() for a in _inputs(oracle_model_from_export(m), B, N, narm, seed=90))
    sizes = [(kin + 3 * n) * U, U, n * 3 * narm * U, n * U, kin * (n + 3 * narm) * U]
    pool = torch.full((_carve(np.empty(0), sizes)[2],), CANARY, dtype=torch.float64, device="cuda")
    (rows, cost, dF, dT, kj), gaps, _ = _carve(pool, sizes)
    o = _capi.RowsOpts((C.c_int * 2)(*([m.frame_id(f) for f in frames] + [-1] * (2 - narm))), 1.0, (C.c_double * 3)(0.0, 0.0, 294.3), 0.04, 0.5,
                       (C.c_double * 3)(0.3, 0.6, 0.4), 1000.0, 100.0, 10.0, 0.5)
    p = lambda t: C.c_void_p(t.data_ptr())
    _capi.check(_capi.lib.mpcf_ocp_rows_batch(m.handle, C.byref(o), B, N, p(q), p(qd), p(F), p(T), p(q_last), p(T_last), p(rp0), p(ro0),
                                              p(rows), p(cost), p(dF), p(dT), p(kj), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    for i, gp in enumerate(gaps):
        assert bool((pool[gp] == CANARY).all()), (name, U, "canary gap %d was written" % i)
    for buf, nm in ((rows, "rows"), (cost, "cost"), (dF, "dtau_dF"), (dT, "dT_dtau"), (kj, "kin_jac")):
        assert not bool((buf == CANARY).any()), (name, U, nm, "has unwritten elements")
        assert bool(torch.isfinite(buf).all()), (name, U, nm)


@pytest.mark.gpu
@pytest.mark.parametrize("name,frames", [("pilz6x2_torso", ["end_effector", "sec_end_effector"]), ("humanoid37", ["larm_ee", "rarm_ee"])])
def test_gpu_tree_ocp_rows_reject_bad_arguments(name, frames):
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    m = _model(name)
    ev = BatchEvaluator(m)
    B, N, n = 4, 2, m.n
    z = lambda r: torch.zeros((r, B * N), dtype=torch.float64, device="cuda")
    ee = [m.frame_id(f) for f in frames]
    with pytest.raises(IndexError):
        ev.ocp_rows(B, N, [ee[0], m.nframes], z(n), z(n), z(6))
    with pytest.raises(IndexError):
        ev.ocp_rows(B, N, [m.nframes + 5], z(n), z(n), z(3))
    with pytest.raises(IndexError):
        ev.ocp_rows(B, N, [ee[0], -2], z(n), z(n), z(6))
    with pytest.raises(ValueError):
        ev.ocp_rows(B, N, [], z(n), z(n), z(3))
    with pytest.raises(ValueError):
        ev.ocp_rows(B, N, ee + [ee[0]], z(n), z(n), z(9))
    # the C entry itself: a frame index out of range is MPCF_EFRAME
    o = _capi.RowsOpts((C.c_int * 2)(ee[0], m.nframes), 1.0, (C.c_double * 3)(), 0.0, 0.0, (C.c_double * 3)(), 0.0, 0.0, 0.0, 0.0)
    rows, cost = z(26 + 3 * n), z(1)
    p = lambda t: C.c_void_p(t.data_ptr())
    assert _capi.lib.mpcf_ocp_rows_batch(m.handle, C.byref(o), B, N, p(z(n)), p(z(n)), p(z(6)), None, None, None, None, None, p(rows), p(cost),
                                         None, None, None, None) == _capi.EFRAME


@pytest.mark.gpu
def test_gpu_compile_time_families_keep_their_frame_checks():
    """On a forest ee_frame[c] must be carried by arm c: swapped frames, a frame on the other arm and a world-fixed frame are
    MPCF_EFRAME.  On a one-arm chain ee_frame[1] is ignored, whatever it holds."""
    import torch
    m = _model("pilz6x2")
    B, N, n = 4, 2, m.n
    z = lambda r: torch.zeros((r, B * N), dtype=torch.float64, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    L, R = m.frame_id("end_effector"), m.frame_id("sec_end_effector")
    world = m.export("fparent").tolist().index(-1)

    def call(model, frames, kin, narm):
        o = _capi.RowsOpts((C.c_int * 2)(*frames), 1.0, (C.c_double * 3)(), 0.0, 0.0, (C.c_double * 3)(), 0.0, 0.0, 0.0, 0.0)
        rows, cost = z(kin + 3 * model.n), z(1)
        rc = _capi.lib.mpcf_ocp_rows_batch(model.handle, C.byref(o), B, N, p(z(model.n)), p(z(model.n)), p(z(3 * narm)), None, None,
                                           None, None, None, p(rows), p(cost), None, None, None, None)
        torch.cuda.synchronize()
        return rc
    assert call(m, (L, R), 26, 2) == _capi.OK
    for frames in ((R, L), (L, L), (R, R), (world, R), (L, world)):
        assert call(m, frames, 26, 2) == _capi.EFRAME, frames
    one = _model("pilz6")
    tip = one.frame_id("prbt_flange")
    for second in (-1, tip, one.nframes + 5):
        assert call(one, (tip, second), 3, 1) == _capi.OK, second
    assert call(one, (one.export("fparent").tolist().index(-1), -1), 3, 1) == _capi.EFRAME
