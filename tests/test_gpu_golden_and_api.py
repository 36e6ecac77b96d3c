"""GPU tests beyond raw kernel parity (run with -m gpu on a B200):
  * the reference's golden vectors (SURVEY.md §4 table) reproduced ON THE GPU through the batched OCP layer;
  * the CasADi-Function look-alike (reference call convention) against the oracle;
  * the host pipeline (pinned host in / host out) against direct device calls;
  * size-independent properties at the BASELINE.json full size (C2: 100 nodes x 65,536 scenarios):
    RNEA(FD(tau)) = tau, Jacobian-vector consistency, shard invariance, per-scenario reduction vs torch.
"""
import os

import numpy as np
import pytest

from conftest import rel_err, rel_err_rows

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-9


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


def test_golden_solutions_on_gpu(torch_mod):
    torch = torch_mod
    from mpc_fatigue_b200.model import data_urdf
    from mpc_fatigue_b200.ocp import DualArmBoxOCP
    sols = np.load(os.path.join(GOLD, "plotter_solutions.npz"))
    ocp = DualArmBoxOCP(data_urdf("pilz6_first"), data_urdf("pilz6_second"))
    for key, euler_tol in (("Result_1", 1e-12), ("Result_2", 1e-12), ("Result_4", 5e-10), ("plotter", 1e-9)):
        s = DualArmBoxOCP.parse_solution(sols[key])
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda().unsqueeze(0)
        r = ocp.evaluate(t(s["q"]), t(s["qd"]), t(s["F_LR"]), t(s["F_RR"]))
        assert float(r["defect_L"].abs().max()) < euler_tol and float(r["defect_R"].abs().max()) < euler_tol
        assert float((r["dist2"] - 0.04).abs().max()) < 1e-7
        assert float(r["force_eq"].abs().max()) < 1.1e-4 and float(r["moment_eq"].abs().max()) < 1.1e-4
        if key != "plotter":
            E1, E2 = r["E_L"][0, 0].cpu().numpy(), r["E_R"][0, 0].cpu().numpy()
            assert np.abs(E1 - [0.2, 0.6, 0.4]).max() < 2e-6 and np.abs(E2 - [0.4, 0.6, 0.4]).max() < 2e-6
            R1 = r["R_L"][0, 0].cpu().numpy()
            assert np.abs(R1 - [[0, 0, 1], [0, 1, 0], [-1, 0, 0]]).max() < 2e-3
        if key == "Result_2":  # active torque bounds, nodes 53..79 (right arm)
            tr = r["tau_R"][0, 53:, :3].cpu().numpy()
            assert np.abs(tr - [-5.0, 5.0, 5.0]).max() < 4e-7
        if key == "Result_4":  # left arm rows on +5
            assert float((r["tau_L"][0, 53:, :2] - 5.0).abs().max()) < 2e-7


def test_function_lookalike_matches_oracle(torch_mod):
    torch = torch_mod
    from mpc_fatigue_b200.model import data_urdf
    from mpc_fatigue_b200.pynocchio_casadi import (Function, generate_forward_kin, generate_fwd_dyn_fatigue_step, generate_inv_dyn,
                                                   generate_jacobian)
    from oracle.pyoracle import Oracle
    from oracle.urdf_model import load_urdf
    xml = data_urdf("pilz6_second")
    om = load_urdf(xml, armature=1e-2)
    orc = Oracle(om)
    rng = np.random.default_rng(0)
    Idyn = Function.deserialize(generate_inv_dyn(xml))
    fk = Function.deserialize(generate_forward_kin(xml, "end_effector"))
    jac = Function.deserialize(generate_jacobian(xml, "end_effector"))
    fid = om.frame_id("end_effector")
    # single node, keyword call -> dict (the reference idiom), numpy in -> numpy out
    q, qd, qdd = rng.uniform(-2, 2, 6), rng.uniform(-1, 1, 6), np.zeros(6)
    out = Idyn(q=q, qdot=qd, qddot=qdd)
    c = lambda v: np.ascontiguousarray(np.asarray(v, dtype=float).reshape(-1, 6).T)
    assert set(out) == {"tau"} and out["tau"].shape == (6,)
    assert rel_err(out["tau"], orc.rnea(c(q), c(qd), c(qdd))[:, 0]) < TOL
    # positional call -> bare output; CasADi column vectors [n, 1] accepted
    J = jac(q.reshape(6, 1))
    assert J.shape == (6, 6) and rel_err(J, orc.jacobian(fid, c(q))[:, 0].reshape(6, 6)) < TOL
    assert rel_err(jac(q=q)["J"][0:6, 0:6], J) == 0.0  # the callers' slicing idiom (force_optimization_pilz_6DOF.py:130)
    pos, rot = fk(q)
    rp, rr = orc.fk(fid, c(q))
    assert rel_err(pos, rp[:, 0]) < TOL and rel_err(rot, rr[:, 0].reshape(3, 3)) < TOL
    # batched [B, N, n] in one call; torch CUDA in -> torch CUDA out
    Q = torch.from_numpy(rng.uniform(-2, 2, (3, 5, 6))).cuda()
    QD = torch.from_numpy(rng.uniform(-1, 1, (3, 5, 6))).cuda()
    tau = Idyn(Q, QD, torch.zeros_like(Q))
    assert tau.is_cuda and tuple(tau.shape) == (3, 5, 6)
    ref = orc.rnea(c(Q.cpu().numpy()), c(QD.cpu().numpy()), None).T.reshape(3, 5, 6)
    assert rel_err(tau.cpu().numpy(), ref) < TOL
    # omitted keyword input defaults to zero (CasADi semantics): qddot omitted == qddot = 0
    assert rel_err(Idyn(q=q, qdot=qd)["tau"], out["tau"]) == 0.0
    # north-star Function and its Jacobian
    step = Function.deserialize(generate_fwd_dyn_fatigue_step(xml, {"armature": 1e-2}))
    tq, f = rng.uniform(-5, 5, (4, 6)), rng.uniform(20, 80, (4, 6))
    q4, qd4 = rng.uniform(-2, 2, (4, 6)), rng.uniform(-1, 1, (4, 6))
    res = step(q=q4, qd=qd4, tau=tq, f=f, dt=0.02)
    rq, rqd, rf, rj = orc.step_rk4_jvp(c(q4), c(qd4), c(tq), c(f), 0.02)
    assert rel_err_rows(res["q_next"].T, rq) < TOL and rel_err_rows(res["qd_next"].T, rqd) < TOL and rel_err_rows(res["f_next"].T, rf) < TOL
    Jd = step.jacobian()(q4, qd4, tq, f, 0.02)
    assert Jd.shape == (4, 18, 25) and rel_err(Jd, np.moveaxis(rj, 2, 0)) < TOL


def test_pilz_force_ocp_rows_and_their_jacobian(torch_mod):
    """The batched 6-DOF force OCP (force_optimization_pilz_6DOF.py:103-178): g-rows vs the oracle, and the Jacobian
    blocks an NLP solver needs vs central differences of the rows themselves."""
    torch = torch_mod
    from mpc_fatigue_b200.model import data_urdf
    from mpc_fatigue_b200.ocp import PilzForceOCP
    from oracle.pyoracle import Oracle
    from oracle.urdf_model import load_urdf
    xml = data_urdf("pilz6")
    ocp = PilzForceOCP(xml, frame="prbt_link_5", N=6, T=2.0)
    om = load_urdf(xml)
    orc = Oracle(om)
    g = torch.Generator(device="cuda").manual_seed(3)
    B, N = 4, 6
    q = (torch.rand((B, N + 1, 6), generator=g, dtype=torch.float64, device="cuda") - 0.5) * 3.0
    qd = (torch.rand((B, N, 6), generator=g, dtype=torch.float64, device="cuda") - 0.5) * 2.0
    Fx = (torch.rand((B, N), generator=g, dtype=torch.float64, device="cuda") - 0.5) * 80.0
    rows = ocp.evaluate(q, qd, Fx, ref_xy=(0.1, 0.2))
    # rows against the oracle
    c = lambda t: np.ascontiguousarray(t.reshape(-1, t.shape[-1]).T.cpu().numpy())
    W = np.zeros((6, B * N)); W[0] = Fx.reshape(-1).cpu().numpy()
    fr = om.frame_id("prbt_link_5")
    rt, rqn, _ = orc.node_eval_ref([fr], -1.0, c(q[:, :N]), c(qd), W, np.zeros((6, B * N)), ocp.h)
    assert rel_err(c(rows["tau"]), rt) < TOL
    assert rel_err(c(rows["defect"]), rqn - c(q[:, 1:])) < TOL
    pos, _ = orc.fk(fr, c(q[:, :N]))
    assert rel_err(c(rows["line"]), pos[:2] - np.array([[0.1], [0.2]])) < TOL
    assert rows["tau_bound"][0] == 50.0 and float(rows["cost"][0]) == float(-(Fx[0] ** 2).sum())
    # Jacobian blocks against central differences of the rows
    jac = ocp.jacobian(q, qd, Fx)
    eps = 1e-6
    for j in range(6):
        dq = torch.zeros_like(q); dq[:, :N, j] = eps
        rp, rm = ocp.evaluate(q + dq, qd, Fx, (0.1, 0.2)), ocp.evaluate(q - dq, qd, Fx, (0.1, 0.2))
        assert float(((rp["tau"] - rm["tau"]) / (2 * eps) - jac["dtau_dq"][..., j]).abs().max()) < 2e-5
        assert float(((rp["line"] - rm["line"]) / (2 * eps) - jac["dline_dq"][..., j]).abs().max()) < 1e-7
        dv = torch.zeros_like(qd); dv[..., j] = eps
        rp, rm = ocp.evaluate(q, qd + dv, Fx, (0.1, 0.2)), ocp.evaluate(q, qd - dv, Fx, (0.1, 0.2))
        assert float(((rp["tau"] - rm["tau"]) / (2 * eps) - jac["dtau_dqd"][..., j]).abs().max()) < 2e-6
    rp, rm = ocp.evaluate(q, qd, Fx + eps, (0.1, 0.2)), ocp.evaluate(q, qd, Fx - eps, (0.1, 0.2))
    assert float(((rp["tau"] - rm["tau"]) / (2 * eps) - jac["dtau_dFx"]).abs().max()) < 1e-7


def test_singular_forward_dynamics_is_an_error_not_a_nan(torch_mod):
    torch = torch_mod
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from mpc_fatigue_b200.model import Model, data_urdf
    m = Model.from_urdf(data_urdf("pilz6"), armature=0.0)  # zero-inertia flange
    ev = BatchEvaluator(m)
    z = torch.zeros((6, 4), dtype=torch.float64, device="cuda")
    with pytest.raises(ZeroDivisionError, match="armature"):
        ev.aba(z, z, z)
    with pytest.raises(ZeroDivisionError):
        ev.step_rk4(z, z, z, z, 0.01)
    ev.rnea(z, z)  # inverse dynamics is fine without armature (the reference's case)
    with pytest.raises(ValueError):
        ev.rnea(z.cpu(), z)
    with pytest.raises(ValueError):
        ev.rnea(z[:, :3], z)
    assert tuple(ev.rnea(z[:, :0].contiguous(), z[:, :0].contiguous()).shape) == (6, 0)  # empty batch


# Host pipeline cases beyond the three of test_host_pipeline_matches_direct_calls:
# (B, N, chunk_units, skip_structural_zeros, outputs, with_jacobian).  B = 1009, N = 5, chunk_units = 505: Bc = 101 scenarios and
# 505 units per chunk, odd, so the plane gather takes its scalar path and the 2-D copies odd pitches; chunk_units < N: one
# scenario per chunk (Bc = 1); "reused": one pipeline object run again with the same (B, N), then another (B, N), then the first.
PIPELINE_CASES = {
    "1009x5": (1009, 5, 505, False, "all", True),
    "1009x5_skip": (1009, 5, 505, True, "all", True),
    "1009x5_reduced": (1009, 5, 505, False, "reduced", True),
    "1009x5_skip_reduced": (1009, 5, 505, True, "reduced", True),
    "no_jacobian": (300, 6, 6 * 64, False, "all", False),
    "no_jacobian_reduced": (300, 6, 6 * 64, True, "reduced", False),
    "one_scenario_per_chunk": (9, 7, 3, False, "all", True),
    "one_scenario_per_chunk_skip": (9, 7, 3, True, "all", True),
    "reused": (1009, 5, 505, False, "all", True),
    "reused_skip": (1009, 5, 505, True, "all", True),
}


def _pipeline_check(torch, pipe, m, B, N, seed):
    """One run of `pipe` against direct step_rk4_jvp (step_rk4 without Jacobian) plus cost_residual calls on the device:
    every returned chunk and the reduced rows bit for bit, and the byte counts."""
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from mpc_fatigue_b200.synth import synth_batch
    ev = BatchEvaluator(m)
    n, dt = m.n, 0.02
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    q, qd, tau, f = synth_batch(lim, 0, B, N, seed=seed, device="cuda")
    if pipe.with_jacobian:
        qn, qdn, fn, jac = ev.step_rk4_jvp(q, qd, tau, f, dt)
        full = torch.cat([qn, qdn, fn, jac.reshape(-1, B * N)])
    else:
        qn, qdn, fn = ev.step_rk4(q, qd, tau, f, dt)
        full = torch.cat([qn, qdn, fn])
    red = ev.cost_residual(B, N, q, qd, f, tau, qn, qdn, fn, dt)
    full = full.reshape(-1, N, B).cpu()
    host = [t.cpu().pin_memory() for t in (q, qd, tau, f)]
    got = {}
    stats = pipe.run(*host, dt, B, N, consume=lambda v, b0, b1: got.__setitem__((b0, b1), v.clone()))
    Bc = max(1, min(B, pipe.chunk_units // N))
    bounds = [(b0, min(B, b0 + Bc)) for b0 in range(0, B, Bc)]
    hrows = len(pipe.plane_map)
    assert stats["chunks"] == len(bounds) and stats["h2d_bytes"] == 4 * n * B * N * 8
    assert torch.equal(pipe.h_red, red.cpu())
    if pipe.outputs == "reduced":
        assert not got and stats["d2h_bytes"] == 4 * B * 8
        return full, stats
    assert sorted(got) == bounds and stats["d2h_bytes"] == hrows * B * N * 8 + 4 * B * 8
    sel = torch.tensor(pipe.plane_map)
    for (b0, b1), v in got.items():
        assert torch.equal(v, full[sel][:, :, b0:b1]), (b0, b1)
    return full, stats


def _pipeline_case(torch, m, B, N, chunk, skip, outputs, with_jac):
    """a pipeline of these options against the direct calls, plus what its plane selection implies"""
    from mpc_fatigue_b200.pipeline import HostStepPipeline
    pipe = HostStepPipeline(m, "cuda:0", chunk_units=chunk, with_jacobian=with_jac, skip_structural_zeros=skip, outputs=outputs)
    full, stats = _pipeline_check(torch, pipe, m, B, N, seed=B + N)
    if skip and with_jac:  # structural zeros stay on the device: 348 of 450 Jacobian planes travel, packed on the device
        assert len(pipe.plane_map) == 18 + 348 and not pipe.identity_map
        if outputs == "all":
            dropped = sorted(set(range(468)) - set(pipe.plane_map))
            assert len(dropped) == 102 and float(full[torch.tensor(dropped)].abs().max()) == 0.0
    if not with_jac:
        assert pipe.plane_map == list(range(18)) and pipe.identity_map
    return pipe, stats


def test_host_pipeline_matches_direct_calls(torch_mod):
    torch = torch_mod
    from mpc_fatigue_b200.model import Model, data_urdf
    from mpc_fatigue_b200.pipeline import HostStepPipeline
    m = Model.from_urdf(data_urdf("pilz6"), armature=1e-2)
    B, N = 700, 7
    pipe, stats = _pipeline_case(torch, m, B, N, N * 256, False, "all", True)
    assert stats["chunks"] == 3 and pipe.identity_map  # 3 ragged chunks
    assert stats["d2h_bytes"] == (18 + 450) * B * N * 8 + 4 * B * 8
    _, st2 = _pipeline_case(torch, m, B, N, N * 256, True, "all", True)
    assert st2["d2h_bytes"] == (18 + 348) * B * N * 8 + 4 * B * 8
    # outputs="reduced": same computation, only the per-scenario rows come back
    _, st3 = _pipeline_case(torch, m, B, N, N * 256, False, "reduced", True)
    assert st3["d2h_bytes"] == 4 * B * 8 and st3["h2d_bytes"] == stats["h2d_bytes"]
    with pytest.raises(ValueError):
        HostStepPipeline(m, "cuda:0", outputs="none")


@pytest.mark.parametrize("case", list(PIPELINE_CASES))
def test_host_pipeline_edge_cases_match_direct_calls(torch_mod, case):
    torch = torch_mod
    from mpc_fatigue_b200.model import Model, data_urdf
    B, N, chunk, skip, outputs, with_jac = PIPELINE_CASES[case]
    m = Model.from_urdf(data_urdf("pilz6"), armature=1e-2)
    pipe, stats = _pipeline_case(torch, m, B, N, chunk, skip, outputs, with_jac)
    if case.startswith("reused"):
        for B2, N2, seed in ((B, N, 2), (257, 3, 3), (B, N, 4)):
            _pipeline_check(torch, pipe, m, B2, N2, seed)
    if case.startswith("one_scenario_per_chunk"):
        assert stats["chunks"] == B


def test_full_size_properties(torch_mod):
    """BASELINE.json config 2 size (U = 6,553,600): properties that need no oracle run."""
    torch = torch_mod
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from mpc_fatigue_b200.model import Model, data_urdf
    from mpc_fatigue_b200.synth import synth_batch
    m = Model.from_urdf(data_urdf("pilz6"), armature=1e-2)
    ev = BatchEvaluator(m)
    B, N, dt = 65536, 100, 0.02
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    q, qd, tau, f = synth_batch(lim, 0, B, N, device="cuda")
    # (1) inverse o forward dynamics = identity on every unit
    back = ev.rnea(q, qd, ev.aba(q, qd, tau))
    assert float(((back - tau).abs().amax(1) / tau.abs().amax(1)).max()) < 1e-9
    # (2) values-only step == primal outputs of the Jacobian kernel, bit for bit or within 1e-12 relative
    qn, qdn, fn = ev.step_rk4(q, qd, tau, f, dt)
    U = B * N
    sl = slice(U - 131072 - 17, U)  # ragged tail slice through the Jacobian kernel
    cq, cqd, ctau, cf = (t[:, sl].contiguous() for t in (q, qd, tau, f))
    jq, jqd, jf, jac = ev.step_rk4_jvp(cq, cqd, ctau, cf, dt)
    for a, b in ((jq, qn[:, sl]), (jqd, qdn[:, sl]), (jf, fn[:, sl])):
        assert float(((a - b).abs().amax(1) / b.abs().amax(1).clamp_min(1.0)).max()) < 1e-12
    # (3) Jacobian-vector product vs a central difference of the GPU step along a random direction
    g = torch.Generator(device="cuda").manual_seed(5)
    d = [torch.randn(cq.shape, generator=g, dtype=torch.float64, device="cuda") for _ in range(4)]
    eps = 1e-6
    p = ev.step_rk4(cq + eps * d[0], cqd + eps * d[1], ctau + eps * d[2], cf + eps * d[3], dt)
    mns = ev.step_rk4(cq - eps * d[0], cqd - eps * d[1], ctau - eps * d[2], cf - eps * d[3], dt)
    fd = torch.cat([(a - b) / (2 * eps) for a, b in zip(p, mns)])
    jv = torch.einsum("rcu,cu->ru", jac[:, :24], torch.cat(d))
    err = (fd - jv).abs().amax(1) / jv.abs().amax(1).clamp_min(1.0)
    assert float(err.max()) < 5e-6, err
    # (4) shard invariance: scenario block evaluated alone == the same scenarios inside the big batch
    b0, b1 = 40000, 40000 + 4096
    blk = synth_batch(lim, b0, b1 - b0, N, device="cuda")
    sq, sqd, sf = ev.step_rk4(*blk, dt)
    view = lambda t: t.reshape(6, N, B)[:, :, b0:b1].reshape(6, -1)
    assert torch.equal(sq, view(qn)) and torch.equal(sqd, view(qdn)) and torch.equal(sf, view(fn))
    # (5) per-scenario reduction vs torch
    red = ev.cost_residual(B, N, q, qd, f, tau, qn, qdn, fn, dt)
    cost = (1.0 * qd.reshape(6, N, B) ** 2 + 1e-2 * tau.reshape(6, N, B) ** 2).sum((0, 1))
    assert float(((red[0] - cost).abs() / cost).max()) < 1e-12
    defect = torch.cat([(a.reshape(6, N, B)[:, :-1] - b.reshape(6, N, B)[:, 1:]).abs() for a, b in ((qn, q), (qdn, qd), (fn, f))]).amax((0, 1))
    assert torch.equal(red[1], defect)
    bound = torch.clamp(50.0 * torch.exp(-2.0 * dt * torch.arange(N, dtype=torch.float64, device="cuda")), min=15.0).reshape(1, N, 1)
    viol = (tau.reshape(6, N, B).abs() - bound).amax((0, 1)).clamp_min(0.0)
    assert float((red[2] - viol).abs().max()) < 1e-12
    assert torch.equal(red[3], (fn - 80.0).reshape(6, N, B).amax((0, 1)).clamp_min(0.0))
