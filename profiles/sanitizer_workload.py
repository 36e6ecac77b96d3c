import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from mpc_fatigue_b200.evaluator import BatchEvaluator
from mpc_fatigue_b200.model import Model, data_urdf
from mpc_fatigue_b200.synth import synth_batch
for name, arm in (("pilz6", 1e-2), ("pilz3", 0.0), ("pilz6x2", 1e-2)):
    m = Model.from_urdf(data_urdf(name), armature=arm)
    ev = BatchEvaluator(m)
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    B, N = 77, 3
    q, qd, tau, f = synth_batch(lim, 0, B, N, device="cuda")
    ev.rnea(q, qd); ev.aba(q, qd, tau); ev.step_rk4(q, qd, tau, f, 0.02)
    qn, qdn, fn, jac = ev.step_rk4_jvp(q, qd, tau, f, 0.02)
    ev.step_rk4_jvp(q, qd, tau, f, 0.02, direct=True)
    ev.fd_derivs(q, qd, tau)
    ev.cost_residual(B, N, q, qd, f, tau, qn, qdn, fn, 0.02)
    fr = m.nframes - 1
    ev.fk(fr, q); ev.jacobian(fr, q)
    ev.node_eval_ref([fr], -1.0, q, qd, torch.zeros((6, B*N), dtype=torch.float64, device="cuda"), f, 0.02)
h = Model.synthetic("humanoid", 37, seed=7, armature=1e-2)
ev = BatchEvaluator(h)
lim = {k: h.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
q, qd, tau, f = synth_batch(lim, 0, 40, 1, device="cuda")
ev.rnea(q, qd); ev.step_rk4(q, qd, tau, f, 0.02); ev.step_rk4_jvp(q, qd, tau, f, 0.02)
torch.cuda.synchronize()
print("sanitizer workload done")
