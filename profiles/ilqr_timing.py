"""The parts of one iLQR iteration (mpc_fatigue_b200.ilqr.solve_ilqr), each timed on its own:

  jvp       step_rk4_jvp at nodes 0..N-1 of the current trajectory (the Jacobians of the Gauss-Newton model)
  gains     riccati_gains with the tracking cost's gradient and curvature planes (backward pass only)
  costs     ilqr_costs with na = 8 step lengths (the line search: 8 closed-loop rollouts per scenario, no trajectory stored)
  accept    feedback_rollout with per-scenario step lengths and the cost's derivative planes (the next iteration's inputs)
  select    the torch step-length rule on the [8, B] costs

on two workloads: pilz6 (armature 1e-2) at 65,536 scenarios x 100 nodes and dual_arm14 at 16,384 x 100.  Timed with CUDA events
after a warm-up, over enough calls for about one second each; prints ms per call and the device name and power limit.
GPU only: there is no CPU path.

    python profiles/ilqr_timing.py [--seconds 1.0] [--out ilqr_timing.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from mpc_fatigue_b200.evaluator import BatchEvaluator  # noqa: E402
from mpc_fatigue_b200.ilqr import TrackingCost, select_alpha  # noqa: E402
from mpc_fatigue_b200.model import Model, data_urdf  # noqa: E402
from mpc_fatigue_b200.synth import synth_batch  # noqa: E402
from profiles.vjp_timing import device_info, timed  # noqa: E402

ALPHAS = tuple(0.5 ** i for i in range(8))


def case(name, m, B, N, seconds, dt=0.0125):
    n = m.n
    nx, U = 3 * n, B * N
    ev = BatchEvaluator(m)
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    q, qd, tau, f = synth_batch(lim, 0, B, N, seed=1234, device="cuda")
    x0 = torch.cat([q[:, :B], qd[:, :B], f[:, :B]]).contiguous()
    del q, qd, f
    f64 = dict(dtype=torch.float64, device="cuda")
    zero = TrackingCost()
    xref = ev.feedback_rollout(zero, x0, tau, N, dt)[0]
    cost = TrackingCost(x_ref=xref, tau_ref=tau, wx=torch.ones(nx, **f64), wu=torch.full((n,), 1e-2, **f64), wN=torch.ones(nx, **f64),
                        f_max=60.0, rho_f=1.0)
    taub = (tau * 1.01).contiguous()
    x, _, J, dv = ev.feedback_rollout(cost, x0, taub, N, dt, derivatives=True)
    out = {"model": name, "family": m.kernel_family, "n": n, "B": B, "N": N, "na": len(ALPHAS)}
    xs = [x[r * n:(r + 1) * n, :U].contiguous() for r in range(3)]
    jac = torch.empty((nx, 4 * n + 1, U), **f64)
    outs = tuple(torch.empty((n, U), **f64) for _ in range(3))
    out["jvp_ms"] = timed(lambda: ev.step_rk4_jvp(xs[0], xs[1], taub, xs[2], dt, out=outs, jac=jac), seconds)
    del xs, outs
    kw = dict(wx=dv["wx"], wu=dv["wu"] + 1e-8, gx=dv["gx"], gu=dv["gu"], wN=dv["wN"], gN=dv["gN"])
    K = ev.riccati_gains(jac, B, N, **kw)
    out["gains_ms"] = timed(lambda: ev.riccati_gains(jac, B, N, **kw), seconds)
    del jac
    Jc = ev.ilqr_costs(cost, x0, x, taub, K, ALPHAS, N, dt)
    out["costs_ms"] = timed(lambda: ev.ilqr_costs(cost, x0, x, taub, K, ALPHAS, N, dt), seconds)
    alpha, acc = select_alpha(Jc, J, ALPHAS)
    out["select_ms"] = timed(lambda: select_alpha(Jc, J, ALPHAS), seconds)
    out["accept_ms"] = timed(lambda: ev.feedback_rollout(cost, x0, taub, N, dt, xbar=x, K=K, alpha=alpha, derivatives=True), seconds)
    torch.cuda.synchronize()
    out["accepted_fraction"] = float(acc.double().mean())
    out["iteration_ms"] = sum(out[k] for k in ("jvp_ms", "gains_ms", "costs_ms", "select_ms", "accept_ms"))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "ilqr_timing.py needs a CUDA device"
    res = {"device": device_info(), "cases": []}
    res["cases"].append(case("pilz6", Model.from_urdf(data_urdf("pilz6"), armature=1e-2), 65536, 100, a.seconds))
    torch.cuda.empty_cache()
    res["cases"].append(case("dual_arm14", Model.synthetic("dual_arm", 14, seed=3, armature=1e-2), 16384, 100, a.seconds))
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
