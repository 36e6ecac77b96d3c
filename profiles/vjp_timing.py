"""Reverse mode against the dense forward-mode Jacobian.

  C2  pilz6 (armature 1e-2), 65,536 scenarios x 100 nodes = 6,553,600 units: step_rk4_vjp against step_rk4_jvp
  C4  humanoid37, 32,768 x 40 units in the library's chunks of 32,768 units: step_rk4_vjp against step_rk4_jvp, per chunk
  R   rollout_rk4_vjp at B = 65,536, N = 100 (pilz6) against rollout_rk4 alone

Timed with CUDA events after a warm-up, over enough calls for about one second each.  Prints ms per call, units/s and the
compulsory bytes per unit (inputs read once, outputs written once, from the shapes; the workspace round trip is not counted),
checks in the same run that the VJP equals lambda^T jac of the dense call on a sample of units, and reads the device name and
power limit.  GPU only: there is no CPU path.

    python profiles/vjp_timing.py [--seconds 1.0]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from mpc_fatigue_b200.evaluator import BatchEvaluator  # noqa: E402
from mpc_fatigue_b200.model import Model, data_urdf  # noqa: E402
from mpc_fatigue_b200.synth import synth_batch  # noqa: E402


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = "unavailable (%s)" % e
    return {"device": name, "power_limit, max_sm_clock": out}


def timed(fn, seconds):
    """ms per call: warm-up, a calibration call, then enough calls for ~`seconds` between two CUDA events"""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    reps = max(1, int(seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def check_sample(ev, inputs, dt, lam, jac, cols):
    """max over the sample of |vjp - lambda^T jac| / max(S, 1e-6 max S), S = sum_r |lambda_r| |jac_rc|"""
    g = ev.step_rk4_vjp(*inputs, dt, *lam, want_dt=True)
    got = torch.cat([g[0], g[1], g[2], g[3], g[4][None]])[:, cols]
    L = torch.cat(lam)[:, cols]
    J = jac[:, :, cols]
    ref = torch.einsum("ru,rcu->cu", L, J)
    S = torch.einsum("ru,rcu->cu", L.abs(), J.abs())
    return float(((got - ref).abs() / torch.clamp(S, min=1e-6 * float(S.max()))).max())


def step_case(name, m, B, N, dt, U, seconds):
    ev = BatchEvaluator(m)
    n = m.n
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    inputs = synth_batch(lim, 0, B, N, seed=1234, device="cuda")
    inputs = [t[:, :U].contiguous() for t in inputs]
    gen = torch.Generator(device="cuda").manual_seed(5)
    lam = [torch.randn((n, U), dtype=torch.float64, device="cuda", generator=gen) for _ in range(3)]
    jac = torch.empty((3 * n, 4 * n + 1, U), dtype=torch.float64, device="cuda")
    outs = tuple(torch.empty((n, U), dtype=torch.float64, device="cuda") for _ in range(3))
    t_jvp = timed(lambda: ev.step_rk4_jvp(*inputs, dt, out=outs, jac=jac), seconds)
    t_vjp = timed(lambda: ev.step_rk4_vjp(*inputs, dt, *lam, want_dt=True), seconds)
    cols = torch.linspace(0, U - 1, 512, device="cuda").long()
    err = check_sample(ev, inputs, dt, lam, jac, cols)
    bytes_jvp = 8 * (4 * n + 3 * n + 3 * n * (4 * n + 1))
    bytes_vjp = 8 * (4 * n + 3 * n + 4 * n + 1)
    del jac
    torch.cuda.empty_cache()
    return {"case": name, "units": U, "family": m.kernel_family,
            "jvp_ms": round(t_jvp, 3), "vjp_ms": round(t_vjp, 3), "speedup": round(t_jvp / t_vjp, 2),
            "jvp_units_per_s": "%.3e" % (U / t_jvp * 1e3), "vjp_units_per_s": "%.3e" % (U / t_vjp * 1e3),
            "jvp_bytes_per_unit": bytes_jvp, "vjp_bytes_per_unit": bytes_vjp, "sample_err_vs_lambdaT_jac": "%.2e" % err}


def rollout_case(m, B, N, dt, seconds):
    ev = BatchEvaluator(m)
    n = m.n
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    q, qd, tau, f = synth_batch(lim, 0, B, N, seed=1234, device="cuda")
    q0, qd0, f0 = (t[:, :B].contiguous() for t in (q, qd, f))
    traj = ev.rollout_rk4(q0, qd0, f0, tau, N, dt)
    gen = torch.Generator(device="cuda").manual_seed(6)
    g = [torch.randn((n, N * B), dtype=torch.float64, device="cuda", generator=gen) for _ in range(3)]
    t_fwd = timed(lambda: ev.rollout_rk4(q0, qd0, f0, tau, N, dt), seconds)
    t_adj = timed(lambda: ev.rollout_rk4_vjp(q0, qd0, f0, tau, N, dt, traj, *g), seconds)
    return {"case": "rollout B=%d N=%d" % (B, N), "rollout_ms": round(t_fwd, 3), "rollout_vjp_ms": round(t_adj, 3),
            "vjp_units_per_s": "%.3e" % (B * N / t_adj * 1e3),
            "vjp_bytes_per_unit": 8 * (3 * n + n + 3 * n + n), "ms_per_node": round(t_adj / N, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    print(json.dumps(device_info()))
    pilz6 = Model.from_urdf(data_urdf("pilz6"), armature=1e-2)
    print(json.dumps(step_case("C2 pilz6 65536x100", pilz6, 65536, 100, 0.005, 65536 * 100, a.seconds)), flush=True)
    hum = Model.synthetic("humanoid", 37, seed=7, armature=1e-2)
    print(json.dumps(step_case("C4 humanoid37 one 32768-unit chunk", hum, 32768, 40, 0.5 / 40, 32768, a.seconds)), flush=True)
    print(json.dumps(rollout_case(pilz6, 65536, 100, 0.005, a.seconds)), flush=True)


if __name__ == "__main__":
    main()
