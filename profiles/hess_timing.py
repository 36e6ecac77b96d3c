"""Second order of the RK4 step: Hessian-vector product and dense adjoint-weighted Hessian.

  HVP C2  pilz6 (armature 1e-2), 65,536 scenarios x 100 nodes = 6,553,600 units: step_rk4_hvp next to step_rk4_vjp
  H   C2  pilz6, 65,536 units: step_rk4_hess (the dense [25, 25, U] Hessian)
  HVP C4  humanoid37, 32,768 units: step_rk4_hvp next to step_rk4_vjp

Timed with CUDA events after a warm-up, over enough calls for about one second each.  Prints ms per call, units/s and the
compulsory bytes per unit (inputs read once, outputs written once, from the shapes), checks in the same run that the HVP equals the
dense Hessian times v on a sample of units, and reads the device name and power limit.  GPU only: there is no CPU path.

    python profiles/hess_timing.py [--seconds 1.0]
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
from mpc_fatigue_b200.model import Model, data_urdf  # noqa: E402
from mpc_fatigue_b200.synth import synth_batch  # noqa: E402
from profiles.vjp_timing import device_info, timed  # noqa: E402


def _inputs(m, B, N, U, seed):
    n = m.n
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    inputs = [t[:, :U].contiguous() for t in synth_batch(lim, 0, B, N, seed=1234, device="cuda")]
    gen = torch.Generator(device="cuda").manual_seed(seed)
    lam = [torch.randn((n, U), dtype=torch.float64, device="cuda", generator=gen) for _ in range(3)]
    v = [torch.randn((n, U), dtype=torch.float64, device="cuda", generator=gen) for _ in range(4)]
    v.append(1e-3 * torch.randn(U, dtype=torch.float64, device="cuda", generator=gen))
    return inputs, lam, v


def check_sample(ev, inputs, dt, lam, v, cols):
    """max over the sample of |H v - (dense H) v| / max(S, 1e-6 max S), S = sum_c |H_rc| |v_c|"""
    pick = lambda t: t[..., cols].contiguous()
    si, sl, sv = [pick(t) for t in inputs], [pick(t) for t in lam], [pick(t) for t in v]
    H = ev.step_rk4_hess(*si, dt, *sl)
    h = ev.step_rk4_hvp(*si, dt, sl, sv, want_dt=True)
    got = torch.cat([*h[:4], h[4][None]])
    V = torch.cat([*sv[:4], sv[4][None]])
    ref = torch.einsum("rcu,cu->ru", H, V)
    S = torch.einsum("rcu,cu->ru", H.abs(), V.abs())
    return float(((got - ref).abs() / torch.clamp(S, min=1e-6 * float(S.max()))).max())


def hvp_case(name, m, B, N, dt, U, seconds):
    ev = BatchEvaluator(m)
    n = m.n
    inputs, lam, v = _inputs(m, B, N, U, 5)
    t_vjp = timed(lambda: ev.step_rk4_vjp(*inputs, dt, *lam, want_dt=True), seconds)
    t_hvp = timed(lambda: ev.step_rk4_hvp(*inputs, dt, lam, v, want_dt=True), seconds)
    t_hvp_jv = timed(lambda: ev.step_rk4_hvp(*inputs, dt, lam, v, want_dt=True, want_jv=True), seconds)
    err = check_sample(ev, inputs, dt, lam, v, torch.linspace(0, U - 1, 256, device="cuda").long())
    torch.cuda.empty_cache()
    return {"case": name, "units": U, "family": m.kernel_family, "vjp_ms": round(t_vjp, 3), "hvp_ms": round(t_hvp, 3),
            "hvp_with_jv_ms": round(t_hvp_jv, 3), "hvp_over_vjp": round(t_hvp / t_vjp, 2),
            "hvp_units_per_s": "%.3e" % (U / t_hvp * 1e3), "hvp_bytes_per_unit": 8 * (4 * n + 3 * n + 4 * n + 1 + 4 * n + 1),
            "sample_err_vs_dense_H_v": "%.2e" % err}


def hess_case(name, m, U, dt, seconds):
    ev = BatchEvaluator(m)
    n, P = m.n, 4 * m.n + 1
    inputs, lam, _ = _inputs(m, U, 1, U, 6)
    t = timed(lambda: ev.step_rk4_hess(*inputs, dt, *lam), seconds)
    torch.cuda.empty_cache()
    return {"case": name, "units": U, "family": m.kernel_family, "hess_ms": round(t, 3), "hess_units_per_s": "%.3e" % (U / t * 1e3),
            "sweeps_per_unit": (3 * n + 1) * (3 * n + 2) // 2, "hess_bytes_per_unit": 8 * (4 * n + 3 * n + P * P),
            "write_GB_per_s": round(8 * P * P * U / t * 1e-6, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    print(json.dumps(device_info()))
    pilz6 = Model.from_urdf(data_urdf("pilz6"), armature=1e-2)
    print(json.dumps(hvp_case("HVP C2 pilz6 65536x100", pilz6, 65536, 100, 0.005, 65536 * 100, a.seconds)), flush=True)
    print(json.dumps(hess_case("H pilz6 65536", pilz6, 65536, 0.005, a.seconds)), flush=True)
    hum = Model.synthetic("humanoid", 37, seed=7, armature=1e-2)
    print(json.dumps(hvp_case("HVP humanoid37 32768", hum, 32768, 1, 0.5 / 40, 32768, a.seconds)), flush=True)


if __name__ == "__main__":
    main()
