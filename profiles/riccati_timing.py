"""Riccati solve of the multiple-shooting LQ subproblem (BatchEvaluator.riccati) next to the step Jacobian that feeds it.

  C2  pilz6 (armature 1e-2), 65,536 scenarios x 100 nodes: step_rk4_jvp (produces jac), then riccati with diagonal weights,
      with the costates, and with a dense H [25, 25, U] as well
  C3  dual_arm14, 16,384 scenarios x 100 nodes (the C3 batch's Jacobian would not fit): step_rk4_jvp, riccati (+ costates)

Timed with CUDA events after a warm-up, over enough calls for about one second each.  Prints ms per call, ns per (scenario, node),
the bytes the solve must read at least (A and B twice: backward and forward pass; the diagonal weights, gradients, defects once;
H once when given) as an effective bandwidth, the FP64 work of the one-warp kernel counted from its loops (FMA per node), and the
device name and power limit.  GPU only: there is no CPU path.

    python profiles/riccati_timing.py [--seconds 1.0] [--out riccati_timing.json]
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


def fma_per_node(n):
    """FMA of one node of k_riccati's backward and forward pass, from its loops (the Z block: upper triangle only)"""
    nx, nu, nc = 3 * n, n, 4 * n
    back = nx * nx + nx * nx * nc + nx * nc * (nc + 1) // 2 + nx * nc
    back += sum((nc - t - 1) * (nc - t) for t in range(nu)) + (nx + 1) * nu * (nu - 1) // 2
    fwd = nu * (nx + 1) + nx * nc
    return back + fwd


def bytes_per_node(n, with_H):
    nx, nu, nc = 3 * n, n, 4 * n
    b = 2 * nx * nc + nc + nx + nc  # A, B twice; wx, wu; d; gx, gu
    if with_H:
        b += nc * nc
    return 8 * b


def case(name, m, B, N, seconds, dense_H):
    n = m.n
    nx, U = 3 * n, B * N
    ev = BatchEvaluator(m)
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    q, qd, tau, f = synth_batch(lim, 0, B, N, seed=1234, device="cuda")
    out = {"model": name, "family": m.kernel_family, "n": n, "B": B, "N": N}
    jac = torch.empty((nx, 4 * n + 1, U), dtype=torch.float64, device="cuda")
    qn, qdn, fn = (torch.empty((n, U), dtype=torch.float64, device="cuda") for _ in range(3))
    out["step_rk4_jvp_ms"] = timed(lambda: ev.step_rk4_jvp(q, qd, tau, f, 0.0125, out=(qn, qdn, fn), jac=jac), seconds)
    del q, qd, tau, f
    g = torch.Generator(device="cuda").manual_seed(7)
    rnd = lambda r, c, lo, hi: torch.rand((r, c), generator=g, dtype=torch.float64, device="cuda") * (hi - lo) + lo
    w = dict(wx=rnd(nx, U, 0.1, 1.0), wu=rnd(n, U, 0.1, 1.0), gx=rnd(nx, U, -1, 1), gu=rnd(n, U, -1, 1), d=rnd(nx, U, -1e-3, 1e-3),
             wN=rnd(nx, B, 0.1, 1.0), gN=rnd(nx, B, -1, 1), dx0=rnd(nx, B, -1e-2, 1e-2))
    ev.riccati(jac, B, N, **w)  # workspace allocation outside the timed window
    items = [("riccati", dict(w)), ("riccati_lam", dict(w, want_lam=True))]
    if dense_H:
        P = 4 * n + 1
        items.append(("riccati_H", dict(w, H=torch.zeros((P, P, U), dtype=torch.float64, device="cuda"))))
    for key, kw in items:
        dx, du = ev.riccati(jac, B, N, **kw)[:2]
        torch.cuda.synchronize()
        assert bool(torch.isfinite(dx).all() and torch.isfinite(du).all()), key
        ms = timed(lambda: ev.riccati(jac, B, N, **kw), seconds)
        nbytes = bytes_per_node(n, "H" in kw) * U
        out[key] = {"ms": ms, "ns_per_node": ms * 1e6 / U, "min_bytes_GB": nbytes / 1e9, "effective_TB_s": nbytes / (ms * 1e-3) / 1e12,
                    "fma_per_node": fma_per_node(n), "TFLOP_s_of_counted_work": 2 * fma_per_node(n) * U / (ms * 1e-3) / 1e12}
        kw.pop("H", None)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "riccati_timing.py needs a CUDA device"
    res = {"device": device_info(), "cases": []}
    res["cases"].append(case("pilz6", Model.from_urdf(data_urdf("pilz6"), armature=1e-2), 65536, 100, a.seconds, True))
    torch.cuda.empty_cache()
    res["cases"].append(case("dual_arm14", Model.synthetic("dual_arm", 14, seed=3, armature=1e-2), 16384, 100, a.seconds, False))
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
