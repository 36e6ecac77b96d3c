"""Fused OCP node rows on every kernel family, and on run-time-topology models against the torch composition users need
without them.

Two-arm models: the 37-joint humanoid carrying a box with both hands (generic64), both Pilz arms on a torso yaw joint
(tests/golden/pilz6x2_torso.urdf, generic16), the two Pilz arms side by side (pilz6x2, forest12x6) and a synthetic 2 x 7 dual
arm (forest14x7).  One-arm models: pilz3 (chain3) and pilz6 (chain6), frame on the last joint.  Each at B = 16,384 scenarios x
N = 40 nodes.  Timed with CUDA events after a warm-up, over enough launches for about one second each:
  (a)  FusedBoxOCP.evaluate: the fused row kernel from [B, N(+1), n] trajectories (one launch + the layout permutes)
  (a0) BatchEvaluator.ocp_rows on SoA planes: the row kernel alone
  (b)  (a) with every derivative output (dtau_dF, dT_dtau, kin_jac: a second launch)
  (b0) (a0) with every derivative output (one-arm models)
  (c)  ThermalMPCNodes.evaluate + box_rows: node_eval_ref, two fk launches and the torch arithmetic around them
One-arm models run (a0) and (b0), two-arm models (a), (a0), (b) and (c).  Prints units/s and the compulsory bytes per unit
(inputs read once, outputs written once, from the shapes), checks in the same run that (a) and (c) agree, and reads the device
name and power limit.  MPCF_LIB=<path to libmpcf.so> times another build.  GPU only: there is no CPU path.

    python profiles/ocp_rows_tree_timing.py [--B 16384] [--N 40] [--seconds 1.0]
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

from mpc_fatigue_b200.model import Model, data_urdf  # noqa: E402
from mpc_fatigue_b200.ocp import FusedBoxOCP, ThermalMPCNodes  # noqa: E402


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
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    reps = max(3, int(seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, reps


def report(tag, m, B, N, label, ms, reps, nbytes):
    U = B * N
    print(json.dumps({"model": tag, "kernel_family": m.kernel_family, "n": m.n, "B": B, "N": N, "what": label, "ms": round(ms, 4),
                      "launches_timed": reps, "units_per_s": round(U / ms * 1e3), "bytes_per_unit": nbytes,
                      "GB_per_s_compulsory": round(nbytes * U / ms * 1e-6, 1)}), flush=True)


def one_arm(tag, m, B, N, seconds):
    """(a0) and (b0) on a one-arm model, frame on the last joint"""
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    n, U = m.n, B * N
    ev = BatchEvaluator(m)
    fpar = m.export("fparent").tolist()
    frame = max(i for i, p in enumerate(fpar) if p == n - 1)
    g = torch.Generator(device="cuda").manual_seed(11)
    r = lambda *s: torch.rand(*s, dtype=torch.float64, device="cuda", generator=g)
    q, qd, F, T = 2 * r(n, U) - 1, r(n, U) - 0.5, 40 * (r(3, U) - 0.5), 20 + 40 * r(n, U)
    q_last, T_last = 2 * r(n, B) - 1, 20 + 40 * r(n, B)
    kw = dict(wsign=-1.0, p_ref=(0.3, 0.2, 0.0), w_qd=1.0, w_F=-1.0, h=0.05)
    rows_bytes = 8 * ((3 * n + 3) + (3 + 3 * n) + 1)        # q, qd, T, F read; rows, cost written
    deriv_bytes = 8 * (n * 3 + n + 3 * (n + 3))              # dtau_dF, dT_dtau, kin_jac written
    for label, deriv, nbytes in (("a0_fused_rows_soa_kernel_only", False, rows_bytes),
                                 ("b0_fused_rows_soa_kernel_with_derivatives", True, rows_bytes + deriv_bytes)):
        ms, reps = timed(lambda: ev.ocp_rows(B, N, [frame], q, qd, F, T, q_last, T_last, derivatives=deriv, **kw), seconds)
        report(tag, m, B, N, label, ms, reps, nbytes)
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=16384)
    ap.add_argument("--N", type=int, default=40)
    ap.add_argument("--seconds", type=float, default=1.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ocp_rows_tree_timing.py needs a CUDA device")
    print(json.dumps(device_info()), flush=True)
    with open(os.path.join(ROOT, "tests", "golden", "pilz6x2_torso.urdf")) as fh:
        torso = fh.read()
    cases = [("humanoid37_hands", Model.synthetic("humanoid", 37, seed=7, armature=1e-2), ["larm_ee", "rarm_ee"]),
             ("pilz6x2_torso", Model.from_urdf(torso, armature=1e-2), ["end_effector", "sec_end_effector"]),
             ("pilz6x2", Model.from_urdf(data_urdf("pilz6x2"), armature=1e-2), ["end_effector", "sec_end_effector"]),
             ("dual_arm14", Model.synthetic("dual_arm", 14, seed=3, armature=1e-2), ["left_ee", "right_ee"])]
    B, N = args.B, args.N
    U = B * N
    for tag in ("pilz3", "pilz6"):
        one_arm(tag, Model.from_urdf(data_urdf(tag), armature=1e-2), B, N, args.seconds)
    for tag, m, names in cases:
        n = m.n
        g = torch.Generator(device="cuda").manual_seed(11)
        r = lambda *s: torch.rand(*s, dtype=torch.float64, device="cuda", generator=g)
        q, qd = 2 * r(B, N + 1, n) - 1, r(B, N, n) - 0.5
        FL, FR = 40 * (r(B, N, 3) - 0.5), 40 * (r(B, N, 3) - 0.5)
        Temp = 20 + 40 * r(B, N + 1, n)
        rp0, ro0, box0 = r(B, 3) - 0.5, r(B, 3) - 0.5, (0.2, 0.1, 0.5)
        fused = FusedBoxOCP(m, names, p_ref=box0, T=20.0, N=N)
        old = ThermalMPCNodes(m, names, T=20.0, N=N)
        W = torch.cat([FL, torch.zeros_like(FL), FR, torch.zeros_like(FR)], dim=-1)

        def composition():
            return old.evaluate(q, qd, W, Temp), old.box_rows(q, qd, FL, FR, 30.0, rp0, ro0, box0)

        # same run: (a) against (c)
        a = fused.evaluate(q, qd, FL, FR, Temp, rp0, ro0)
        c0, c1 = composition()
        err = {}
        for k, ref in (("tau", c0["tau"]), ("q_defect", c0["q_defect"]), ("T_defect", c0["T_defect"]), ("force_eq", c1["force_eq"]),
                       ("moment_eq", c1["moment_eq"]), ("rel_pos", c1["rel_pos"]), ("rel_ori", c1["rel_ori"]), ("cost", c1["cost"])):
            err[k] = float((a[k] - ref).abs().max()) / max(1.0, float(ref.abs().max()))
        agree = max(err.values()) < 1e-9
        del a, c0, c1
        # SoA planes for (a0), as the fused path lays them out
        nm = lambda x: x.permute(2, 1, 0).reshape(x.shape[2], -1).contiguous()
        soa = dict(q=nm(q[:, :N]), qd=nm(qd), F=torch.cat([nm(FL), nm(FR)]), T=nm(Temp[:, :N]), q_last=q[:, N].t().contiguous(),
                   T_last=Temp[:, N].t().contiguous(), rp0=rp0.t().contiguous(), ro0=ro0.t().contiguous())
        frames = [m.frame_id(f) for f in names]

        def kernel_only():
            return fused.ev.ocp_rows(B, N, frames, soa["q"], soa["qd"], soa["F"], soa["T"], soa["q_last"], soa["T_last"], soa["rp0"],
                                     soa["ro0"], **fused.kw)

        nrows = 26 + 3 * n
        rows_bytes = 8 * ((3 * n + 6) + nrows + 1)              # q, qd, T, F read; rows, cost written
        deriv_bytes = 8 * (n * 6 + n + 26 * (n + 6))            # dtau_dF, dT_dtau, kin_jac written
        runs = [("a_fused_rows", lambda: fused.evaluate(q, qd, FL, FR, Temp, rp0, ro0), rows_bytes),
                ("a0_fused_rows_soa_kernel_only", kernel_only, rows_bytes),
                ("b_fused_rows_with_derivatives", lambda: fused.evaluate(q, qd, FL, FR, Temp, rp0, ro0, derivatives=True), rows_bytes + deriv_bytes),
                ("c_torch_composition", composition, rows_bytes)]
        for label, fn, nbytes in runs:
            ms, reps = timed(fn, args.seconds)
            report(tag, m, B, N, label, ms, reps, nbytes)
            torch.cuda.empty_cache()
        print(json.dumps({"model": tag, "a_vs_c_agree_1e-9": agree, "max_rel_err": {k: float("%.2e" % v) for k, v in err.items()}}), flush=True)
        if not agree:
            sys.exit(1)


if __name__ == "__main__":
    main()
