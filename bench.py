#!/usr/bin/env python3
"""bench.py — rollout-steps/s of the RK4 dynamics+fatigue step WITH forward-mode Jacobians (SURVEY.md §8d).

    python bench.py --gpus N --steps K --warmup W          (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --config C1|C2|C3|C4|C5 ...            one BASELINE.json config as the headline line (default C2)
    python bench.py --impl reference ...                   CPU arm: the oracle port on all host cores
    python bench.py --dump-outputs DIR ...                 also write the headline's last-step outputs as DIR/<name>.npy

Headline (default): config C2 = BASELINE.json configs[1] (Pilz 6-DOF + armature 1e-2, N = 100 nodes x B = 65,536 scenarios per
GPU, fp64, dense Jacobians; weak scaling).  One "step" = one pass of the hot path over the rank's whole batch: the Jacobian
pipeline (states + dense Jacobian for U = B*N units) + the per-scenario cost/residual reduction, and for N > 1 the NCCL
all-gather of the [4, B] cost/residual rows.  Inputs + outputs (25.8 GB) >> 126 MB L2, so no flush between iterations.

The same JSON line carries the other configs under "configs" (each measured in this run with the same timing rules):
C1 (3-DOF reference-mode node evaluation with its CPU reference run), C3 (dual-arm 12-DOF with the coupled fatigue states,
131,072 scenarios), C4 (37-DOF branched tree, 32,768 scenarios x 40 nodes) at N = 1, and C5 (1,048,576 scenarios of the C2
model, STRONG-scaled over the N ranks, scenario chunks reusing one Jacobian buffer, per-chunk all-gather on a side stream).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rollout_steps_per_s_with_jacobians"
UNIT = "rollout-steps/s"
ARMATURE = 1e-2
JAC_CHUNK_BYTES = 24 << 30  # Jacobian buffer reused over the scenario chunks of a config (C2's own Jacobian is 23.6 GB)
DUMP_BYTES = 48 << 20  # --dump-outputs: all arrays together stay under 64 MB

# name -> (model, nodes N, scenarios, dt, scaling)   scenarios: per GPU for "weak", total for "strong"
CONFIGS = {
    "C2": dict(model="pilz6", N=100, B=65536, dt=0.02, scaling="weak",
               workload="C2: Pilz 6-DOF (urdf pilz_robot_6DOF, armature 1e-2), RK4 dyn+fatigue step with dense forward-mode "
                        "Jacobian, N=100 nodes x 65536 scenarios per GPU, dt=0.02"),
    "C3": dict(model="pilz6x2", N=100, B=131072, dt=0.02, scaling="strong", coupled=True,
               workload="C3: dual-arm 2 x Pilz 6-DOF (12 DOF, two-tree model) with coupled fatigue states (shared box load split "
                        "between the arms), N=100 nodes x 131072 scenarios, dt=0.02, dense Jacobian in scenario chunks"),
    "C4": dict(model="humanoid37", N=40, B=32768, dt=0.5 / 40, scaling="strong",
               workload="C4: synthetic 37-DOF branched tree (6-joint root chain + torso + 2x7 arms + 4x4 legs), N=40 nodes x 32768 "
                        "scenarios, dt=0.0125, dense Jacobian (132 KB/unit) in scenario chunks"),
    "C5": dict(model="pilz6", N=100, B=1048576, dt=0.02, scaling="strong",
               workload="C5: 1,048,576-scenario Pilz 6-DOF sweep (N=100 nodes), strong-scaled over the ranks, scenario chunks of "
                        "65536 reusing one Jacobian buffer, NCCL all-gather of the per-scenario cost/residual rows per chunk"),
}


# ---- work models -------------------------------------------------------------------------------------------------------
def frozen_flop_model(n: int) -> dict:
    """BASELINE.md §3 / SURVEY.md §8d: the dual-number formulation (1 + 4n + 1 sweeps of RK4(ABA))."""
    aba = (224 * n - 259) + (205 * n - 248)
    step_values = 4 * (aba + 7 * n) + 24 * n
    P = 4 * n + 1
    return dict(aba=aba, step_values=step_values, step_jac=step_values * (1 + P),
                bytes_values=(4 * n + 1 + 3 * n) * 8, bytes_jac=(4 * n + 1 + 3 * n) * 8 + 3 * n * P * 8)


flop_model = frozen_flop_model  # the name tests and round-1 tooling use


def work_model() -> dict:
    """profiles/work_model.json: FP64 operations the shipped kernels EXECUTE per unit (ncu counters dadd / dmul / dfma of a
    tracked capture, written by profiles/make_work_model.py) — the re-frozen work model SURVEY.md §8(d) asks for
    ("instrumented count, whichever is smaller")."""
    try:
        with open(os.path.join(ROOT, "profiles", "work_model.json")) as fh:
            return json.load(fh)
    except OSError:
        return {}


def roofline_for(family: str, n: int, units: float, kernel_ms: dict, peak_tflops: float, hbm_peak: float, peak_src: str, total_ms: float | None = None) -> dict:
    """FP64 roofline of one config.  achieved = ALGORITHMIC FLOP per unit x units / device time of the pipeline kernels,
    with FLOP per unit = min(frozen dual-number model, instrumented count of the shipped algorithm) (SURVEY §8d: "whichever
    is smaller"); `fp64_pipe` = executed FP64 instructions (every DADD/DMUL/DFMA occupies one issue slot of the pipe whose
    peak is the DFMA rate) / time / peak instruction rate: the utilisation ncu reports as sm__pipe_fp64_cycles_active,
    recomputed from this run's own kernel times."""
    fm = frozen_flop_model(n)
    wm = work_model().get(family)
    total_ms = total_ms if total_ms is not None else sum(kernel_ms.values())  # device time of the whole Jacobian call (events around it)
    out = {"bound": "fp64", "unit": "TFLOP/s", "peak": peak_tflops, "peak_source": peak_src, "kernel_ms": total_ms, "kernels_ms": kernel_ms}
    flop_frozen = fm["step_jac"]
    if wm:
        flop_exec = sum(k["dadd"] + k["dmul"] + 2 * k["dfma"] for k in wm["kernels"].values())
        inst_exec = sum(k["dadd"] + k["dmul"] + k["dfma"] for k in wm["kernels"].values())
        flop = min(flop_frozen, flop_exec)
        out["flop_model"] = ("instrumented: %d FLOP/unit executed by the shipped kernels (%s); frozen dual-number model %d"
                             % (flop_exec, wm["source"], flop_frozen))
        out["fp64_pipe"] = {"frac": inst_exec * units / (total_ms * 1e-3) / (peak_tflops * 1e12 / 2),
                            "fp64_thread_instructions_per_unit": inst_exec,
                            "per_kernel": {k: v["dadd"] + v["dmul"] + v["dfma"] for k, v in wm["kernels"].items()},
                            "what": "executed FP64 instructions / time / DFMA issue rate of the probe (= sm__pipe_fp64_cycles_active)"}
        tc = wm.get("tensor_core_pipeline")
        if tc:  # DMMA.8x8x4 = 256 FMA = the work of 8 warp-wide DFMA on the same 64 FMA / clk / SM peak
            dmma = sum(k.get("dmma_warp_instr", 0) for k in tc["kernels"].values())
            out["tensor_pipe"] = {"frac": dmma * 256 * units / (total_ms * 1e-3) / (peak_tflops * 1e12 / 2), "dmma_warp_instructions_per_unit": dmma,
                                  "source": tc["source"], "what": "DMMA.8x8x4 issued (operands padded to 40 x 80 x 64-column slabs) x 256 FMA / time / FMA peak"}
        traffic = wm.get("dram_bytes_per_unit")
        out["traffic"] = traffic * units if traffic else None
        out["traffic_source"] = wm["source"] if traffic else None
    else:
        flop = flop_frozen
        out["flop_model"] = "frozen BASELINE.md §3 model: %d FLOP/unit (no instrumented count for family %s)" % (flop_frozen, family)
        out["traffic"] = None
    ach = flop * units / (total_ms * 1e-3) / 1e12
    out.update({"achieved": ach, "frac": ach / peak_tflops, "flop_per_unit": flop})
    if kernel_ms:
        dom = max(kernel_ms, key=kernel_ms.get)
        out.update({"dominant_kernel": dom, "dominant_share": kernel_ms[dom] / max(total_ms, 1e-9)})
    gbs = fm["bytes_jac"] * units / (total_ms * 1e-3) / 1e9
    out["hbm"] = {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "algorithmic_bytes_per_unit": fm["bytes_jac"]}
    return out


# ---- clocks sampler (B200_PROFILING.md recipe) ----
class ClockSampler:
    """SM clock and clock-event reasons of one GPU, sampled every 50 ms by a thread through NVML (what nvidia-smi itself
    reads; no subprocess, so no start-up delay and no pipe buffering: every sample carries its own time stamp).  Falls back
    to one `nvidia-smi --query-gpu` call per sample when the NVML python module is missing."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index, self.rows, self.thread, self.stop_flag, self.src = index, [], None, threading.Event(), None

    def _nvml_reader(self):
        import pynvml
        pynvml.nvmlInit()
        import torch
        p = torch.cuda.get_device_properties(self.index)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)).encode())
        mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        bits = [pynvml.nvmlClocksEventReasonHwSlowdown, pynvml.nvmlClocksEventReasonHwThermalSlowdown,
                pynvml.nvmlClocksEventReasonSwThermalSlowdown, pynvml.nvmlClocksEventReasonSwPowerCap]

        def read():
            r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
            return float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), mx, [bool(r & b) for b in bits]
        return read

    def _smi_reader(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

        def read():
            out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=10).stdout.strip().split(",")
            return float(out[0]), float(out[1]), [c.strip().lower().startswith("active") for c in out[2:6]]
        return read

    def start(self):
        read = None
        for name, make in (("nvml", self._nvml_reader), ("nvidia-smi", self._smi_reader)):
            try:
                read = make()
                read()
                self.src = name
                break
            except Exception:  # noqa: BLE001 - any failure of one source just selects the next
                read = None
        if read is None:
            return

        def loop():
            while not self.stop_flag.is_set():
                try:
                    self.rows.append((time.perf_counter(),) + read())
                except Exception:  # noqa: BLE001
                    pass
                self.stop_flag.wait(0.05)
        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    @staticmethod
    def mark() -> float:
        return time.perf_counter()

    def stop(self, t0: float | None = None, t1: float | None = None) -> dict:
        """Statistics over the samples taken inside [t0, t1] (the timed region); if none fell inside it (a very short
        region), over everything sampled since start(), i.e. warm-up + timed steps of the same kernels, and says so."""
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable (no NVML module, no nvidia-smi)"], "samples": 0}
        self.stop_flag.set()
        self.thread.join(timeout=15)
        rows = [r for r in self.rows if t0 is not None and t1 is not None and t0 <= r[0] <= t1]
        window = "timed region"
        if not rows:
            rows, window = list(self.rows), "warm-up + timed region (no sample fell inside the timed region)"
        mhz = sorted(r[1] for r in rows)
        reasons = sorted({nm for r in rows for nm, on in zip(self.NAMES, r[3]) if on})
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": rows[-1][2] if rows else None, "reasons": reasons,
                "samples": len(mhz), "window": window, "source": self.src}


def measured_peaks() -> dict:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh)
    except OSError:
        return {}


# =================================================================================================
# CPU arm: the oracle (test infrastructure) timed on the host cores
# =================================================================================================
def cpu_model(name: str):
    from oracle.urdf_model import load_urdf
    with open(os.path.join(ROOT, "mpc_fatigue_b200", "data", "models", name + ".urdf")) as fh:
        return load_urdf(fh.read(), armature=ARMATURE)


def cpu_inputs(np, om, U, seed=1234):
    rng = np.random.default_rng(seed)
    n = om.n
    lo, hi = np.array(om.q_lo)[:, None], np.array(om.q_hi)[:, None]
    q = np.ascontiguousarray(rng.uniform(lo, hi, (n, U)))
    qd = np.ascontiguousarray(rng.uniform(-1, 1, (n, U)) * np.array(om.v_max)[:, None])
    tau = np.ascontiguousarray(rng.uniform(-1, 1, (n, U)) * np.array(om.tau_max)[:, None] * 0.25)
    f = np.ascontiguousarray(rng.uniform(20, 80, (n, U)))
    return q, qd, tau, f


def cpu_arms(target_seconds: float, steps: int = 3):
    """Both CPU implementations of the C2 step-with-Jacobian on all host cores, same inputs:
      forward : forward-mode AD with all 19 tangent directions carried as one SIMD vector per value (the algorithm class of the
                reference: CasADi differentiates the traced graph by forward/reverse sweeps), -O3 -march=native, OpenMP over
                units — the BASELINE;
      complex : the checker the parity tests use (25 complex-step sweeps, no FMA contraction) — reported for continuity with
                round 1, 10-20x slower than a tuned CPU code.
    Returns (np, dict per arm of callables and unit counts)."""
    import numpy as np
    from oracle import pyoracle
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "-s"], check=True)
    om = cpu_model("pilz6")
    cores = len(os.sched_getaffinity(0))
    orc = pyoracle.Oracle(om, fast=True, threads=cores)
    arms = {}
    for name, fn in (("forward", getattr(orc, "step_rk4_jvp_forward", None)), ("complex", orc.step_rk4_jvp)):
        if fn is None:
            continue
        U0 = 4096
        x = cpu_inputs(np, om, U0)
        fn(*x, 0.02)
        t0 = time.perf_counter()
        fn(*x, 0.02)
        rate0 = U0 / (time.perf_counter() - t0)
        U = int(max(U0, min(1 << 21, rate0 * target_seconds / max(steps, 1))))
        arms[name] = (fn, U, cpu_inputs(np, om, U))
    return np, cores, arms


CPU_KIND = {"forward": "port", "complex": "port"}
CPU_WHAT = {"forward": "oracle C port, forward-mode AD with the 19 tangent directions as one SIMD vector per value, -O3 -march=native + OpenMP",
            "complex": "oracle C port, Jacobians by 25 complex-step sweeps (the parity checker), -O3 -march=native + OpenMP"}


def cpu_baseline(target_seconds: float = 10.0) -> dict:
    """Bounded sample of the C2 workload on the host cores; headline = the forward-mode build, the complex-step checker beside it."""
    np, cores, arms = cpu_arms(target_seconds / 2)
    res = {}
    for name, (fn, U, x) in arms.items():
        best = 0.0
        for _ in range(3):
            t0 = time.perf_counter()
            fn(*x, 0.02)
            best = max(best, U / (time.perf_counter() - t0))
        res[name] = {"value": best, "units": U}
    head = "forward" if "forward" in res else "complex"
    out = {"value": res[head]["value"], "unit": UNIT, "cores": cores, "kind": CPU_KIND[head],
           "sample": "%d units of the C2 workload (same model, dt, value distributions), best of 3; %s" % (res[head]["units"], CPU_WHAT[head]),
           "per_core": res[head]["value"] / cores}
    if head != "complex" and "complex" in res:
        out["complex_step_checker"] = {"value": res["complex"]["value"], "unit": UNIT, "sample": "%d units; %s" % (res["complex"]["units"], CPU_WHAT["complex"])}
    return out


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    total = max(1, args.steps + args.warmup)
    budget_s = 2.0 if os.environ.get("MPCF_BENCH_QUICK") else 90.0  # whole run ~ 90 s (a few seconds in the contract test)
    np, cores, arms = cpu_arms(budget_s * 0.8, total)
    head = "forward" if "forward" in arms else "complex"
    fn, U, x = arms[head]
    for _ in range(args.warmup):
        fn(*x, 0.02)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn(*x, 0.02)
    el = time.perf_counter() - t0
    value = U * args.steps / el
    sample = "%d units per step (bounded sample of the C2 workload), %d host threads; %s" % (U, cores, CPU_WHAT[head])
    extra = {}
    if head != "complex" and "complex" in arms:
        fc, Uc, xc = arms["complex"]
        Uc = min(Uc, 1 << 16)
        xc = tuple(a[:, :Uc].copy() for a in xc)
        t0 = time.perf_counter()
        fc(*xc, 0.02)
        extra["complex_step_checker"] = {"value": Uc / (time.perf_counter() - t0), "unit": UNIT, "sample": "%d units, one pass; %s" % (Uc, CPU_WHAT["complex"])}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config("C2", args.gpus),
        "cpu_baseline": dict({"value": value, "unit": UNIT, "cores": cores, "kind": CPU_KIND[head], "sample": sample}, **extra),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference CasADi/Pinocchio path cannot be built in this image (no casadi/pinocchio/Eigen/urdfdom); this arm times "
                "the compiled oracle port in the reference's algorithm class (forward-mode AD of RK4(ABA) + fatigue), on all host "
                "cores — at least as fast as CasADi's single-threaded SX interpreter",
    }))


# =================================================================================================
# GPU arm
# =================================================================================================
def workload_config(name: str, n_gpus: int) -> dict:
    c = CONFIGS[name]
    per_gpu = c["B"] if c["scaling"] == "weak" else c["B"] // n_gpus
    return {"workload": c["workload"], "config": name, "robot": c["model"], "nodes": c["N"], "dt": c["dt"],
            "scenarios_per_gpu": per_gpu, "scenarios_total": per_gpu * n_gpus, "units_per_gpu": per_gpu * c["N"],
            "parallelism": "scenario-sharded x%d" % n_gpus, "l2": "inputs+outputs >> 126 MB L2, no flush needed", "seed": 1234}


def make_model(name: str):
    from mpc_fatigue_b200.model import Model, data_urdf
    if name == "humanoid37":
        return Model.synthetic("humanoid", 37, seed=7, armature=ARMATURE)
    return Model.from_urdf(data_urdf(name), armature=ARMATURE)


class ConfigRunner:
    """One config on one rank: the rank's scenarios cut into chunks of Bc scenarios (x all N nodes, node-major units), every
    chunk a stand-alone batch [n, N*Bc] of inputs and states; ONE Jacobian buffer (<= JAC_CHUNK_BYTES) and one workspace are
    reused by all chunks.  step(): per chunk Jacobian pipeline + per-scenario reduction (+ all-gather of the chunk's [4, Bc]
    rows on a side stream, overlapped with the next chunk's kernels)."""

    def __init__(self, name: str, dev, rank: int, world: int):
        import torch
        from mpc_fatigue_b200.evaluator import BatchEvaluator
        from mpc_fatigue_b200.synth import synth_batch
        self.torch, self.name, self.dev, self.rank, self.world = torch, name, dev, rank, world
        c = CONFIGS[name]
        self.c = c
        self.model = make_model(c["model"])
        if c.get("coupled"):
            from mpc_fatigue_b200.coupling import box_load_coupling
            self.model.set_coupling(box_load_coupling(self.model))
        self.ev = BatchEvaluator(self.model, dev)
        n, N = self.model.n, c["N"]
        self.n, self.N = n, N
        B_local = c["B"] if c["scaling"] == "weak" else c["B"] // world
        b_start = rank * B_local
        jac_unit = 3 * n * (4 * n + 1) * 8
        Bc = max(1, min(B_local, JAC_CHUNK_BYTES // (jac_unit * N)))
        while B_local % Bc:  # equal chunks (every config's B is a power of two)
            Bc -= 1
        self.B_local, self.Bc, self.nchunks = B_local, Bc, B_local // Bc
        self.U = B_local * N
        limits = {k: self.model.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
        self.inp = [synth_batch(limits, b_start + i * Bc, Bc, N, seed=1234, device=dev) for i in range(self.nchunks)]
        self.out = [tuple(torch.empty_like(self.inp[i][0]) for _ in range(3)) for i in range(self.nchunks)]
        self.jac = torch.empty((3 * n, 4 * n + 1, Bc * N), dtype=torch.float64, device=dev)
        self.red = torch.empty((self.nchunks, 4, Bc), dtype=torch.float64, device=dev)  # all-gather send buffers, written by the kernel
        from mpc_fatigue_b200.ocp import f0_bound_table
        self.table = torch.from_numpy(f0_bound_table(N, n, c["dt"])).to(dev)
        if world > 1:
            self.recv = torch.empty((self.nchunks, world, 4, Bc), dtype=torch.float64, device=dev)  # preallocated once
            self.side = torch.cuda.Stream(dev)
        self.family = self.model.kernel_family

    def step(self, pairs=None):
        torch, ev = self.torch, self.ev
        for i in range(self.nchunks):
            q, qd, tau, f = self.inp[i]
            qn, qdn, fn = self.out[i]
            if pairs is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            ev.step_rk4_jvp(q, qd, tau, f, self.c["dt"], out=(qn, qdn, fn), jac=self.jac)
            if pairs is not None:
                e1.record()
                pairs.append((e0, e1))
            ev.cost_residual_table(self.Bc, self.N, q, qd, f, tau, qn, qdn, fn, self.table, out=self.red[i])
            if self.world > 1:
                import torch.distributed as dist
                done = torch.cuda.Event()
                done.record()
                self.side.wait_event(done)
                with torch.cuda.stream(self.side):
                    dist.all_gather_into_tensor(self.recv[i].view(-1), self.red[i].view(-1))
        if self.world > 1:
            torch.cuda.current_stream().wait_stream(self.side)
            return self.recv
        return self.red

    def launches_per_step(self) -> int:
        return -1

    def outputs(self, gathered) -> dict:
        """What a caller of step() holds after it: q+, qd+, f+ of every chunk, the Jacobian of the last chunk (one buffer is
        reused by all chunks) and the per-scenario cost / residual rows (of every rank after the all-gather)."""
        return {"q_next": [o[0] for o in self.out], "qd_next": [o[1] for o in self.out], "f_next": [o[2] for o in self.out],
                "jacobian": [self.jac], "cost_residual": list(gathered.reshape(-1, 4, self.Bc))}


def dump_outputs(path: str, arrays: dict) -> None:
    """Write every array as <path>/<name>.npy in float64.  `arrays` maps a name to a list of equally wide chunks whose last
    axes together make the unit axis.  An array larger than its share of DUMP_BYTES keeps a fixed, seeded sample of its unit
    columns (in ascending order), so runs with the same arguments write the same elements and two builds compare one to one."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, chunks in arrays.items():
        width = chunks[0].shape[-1]
        total, rows = width * len(chunks), chunks[0].numel() // width
        keep = min(total, max(1, share // (8 * rows)))
        idx = np.sort(np.random.default_rng(0).choice(total, keep, replace=False)) if keep < total else np.arange(total)
        cols = [torch.from_numpy(idx[idx // width == i] % width).to(c.device) for i, c in enumerate(chunks)]
        out = torch.cat([c.index_select(c.dim() - 1, k) for c, k in zip(chunks, cols)], -1)
        np.save(os.path.join(path, name + ".npy"), out.to(torch.float64).cpu().numpy())


def warmup_steps(steps: int, warmup: int) -> int:
    """Warm-up steps actually run before K timed steps: W, but at least one (module load, first-touch allocations) and at
    least three when more than one step is timed."""
    return max(warmup, 3) if steps > 1 else max(warmup, 1)


def time_config(runner: ConfigRunner, steps: int, warmup: int, fence, sampler=None):
    """warmup_steps(K, W) warm-up steps, then exactly K timed steps bracketed by fence(); device time by CUDA events; per-kernel
    times of the pipeline through the library's event hooks (compile-time families) or the events around the whole Jacobian call."""
    import ctypes as C
    import torch
    from mpc_fatigue_b200 import _capi
    for _ in range(warmup_steps(steps, warmup)):
        runner.step()
    fence()
    launches0 = _capi.lib.mpcf_launch_count()
    pairs = []
    _capi.lib.mpcf_profile_enable(1)
    fence()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    mark0 = sampler.mark() if sampler else None
    t0.record()
    for _ in range(steps):
        gathered = runner.step(pairs)
    t1.record()
    fence()
    mark1 = sampler.mark() if sampler else None
    launches = _capi.lib.mpcf_launch_count() - launches0
    el_ms = t0.elapsed_time(t1)
    ms3 = (C.c_double * 3)()
    nprof = C.c_long()
    _capi.lib.mpcf_profile_read(ms3, C.byref(nprof))
    _capi.lib.mpcf_profile_enable(0)
    jvp_ms = sum(a.elapsed_time(b) for a, b in pairs) / steps
    if nprof.value:
        kern = {"step_stages": ms3[0] / steps, "stage_derivs": ms3[1] / steps, "chain_rule": ms3[2] / steps}
    else:
        kern = {"step_rk4_jvp": jvp_ms}
    return {"el_ms": el_ms, "kern": kern, "jvp_ms": jvp_ms, "launches": int(launches), "gathered": gathered, "marks": (mark0, mark1)}


def fp64_probe(dev) -> float:
    """DFMA-chain probe: the FP64 roofline denominator (MEASURED_PEAKS.json carries no FP64 figure; nominal 37.2 TFLOP/s)."""
    import ctypes as C
    import torch
    from mpc_fatigue_b200 import _capi
    blocks, iters = 148 * 16, 200000
    pout = torch.empty(blocks * 256, dtype=torch.float64, device=dev)
    best = 0.0
    for _ in range(4):
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        _capi.check(_capi.lib.mpcf_probe_fp64(iters, blocks, C.c_void_p(pout.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        p1.record()
        torch.cuda.synchronize()
        best = max(best, blocks * 256 * iters * 16 / (p0.elapsed_time(p1) * 1e-3) / 1e12)
    return best


def pcie_probe(dev) -> dict:
    """Measured host<->device copy bandwidth of this box (pinned memory, 1 GiB transfers, best of 3): the denominator of the
    end-to-end path, which is copy-bound."""
    import torch
    nbytes = 1 << 30
    h = torch.empty(nbytes // 8, dtype=torch.float64).pin_memory()
    d = torch.empty(nbytes // 8, dtype=torch.float64, device=dev)
    res = {}
    for name, dst, src in (("d2h_gbs", h, d), ("h2d_gbs", d, h)):
        best = 0.0
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dst.copy_(src, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            best = max(best, nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        res[name] = best
    return res


def config_result(name: str, runner: ConfigRunner, t: dict, steps: int, world: int, peak_tf: float, hbm_peak: float, peak_src: str) -> dict:
    units_per_step = world * runner.U
    value = units_per_step * steps / (t["el_ms"] * 1e-3)
    roof = roofline_for(runner.family, runner.n, runner.U, t["kern"], peak_tf, hbm_peak, peak_src, total_ms=t["jvp_ms"])
    return {"metric": METRIC, "value": value, "unit": UNIT, "ms_per_step": t["el_ms"] / steps, "steps": steps,
            "scaling": CONFIGS[name]["scaling"], "config": workload_config(name, world), "chunks_per_step": runner.nchunks,
            "scenarios_per_chunk": runner.Bc, "kernel_family": runner.family, "gpu_launches": t["launches"], "roofline": roof,
            "checksum_cost": float(t["gathered"].reshape(-1, 4, runner.Bc)[:, 0].sum().item())}


def run_c1(dev, steps: int = 10, warmup: int = 3, outputs: dict | None = None) -> dict:
    """C1: Pilz 3-DOF fatigue OCP (python/Pilz_3_DOF/inverse_dynamics_pilz_3DOF.py:78-89,124-146: N=20, T=4; per node
    tau = RNEA(q, qd, 0), F0 bound tau0=50, alpha=2, floor=10, Euler).  "CPU CasADi reference run" stand-in: the oracle's
    reference-mode node evaluation of ONE OCP (20 nodes, one thread), timed; beside it the GPU evaluating 65,536 such OCPs
    per launch (`steps` timed launches after warmup_steps(steps, warmup)), and the agreement of the two on the first OCP.
    `outputs` receives the GPU results of the last timed launch."""
    import numpy as np
    import torch
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    from mpc_fatigue_b200.ocp import f0_bound_schedule
    from mpc_fatigue_b200.synth import synth_batch
    from oracle.pyoracle import Oracle
    N, T = 20, 4.0
    h = T / N
    model = make_model("pilz3")
    ev = BatchEvaluator(model, dev)
    om = cpu_model("pilz3")
    orc = Oracle(om, fast=True, threads=1)
    B = 65536
    limits = {k: model.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    q, qd, _, f = synth_batch(limits, 0, B, N, seed=1234, device=dev)
    bound = f0_bound_schedule(N, h, 50.0, 2.0, 10.0)
    # CPU: one OCP = units b = 0 of every node
    idx = torch.arange(N, device=dev) * B
    hq, hqd, hf = (np.ascontiguousarray(t[:, idx].cpu().numpy()) for t in (q, qd, f))

    def cpu_once():
        tau, qn, Tn = orc.node_eval_ref([], -1.0, hq, hqd, None, hf, h)
        return tau, qn, Tn, float(np.maximum(np.abs(tau) - bound[None, :], 0.0).max())
    cpu_once()
    reps, t0 = 200, time.perf_counter()
    for _ in range(reps):
        tau_c, qn_c, Tn_c, viol_c = cpu_once()
    cpu_s = (time.perf_counter() - t0) / reps
    # GPU: all B OCPs
    warm = warmup_steps(steps, warmup)
    for _ in range(warm):
        tau_g, qn_g, Tn_g = ev.node_eval_ref([], -1.0, q, qd, None, f, h)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        tau_g, qn_g, Tn_g = ev.node_eval_ref([], -1.0, q, qd, None, f, h)
    e1.record()
    torch.cuda.synchronize()
    gpu_ms = e0.elapsed_time(e1) / steps
    if outputs is not None:
        outputs.update(tau=[tau_g], q_next=[qn_g], T_next=[Tn_g])
    err = max(float(np.abs(a[:, idx].cpu().numpy() - b).max() / max(1.0, np.abs(b).max())) for a, b in ((tau_g, tau_c), (qn_g, qn_c), (Tn_g, Tn_c)))
    return {"config": {"workload": "C1: Pilz 3-DOF fatigue OCP, reference-mode node evaluation (RNEA(q,qd,0), Euler, thermal ZOH, F0 bound), "
                                   "N=20 nodes, T=4", "robot": "pilz3", "nodes": N},
            "steps": steps, "warmup": warm,
            "cpu_reference_run": {"seconds_per_ocp_evaluation": cpu_s, "node_evaluations_per_s": N / cpu_s, "cores": 1, "kind": "port",
                                  "what": "oracle reference-mode node evaluation of one OCP (20 nodes), the stand-in for the per-node CasADi "
                                          "calls of inverse_dynamics_pilz_3DOF.py:124-146 (casadi is not installable here)",
                                  "max_torque_bound_violation": viol_c},
            "gpu": {"ocps_per_launch": B, "ms_per_launch": gpu_ms, "node_evaluations_per_s": B * N / (gpu_ms * 1e-3)},
            "max_rel_err_gpu_vs_cpu": err}


def run_gpu(args) -> None:
    import torch
    import torch.distributed as dist
    from mpc_fatigue_b200.dist import bind_to_gpu_numa_node

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # multi-GPU: every rank's pinned staging buffers on the NUMA node of its own GPU (N = 1 keeps all host cores, which
    # the cpu_baseline leg uses)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 and os.environ.get("MPCF_NUMA_BIND", "1") != "0" else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    head = args.config
    peaks = measured_peaks()
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---- headline config ----
    if head == "C1":
        outputs = {}
        line = run_c1(dev, args.steps, args.warmup, outputs) if rank == 0 else None
        if rank == 0:
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, outputs)
            print(json.dumps(dict(line, metric="reference_mode_node_evaluations_per_s", value=line["gpu"]["node_evaluations_per_s"],
                                  unit="node-evaluations/s", n_gpus=world, higher_is_better=True, dtype="f64", data="synthetic")))
        if world > 1:
            dist.destroy_process_group()
        return
    runner = ConfigRunner(head, dev, rank, world)
    t = time_config(runner, args.steps, args.warmup, fence, sampler)
    if args.dump_outputs and rank == 0:  # before the legs below overwrite the first chunk's states and free the Jacobian
        dump_outputs(args.dump_outputs, runner.outputs(t["gathered"]))
    t["el_ms"] = max_over_ranks(t["el_ms"])
    clocks = sampler.stop(*t["marks"]) if rank == 0 else None
    peak_tf = fp64_probe(dev)
    peak_src = "DFMA-chain probe measured in this run (MEASURED_PEAKS.json has no FP64 figure; nominal 37.2)"
    res = config_result(head, runner, t, args.steps, world, peak_tf, hbm_peak, peak_src)
    q, qd, tau, f = runner.inp[0]
    qn, qdn, fn = runner.out[0]
    model, n, N = runner.model, runner.n, runner.N

    # ---- values-only kernel on the first chunk (reported next to the headline; same units) ----
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        runner.ev.step_rk4(q, qd, tau, f, runner.c["dt"], out=(qn, qdn, fn))
    torch.cuda.synchronize()
    e0.record()
    for _ in range(3):
        runner.ev.step_rk4(q, qd, tau, f, runner.c["dt"], out=(qn, qdn, fn))
    e1.record()
    torch.cuda.synchronize()
    values_ms = e0.elapsed_time(e1) / 3
    Uc = runner.Bc * N

    # ---- end to end through the host-facing API (C2 headline only): pinned host in -> H2D -> kernels -> D2H ----
    e2e = e2e_reduced = None
    if head == "C2":
        from mpc_fatigue_b200.dist import allgather_rows
        from mpc_fatigue_b200.pipeline import HostStepPipeline
        B = runner.Bc
        U = runner.U
        hq, hqd, htau, hf = (torch.empty((n, U), dtype=torch.float64).pin_memory() for _ in range(4))
        for h_, d_ in ((hq, q), (hqd, qd), (htau, tau), (hf, f)):
            h_.copy_(d_)
        del runner.jac
        runner.jac = None
        torch.cuda.empty_cache()
        link = pcie_probe(dev)
        e2e_steps = max(1, min(args.steps, 3))

        def timed_pipe(pipe):
            pipe.run(hq, hqd, htau, hf, runner.c["dt"], B, N)  # warm-up pass
            fence()
            w0 = time.perf_counter()
            for _ in range(e2e_steps):
                stats = pipe.run(hq, hqd, htau, hf, runner.c["dt"], B, N)
                if world > 1:
                    allgather_rows(pipe.reduced)
            fence()
            return max_over_ranks(time.perf_counter() - w0), stats

        pipe = HostStepPipeline(model, dev, chunk_units=1 << 19, skip_structural_zeros=True)
        e2e_s, stats = timed_pipe(pipe)
        d2h_gbs = stats["d2h_bytes"] * e2e_steps / e2e_s / 1e9
        e2e = {"value": world * U * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(stats["h2d_bytes"]),
               "d2h_bytes_per_step": int(stats["d2h_bytes"]), "steps": e2e_steps, "numa_node_rank0": numa,
               "d2h_gbs": d2h_gbs, "link_peak": link, "d2h_frac_of_link_peak": d2h_gbs / max(link["d2h_gbs"], 1e-9),
               "what": "HostStepPipeline.run: pinned host q,qd,tau,f -> chunked H2D -> step_rk4_jvp + cost_residual -> one gather "
                       "kernel packs q+,qd+,f+ and the 348 structurally non-zero Jacobian planes (of 450: d(q+,qd+)/df = 0, df+/df "
                       "diagonal) into a contiguous staging buffer -> ONE D2H copy per chunk into pinned host memory (copy-bound: "
                       "2.9 KB per unit over PCIe)"}
        del pipe
        torch.cuda.empty_cache()
        # same host-facing call, only the per-scenario cost / residual rows return (device-resident consumer): beside e2e, never instead
        pipe_r = HostStepPipeline(model, dev, chunk_units=1 << 19, outputs="reduced")
        e2e_r_s, stats_r = timed_pipe(pipe_r)
        e2e_reduced = {"value": world * U * e2e_steps / e2e_r_s, "unit": UNIT, "h2d_bytes_per_step": int(stats_r["h2d_bytes"]),
                       "d2h_bytes_per_step": int(stats_r["d2h_bytes"]),
                       "what": "HostStepPipeline(outputs='reduced'): pinned host inputs -> H2D -> step_rk4_jvp + cost_residual -> D2H of the "
                               "[4, B] per-scenario cost/residual rows only"}
        del pipe_r
    del runner
    torch.cuda.empty_cache()

    # ---- the other configs, measured in the same run (short: 1-3 timed steps each) ----
    others = {}
    if head == "C2" and not args.only_headline:
        names = ["C5"] if world > 1 else ["C3", "C4", "C5"]
        for name in names:
            try:
                r = ConfigRunner(name, dev, rank, world)
                k = 1 if name == "C4" else 3
                tt = time_config(r, k, 1, fence)
                tt["el_ms"] = max_over_ranks(tt["el_ms"])
                others[name] = config_result(name, r, tt, k, world, peak_tf, hbm_peak, peak_src)
                del r
            except Exception as exc:  # noqa: BLE001 - a failing side config must not take the headline line with it
                others[name] = {"error": "%s: %s" % (type(exc).__name__, exc)}
            torch.cuda.empty_cache()
        if world == 1:
            try:
                others["C1"] = run_c1(dev)
            except Exception as exc:  # noqa: BLE001
                others["C1"] = {"error": "%s: %s" % (type(exc).__name__, exc)}

    if rank == 0:
        fmv = frozen_flop_model(n)
        cpu = cpu_baseline() if world == 1 and not args.no_cpu else None
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup_steps(args.steps, args.warmup),
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": CONFIGS[head]["scaling"], "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": res["config"], "clocks": clocks, "gpu_launches": res["gpu_launches"],
            "e2e": e2e, "e2e_reduced_rows": e2e_reduced, "roofline": res["roofline"],
            "values_only": {"value": Uc / (values_ms * 1e-3), "unit": UNIT, "kernel_ms": values_ms, "units": Uc,
                            "roofline_frac_fp64_frozen_model": fmv["step_values"] * Uc / (values_ms * 1e-3) / 1e12 / peak_tf},
            "cpu_baseline": cpu, "checksum_cost": res["checksum_cost"], "chunks_per_step": res["chunks_per_step"],
            "kernel_family": res["kernel_family"], "configs": others,
        }
        if e2e is None:
            line["e2e"] = {"value": None, "unit": UNIT, "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
                           "what": "the host-facing end-to-end leg is measured on the C2 headline only"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=["C1", "C2", "C3", "C4", "C5"])
    ap.add_argument("--only-headline", action="store_true", help="skip the side configs (C1, C3, C4, C5) of the default run")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the headline config's outputs of the last "
                    "step as DIR/<name>.npy (float64, under 64 MB in all: larger outputs keep a fixed, seeded sample of their units)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
