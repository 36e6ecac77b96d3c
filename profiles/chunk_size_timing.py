"""Throughput of the tree Jacobian pipeline (37-joint tree, 113,664 units) against the chunk size the caller's workspace allows:
the entry cuts its chunks to whole waves of the derivative kernel (kernels_tree.cu: run_tree), this script shows why.
    python profiles/chunk_size_timing.py        (GPU)"""
import ctypes as C, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from mpc_fatigue_b200 import _capi
from mpc_fatigue_b200.model import Model
from mpc_fatigue_b200.synth import synth_batch
m = Model.synthetic("humanoid", 37, seed=7, armature=1e-2)
n = m.n
lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
U = 113664
q, qd, tau, f = synth_batch(lim, 0, U // 32, 32, seed=3, device="cuda")
out = [torch.empty_like(q) for _ in range(3)]
jac = torch.empty((3 * n, 4 * n + 1, U), dtype=torch.float64, device="cuda")
p = lambda t: C.c_void_p(t.data_ptr())
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
for chunk in (32768, 28416, 14208, 30720, 24576, 21312, 18944):
    need = int(_capi.lib.mpcf_step_rk4_jvp_workspace_bytes(m.handle, chunk))
    # the entry sizes its chunk from the bytes it is given: trim the slack so that exactly `chunk` units fit
    per_unit = (need - 148 * 4 * 2 * 40 * 128 * 8) // ((chunk + 31) // 32 * 32)
    scratch = 148 * 2 * 2 * 40 * 128 * 8
    ws_bytes = chunk * per_unit + scratch + 64
    ws = torch.empty(ws_bytes // 8 + 16, dtype=torch.float64, device="cuda")
    def run():
        _capi.check(_capi.lib.mpcf_step_rk4_jvp_ws_batch(m.handle, U, p(q), p(qd), p(tau), p(f), 0.0125, None, p(out[0]), p(out[1]), p(out[2]), p(jac), p(ws), ws_bytes, st))
    run(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3): run()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    print("chunk %6d  %.3f ms  %.3e units/s" % (chunk, ms, U / ms * 1e3))
