"""ctypes binding of the C-ABI in include/mpcf.h (libmpcf.so, built in-tree by csrc/Makefile).

There is no CPU fallback: if the library is missing this module raises at import time, and every
batch call needs CUDA device pointers.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MPCF_LIB") or os.path.join(_HERE, "lib", "libmpcf.so")  # MPCF_LIB: A/B-test another build

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "mpc_fatigue_b200: %s not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C mpc_fatigue_b200/csrc` (nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)

lib = C.CDLL(LIB_PATH)

OK, EINVAL, EPARSE, EJOINT, EFRAME, ESINGULAR, ECUDA, ELIMIT = 0, -1, -2, -3, -4, -5, -6, -7
SYNTH_CHAIN, SYNTH_HUMANOID, SYNTH_DUAL_ARM = 0, 1, 2
MAX_DOF, MAX_EE = 64, 4


class Opts(C.Structure):
    _fields_ = [("armature", C.c_double), ("gravity", C.c_double * 3), ("lambda_", C.c_double),
                ("kappa", C.c_double), ("ctau", C.c_double), ("cv", C.c_double)]


class Coupling(C.Structure):
    _fields_ = [("ee_frame", C.c_int * 2), ("weight", C.c_double)]


class RowsOpts(C.Structure):
    _fields_ = [("ee_frame", C.c_int * 2), ("wsign", C.c_double), ("fdes", C.c_double * 3), ("dist2_ref", C.c_double), ("mu", C.c_double),
                ("p_ref", C.c_double * 3), ("w_box", C.c_double), ("w_qd", C.c_double), ("w_F", C.c_double), ("h", C.c_double)]


_dp = C.c_void_p  # device pointers travel as integers
_sig = {
    "mpcf_opts_default": (None, [C.POINTER(Opts)]),
    "mpcf_model_create_from_urdf": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(Opts), C.POINTER(C.c_void_p)]),
    "mpcf_model_create_synthetic": (C.c_int, [C.c_int, C.c_int, C.c_ulonglong, C.POINTER(Opts), C.POINTER(C.c_void_p)]),
    "mpcf_model_destroy": (C.c_int, [C.c_void_p]),
    "mpcf_model_info": (C.c_int, [C.c_void_p] + [C.POINTER(C.c_int)] * 4),
    "mpcf_frame_id": (C.c_int, [C.c_void_p, C.c_char_p]),
    "mpcf_joint_name": (C.c_char_p, [C.c_void_p, C.c_int]),
    "mpcf_frame_name": (C.c_char_p, [C.c_void_p, C.c_int]),
    "mpcf_model_export": (C.c_long, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t]),
    "mpcf_model_set_armature": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "mpcf_model_set_fatigue": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "mpcf_model_set_coupling": (C.c_int, [C.c_void_p, C.POINTER(Coupling)]),
    "mpcf_model_kernel_family": (C.c_char_p, [C.c_void_p]),
    "mpcf_rnea_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, C.c_void_p]),
    "mpcf_fk_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_long, _dp, _dp, _dp, C.c_void_p]),
    "mpcf_frame_jac_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_long, _dp, _dp, C.c_void_p]),
    "mpcf_frame_jac_t_wrench_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_long, _dp, _dp, _dp, C.c_void_p]),
    "mpcf_node_eval_ref_batch": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_double, C.c_long, _dp, _dp, _dp,
                                           _dp, _dp, C.c_double, _dp, _dp, _dp, C.c_void_p]),
    "mpcf_node_eval_ref_jvp_batch": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_double, C.c_long, _dp, _dp, _dp, _dp, _dp, _dp,
                                               C.c_void_p]),
    "mpcf_aba_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, C.c_void_p]),
    "mpcf_step_rk4_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, _dp, C.c_void_p]),
    "mpcf_rollout_rk4_batch": (C.c_int, [C.c_void_p, C.c_long, C.c_int, _dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, C.c_void_p]),
    "mpcf_step_rk4_jvp_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, _dp, _dp,
                                          C.c_void_p]),
    "mpcf_step_rk4_jvp_dual_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, _dp, _dp,
                                               C.c_void_p]),
    "mpcf_step_rk4_jvp_strided_batch": (C.c_int, [C.c_void_p, C.c_long, C.c_long, _dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, _dp, _dp,
                                                  C.c_long, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpcf_step_rk4_jvp_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_long]),
    "mpcf_step_rk4_jvp_ws_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, _dp, _dp,
                                             C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpcf_step_rk4_vjp_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, C.c_double, _dp] + [_dp] * 11
                                + [C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpcf_rollout_rk4_vjp_batch": (C.c_int, [C.c_void_p, C.c_long, C.c_int, _dp, _dp, _dp, _dp, C.c_double] + [_dp] * 10
                                   + [C.c_void_p, C.c_size_t, C.c_void_p]),
    "mpcf_step_rk4_hess_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, C.c_double, _dp] + [_dp] * 4 + [C.c_void_p]),
    "mpcf_step_rk4_hvp_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, C.c_double, _dp] + [_dp] * 16 + [C.c_void_p]),
    "mpcf_fd_derivs_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, _dp, _dp, C.c_void_p]),
    "mpcf_rnea_derivs_batch": (C.c_int, [C.c_void_p, C.c_long, _dp, _dp, _dp, _dp, _dp, _dp, C.c_void_p]),
    "mpcf_cost_residual_batch": (C.c_int, [C.c_void_p, C.c_long, C.c_int] + [_dp] * 7 + [C.c_double] * 7 + [_dp, C.c_void_p]),
    "mpcf_cost_residual_table_batch": (C.c_int, [C.c_void_p, C.c_long, C.c_int] + [_dp] * 7 + [C.c_double] * 2 + [_dp, C.c_double, _dp, C.c_long,
                                                                                                         C.c_void_p]),
    "mpcf_ocp_rows_count": (C.c_int, [C.c_void_p]),
    "mpcf_ocp_rows_count_arms": (C.c_int, [C.c_void_p, C.c_int]),
    "mpcf_ocp_rows_batch": (C.c_int, [C.c_void_p, C.POINTER(RowsOpts), C.c_long, C.c_int] + [_dp] * 13 + [C.c_void_p]),
    "mpcf_probe_fp64": (C.c_int, [C.c_long, C.c_int, _dp, C.c_void_p]),
    "mpcf_memcpy2d_async": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_void_p]),
    "mpcf_gather_planes": (C.c_int, [_dp, C.c_long, C.c_void_p, C.c_int, C.c_long, _dp, C.c_void_p]),
    "mpcf_profile_enable": (C.c_int, [C.c_int]),
    "mpcf_profile_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_long)]),
    "mpcf_last_error": (C.c_char_p, []),
    "mpcf_launch_count": (C.c_long, []),
}
for _name, (_res, _args) in _sig.items():
    _fn = getattr(lib, _name)  # AttributeError here means the library does not export what mpcf.h declares
    _fn.restype = _res
    _fn.argtypes = _args

EXPORTED_SYMBOLS = tuple(_sig)


def last_error() -> str:
    return (lib.mpcf_last_error() or b"").decode()


def check(rc: int) -> None:
    """Map C error codes to Python exceptions (reference behaviour: C++ exceptions -> RuntimeError/IndexError)."""
    if rc >= 0:
        return
    msg = last_error()
    if rc in (EINVAL, EPARSE, EJOINT, ELIMIT):
        raise ValueError(msg)
    if rc == EFRAME:
        raise IndexError(msg)
    if rc == ESINGULAR:
        raise ZeroDivisionError(msg)
    raise RuntimeError(msg)
