"""ctypes binding of the C ABI declared in include/nlml_hpe_b200.h.

There is deliberately no fallback: if the shared library is missing or a call fails, an
exception is raised.  Nothing here imports oracle/.
"""
from __future__ import annotations

import ctypes
import os

from . import _build

c_float_p = ctypes.POINTER(ctypes.c_float)
c_double_p = ctypes.POINTER(ctypes.c_double)

EXPORTS = [
    "nlml_abi_version", "nlml_last_error",
    "nlml_tucker_plan_create", "nlml_tucker_plan_destroy", "nlml_tucker_fit_f32",
    "nlml_tucker_fit_host_f32", "nlml_tucker_solve_f32", "nlml_tucker_solve_host_f32", "nlml_tucker_launch_count",
    "nlml_tucker_fit_landmarks_f32", "nlml_tucker_fit_landmarks_host_f32", "nlml_tucker_solve_landmarks_f32",
    "nlml_tucker_solve_landmarks_host_f32", "nlml_tucker_powell_landmarks_f64",
    "nlml_tucker_powell_f64", "nlml_debug_powell_objective", "nlml_debug_project_tc", "nlml_cosine_fit_f64", "nlml_core_times_features_f32",
    "nlml_mlp_plan_create", "nlml_mlp_plan_destroy", "nlml_mlp_forward_f32",
    "nlml_mlp_forward_host_f32", "nlml_mlp_forward_landmarks_f32", "nlml_mlp_forward_landmarks_host_f32", "nlml_pose_postprocess_f64", "nlml_mlp_latent_f32", "nlml_mlp_launch_count", "nlml_mlp_set_path",
    "nlml_measure_fp32_tflops", "nlml_measure_fp32_tflops_3reg", "nlml_measure_tf32_tflops", "nlml_debug_tf32_gemm", "nlml_debug_tf32_gemm_mode",
]

_lib = None


class NlmlError(RuntimeError):
    pass


def load():
    """Load libnlml_hpe_b200.so (built in-tree by __graft_entry__.build / _build.build)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("NLML_HPE_LIB") or _build.LIB_PATH   # override: development builds only
    if not os.path.exists(path):
        raise NlmlError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a).  nlml_hpe_b200 has no CPU fallback.")
    lib = ctypes.CDLL(path)
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float
    lib.nlml_abi_version.restype = i32
    lib.nlml_last_error.restype = ctypes.c_char_p
    lib.nlml_tucker_plan_create.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, ctypes.POINTER(vp)]
    lib.nlml_tucker_plan_destroy.argtypes = [vp]
    lib.nlml_tucker_plan_destroy.restype = None
    lib.nlml_tucker_fit_f32.argtypes = [vp, vp, i64, i64, i32, f32, f32, vp, i64, i32, vp]
    lib.nlml_tucker_fit_host_f32.argtypes = [vp, vp, i64, i64, i32, f32, f32, vp, i64]
    lib.nlml_tucker_solve_f32.argtypes = [vp, vp, i64, i64, i32, vp, i64, vp, vp]
    lib.nlml_tucker_solve_host_f32.argtypes = [vp, vp, i64, i64, i32, vp, i64]
    lib.nlml_tucker_powell_f64.argtypes = [vp, vp, i64, i64, vp, i64, vp, vp, vp]
    lib.nlml_tucker_fit_landmarks_f32.argtypes = lib.nlml_tucker_fit_f32.argtypes
    lib.nlml_tucker_fit_landmarks_host_f32.argtypes = lib.nlml_tucker_fit_host_f32.argtypes
    lib.nlml_tucker_solve_landmarks_f32.argtypes = lib.nlml_tucker_solve_f32.argtypes
    lib.nlml_tucker_solve_landmarks_host_f32.argtypes = lib.nlml_tucker_solve_host_f32.argtypes
    lib.nlml_tucker_powell_landmarks_f64.argtypes = lib.nlml_tucker_powell_f64.argtypes
    lib.nlml_debug_powell_objective.argtypes = [vp, vp, vp, i32, vp]
    lib.nlml_debug_project_tc.argtypes = [vp, vp, i64, i64, vp]
    lib.nlml_cosine_fit_f64.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, i32]
    lib.nlml_core_times_features_f32.argtypes = [vp, vp, i64, i32, i32, vp, i32]
    lib.nlml_tucker_launch_count.argtypes = [vp]
    lib.nlml_tucker_launch_count.restype = i64
    lib.nlml_mlp_plan_create.argtypes = [vp, vp, vp, vp, i32, ctypes.POINTER(vp)]
    lib.nlml_mlp_plan_destroy.argtypes = [vp]
    lib.nlml_mlp_plan_destroy.restype = None
    lib.nlml_mlp_forward_f32.argtypes = [vp, vp, i64, i64, vp, vp]
    lib.nlml_mlp_forward_host_f32.argtypes = [vp, vp, i64, i64, vp]
    lib.nlml_mlp_latent_f32.argtypes = [vp, vp, i64, i64, vp, vp]
    lib.nlml_mlp_forward_landmarks_f32.argtypes = [vp, vp, i64, i64, vp, vp]
    lib.nlml_mlp_forward_landmarks_host_f32.argtypes = [vp, vp, i64, i64, vp]
    lib.nlml_pose_postprocess_f64.argtypes = [vp, i64, i32, ctypes.c_double, vp, vp]
    lib.nlml_mlp_launch_count.argtypes = [vp]
    lib.nlml_mlp_launch_count.restype = i64
    lib.nlml_mlp_set_path.argtypes = [vp, i32]
    lib.nlml_measure_fp32_tflops.argtypes = [i32, c_double_p]
    lib.nlml_measure_fp32_tflops_3reg.argtypes = [i32, c_double_p]
    lib.nlml_measure_tf32_tflops.argtypes = [i32, c_double_p]
    lib.nlml_debug_tf32_gemm.argtypes = [vp, vp, i32, i32, vp]
    lib.nlml_debug_tf32_gemm_mode.argtypes = [vp, vp, i32, i32, vp, i32]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().nlml_last_error().decode(errors="replace")
        raise NlmlError(f"nlml_hpe_b200 call failed (code {rc}): {msg}")
