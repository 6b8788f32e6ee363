"""ctypes binding of libtneq_b200.so (include/tneq_b200.h).

The product has no CPU path: if the library is missing, or no B200 is
visible, everything that would compute raises RuntimeError.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, byref, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtneq_b200.so")

EXPORTS = ["tnq_device_check", "tnq_plan_create", "tnq_plan_destroy", "tnq_plan_num_inputs",
           "tnq_plan_num_outputs", "tnq_plan_query", "tnq_plan_run", "tnq_gemm_tf32x3", "tnq_gemm_tf32x3_view", "tnq_gemm_tf32x3_bk", "tnq_gemm_kernel_attrs", "tnq_permute_f32", "tnq_fold_vec_f32", "tnq_outer_acc_f32", "tnq_cplx_expand_f32",
           "tnq_cplx_fold_f32", "tnq_gemm_f64", "tnq_permute_f64", "tnq_fold_vec_f64", "tnq_outer_acc_f64", "tnq_cplx_expand_f64",
           "tnq_cplx_fold_f64", "tnq_mps_chain", "tnq_mps_chain_workspace_bytes", "tnq_mps_chain_x", "tnq_mps_chain_sample", "tnq_mps_ladder",
           "tnq_mps_ladder_workspace_bytes", "tnq_mps_ladder2", "tnq_mps_ladder2_workspace_bytes", "tnq_mps_ladder2_geometry", "tnq_allreduce_oneshot", "tnq_allreduce_oneshot_words", "tnq_allreduce_set_timeout_ms", "tnq_sgdg_step", "tnq_sgdg_step_flat",
           "tnq_sgdg_step_c64", "tnq_sgdg_step_flat_c64", "tnq_sgdg_step_f64", "tnq_sgdg_step_flat_f64", "tnq_sgdg_step_c128",
           "tnq_sgdg_step_flat_c128", "tnq_launch_count",
           "tnq_last_error"]


class RunInfo(ctypes.Structure):
    _fields_ = [("tile_samples", c_int32), ("grid", c_int32), ("frame_in_smem", c_int32), ("launches", c_int32),
                ("smem_bytes", c_int64), ("workspace_bytes", c_int64)]


_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  tneq_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.tnq_last_error.restype = c_char_p
    lib.tnq_launch_count.restype = c_int64
    lib.tnq_device_check.restype = c_int
    lib.tnq_plan_create.argtypes = [POINTER(c_int64), c_int64, POINTER(c_void_p)]
    lib.tnq_plan_destroy.argtypes = [c_void_p]
    lib.tnq_plan_destroy.restype = None
    lib.tnq_plan_num_inputs.argtypes = [c_void_p]
    lib.tnq_plan_num_outputs.argtypes = [c_void_p]
    lib.tnq_plan_query.argtypes = [c_void_p, c_int64, POINTER(RunInfo)]
    lib.tnq_plan_run.argtypes = [c_void_p, c_int64, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int64),
                                 POINTER(c_void_p), POINTER(c_double), c_void_p, c_int64, c_void_p]
    lib.tnq_gemm_tf32x3.argtypes = [c_void_p, c_void_p, c_void_p] + [c_int64] * 10 + [c_int, c_void_p]
    lib.tnq_gemm_tf32x3_view.argtypes = [c_void_p] + [c_int64] * 7 + [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p]
    lib.tnq_gemm_tf32x3_bk.argtypes = [c_void_p, c_int, c_int64, c_void_p, c_int, c_int64, c_void_p, c_int64, c_int64, c_int64,
                                       c_int64, c_void_p]
    lib.tnq_fold_vec_f32.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]
    lib.tnq_outer_acc_f32.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]
    lib.tnq_permute_f32.argtypes = [c_void_p, c_void_p, c_int, POINTER(c_int64), POINTER(c_int64), c_int, c_int, c_void_p]
    lib.tnq_cplx_expand_f32.argtypes = [c_void_p, c_void_p, c_int, POINTER(c_int64), POINTER(c_int64), c_int, c_int,
                                        c_int, c_void_p]
    lib.tnq_cplx_fold_f32.argtypes = [c_void_p, c_void_p, c_int, POINTER(c_int64), POINTER(c_int64), c_int64, c_int64,
                                      c_int, c_int, c_void_p]
    # float64 / complex128 siblings: same arguments, element strides in doubles
    lib.tnq_gemm_f64.argtypes = lib.tnq_gemm_tf32x3.argtypes
    for name in ("permute", "fold_vec", "outer_acc", "cplx_expand", "cplx_fold"):
        getattr(lib, f"tnq_{name}_f64").argtypes = getattr(lib, f"tnq_{name}_f32").argtypes
    lib.tnq_mps_chain_workspace_bytes.argtypes = [c_int, c_int, c_int64]
    lib.tnq_mps_chain_workspace_bytes.restype = c_int64
    lib.tnq_mps_chain.argtypes = [c_int, c_int, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64),
                                  c_int64, c_int, c_void_p, c_void_p, c_void_p, POINTER(c_void_p), c_double, c_void_p,
                                  c_int64, c_void_p]
    lib.tnq_mps_chain_x.argtypes = [c_int, c_int, POINTER(c_void_p), POINTER(c_void_p), c_void_p, c_int64, c_int64,
                                    POINTER(c_float), c_int64, c_void_p, c_void_p, c_void_p]
    lib.tnq_mps_chain_sample.argtypes = [c_int, c_int, POINTER(c_void_p), POINTER(c_void_p), c_int64, c_int, c_void_p,
                                         c_void_p, c_void_p, POINTER(c_float), c_void_p, c_void_p]
    lib.tnq_mps_ladder_workspace_bytes.argtypes = [c_int, c_int, c_int64, c_int]
    lib.tnq_mps_ladder_workspace_bytes.restype = c_int64
    lib.tnq_mps_ladder.argtypes = [c_int, c_int, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p),
                                   POINTER(c_int64), c_int64, c_int, c_void_p, c_void_p, c_void_p, POINTER(c_void_p),
                                   POINTER(c_void_p), c_double, c_void_p, c_int64, c_void_p]
    lib.tnq_mps_ladder2_workspace_bytes.argtypes = [c_int, c_int64, c_int]
    lib.tnq_mps_ladder2_workspace_bytes.restype = c_int64
    lib.tnq_mps_ladder2_geometry.argtypes = [c_int, c_int64, c_int, POINTER(c_int64)]
    lib.tnq_mps_ladder2.argtypes = [c_int, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p),
                                    POINTER(c_int64), c_int64, c_int, c_void_p, c_void_p, c_void_p, POINTER(c_void_p),
                                    POINTER(c_void_p), c_double, c_void_p, c_int64, c_void_p]
    lib.tnq_allreduce_oneshot_words.argtypes = [c_int64]
    lib.tnq_allreduce_oneshot_words.restype = c_int64
    lib.tnq_allreduce_set_timeout_ms.argtypes = [c_int64]
    lib.tnq_allreduce_oneshot.argtypes = [c_void_p, c_int, c_int, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                          c_float, c_void_p]
    lib.tnq_sgdg_step_flat.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float,
                                       c_float, c_void_p]
    lib.tnq_sgdg_step.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_float,
                                  c_void_p]
    # complex64 / float64 / complex128 siblings: the same arguments, lr and momentum in double for the double types
    for sfx, real in (("c64", c_float), ("f64", c_double), ("c128", c_double)):
        getattr(lib, f"tnq_sgdg_step_{sfx}").argtypes = lib.tnq_sgdg_step.argtypes[:7] + [real, real, c_void_p]
        getattr(lib, f"tnq_sgdg_step_flat_{sfx}").argtypes = lib.tnq_sgdg_step_flat.argtypes[:8] + [real, real, c_void_p]
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise RuntimeError("tneq_b200: " + load().tnq_last_error().decode("utf-8", "replace"))


_graph_launches = 0


def add_graph_launches(n: int) -> None:
    """Kernels of this library that ran through a CUDA-graph replay (they are launched by
    cudaGraphLaunch, not by the library's own launch sites)."""
    global _graph_launches
    _graph_launches += int(n)


def launch_count() -> int:
    """Kernels of this library launched so far, directly or by graph replay."""
    return int(load().tnq_launch_count()) + _graph_launches
