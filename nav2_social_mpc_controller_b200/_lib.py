"""Loader of libsmpc.so (built in-tree by `make -C nav2_social_mpc_controller_b200/csrc`).

There is deliberately no fallback: if the library is missing or cannot be loaded, every
entry point of this package raises."""
from __future__ import annotations

import ctypes as C
import os

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# SMPC_LIB_PATH: load another build of the same library (csrc `make DEV=1` experiment builds); still no fallback
LIB_PATH = os.environ.get("SMPC_LIB_PATH") or os.path.join(_HERE, "libsmpc.so")
_lib = None


class SmpcError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libsmpc error {code}: {message}")
        self.code = code
        self.message = message


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    P = C.POINTER
    L.smpc_abi_version.restype = C.c_int
    L.smpc_last_error.restype = C.c_char_p
    L.smpc_params_default.argtypes = [P(abi.SmpcParams)]
    L.smpc_params_default.restype = None
    L.smpc_params_from_yaml.argtypes = [C.c_char_p, C.c_char_p, P(abi.SmpcParams)]
    L.smpc_params_from_yaml.restype = C.c_int
    L.smpc_problem_dims.argtypes = [P(abi.SmpcParams), C.c_int, P(C.c_int), P(C.c_int), P(C.c_int), P(C.c_int)]
    L.smpc_problem_dims.restype = C.c_int
    L.smpc_create.argtypes = [P(abi.SmpcParams), C.c_int, P(C.c_void_p)]
    L.smpc_create.restype = C.c_int
    L.smpc_destroy.argtypes = [C.c_void_p]
    L.smpc_destroy.restype = None
    L.smpc_solve_batch.argtypes = [C.c_void_p, P(abi.SmpcBatch), P(abi.SmpcResult)]
    L.smpc_solve_batch.restype = C.c_int
    L.smpc_solve_batch_device.argtypes = [C.c_void_p, P(abi.SmpcBatch), P(abi.SmpcResult), C.c_void_p]
    L.smpc_solve_batch_device.restype = C.c_int
    L.smpc_eval_batch_device.argtypes = [C.c_void_p, P(abi.SmpcBatch), C.c_void_p, P(abi.SmpcEvalOut), C.c_void_p]
    L.smpc_eval_batch_device.restype = C.c_int
    L.smpc_eval_batch.argtypes = [C.c_void_p, P(abi.SmpcBatch), C.c_void_p, P(abi.SmpcEvalOut)]
    L.smpc_eval_batch.restype = C.c_int
    L.smpc_multistart_argmin_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.smpc_multistart_argmin_device.restype = C.c_int
    L.smpc_last_kernel_ms.argtypes = [C.c_void_p]
    L.smpc_last_kernel_ms.restype = C.c_double
    L.smpc_launch_count.argtypes = [C.c_void_p]
    L.smpc_launch_count.restype = C.c_longlong
    L.smpc_measure_fp64_peak.argtypes = [C.c_void_p, P(C.c_double)]
    L.smpc_measure_fp64_peak.restype = C.c_int
    L.smpc_optimize.argtypes = [C.c_void_p, P(abi.SmpcOptimizeIo)]
    L.smpc_optimize.restype = C.c_int
    L.smpc_optimize_batch.argtypes = [C.c_void_p, P(abi.SmpcFleetIo)]
    L.smpc_optimize_batch.restype = C.c_int
    L.smpc_run_episodes.argtypes = [C.c_void_p, P(abi.SmpcEpisodeIo)]
    L.smpc_run_episodes.restype = C.c_int
    L.smpc_run_crowd_episodes.argtypes = [C.c_void_p, P(abi.SmpcEpisodeIo), P(abi.SmpcCrowdIo)]
    L.smpc_run_crowd_episodes.restype = C.c_int
    L.smpc_run_shared_episodes.argtypes = [C.c_void_p, P(abi.SmpcEpisodeIo), P(abi.SmpcCrowdIo), P(abi.SmpcSceneIo)]
    L.smpc_run_shared_episodes.restype = C.c_int
    L.smpc_reset_memory.argtypes = [C.c_void_p]
    L.smpc_reset_memory.restype = C.c_int
    L.smpc_project_people_batch.argtypes = [C.c_void_p, P(abi.SmpcProjectArgs)]
    L.smpc_project_people_batch.restype = C.c_int
    L.smpc_project_people_batch_device.argtypes = [C.c_void_p, P(abi.SmpcProjectArgs), C.c_void_p]
    L.smpc_project_people_batch_device.restype = C.c_int
    L.smpc_format_batch_device.argtypes = [C.c_void_p, P(abi.SmpcFormatArgs), C.c_void_p]
    L.smpc_format_batch_device.restype = C.c_int
    L.smpc_people_to_status_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p]
    L.smpc_people_to_status_device.restype = C.c_int
    L.smpc_memory_update_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
    L.smpc_memory_update_device.restype = C.c_int
    L.smpc_trajectorize_batch_device.argtypes = [C.c_void_p, P(abi.SmpcTrajectorizeArgs), C.c_void_p]
    L.smpc_trajectorize_batch_device.restype = C.c_int
    L.smpc_fov_filter_batch_device.argtypes = [C.c_void_p, P(abi.SmpcFovArgs), C.c_void_p]
    L.smpc_fov_filter_batch_device.restype = C.c_int
    L.smpc_multi_create.argtypes = [P(abi.SmpcParams), C.c_int, P(C.c_int), P(C.c_void_p)]
    L.smpc_multi_create.restype = C.c_int
    L.smpc_multi_destroy.argtypes = [C.c_void_p]
    L.smpc_multi_destroy.restype = None
    L.smpc_multi_device_count.argtypes = [C.c_void_p]
    L.smpc_multi_device_count.restype = C.c_int
    L.smpc_solve_batch_multi.argtypes = [C.c_void_p, P(abi.SmpcBatch), P(abi.SmpcResult), C.c_int]
    L.smpc_solve_batch_multi.restype = C.c_int
    L.smpc_debug_shard_bounds.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, P(C.c_int), P(C.c_int)]
    L.smpc_debug_shard_bounds.restype = C.c_int
    L.smpc_set_group.argtypes = [C.c_void_p, C.c_int]
    L.smpc_set_group.restype = C.c_int
    L.smpc_debug_polymin.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.smpc_debug_polymin.restype = C.c_int
    L.smpc_debug_math.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.smpc_debug_math.restype = C.c_int
    if L.smpc_abi_version() != abi.SMPC_ABI_VERSION:
        raise ImportError("libsmpc.so ABI version mismatch")
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise SmpcError(rc, lib().smpc_last_error().decode(errors="replace"))


EXPORTED_SYMBOLS = (
    "smpc_abi_version", "smpc_last_error", "smpc_params_default", "smpc_params_from_yaml", "smpc_problem_dims",
    "smpc_create", "smpc_destroy", "smpc_solve_batch", "smpc_solve_batch_device", "smpc_eval_batch_device",
    "smpc_eval_batch", "smpc_multistart_argmin_device", "smpc_last_kernel_ms", "smpc_launch_count",
    "smpc_measure_fp64_peak", "smpc_debug_polymin", "smpc_debug_math", "smpc_debug_plan_chunks", "smpc_set_group",
    "smpc_optimize", "smpc_optimize_batch", "smpc_run_episodes", "smpc_run_crowd_episodes",
    "smpc_run_shared_episodes",
    "smpc_reset_memory", "smpc_project_people_batch", "smpc_project_people_batch_device",
    "smpc_format_batch_device", "smpc_people_to_status_device", "smpc_memory_update_device",
    "smpc_trajectorize_batch_device", "smpc_fov_filter_batch_device", "smpc_multi_create", "smpc_multi_destroy",
    "smpc_multi_device_count", "smpc_solve_batch_multi", "smpc_debug_shard_bounds",
)
