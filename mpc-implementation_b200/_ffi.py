"""ctypes binding of include/nmpc_b200.h (libnmpc_b200.so, built in-tree under csrc/).

There is deliberately no fallback: if the CUDA library is missing or cannot be loaded the import of
`lib()` raises, and `nmpc_create` itself fails on a machine without an sm_100 device.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

_CSRC = Path(__file__).resolve().parent / "csrc"
LIB_PATH = Path(__import__("os").environ.get("NMPC_B200_LIB", _CSRC / "libnmpc_b200.so"))     # override: A/B timing of library builds

NMPC_OBS_PER_INSTANCE = 1
NMPC_PREDICT_TARGET = 2      # nmpc_solve_and_step / nmpc_run_closed_loop: the target's own Euler prediction, made in the kernel
NMPC_KEEP_BARRIER = 4        # nmpc_solve(_host): keep the final iterate's barrier data for nmpc_sensitivity

# CasADi's stats()['return_status'] strings of the IPOPT plugin
STATUS_NAMES = {0: "Solve_Succeeded", 1: "Maximum_Iterations_Exceeded", 2: "Restoration_Failed",
                3: "Search_Direction_Becomes_Too_Small", 4: "Invalid_Number_Detected", 5: "Error_In_Step_Computation",
                6: "Infeasible_Problem_Detected"}


class NmpcSpec(C.Structure):
    """struct nmpc_spec (include/nmpc_b200.h)."""
    _fields_ = [("T", C.c_double), ("N", C.c_int32), ("n_obs", C.c_int32),
                ("w1", C.c_double), ("w2", C.c_double), ("vfov", C.c_double), ("hfov", C.c_double),
                ("max_iter", C.c_int32), ("scaling", C.c_int32), ("tol", C.c_double),
                ("max_batch", C.c_int32), ("fill", C.c_int32), ("model", C.c_int32)]


class NmpcWarmOpts(C.Structure):
    """struct nmpc_warm_opts"""
    _fields_ = [("mu_init", C.c_double), ("bound_push", C.c_double), ("bound_frac", C.c_double),
                ("slack_bound_push", C.c_double), ("slack_bound_frac", C.c_double), ("mult_bound_push", C.c_double)]


class NmpcStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("factorizations", C.c_int64),
                ("ls_trials", C.c_int64), ("soc_accepted", C.c_int64), ("resto_calls", C.c_int64), ("resto_iters", C.c_int64),
                ("watchdog_starts", C.c_int64), ("soft_resto_steps", C.c_int64), ("filter_resets", C.c_int64),
                ("trial_passes", C.c_int64)]


EXPORTS = ["nmpc_create", "nmpc_destroy", "nmpc_solve", "nmpc_solve_host", "nmpc_solve_host_async", "nmpc_synchronize", "nmpc_query", "nmpc_solve_and_step", "nmpc_run_closed_loop", "nmpc_eval", "nmpc_lam_p", "nmpc_sensitivity", "nmpc_sensitivity_obstacles", "nmpc_barrier_data", "nmpc_step",
           "nmpc_get_stats", "nmpc_set_debug_log", "nmpc_set_order", "nmpc_set_weights", "nmpc_set_target_trajectory", "nmpc_set_obstacle_motion", "nmpc_set_schedule", "nmpc_set_warm_start", "nmpc_measure_fp64_peak", "nmpc_n_w", "nmpc_n_g", "nmpc_n_p",
           "nmpc_last_error", "nmpc_version"]

_lib = None


def build(force: bool = False) -> Path:
    """Compile csrc/ for sm_100a with nvcc (cross-compiles without a GPU)."""
    args = ["make", "-C", str(_CSRC), "-s"] + (["-B"] if force else [])   # the Makefile runs itself with -j8
    subprocess.check_call(args)
    return LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(f"{LIB_PATH} is missing: run __graft_entry__.build() (there is no CPU fallback)")
    L = C.CDLL(str(LIB_PATH))
    dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_void_p
    L.nmpc_create.argtypes = [C.POINTER(NmpcSpec), C.c_int, C.POINTER(vp)]
    L.nmpc_destroy.argtypes = [vp]
    # pointers are passed as integers (device or host addresses)
    L.nmpc_solve.argtypes = [vp, C.c_int32] + [vp] * 7 + [C.c_uint32] + [vp] * 7 + [vp]
    L.nmpc_solve_host.argtypes = [vp, C.c_int32] + [vp] * 7 + [C.c_uint32] + [vp] * 7
    L.nmpc_solve_host_async.argtypes = [vp, C.c_int32] + [vp] * 7 + [C.c_uint32] + [vp] * 7
    L.nmpc_synchronize.argtypes = [vp]
    L.nmpc_query.argtypes = [vp, C.POINTER(C.c_int32)]
    L.nmpc_solve_and_step.argtypes = [vp, C.c_int32] + [vp] * 7 + [C.c_uint32] + [vp] * 7 + [vp]
    if hasattr(L, "nmpc_run_closed_loop"):
        L.nmpc_run_closed_loop.argtypes = [vp, C.c_int32, C.c_int32] + [vp] * 7 + [C.c_uint32] + [vp] * 8 + [vp]
    L.nmpc_eval.argtypes = [vp, C.c_int32, vp, vp, vp, C.c_uint32, C.c_double, vp, vp] + [vp] * 5 + [vp]
    L.nmpc_step.argtypes = [vp, C.c_int32] + [vp] * 6 + [vp]
    if hasattr(L, "nmpc_lam_p"):
        L.nmpc_lam_p.argtypes = [vp, C.c_int32, vp, vp, vp, C.c_uint32, vp, vp, vp]
    if hasattr(L, "nmpc_sensitivity"):
        L.nmpc_sensitivity.argtypes = [vp, C.c_int32, vp, vp, vp, vp, C.c_uint32, vp, vp, vp, vp]
        L.nmpc_barrier_data.argtypes = [vp, vp, vp, vp]
    if hasattr(L, "nmpc_sensitivity_obstacles"):
        L.nmpc_sensitivity_obstacles.argtypes = [vp, C.c_int32, vp, vp, vp, vp, C.c_uint32, vp, vp, vp]
    L.nmpc_get_stats.argtypes = [vp, C.POINTER(NmpcStats)]
    L.nmpc_set_debug_log.argtypes = [vp, vp, C.c_int32]
    L.nmpc_set_order.argtypes = [vp, vp]
    L.nmpc_set_weights.argtypes = [vp, vp]
    L.nmpc_set_target_trajectory.argtypes = [vp, vp]
    if hasattr(L, "nmpc_set_warm_start"):
        L.nmpc_set_warm_start.argtypes = [vp, vp, vp, C.POINTER(NmpcWarmOpts)]
    if hasattr(L, "nmpc_set_schedule"):      # (absent only in old builds loaded through NMPC_B200_LIB for A/B timing)
        L.nmpc_set_schedule.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp, C.c_int32]
    if hasattr(L, "nmpc_set_obstacle_motion"):
        L.nmpc_set_obstacle_motion.argtypes = [vp, vp, vp]
    L.nmpc_measure_fp64_peak.argtypes = [C.c_int, C.POINTER(C.c_double)]
    L.nmpc_n_w.argtypes = [C.POINTER(NmpcSpec)]
    L.nmpc_n_g.argtypes = [C.POINTER(NmpcSpec)]
    L.nmpc_n_p.argtypes = [C.POINTER(NmpcSpec)]
    for name in EXPORTS:
        if hasattr(L, name):
            getattr(L, name).restype = C.c_int
    L.nmpc_last_error.restype = C.c_char_p
    L.nmpc_version.restype = C.c_char_p
    L.nmpc_n_w.restype = C.c_int32
    L.nmpc_n_g.restype = C.c_int32
    L.nmpc_n_p.restype = C.c_int32
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what} failed: {lib().nmpc_last_error().decode()}")
