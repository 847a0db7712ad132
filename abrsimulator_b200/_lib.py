"""ctypes binding of libabr_b200.so (C-ABI declared in include/abr_b200.h).

There is no CPU fallback: if the library cannot be loaded, or no CUDA device is
present, every compute call raises.
"""
from __future__ import annotations

import ctypes as C
import os

from . import _build

NUM_ACC = 11
NUM_STATS = 11
POLICY_FIXED, POLICY_RANDOM, POLICY_BBA, POLICY_RATE, POLICY_BOLA = 0, 1, 2, 3, 4
MPC_REF, MPC_ROBUST = 0, 1
MPC_TRUNCATE, MPC_EMPTY_DEFAULT, MPC_PRED_SES, MPC_EXHAUSTIVE = 1, 2, 4, 8
MPC_MODE_EXHAUSTIVE = 0x100
ACC_NAMES = ("reward", "rebuffer", "utility", "smooth", "sleep", "delay", "steps", "episodes", "startup", "latency",
             "played")
FIELDS = dict(seg=(0, "int32"), chunk=(1, "int32"), last_q=(2, "int32"), trace_id=(3, "int32"),
              hist_len=(4, "int32"), done=(5, "uint8"), err_len=(6, "int32"), phase=(10, "float64"), pos=(18, "float64"),
              buffer=(11, "float64"), bw_hist=(12, "float64"), last_pred=(13, "float64"),
              err_ring=(14, "float64"), acc=(15, "float64"), t_now=(16, "float64"), play_time=(17, "float64"),
              started=(7, "uint8"), play_id=(8, "int32"), play_len=(19, "float64"), sizes=(20, "float64"), utility=(21, "float64"),
              trace_bw=(22, "float64"), order=(23, "int32"))


class AbrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libabr_b200 error {code}: {msg}")
        self.code = code


class AbrParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "chunk_length", "max_buffer", "rtt", "payload", "sleep_quantum", "rebuf_penalty",
        "smooth_penalty", "utility_scale", "bba_reservoir", "bba_cushion", "start_up_length",
        "startup_penalty", "latency_penalty", "latency_tick")] + [
        (n, C.c_int32) for n in ("utility_mode", "default_quality", "auto_reset", "hist_k",
                                 "track_history", "track_acc", "live", "smooth_prev_ladder")]


class AbrPolicyParams(C.Structure):
    """Parameters of the RATE and BOLA policies (SPEC §4.2, §4.3)."""
    _fields_ = [(n, C.c_double) for n in ("rb_safety", "bola_min_buffer", "bola_target_buffer")]


class AbrObsSpec(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("buffer_scale", "throughput_scale", "delay_scale", "size_scale")]


# every symbol include/abr_b200.h declares (tests check that the .so exports all of them)
SYMBOLS = ("abr_version", "abr_last_error", "abr_launch_count", "abr_device_info", "abr_params_default",
           "abr_env_create", "abr_env_destroy", "abr_env_num_sessions", "abr_sort_by_trace", "abr_env_set_order", "abr_env_reset", "abr_env_reset_sorted", "abr_env_get_order", "abr_env_reset_host",
           "abr_env_step", "abr_env_step_live", "abr_env_step_f32", "abr_env_step_policy", "abr_env_qoe_cost", "abr_env_rollout_fused",
           "abr_env_rollout_fused_live", "abr_env_rollout_fused_f32", "abr_env_run", "abr_env_mpc_decide", "abr_stats_partial",
           "abr_env_state_ptr", "abr_policy_params_default", "abr_env_set_policy_params", "abr_env_policy_decide",
           "abr_env_error_count", "abr_env_run_host", "abr_mpc_decide", "abr_mpc_decide_host", "abr_mpc_decide_startup",
           "abr_mpc_decide_startup_host", "abr_mpc_score_host",
           "abr_fp64_probe")

_lib = None


def library_path() -> str:
    return _build.LIB


def load():
    """Load the in-tree library (building it first if it is missing and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if _build.is_stale():
        # missing or built from other sources: rebuild (raises if there is no nvcc — loud failure, no fallback)
        # under a file lock: concurrent ranks build once, the rest wait and load the finished file
        _build.build_library()
    lib = C.CDLL(path)
    lib.abr_last_error.restype = C.c_char_p
    lib.abr_launch_count.restype = C.c_longlong
    lib.abr_version.restype = C.c_int
    # argtypes for the host-buffer entry point: plain Python ints / None convert without per-call ctypes objects
    vp = C.c_void_p
    lib.abr_env_run_host.argtypes = [vp, C.c_int, C.c_uint64, C.c_int, vp, vp, C.c_int, C.c_longlong, vp, vp, vp, vp, vp, vp]
    lib.abr_env_run_host.restype = C.c_int
    lib.abr_env_step_policy.argtypes = [vp, vp, C.c_int, C.c_uint64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.abr_env_step_policy.restype = C.c_int
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise AbrError(rc, load().abr_last_error().decode("utf-8", "replace"))


def default_params(**kw) -> AbrParams:
    p = AbrParams()
    load().abr_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise TypeError(f"unknown ABR parameter {k!r}")
        setattr(p, k, v)
    return p


def launch_count() -> int:
    return int(load().abr_launch_count())
