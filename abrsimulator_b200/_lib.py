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


class AbrObsWindowSpec(C.Structure):
    """The window length and the scales of the windowed observation (SPEC §4.5, include/abr_b200_obs.h)."""
    _fields_ = [("window", C.c_int32)] + [(n, C.c_double) for n in (
        "util_scale", "buffer_scale", "throughput_scale", "delay_scale", "size_scale")]


# The signature of every symbol include/abr_b200.h declares, in the header's order: (restype, argtypes).  Buffers,
# streams and the AbrEnv handle are c_void_p; tests check the table against the header and the .so's exports.
_P, _I, _LL, _U64, _D = C.c_void_p, C.c_int, C.c_longlong, C.c_uint64, C.c_double
_PARAMS, _POLICY_PARAMS, _OBS_SPEC = C.POINTER(AbrParams), C.POINTER(AbrPolicyParams), C.POINTER(AbrObsSpec)
_RUN = [_P, _I, _U64, _I, _P, _P, _I, _LL, _P]                   # env, policy, seed, steps, trace ids, offsets, N, base, actions
_MPC = [_P, _P, _I, _I, _PARAMS, _I] + [_P] * 5 + [_I] + [_P] * 3 + [_I] * 3   # tables .. robust state, horizon, mode, flags
_STARTUP = [_P, _I, _D]                                            # startup, n_ts, ts_step
SIGNATURES = {
    "abr_version": (_I, []),
    "abr_last_error": (C.c_char_p, []),
    "abr_launch_count": (_LL, []),
    "abr_device_info": (_I, [_P] * 4),
    "abr_params_default": (None, [_PARAMS]),
    "abr_env_create": (_I, [_P, _P, _P, _I, _I, _P, _P, _I, _I, _PARAMS, _I, _P]),
    "abr_env_destroy": (None, [_P]),
    "abr_env_num_sessions": (_I, [_P]),
    "abr_sort_by_trace": (_I, [_P, _I, _I, _P, _P]),
    "abr_env_set_order": (_I, [_P, _P, _I, _P]),
    "abr_env_reset": (_I, [_P, _P, _P, _I, _LL, _P]),
    "abr_env_reset_sorted": (_I, [_P, _P, _P, _I, _LL, _P]),
    "abr_env_get_order": (_I, [_P, _P, _I, _P]),
    "abr_env_reset_host": (_I, [_P, _P, _P, _I, _LL, _P]),
    "abr_env_step": (_I, [_P] * 11),
    "abr_env_step_policy": (_I, [_P, _P, _I, _U64, _OBS_SPEC] + [_P] * 10),
    "abr_env_step_live": (_I, [_P] * 13),
    "abr_env_rollout_fused": (_I, [_P, _I, _U64, _I] + [_P] * 9),
    "abr_env_rollout_fused_live": (_I, [_P, _I, _U64, _I] + [_P] * 11),
    "abr_env_run": (_I, _RUN + [_P] * 10),
    "abr_env_step_f32": (_I, [_P] * 13),
    "abr_env_rollout_fused_f32": (_I, [_P, _I, _U64, _I] + [_P] * 11),
    "abr_policy_params_default": (None, [_POLICY_PARAMS]),
    "abr_env_set_policy_params": (_I, [_P, _POLICY_PARAMS]),
    "abr_env_policy_decide": (_I, [_P, _I, _P, _P]),
    "abr_env_mpc_decide": (_I, [_P, _I, _I, _P, _P, _P]),
    "abr_env_qoe_cost": (_I, [_P, _P, _P]),
    "abr_stats_partial": (_I, [_P, _P, _P]),
    "abr_env_state_ptr": (_I, [_P, _I, _P]),
    "abr_env_error_count": (_I, [_P, _P, _P]),
    "abr_env_run_host": (_I, _RUN + [_P] * 5),
    "abr_mpc_decide": (_I, _MPC + [_P] * 6),
    "abr_mpc_decide_startup": (_I, _MPC + _STARTUP + [_P] * 7),
    "abr_mpc_decide_startup_host": (_I, _MPC + _STARTUP + [_P] * 6),
    "abr_mpc_decide_host": (_I, _MPC + [_P] * 5),
    "abr_mpc_score_host": (_I, [_P, _P, _I, _I, _PARAMS, _I, _I, _D, _P, _I, _I, _I, _D, _P, _I, _P]),
    "abr_fp64_probe": (_I, [_I, _I, _P, _P, _P]),
}
SYMBOLS = tuple(SIGNATURES)
# Entry points declared in the companion headers of abr_b200.h (include/abr_b200_lookahead.h), bound the same way.
EXTRA_SIGNATURES = {
    "abr_env_lookahead_decide": (_I, [_P, _I, _P, _P, _P, _P]),
}
# include/abr_b200_mpc_pred.h: MPC over caller-supplied throughput predictions (SPEC §5.6).
MPC_PRED_SIGNATURES = {
    "abr_env_mpc_decide_pred": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
}
# include/abr_b200_obs.h: the windowed observation of the policy-in-the-loop step (SPEC §4.5).
_OBS_WINDOW_SPEC = C.POINTER(AbrObsWindowSpec)
OBS_SIGNATURES = {
    "abr_env_step_policy_window": (_I, [_P, _P, _I, _U64, _OBS_WINDOW_SPEC] + [_P] * 10),
    "abr_env_observe_window": (_I, [_P, _OBS_WINDOW_SPEC, _P, _P]),
}
# include/abr_b200_mpc_scen.h: MPC over caller-supplied throughput scenarios (SPEC §5.7).
MPC_SCEN_MEAN, MPC_SCEN_WORST, MPC_SCEN_MAX = 0, 1, 16
MPC_SCEN_SIGNATURES = {
    "abr_env_mpc_decide_scen": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P]),
}

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
    for name, (restype, argtypes) in {**SIGNATURES, **EXTRA_SIGNATURES, **MPC_PRED_SIGNATURES, **OBS_SIGNATURES,
                                   **MPC_SCEN_SIGNATURES}.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = lib
    return lib


def _addr(x):
    """The address of a buffer for a c_void_p argument: None, a torch tensor or a numpy array."""
    if x is None:
        return None
    return x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data


def check(rc: int):
    if rc != 0:
        raise AbrError(rc, load().abr_last_error().decode("utf-8", "replace"))


def default_params(**kw) -> AbrParams:
    p = AbrParams()
    load().abr_params_default(p)
    for k, v in kw.items():
        if not hasattr(p, k):
            raise TypeError(f"unknown ABR parameter {k!r}")
        setattr(p, k, v)
    return p


def launch_count() -> int:
    return int(load().abr_launch_count())
