"""ctypes binding of libflexgpu.so (the C ABI declared in include/flexgpu.h).

There is deliberately no fallback: if the shared library has not been built
(`python __graft_entry__.py build` or `safe-marl_b200/csrc/build.sh`) importing this
module raises, and if no CUDA device is present `fp_create` fails.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# FLEXGPU_LIB: tuning builds of the same library (tools/); the product path is the in-tree default
LIB_PATH = os.environ.get("FLEXGPU_LIB") or os.path.join(_HERE, "libflexgpu.so")

FP_MAX_BUS = 33
FP_MAX_AGENTS = 5
FP_INFO_STRIDE = 8
FP_NSTATS = 16
FP_REC_STRIDE = 16
FP_F32, FP_F64, FP_F32_POLICY = 0, 1, 2
VARIANT_THREAD, VARIANT_WARP = 0, 1
VARIANTS = {"thread": VARIANT_THREAD, "warp": VARIANT_WARP}
# MLP activations (include/flexgpu.h FP_ACT_*), by scikit-learn's names
ACTIVATIONS = {"identity": 0, "relu": 1, "tanh": 2, "logistic": 3}

# record slots (include/flexgpu.h FP_REC_*)
REC_E_INIT, REC_E_CUR, REC_CUM, REC_TIME, REC_HIST, REC_VMASK, REC_COUNTS, REC_LINES = 0, 5, 10, 11, 12, 13, 14, 15
FLAG_DONE, FLAG_FAILED, FLAG_RESET_FAILED = 1, 2, 4

INFO_KEYS = ("reward", "revenue", "der_cost", "ess_cost", "discomfort_penalty", "voltage_penalty",
             "cumulative_reward", "solver_failed")
STAT_KEYS = ("reward", "revenue", "der_cost", "ess_cost", "discomfort_penalty", "voltage_penalty",
             "cumulative_reward", "solver_failed", "violation_count", "env_steps", "episodes",
             "line_violation_count")


class FpConfig(C.Structure):
    _fields_ = [
        ("n_bus", C.c_int32), ("n_agents", C.c_int32), ("history", C.c_int32),
        ("episode_limit", C.c_int32), ("raw_actions", C.c_int32), ("pf_max_iter", C.c_int32),
        ("variant", C.c_int32), ("pf_f32_passes", C.c_int32),
        ("pf_tol", C.c_double), ("v_min", C.c_double), ("v_max", C.c_double),
        ("e_min", C.c_double), ("e_max", C.c_double), ("p_ch_max", C.c_double),
        ("p_dis_max", C.c_double), ("eta_ch", C.c_double), ("eta_dis", C.c_double),
        ("max_power_reduction", C.c_double), ("kappa", C.c_double), ("pv_cost", C.c_double),
        ("ess_cost", C.c_double), ("discomfort_coeff", C.c_double), ("voltage_coeff", C.c_double),
        ("delta_t", C.c_double), ("fail_penalty", C.c_double), ("e_next_lb", C.c_double),
        ("parent", C.c_int32 * FP_MAX_BUS), ("r", C.c_double * FP_MAX_BUS),
        ("x", C.c_double * FP_MAX_BUS), ("imax", C.c_double * FP_MAX_BUS),
        ("agent_bus", C.c_int32 * FP_MAX_AGENTS), ("reserved2_", C.c_int32 * 3),
        ("action_low", C.c_double), ("action_high", C.c_double),
    ]


class FlexGpuError(RuntimeError):
    pass


_P = C.c_void_p
_PROTOS = {
    "fp_create": (C.c_int, [C.POINTER(FpConfig), C.c_int64, C.c_int, C.POINTER(_P)]),
    "fp_destroy": (C.c_int, [_P]),
    "fp_last_error": (C.c_char_p, [_P]),
    "fp_n_envs": (C.c_int64, [_P]),
    "fp_load_profiles": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64]),
    "fp_reset": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "fp_reset_random": (C.c_int, [_P, C.c_uint64, C.c_int64, _P, _P]),
    "fp_reset_random_retry": (C.c_int, [_P, C.c_uint64, C.c_int64, _P, C.c_int32, _P, _P]),
    "fp_step": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, _P]),
    "fp_step_preview": (C.c_int, [_P, C.c_int32, _P, C.c_int, _P, _P, _P, _P, _P, _P]),
    "fp_step_host": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P]),
    "fp_get_obs": (C.c_int, [_P, _P, C.c_int, C.c_int, _P]),
    "fp_get_obs_view": (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(C.c_int64), C.POINTER(C.c_int64), _P]),
    "fp_step_obs": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, C.POINTER(_P), C.POINTER(C.c_int64), C.POINTER(C.c_int64), _P]),
    "fp_step_ring": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, C.POINTER(_P), C.POINTER(C.c_int32), C.POINTER(C.c_int64), _P]),
    "fp_obs_ring": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int32), C.POINTER(C.c_int64), _P]),
    "fp_obs_ring_reset_push": (C.c_int, [_P, _P, _P]),
    "fp_obs_ring_gather": (C.c_int, [_P, _P, _P]),
    "fp_set_obs_history": (C.c_int, [_P, C.c_int]),
    "fp_get_state": (C.c_int, [_P, _P, C.c_int, _P]),
    "fp_state_ptrs": (C.c_int, [_P] + [C.POINTER(_P)] * 6),
    "fp_set_keep_flows": (C.c_int, [_P, C.c_int]),
    "fp_history_ptr": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int64), C.c_int32]),
    "fp_power_flow": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "fp_stats_read": (C.c_int, [_P, _P, _P]),
    "fp_stats_reset": (C.c_int, [_P, _P]),
    "fp_inject_failure": (C.c_int, [_P, _P]),
    "fp_launch_count": (C.c_int64, [_P]),
    "fp_sizeof_config": (C.c_int32, []),
    "fp_replay_create": (C.c_int, [C.c_int64, C.c_int32, C.POINTER(C.c_int32), C.c_int, C.POINTER(_P)]),
    "fp_replay_destroy": (C.c_int, [_P]),
    "fp_replay_last_error": (C.c_char_p, [_P]),
    "fp_replay_len": (C.c_int64, [_P]),
    "fp_replay_capacity": (C.c_int64, [_P]),
    "fp_replay_clear": (C.c_int, [_P]),
    "fp_replay_reserve": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_int64)]),
    "fp_replay_write": (C.c_int, [_P, C.c_int32, C.c_int64, C.c_int64, _P, _P]),
    "fp_replay_sample": (C.c_int, [_P, C.c_int64, C.c_int64, C.POINTER(_P), _P]),
    "fp_replay_field_ptr": (C.c_int, [_P, C.c_int32, C.POINTER(_P)]),
    "fp_predictor_load": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, C.c_double, C.c_double, C.c_double]),
    "fp_predict": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, _P]),
    "fp_predictor_load_mlp": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_int32, C.c_double, C.c_double, C.c_double]),
    "fp_predict_mlp": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, _P]),
    "fp_safety_load": (C.c_int, [_P, _P, _P, C.c_double, C.c_double, C.c_double]),
    "fp_safety_project": (C.c_int, [_P, _P, C.c_int, _P, C.c_int32, _P, _P, _P]),
    "fp_safety_load_affine": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, C.c_double, C.c_double, C.c_double]),
    "fp_safety_project_affine": (C.c_int, [_P, _P, C.c_int, _P, C.c_int32, _P, _P, _P, _P]),
    "fp_policy_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "fp_policy_create_agents": (C.c_int, [C.c_int, C.c_int32, C.POINTER(_P)]),
    "fp_policy_destroy": (C.c_int, [_P]),
    "fp_policy_last_error": (C.c_char_p, [_P]),
    "fp_policy_launch_count": (C.c_int64, [_P]),
    "fp_policy_load": (C.c_int, [_P] * 11),
    "fp_policy_act": (C.c_int, [_P, _P, C.c_int32, C.c_int64, C.c_int64, _P, _P, _P, C.c_int32, _P, _P, _P, _P, C.c_uint64, C.c_uint64,
                                C.c_float, C.c_int32, _P]),
    "fp_policy_hidden_to_ring": (C.c_int, [_P, _P, C.c_int64, C.c_int64, _P, C.c_int64, C.c_int64, _P, _P]),
    "fp_policy_gather_windows": (C.c_int, [_P, _P, C.c_int32, C.c_int64, C.c_int64, _P, C.c_int64, C.c_int64, C.c_int64, _P]),
    "fp_policy_rows_to_ring": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, C.c_int64, C.c_int64, _P]),
    "fp_policy_scalars_to_ring": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, _P, _P, _P, _P, C.c_int64, C.c_int64, _P]),
    "fp_policy_state_sink": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int64]),
    "fp_policy_sample": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P, C.c_uint64, C.c_uint64, C.c_float, C.c_int32, _P]),
    "fp_critic_load": (C.c_int, [_P] * 9),
    "fp_critic_value": (C.c_int, [_P, _P, C.c_int32, C.c_int64, C.c_int64, _P, _P, _P]),
    "fp_policy_transition_tail": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P,
                                            C.c_int64, C.c_int64, _P]),
    "fp_learner_feed": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P]),
}

EXPORTED_SYMBOLS = tuple(_PROTOS.keys())

_lib = None


def lib():
    """Load (once) and return the shared library; raise FlexGpuError if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FlexGpuError(
                f"{LIB_PATH} not found: build the CUDA extension first "
                "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        if l.fp_sizeof_config() != C.sizeof(FpConfig):
            raise FlexGpuError("FpConfig layout mismatch between flexgpu/_lib.py and libflexgpu.so")
        _lib = l
    return _lib


def check(rc, handle=None, what="", last_error=None):
    """Raise FlexGpuError for a failed entry point.  last_error: the *_last_error function of the handle's kind
    (default fp_last_error, the env handle's); a NULL handle reads the last failed create of that kind."""
    if rc != 0:
        msg = (last_error or lib().fp_last_error)(handle)
        raise FlexGpuError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def stream(device):
    """torch's current stream on `device` (the handle's device, whatever torch's current device is) as a cudaStream_t."""
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
