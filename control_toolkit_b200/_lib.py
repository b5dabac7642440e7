"""ctypes binding of libctk_b200.so (include/ctk_b200.h).

The reference itself calls C through ctypes (reference Controllers/controller_C.py:222-248); this is the same
mechanism.  There is NO CPU fallback: if the library is missing or no CUDA device is usable the import of an
optimizer works (so CPU-only tooling can inspect configs) but creating a backend raises ``BackendUnavailable``.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CTK_LIB") or os.path.join(HERE, "libctk_b200.so")  # CTK_LIB: diagnostics builds (tools/build_variants.sh)

CTK_ABI_VERSION = 1
CTK_OK, CTK_EINVAL, CTK_ECUDA, CTK_ESTATE = 0, -1, -2, -3
OPT_MPPI, OPT_CEM, OPT_RPGD = 0, 1, 2
PRED_ODE, PRED_MLP, PRED_GRU = 0, 1, 2
COST_DEFAULT, COST_QUADRATIC_BOUNDARY_GRAD = 0, 1
ENV_CARTPOLE, ENV_DUBINS_CAR = 0, 1
DIST_NORMAL, DIST_UNIFORM = 0, 1
ADAM_KERAS, ADAM_TORCH = 0, 1
MLP_SIMT, MLP_TCGEN05, MLP_TCGEN05_BF16, MLP_TCGEN05_FAST = 0, 1, 2, 3
STATE_U_NOM, STATE_CEM_MU, STATE_CEM_STD, STATE_RPGD_Q, STATE_RPGD_M, STATE_RPGD_V, STATE_RPGD_AGES, STATE_U_PREV, STATE_RNN_H = range(9)
COUNTER_COUNT, COUNTER_ADAM_STEP, COUNTER_TICK = range(3)
STREAM_MPPI, STREAM_CEM, STREAM_RPGD_INIT, STREAM_RPGD_RESAMPLE = range(4)
LOG_Q, LOG_J, LOG_ROLLOUTS, LOG_ELITE_IDX, LOG_U_NOM, LOG_AGES = range(6)


class BackendUnavailable(RuntimeError):
    """The CUDA extension cannot be used (not built, or no GPU).  Never silently replaced by a CPU path."""


class ctk_ode_params(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("u_max", "kp1_Mm", "m", "neg_M_fric", "neg_J_fric", "mg", "L", "kp1", "mL", "g",
                                         "kp1L", "h")] + [("intermediate_steps", C.c_int32)]


class ctk_cost_params(C.Structure):
    _fields_ = [("kind", C.c_int32)] + [(n, C.c_float) for n in (
        "dd_weight", "ep_weight", "ekp_weight", "cc_weight", "ccrc_weight", "R", "MAX_COST", "two_thl", "thl_095", "thl_005",
        "thl_09", "thl_01", "target_position", "target_equilibrium")]


class ctk_mlp_weights(C.Structure):
    _fields_ = [("hidden", C.c_int32)] + [(n, C.POINTER(C.c_float)) for n in ("W1", "b1", "W2", "b2", "W3", "b3")]


class ctk_gru_weights(C.Structure):
    _fields_ = [("hidden", C.c_int32)] + [(n, C.POINTER(C.c_float)) for n in ("Wi1", "Wh1", "bi1", "bh1", "Wi2", "Wh2", "bi2", "bh2", "W3", "b3")]


class ctk_config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("optimizer", C.c_int32), ("predictor", C.c_int32), ("device", C.c_int32),
        ("num_rollouts", C.c_int32), ("num_rollouts_global", C.c_int32), ("rollout_offset", C.c_int32),
        ("mpc_horizon", C.c_int32), ("num_states", C.c_int32), ("num_control_inputs", C.c_int32),
        ("action_low", C.c_float), ("action_high", C.c_float),
        ("seed", C.c_uint64),
        ("logging", C.c_int32), ("freeze_previous_input", C.c_int32), ("period_interpolation_inducing_points", C.c_int32),
        ("mppi_coef_du2", C.c_float), ("mppi_R", C.c_float), ("mppi_half_R", C.c_float), ("mppi_cc_weight", C.c_float),
        ("mppi_neg_inv_LBD", C.c_float), ("mppi_stdev", C.c_float),
        ("cem_outer_it", C.c_int32), ("cem_best_k", C.c_int32), ("cem_warmup", C.c_int32), ("cem_warmup_iterations", C.c_int32),
        ("cem_initial_action_stdev", C.c_float), ("cem_stdev_min", C.c_float),
        ("rpgd_outer_its", C.c_int32), ("rpgd_first_iter_count", C.c_int32), ("rpgd_resamp_per", C.c_int32),
        ("rpgd_shift_previous", C.c_int32), ("rpgd_keep_k", C.c_int32), ("rpgd_distribution", C.c_int32),
        ("rpgd_adam_form", C.c_int32),
        ("rpgd_sample_mean", C.c_float), ("rpgd_sample_stdev", C.c_float), ("rpgd_sample_min", C.c_float),
        ("rpgd_sample_max", C.c_float), ("rpgd_learning_rate", C.c_float), ("rpgd_gradmax_clip", C.c_float),
        ("rpgd_beta_1", C.c_double), ("rpgd_beta_2", C.c_double), ("rpgd_epsilon", C.c_double),
        ("mlp_engine", C.c_int32), ("cem_uniform_actions", C.c_int32), ("rpgd_gradient_mode", C.c_int32), ("num_clients", C.c_int32), ("environment", C.c_int32),
        ("rpgd_sample_whole_space", C.c_int32), ("reserved", C.c_int32 * 2),
    ]


# every symbol include/ctk_b200.h declares: name -> (restype, argtypes)
_H = C.c_void_p
_FP = C.POINTER(C.c_float)
SYMBOLS = {
    "ctk_create": (C.c_int, [C.POINTER(ctk_config), C.POINTER(ctk_ode_params), C.POINTER(ctk_cost_params), C.POINTER(_H)]),
    "ctk_destroy": (C.c_int, [_H]),
    "ctk_reset": (C.c_int, [_H]),
    "ctk_set_cost_params": (C.c_int, [_H, C.POINTER(ctk_cost_params)]),
    "ctk_set_ode_params": (C.c_int, [_H, C.POINTER(ctk_ode_params)]),
    "ctk_set_env_params": (C.c_int, [_H, _FP, C.c_int]),
    "ctk_set_control_limits": (C.c_int, [_H, _FP, _FP, C.c_int]),
    "ctk_set_mlp_weights": (C.c_int, [_H, C.POINTER(ctk_mlp_weights)]),
    "ctk_set_gru_weights": (C.c_int, [_H, C.POINTER(ctk_gru_weights)]),
    "ctk_set_stream": (C.c_int, [_H, C.c_void_p]),
    "ctk_push_injected_noise": (C.c_int, [_H, _FP, C.c_size_t]),
    "ctk_clear_injected_noise": (C.c_int, [_H]),
    "ctk_step": (C.c_int, [_H, _FP, _FP]),
    "ctk_step_state": (C.c_int, [_H, _FP, _FP, C.c_int, _FP, C.c_size_t]),
    "ctk_step_local": (C.c_int, [_H, C.c_void_p]),
    "ctk_partials": (C.c_int, [_H, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "ctk_step_finish": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_void_p]),
    "ctk_step_batch": (C.c_int, [_H, _FP, C.POINTER(C.c_int32), _FP]),
    "ctk_reset_client": (C.c_int, [_H, C.c_int]),
    "ctk_step_device": (C.c_int, [_H, C.c_void_p, C.c_void_p]),
    "ctk_step_device_n": (C.c_int, [_H, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int]),
    "ctk_exchange_barrier": (C.c_int, [_H]),
    "ctk_exchange_export": (C.c_int, [_H, C.c_void_p]),
    "ctk_exchange_connect": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p]),
    "ctk_exchange_mailbox": (C.c_int, [_H, C.POINTER(C.c_void_p)]),
    "ctk_exchange_connect_ptrs": (C.c_int, [_H, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int)]),
    "ctk_get_state": (C.c_int, [_H, C.c_int, _FP, C.c_size_t]),
    "ctk_set_state": (C.c_int, [_H, C.c_int, _FP, C.c_size_t]),
    "ctk_get_counter": (C.c_int, [_H, C.c_int, C.POINTER(C.c_int64)]),
    "ctk_set_counter": (C.c_int, [_H, C.c_int, C.c_int64]),
    "ctk_get_log": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_size_t]),
    "ctk_get_log_view": (C.c_int, [_H, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "ctk_get_log_top": (C.c_int, [_H, C.c_int, C.POINTER(C.c_int32), _FP, _FP, _FP]),
    "ctk_last_kernel": (C.c_char_p, [_H]),
    "ctk_get_launch_count": (C.c_int, [_H, C.POINTER(C.c_int64)]),
    "ctk_enable_kernel_timing": (C.c_int, [_H, C.c_int]),
    "ctk_get_kernel_timing": (C.c_int, [_H, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ctk_debug_trace": (C.c_int, [_H, C.c_int, C.POINTER(C.c_uint64), C.c_size_t, C.POINTER(C.c_int)]),
    "ctk_rollout_single": (C.c_int, [_H, _FP, _FP, _FP, _FP]),
    "ctk_last_error": (C.c_char_p, []),
    "ctk_abi_version": (C.c_int, []),
    "ctk_fp32_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "ctk_fp32_microbench": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "ctk_philox_fill": (C.c_int, [C.c_int, C.c_uint64, C.c_int, _FP, C.c_size_t]),
    "ctk_philox_export": (C.c_int, [_H, C.c_uint32, C.c_int64, C.c_int, C.c_int, C.c_size_t, C.c_size_t, _FP]),
    "ctk_topk": (C.c_int, [C.c_int, _FP, C.c_int, C.c_int, C.POINTER(C.c_int32)]),
}

_lib = None


def load():
    """Load libctk_b200.so (built by ``python -m control_toolkit_b200.build``).  Raises BackendUnavailable."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BackendUnavailable(f"{LIB_PATH} not found: run `python -m control_toolkit_b200.build` (needs nvcc). "
                                 "control_toolkit_b200 has no CPU fallback.")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # e.g. libcudart missing
        raise BackendUnavailable(f"cannot load {LIB_PATH}: {e}") from e
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype, fn.argtypes = res, args
    if lib.ctk_abi_version() != CTK_ABI_VERSION:
        raise BackendUnavailable(f"ABI mismatch: library {lib.ctk_abi_version()} vs binding {CTK_ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int) -> int:
    """Translate a status code into the reference's error conventions (ValueError for bad config, RuntimeError else)."""
    if rc >= 0:
        return rc
    msg = (load().ctk_last_error() or b"").decode()
    if rc == CTK_EINVAL:
        raise ValueError(msg)
    if rc == CTK_ECUDA and ("no CUDA-capable device" in msg or "driver" in msg.lower() and "insufficient" in msg.lower()):
        raise BackendUnavailable(msg)
    raise RuntimeError(msg)


def fptr(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_FP)
