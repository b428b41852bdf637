"""ctypes binding of ``libdronecu.so`` (the C ABI declared in include/dronecu.h).

There is no Python or CPU fallback: if the shared library has not been built, or no CUDA
device is present when an env is created, this raises.  ``python -m drone_rl_b200.build``
(or ``__graft_entry__.build()``) compiles the library in-tree for sm_100a.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DRONECU_LIB", os.path.join(_HERE, "libdronecu.so"))   # DRONECU_LIB: A/B builds for profiling


class DronecuError(RuntimeError):
    pass


class Config(C.Structure):
    """Mirror of ``dronecu_config`` (include/dronecu.h)."""
    _fields_ = [
        ("dt", C.c_double), ("mass", C.c_double), ("gravity", C.c_double),
        ("inertia", C.c_double * 3), ("arm_length", C.c_double), ("k_yaw", C.c_double),
        ("reward_scale", C.c_double), ("bonus_radius", C.c_double), ("bonus", C.c_double),
        ("z_floor", C.c_double), ("r_max", C.c_double),
        ("fixed_target", C.c_double * 3), ("fixed_start", C.c_double * 3),
        ("start_z", C.c_double), ("target_z", C.c_double), ("curriculum_step", C.c_double),
        ("curriculum_period", C.c_int32), ("max_steps", C.c_int32), ("obs_dim", C.c_int32),
        ("flags", C.c_uint32),
    ]


FLAG_RANDOMIZED = 1
FLAG_AUTORESET = 2
ACTIONS_STREAMED = 0
ACTIONS_UNIFORM = 1


class RolloutOut(C.Structure):
    _fields_ = [("d_obs0", C.c_void_p), ("d_next_obs", C.c_void_p), ("d_actions", C.c_void_p),
                ("d_reward", C.c_void_p), ("d_done", C.c_void_p), ("d_truncated", C.c_void_p)]


class StepOut(C.Structure):
    _fields_ = [("d_obs", C.c_void_p), ("d_reward", C.c_void_p), ("d_done", C.c_void_p),
                ("d_truncated", C.c_void_p), ("d_terminal_obs", C.c_void_p),
                ("d_episode_r", C.c_void_p), ("d_episode_l", C.c_void_p)]


class StateView(C.Structure):
    _fields_ = [("d_pos", C.c_void_p), ("d_vel", C.c_void_p), ("d_euler", C.c_void_p),
                ("d_omega", C.c_void_p), ("d_target", C.c_void_p), ("d_step", C.c_void_p),
                ("d_ep_num", C.c_void_p), ("d_ep_len", C.c_void_p), ("d_ep_ret", C.c_void_p)]


class PolicyOut(C.Structure):
    _fields_ = [("d_obs", C.c_void_p), ("d_actions", C.c_void_p), ("d_logp", C.c_void_p), ("d_value", C.c_void_p),
                ("d_reward", C.c_void_p), ("d_done", C.c_void_p), ("d_last_value", C.c_void_p),
                ("d_last_obs", C.c_void_p), ("obs_padded", C.c_int32), ("reserved", C.c_int32)]


class PPOConfig(C.Structure):
    _fields_ = [("learning_rate", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
                ("clip_range", C.c_float), ("vf_coef", C.c_float), ("ent_coef", C.c_float),
                ("max_grad_norm", C.c_float)]


class NormPassArgs(C.Structure):
    """Mirror of ``dronecu_norm_pass_args`` (include/dronecu.h)."""
    _fields_ = [("d_obs", C.c_void_p), ("obs_stride", C.c_int32), ("K", C.c_int32), ("n", C.c_int64),
                ("d_affine", C.c_void_p), ("d_reward", C.c_void_p), ("d_done", C.c_void_p), ("d_returns", C.c_void_p),
                ("d_stats", C.c_void_p), ("gamma", C.c_double), ("epsilon", C.c_double), ("clip_reward", C.c_double),
                ("update", C.c_int32), ("side_env", C.c_int32), ("d_side_obs", C.c_void_p), ("d_partials", C.c_void_p)]


class EvalArgs(C.Structure):
    """Mirror of ``dronecu_eval_args`` (include/dronecu.h)."""
    _fields_ = [("t0", C.c_int64), ("limit", C.c_int32), ("catch_up", C.c_int32), ("deterministic", C.c_int32),
                ("max_eps", C.c_int32), ("env_index0", C.c_int64), ("n_global", C.c_int64), ("n_eval_episodes", C.c_int64),
                ("d_steps", C.c_void_p), ("d_count", C.c_void_p), ("d_ep_return", C.c_void_p), ("d_ep_length", C.c_void_p),
                ("d_pending", C.c_void_p)]


class TimeoutBuf(C.Structure):
    """Mirror of ``dronecu_timeout_buf`` (include/dronecu.h)."""
    _fields_ = [("d_obs", C.c_void_p), ("d_row", C.c_void_p), ("slots_per_env", C.c_int32)]


NORM_AFFINE = 31
NORM_STATS = 34
NORM_MOMENTS = 34
NORM_BLOCK = 256
POLICY_PARAMS = 10697
GRAD_LEN = POLICY_PARAMS + 8
IPC_HANDLE_BYTES = 64
DP_MAX_WORLD = 16


class Stats(C.Structure):
    _fields_ = [("episodes", C.c_uint64), ("terminated", C.c_uint64), ("truncated", C.c_uint64),
                ("length_sum", C.c_uint64), ("return_sum", C.c_double), ("env_steps", C.c_uint64)]


_P = C.c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)
    "dronecu_version": (C.c_int, []),
    "dronecu_last_error": (C.c_char_p, []),
    "dronecu_config_single": (None, [C.POINTER(Config)]),
    "dronecu_config_vector": (None, [C.POINTER(Config)]),
    "dronecu_create": (C.c_int, [C.POINTER(Config), C.c_int, C.c_int64, C.c_int64, C.c_uint64, C.POINTER(_P)]),
    "dronecu_destroy": (C.c_int, [_P]),
    "dronecu_num_envs": (C.c_int64, [_P]),
    "dronecu_obs_dim": (C.c_int, [_P]),
    "dronecu_global_step": (C.c_int64, [_P]),
    "dronecu_set_global_step": (C.c_int, [_P, C.c_int64]),
    "dronecu_motor_max": (C.c_double, [_P]),
    "dronecu_launch_count": (C.c_uint64, [_P]),
    "dronecu_reset": (C.c_int, [_P, _P, _P, _P]),
    "dronecu_step": (C.c_int, [_P, _P, C.POINTER(StepOut), _P]),
    "dronecu_rollout": (C.c_int, [_P, C.c_int, C.c_int, _P, C.POINTER(RolloutOut), _P]),
    "dronecu_step_host": (C.c_int, [_P, _P, C.POINTER(StepOut)]),
    "dronecu_reset_host": (C.c_int, [_P, _P, _P]),
    "dronecu_get_state": (C.c_int, [_P, C.POINTER(StateView), _P]),
    "dronecu_set_state": (C.c_int, [_P, C.POINTER(StateView), _P]),
    "dronecu_get_state_host": (C.c_int, [_P, C.POINTER(StateView)]),
    "dronecu_set_state_host": (C.c_int, [_P, C.POINTER(StateView)]),
    "dronecu_episode_stats": (C.c_int, [_P, C.POINTER(Stats), C.c_int]),
    # PPO half
    "dronecu_rollout_policy": (C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(PolicyOut), _P]),
    "dronecu_policy_forward": (C.c_int, [C.c_int, C.c_int64, _P, _P, _P, _P, _P]),
    "dronecu_set_rollout_kernel": (C.c_int, [C.c_int]),
    "dronecu_rollout_policy_tc": (C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(PolicyOut), _P]),
    "dronecu_policy_forward_tc": (C.c_int, [C.c_int, C.c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "dronecu_rollout_policy_norm": (C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(PolicyOut), _P, C.c_int, _P]),
    "dronecu_rollout_policy_timeouts": (C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(PolicyOut), _P, C.c_int,
                                                  C.POINTER(TimeoutBuf), _P]),
    "dronecu_bootstrap_timeouts": (C.c_int, [C.c_int, _P, C.POINTER(TimeoutBuf), C.c_int64, _P, C.c_float, _P, _P]),
    "dronecu_evaluate_policy": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(EvalArgs), _P]),
    "dronecu_norm_pass": (C.c_int, [C.c_int, C.POINTER(NormPassArgs), _P]),
    "dronecu_norm_reduce": (C.c_int, [C.c_int, _P, C.c_int64, _P, _P]),
    "dronecu_norm_combine": (C.c_int, [C.c_int, _P, _P, C.c_double, C.c_float, _P, _P]),
    "dronecu_gae": (C.c_int, [C.c_int, C.c_int, C.c_int64, _P, _P, _P, _P, C.c_float, C.c_float, _P, _P, _P]),
    "dronecu_ppo_config_default": (None, [C.POINTER(PPOConfig)]),
    "dronecu_ppo_create": (C.c_int, [C.POINTER(PPOConfig), C.c_int, C.POINTER(_P)]),
    "dronecu_ppo_destroy": (C.c_int, [_P]),
    "dronecu_minibatch_permutation": (C.c_int, [C.c_int, C.c_int64, C.c_uint64, C.c_uint64, _P, _P]),
    "dronecu_minibatch_partition": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_uint64, C.c_uint64, _P, _P]),
    "dronecu_ppo_adv_stats_epoch": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    "dronecu_ppo_adv_stats": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    "dronecu_ppo_grad": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_float, C.c_float, _P, _P, _P]),
    "dronecu_ppo_grad_tc": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_float, C.c_float, _P, _P, _P]),
    "dronecu_ppo_grad_bf16": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_float, C.c_float, _P, _P, _P]),
    "dronecu_ppo_grad_strided": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_float, C.c_float, _P, _P, _P]),
    "dronecu_ppo_debug_buffer": (C.c_int, [_P, _P]),
    "dronecu_ppo_apply": (C.c_int, [_P, _P, _P, C.c_double, _P, _P]),
    "dronecu_ppo_num_updates": (C.c_int64, [_P]),
    "dronecu_ppo_get_state": (C.c_int, [_P, _P, C.POINTER(C.c_int64), _P]),
    "dronecu_ppo_set_state": (C.c_int, [_P, _P, C.c_int64, _P]),
    "dronecu_ppo_set_info_accumulator": (C.c_int, [_P, _P]),
    # data-parallel exchange over peer memory
    "dronecu_ppo_dp_alloc": (C.c_int, [_P, C.c_int, C.c_int, _P, C.POINTER(_P)]),
    "dronecu_ppo_dp_connect": (C.c_int, [_P, C.c_int, _P, C.POINTER(_P)]),
    "dronecu_ppo_dp_set_timeout": (C.c_int, [_P, C.c_double]),
    "dronecu_ppo_dp_status": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int64)]),
    "dronecu_ppo_dp_allreduce_f64": (C.c_int, [_P, _P, C.c_int, _P]),
    "dronecu_ppo_apply_dp": (C.c_int, [_P, _P, _P, _P, _P]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen libdronecu.so and type every exported entry point.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise DronecuError(
            f"{LIB_PATH} not found: build it with `python -m drone_rl_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    _register_optional(lib)
    _lib = lib
    return lib


# entry points added by later translation units (policy rollout, GAE, PPO update) register here
_OPTIONAL_SIGNATURES = {}


def _register_optional(lib):
    for name, (restype, argtypes) in _OPTIONAL_SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes


def declared_symbols():
    return list(_SIGNATURES) + list(_OPTIONAL_SIGNATURES)


def check(rc: int, what: str = "dronecu"):
    if rc != 0:
        msg = load().dronecu_last_error()
        raise DronecuError(f"{what} failed (status {rc}): {msg.decode() if msg else ''}")
