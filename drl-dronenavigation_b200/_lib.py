"""ctypes binding of ``libdronenav.so`` (include/dronenav.h).

There is no CPU or PyTorch fallback: if the library is missing or cannot be loaded
the import of this module's :func:`lib` raises, and every product path that touches
the environment fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libdronenav.so")

DN_ABI_VERSION = 4

# enums of include/dronenav.h
DN_ACT_THRUST, DN_ACT_RPM, DN_ACT_ONE_D_RPM, DN_ACT_PID, DN_ACT_VEL, DN_ACT_ONE_D_PID = 0, 1, 2, 3, 4, 5
DN_MODEL_CF2X, DN_MODEL_CF2P, DN_MODEL_RACE = 0, 1, 2
DN_PHYS_DYN, DN_PHYS_DRAG, DN_PHYS_GROUND_EFFECT, DN_PHYS_GROUND_CONTACT = 0, 1, 2, 4
DN_REWARD_DEFAULT, DN_REWARD_DUMMY, DN_REWARD_THRUSTENV, DN_REWARD_HER = 0, 1, 2, 3
DN_REWARD_REACHING, DN_REWARD_PROGRESS, DN_REWARD_HOVER, DN_REWARD_FLYTHRUGATE = 4, 5, 6, 7
DN_REWARD_BOOTSTRAPPED, DN_REWARD_CHAMP = 8, 9
DN_SPAWN_FIXED, DN_SPAWN_LINE, DN_SPAWN_MIDPOINT = 0, 1, 2
DN_DONE_TERMINATED, DN_DONE_TRUNCATED = 1, 2


class dn_config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("num_envs", C.c_int32),
        ("env_id_offset", C.c_int64), ("seed", C.c_uint64),
        ("pyb_freq", C.c_int32), ("ctrl_freq", C.c_int32),
        ("act_type", C.c_int32), ("normalize_actions", C.c_int32),
        ("physics", C.c_int32), ("reward_id", C.c_int32),
        ("include_distance", C.c_int32), ("cylinder", C.c_int32),
        ("circle", C.c_int32), ("max_steps", C.c_int32),
        ("spawn_mode", C.c_int32), ("normalize_obs", C.c_int32),
        ("threshold", C.c_double), ("discount", C.c_double),
        ("aviary_dim", C.c_double * 6), ("init_xyz", C.c_double * 3), ("init_rpy", C.c_double * 3),
        ("num_targets", C.c_int32), ("normalize_reward", C.c_int32),
        ("clip_reward", C.c_double), ("reward_gamma", C.c_double),
        ("targets", C.POINTER(C.c_double)),
        ("drone_model", C.c_int32), ("reserved0", C.c_int32),
    ]


class dn_step_io(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p), ("obs", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
        ("terminal_obs", C.c_void_p), ("found_targets", C.c_void_p),
        ("episode_return", C.c_void_p), ("episode_length", C.c_void_p),
    ]


STATE_FIELDS = ("pos", "quat", "vel", "rpy_rates", "ang_v", "prev_vel", "prev_ang_v", "dist", "prev_dist",
                "target_idx", "steps", "just_found", "ep_return", "ep_length", "episode_count",
                "last_rpm_sum", "obs_rms", "aux", "rew_rms", "spawn", "pid")


class dn_state_view(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in STATE_FIELDS]


class dn_stats(C.Structure):
    _fields_ = [
        ("return_sum", C.c_double), ("length_sum", C.c_uint64), ("episodes", C.c_uint64),
        ("successes", C.c_uint64), ("found_targets", C.c_uint64), ("crashes", C.c_uint64),
        ("truncations", C.c_uint64),
    ]


# ---- include/dnppo.h ------------------------------------------------------------------------------------------
DN_MLP_BF16X3, DN_MLP_BF16 = 0, 1
DN_PPO_MAX_LAYERS = 4


class dn_ppo_config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("max_rows", C.c_int32),
        ("n_pi", C.c_int32), ("n_vf", C.c_int32),
        ("pi_hidden", C.c_int32 * DN_PPO_MAX_LAYERS), ("vf_hidden", C.c_int32 * DN_PPO_MAX_LAYERS),
        ("precision", C.c_int32), ("normalize_advantage", C.c_int32), ("world_size", C.c_int32), ("reserved0", C.c_int32),
        ("clip_range", C.c_float), ("clip_range_vf", C.c_float), ("ent_coef", C.c_float), ("vf_coef", C.c_float),
        ("max_grad_norm", C.c_float), ("target_kl", C.c_float),
        ("learning_rate", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
        ("pi_w_off", C.c_int64 * (DN_PPO_MAX_LAYERS + 1)), ("pi_b_off", C.c_int64 * (DN_PPO_MAX_LAYERS + 1)),
        ("vf_w_off", C.c_int64 * (DN_PPO_MAX_LAYERS + 1)), ("vf_b_off", C.c_int64 * (DN_PPO_MAX_LAYERS + 1)),
        ("log_std_off", C.c_int64), ("n_params", C.c_int64),
    ]


class dn_ppo_rollout(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("actions", C.c_void_p), ("old_log_prob", C.c_void_p), ("old_values", C.c_void_p),
                ("advantages", C.c_void_p), ("returns", C.c_void_p)]


class dn_ppo_stats(C.Structure):
    _fields_ = [("policy_gradient_loss", C.c_double), ("value_loss", C.c_double), ("approx_kl", C.c_double),
                ("clip_fraction", C.c_double), ("minibatches", C.c_int32), ("optimizer_steps", C.c_int32),
                ("early_stop", C.c_int32), ("last_approx_kl", C.c_float), ("last_grad_norm", C.c_float)]


class dn_ppo_sample(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("row_id_offset", C.c_int64), ("counter", C.c_void_p), ("deterministic", C.c_int32),
                ("low", C.c_float), ("high", C.c_float)]


DN_PPO_ACT_TAG = 0x50504F41     # second Philox counter word of dn_ppo_act's draws

# ---- include/dnsac.h ------------------------------------------------------------------------------------------
DN_SAC_MAX_LAYERS = 4
DN_SAC_SAMPLE, DN_SAC_DETERMINISTIC, DN_SAC_UNIFORM = 0, 1, 2
DN_SAC_ACT_TAG = 0x53414341     # "SACA": second Philox counter word of dn_sac_act's draws


class dn_sac_actor_config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("max_rows", C.c_int32),
        ("n_hidden", C.c_int32), ("hidden", C.c_int32 * DN_SAC_MAX_LAYERS), ("precision", C.c_int32),
        ("w_off", C.c_int64 * DN_SAC_MAX_LAYERS), ("b_off", C.c_int64 * DN_SAC_MAX_LAYERS),
        ("mu_w_off", C.c_int64), ("mu_b_off", C.c_int64), ("log_std_w_off", C.c_int64), ("log_std_b_off", C.c_int64),
        ("n_params", C.c_int64),
    ]


class dn_sac_sample(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("row_id_offset", C.c_int64), ("counter", C.c_void_p), ("mode", C.c_int32),
                ("reserved0", C.c_int32)]


# every symbol include/dronenav.h and include/dnppo.h declare: name -> (restype, argtypes)
SYMBOLS = {
    "dn_abi_version": (C.c_int, []),
    "dn_last_error": (C.c_char_p, []),
    "dn_create": (C.c_int, [C.POINTER(dn_config), C.c_int, C.POINTER(C.c_void_p)]),
    "dn_destroy": (C.c_int, [C.c_void_p]),
    "dn_num_envs": (C.c_int, [C.c_void_p]),
    "dn_obs_dim": (C.c_int, [C.c_void_p]),
    "dn_launch_count": (C.c_int64, [C.c_void_p]),
    "dn_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dn_step": (C.c_int, [C.c_void_p, C.POINTER(dn_step_io), C.c_void_p]),
    "dn_step_many": (C.c_int, [C.c_void_p, C.POINTER(dn_step_io), C.c_int, C.c_int, C.c_void_p]),
    "dn_step_host": (C.c_int, [C.c_void_p, C.POINTER(dn_step_io)]),
    "dn_host_buffers": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(dn_step_io)]),
    "dn_step_host_async": (C.c_int, [C.c_void_p, C.POINTER(dn_step_io)]),
    "dn_step_host_wait": (C.c_int, [C.c_void_p]),
    "dn_host_server": (C.c_int, [C.c_void_p, C.c_int]),
    "dn_host_server_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dn_action_to_rpm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "dn_gae": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p,
                         C.c_int32, C.c_int32, C.c_void_p]),
    "dn_get_state": (C.c_int, [C.c_void_p, C.POINTER(dn_state_view), C.c_void_p]),
    "dn_set_state": (C.c_int, [C.c_void_p, C.POINTER(dn_state_view), C.c_void_p]),
    "dn_episode_stats": (C.c_int, [C.c_void_p, C.POINTER(dn_stats), C.c_int, C.c_void_p]),
    # include/dnppo.h
    "dn_mlp_gemm": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dn_ppo_create": (C.c_int, [C.POINTER(dn_ppo_config), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.POINTER(C.c_void_p)]),
    "dn_ppo_destroy": (C.c_int, [C.c_void_p]),
    "dn_ppo_sync_weights": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dn_ppo_begin_update": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dn_ppo_minibatch_grad": (C.c_int, [C.c_void_p, C.POINTER(dn_ppo_rollout), C.c_void_p, C.c_int32, C.c_void_p]),
    "dn_ppo_minibatch_apply": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dn_ppo_get_stats": (C.c_int, [C.c_void_p, C.POINTER(dn_ppo_stats), C.c_void_p]),
    "dn_ppo_comm_create": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "dn_ppo_comm_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dn_ppo_allreduce": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dn_ppo_poll": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dn_ppo_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dn_ppo_act": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(dn_ppo_sample), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_void_p]),
    "dn_ppo_buffer": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
}

# every symbol include/dnsac.h declares
SAC_SYMBOLS = {
    "dn_sac_actor_create": (C.c_int, [C.POINTER(dn_sac_actor_config), C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "dn_sac_actor_destroy": (C.c_int, [C.c_void_p]),
    "dn_sac_actor_sync_weights": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dn_sac_act": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(dn_sac_sample), C.c_void_p, C.c_void_p, C.c_void_p]),
    "dn_sac_actor_buffer": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
}

_lib = None


class DroneNavError(RuntimeError):
    """A libdronenav call returned a negative code."""


def lib() -> C.CDLL:
    """The loaded C-ABI library.  Raises if it was not built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  drl_dronenavigation_b200 has no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (restype, argtypes) in (SYMBOLS | SAC_SYMBOLS).items():
            fn = getattr(handle, name)          # AttributeError if the symbol is not exported
            fn.restype = restype
            fn.argtypes = argtypes
        if handle.dn_abi_version() != DN_ABI_VERSION:
            raise ImportError("libdronenav.so ABI version mismatch; rebuild it")
        _lib = handle
    return _lib


def check(code: int, what: str = "libdronenav") -> None:
    if code < 0:
        msg = lib().dn_last_error()
        raise DroneNavError(f"{what} failed ({code}): {msg.decode() if msg else ''}")
