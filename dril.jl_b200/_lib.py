"""ctypes binding of libdril_b200.so (include/dril_b200.h). There is no CPU fallback: a missing
library or a missing CUDA device raises."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdril_b200.so")

c_i32, c_i64, c_u64, c_f32, c_f64 = C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_double
P = C.c_void_p


class DrilError(RuntimeError):
    pass


class NormCfg(C.Structure):
    _fields_ = [("training", c_i32), ("norm_obs", c_i32), ("norm_reward", c_i32), ("clip_obs", c_f32),
                ("clip_reward", c_f32), ("gamma", c_f32), ("epsilon", c_f32)]


class AdrParam(C.Structure):
    _fields_ = [("index", c_i32), ("init_lo", c_f32), ("init_hi", c_f32), ("limit_lo", c_f32), ("limit_hi", c_f32),
                ("delta", c_f32)]


class PPOHyper(C.Structure):
    _fields_ = [("gamma", c_f32), ("gae_lambda", c_f32), ("clip_range", c_f32), ("clip_range_vf", c_f32),
                ("ent_coef", c_f32), ("vf_coef", c_f32), ("max_grad_norm", c_f32), ("target_kl", c_f32),
                ("normalize_advantage", c_i32), ("learning_rate", c_f32), ("adam_beta1", c_f32),
                ("adam_beta2", c_f32), ("adam_eps", c_f32)]


class IterStats(C.Structure):
    _fields_ = [("entropy_loss", c_f32), ("policy_loss", c_f32), ("value_loss", c_f32), ("approx_kl_div", c_f32),
                ("clip_fraction", c_f32), ("loss", c_f32), ("explained_variance", c_f32), ("grad_norm", c_f32),
                ("learning_rate", c_f32), ("entropy", c_f32), ("ratio", c_f32), ("rollout_ms", c_f32),
                ("update_ms", c_f32), ("n_minibatch_steps", c_i32), ("kl_stopped", c_i32), ("episodes", c_i64),
                ("episode_return_sum", c_f64), ("episode_length_sum", c_f64),
                ("ep_rew_mean", c_f32), ("ep_len_mean", c_f32), ("episodes_in_window", c_i64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol declared in include/dril_b200.h: name -> argtypes (restype is int32 unless noted)
PROTOTYPES = {
    "dril_device_count": [C.POINTER(c_i32)],
    "dril_set_option": [C.c_char_p, c_i32],
    "dril_ctx_create": [c_i32, c_u64, C.POINTER(P)],
    "dril_ctx_destroy": [P],
    "dril_ctx_synchronize": [P],
    "dril_ctx_launch_count": [P, C.POINTER(c_i64)],
    "dril_ctx_set_profiling": [P, c_i32],
    "dril_ctx_reset_profile": [P],
    "dril_ctx_get_profile": [P, c_i32, C.POINTER(c_f64), C.POINTER(c_i64)],
    "dril_ctx_sm_count": [P, C.POINTER(c_i32)],
    "dril_ctx_event_record": [P, c_i32],
    "dril_ctx_event_elapsed_ms": [P, c_i32, c_i32, C.POINTER(c_f32)],
    "dril_ctx_flush_l2": [P],
    "dril_comm_unique_id": [P],
    "dril_comm_init": [P, c_i32, c_i32, P],
    "dril_comm_destroy": [P],
    "dril_comm_p2p_export": [P, c_i64, P],
    "dril_comm_p2p_import": [P, P],
    "dril_env_create": [P, c_i32, c_i64, c_i32, c_i32, c_i32, c_i64, C.POINTER(NormCfg), c_i32, C.POINTER(P)],
    "dril_env_destroy": [P],
    "dril_env_seed": [P, c_u64],
    "dril_env_reset": [P],
    "dril_env_observe": [P, P],
    "dril_env_step": [P, P, P, P, P, P, P, P],
    "dril_env_num_envs": [P, C.POINTER(c_i64)],
    "dril_env_get_state": [P, P, P],
    "dril_env_set_state": [P, P, P],
    "dril_env_get_norm_stats": [P, P, P, C.POINTER(c_i64), C.POINTER(c_f32), C.POINTER(c_f32), C.POINTER(c_i64)],
    "dril_env_set_norm_stats": [P, P, P, c_i64, c_f32, c_f32, c_i64],
    "dril_env_set_training": [P, c_i32],
    "dril_env_set_scaling": [P, c_i32, P, P, P, P],
    "dril_env_get_original": [P, P, P],
    "dril_env_monitor_stats": [P, C.POINTER(c_f32), C.POINTER(c_f32), C.POINTER(c_i64), C.POINTER(c_i64)],
    "dril_env_set_params": [P, c_i32, P, P],
    "dril_env_get_params": [P, c_i32, P],
    "dril_env_set_observe_params": [P, c_i32],
    "dril_env_obs_dim": [P, C.POINTER(c_i32)],
    "dril_env_set_obs_history": [P, c_i32, c_i32],
    "dril_env_set_obs_noise": [P, c_i32, P],
    "dril_env_set_action_delay": [P, P],
    "dril_env_set_adr": [P, c_i32, P, c_f32, c_i64, c_f32, c_f32],
    "dril_env_get_adr": [P, P, P, P, P, C.POINTER(c_i64)],
    "dril_policy_create": [P, c_i32, c_i32, P, c_i32, c_i32, c_i32, P, P, C.POINTER(P)],
    "dril_policy_destroy": [P],
    "dril_policy_num_params": [P, C.POINTER(c_i64)],
    "dril_policy_update_path": [P, C.POINTER(c_i32)],
    "dril_policy_set_params": [P, P, c_i64],
    "dril_policy_get_params": [P, P, c_i64],
    "dril_policy_get_opt_state": [P, P, P, c_i64, C.POINTER(c_i64)],
    "dril_policy_set_opt_state": [P, P, P, c_i64, c_i64],
    "dril_policy_seed": [P, c_u64, c_u64],
    "dril_policy_forward": [P, P, c_i64, c_i32, P, P, P, P],
    "dril_policy_evaluate": [P, P, P, c_i64, P, P, P],
    "dril_policy_predict_values": [P, P, c_i64, P],
    "dril_buffer_create": [P, c_i64, c_i64, c_i32, c_i32, c_i32, C.POINTER(P)],
    "dril_buffer_destroy": [P],
    "dril_buffer_download": [P, c_i32, P, c_i64],
    "dril_buffer_upload": [P, c_i32, P, c_i64],
    "dril_buffer_field_bytes": [P, c_i32, C.POINTER(c_i64)],
    "dril_rollout_collect": [P, P, P, P, C.POINTER(c_f32)],
    "dril_rollout_collect_steps": [P, P, P, c_i64, c_i64, c_i32, P],
    "dril_evaluate": [P, P, c_i64, c_i32, c_i32, P, P, C.POINTER(c_i64), C.POINTER(c_i64)],
    "dril_env_zero_returns": [P],
    "dril_gae": [P, c_f32, c_f32],
    "dril_gae_raw": [P, P, P, P, P, P, P, c_i64, c_i64, c_f32, c_f32, P, P],
    "dril_ppo_loss_grad": [P, P, P, P, P, P, P, c_i64, C.POINTER(PPOHyper), C.POINTER(c_f32), P, P],
    "dril_optimizer_step": [P, P, c_i64, C.POINTER(PPOHyper), C.POINTER(c_f32)],
    "dril_ppo_update": [P, P, C.POINTER(PPOHyper), c_i32, c_i64, c_u64, c_u64, C.POINTER(IterStats)],
    "dril_iteration_prepare": [P, P, P, c_i32, c_i64],
    "dril_ppo_iteration_async": [P, P, P, C.POINTER(PPOHyper), c_i32, c_i64, c_u64, c_u64],
    "dril_iteration_result": [P, C.POINTER(IterStats)],
    "dril_explained_variance": [P, C.POINTER(c_f32)],
}
SPECIAL_RESTYPE = {"dril_last_error": C.c_char_p, "dril_version": c_i32, "dril_source_hash": C.c_char_p}

BUF_FIELDS = dict(obs=0, actions=1, rewards=2, values=3, logprobs=4, advantages=5, returns=6, flags=7, boot=8,
                  last_values=9, episode_r=10, episode_l=11)
KERNEL_KINDS = ["rollout", "gae", "adv_stats", "loss_grad", "grad_reduce", "adam", "explained_var", "monitor",
                "env", "policy", "allreduce", "permute"]

_lib = None


def load(require_device=True):
    """Load libdril_b200.so (building it is __graft_entry__.build()'s job). Raises if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DrilError(f"{LIB_PATH} not found: build it with `python dril.jl_b200/build.py` "
                            "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, args in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = c_i32
        lib.dril_last_error.restype = C.c_char_p
        lib.dril_last_error.argtypes = []
        lib.dril_version.restype = c_i32
        lib.dril_version.argtypes = []
        lib.dril_source_hash.restype = C.c_char_p
        lib.dril_source_hash.argtypes = []
        _lib = lib
    if require_device:
        n = c_i32(0)
        check(_lib.dril_device_count(C.byref(n)))
    return _lib


def check(status):
    if status != 0:
        raise DrilError(_lib.dril_last_error().decode())


def ptr(a):
    """numpy array (C-contiguous) -> void*"""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(P)


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)
