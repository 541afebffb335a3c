"""ctypes binding of libevac_b200.so (the C ABI declared in include/evac_b200.h).

There is deliberately no CPU fallback: if the library is missing or cannot be loaded this
module raises, and every product entry point (`setup_env`, `EvacuationEnv`) fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build
from .build import LIB_PATH

EVAC_ABI_VERSION = 6
NUM_EPISODE_STATS = 9
EPISODE_STAT_KEYS = (  # env.py:115-125
    "episode_intrinsic_reward", "episode_status_reward", "episode_reward", "episode_length",
    "escaped_pedestrians", "exiting_pedestrians", "following_pedestrians", "viscek_pedestrians",
    "overall_timesteps",
)

POS = {"abs": 0, "rel": 1, "grav": 2}
STAT = {"no": 0, "ohe": 1, "cat": 2}
OBS = {"Dict": 0, "Box": 1}
PREC = {"fp32": 0, "fp64": 1}
AGENT = {"table": 0, "random": 1, "rotating": 2, "wacuum": 3}
SEARCH = {"auto": 0, "brute": 1, "cells": 2}


class EvacConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("number_of_pedestrians", C.c_int32),
        ("width", C.c_double), ("height", C.c_double),
        ("step_size", C.c_double), ("noise_coef", C.c_double), ("eps", C.c_double),
        ("enslaving_degree", C.c_double),
        ("is_new_exiting_reward", C.c_int32), ("is_new_followers_reward", C.c_int32),
        ("intrinsic_reward_coef", C.c_double),
        ("is_termination_agent_wall_collision", C.c_int32),
        ("init_reward_each_step", C.c_double),
        ("max_timesteps", C.c_int32),
        ("positions", C.c_int32), ("statuses", C.c_int32), ("obs_type", C.c_int32),
        ("alpha", C.c_double),
        ("to_leader", C.c_double), ("to_pedestrian", C.c_double), ("to_exit", C.c_double), ("to_escape", C.c_double),
        ("auto_reset", C.c_int32), ("precision", C.c_int32), ("neighbor_search", C.c_int32),
    ]


class EvacEnvParams(C.Structure):
    _fields_ = [
        ("noise_coef", C.c_double), ("enslaving_degree", C.c_double), ("alpha", C.c_double),
        ("intrinsic_reward_coef", C.c_double), ("init_reward_each_step", C.c_double),
        ("is_new_exiting_reward", C.c_int32), ("is_new_followers_reward", C.c_int32),
        ("is_termination_agent_wall_collision", C.c_int32), ("max_timesteps", C.c_int32),
    ]


class EvacPolicyConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("seq_len", C.c_int32), ("d_model", C.c_int32), ("num_heads", C.c_int32),
        ("dim_feedforward", C.c_int32), ("num_blocks", C.c_int32), ("use_resid", C.c_int32),
        ("dropout", C.c_float), ("layer_norm_eps", C.c_float), ("num_hidden", C.c_int32), ("action_dim", C.c_int32),
    ]


class EvacPolicyIO(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32), ("obs", C.c_void_p),
        ("norm_mean", C.c_void_p), ("norm_var", C.c_void_p), ("norm_count", C.c_void_p), ("obs_norm", C.c_void_p),
        ("norm_eps", C.c_float), ("norm_clip", C.c_float),
        ("embedding", C.c_void_p), ("mean", C.c_void_p), ("value", C.c_void_p), ("action", C.c_void_p),
        ("action_clipped", C.c_void_p), ("logprob", C.c_void_p), ("entropy", C.c_void_p), ("given_action", C.c_void_p),
        ("sample", C.c_int32), ("training", C.c_int32), ("seed", C.c_uint64), ("offset", C.c_uint64),
        ("offset_device", C.c_void_p), ("env_index_offset", C.c_int64), ("norm_frozen", C.c_int32),
    ]


class EvacPolicyRolloutIO(C.Structure):
    _fields_ = [
        ("obs", C.c_void_p), ("next_done", C.c_void_p),
        ("norm_mean", C.c_void_p), ("norm_var", C.c_void_p), ("norm_count", C.c_void_p),
        ("norm_eps", C.c_float), ("norm_clip", C.c_float), ("norm_update", C.c_int32),
        ("returns", C.c_void_p), ("ret_mean", C.c_void_p), ("ret_var", C.c_void_p), ("ret_count", C.c_void_p),
        ("gamma", C.c_float), ("eps", C.c_float), ("clip", C.c_float),
        ("sample", C.c_int32), ("seed", C.c_uint64), ("offset", C.c_uint64), ("offset_device", C.c_void_p),
        ("env_index_offset", C.c_int64),
        ("obs_norm", C.c_void_p), ("action", C.c_void_p), ("logprob", C.c_void_p), ("value", C.c_void_p),
        ("reward_norm", C.c_void_p), ("dones", C.c_void_p), ("status_counts", C.c_void_p),
        ("reward_sum", C.c_void_p), ("terminated", C.c_void_p), ("truncated", C.c_void_p),
    ]


# every symbol include/evac_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "evac_abi_version": (C.c_int32, []),
    "evac_last_error": (C.c_char_p, []),
    "evac_build_id": (C.c_char_p, []),
    "evac_default_config": (C.c_int, [C.POINTER(EvacConfig)]),
    "evac_create": (C.c_int, [C.POINTER(EvacConfig), C.c_int32, C.c_int32, C.c_uint64, C.c_int64, C.POINTER(_P)]),
    "evac_destroy": (C.c_int, [_P]),
    "evac_obs_dim": (C.c_int32, [_P]),
    "evac_num_envs": (C.c_int32, [_P]),
    "evac_num_cells": (C.c_int32, [_P]),
    "evac_state_elem_size": (C.c_int32, [_P]),
    "evac_reset": (C.c_int, [_P, _P, _P, _P]),
    "evac_set_state": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "evac_get_state": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "evac_observe": (C.c_int, [_P, _P, _P]),
    "evac_step": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "evac_step_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "evac_rollout": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P]),
    "evac_episode_stats": (C.c_int, [_P, _P, _P, _P, _P]),
    "evac_get_accumulators": (C.c_int, [_P, _P, _P, _P]),
    "evac_launch_count": (C.c_int64, [_P]),
    "evac_state_bytes": (C.c_int64, [_P]),
    "evac_save_state": (C.c_int, [_P, _P, _P]),
    "evac_load_state": (C.c_int, [_P, _P, _P]),
    "evac_set_env_params": (C.c_int, [_P, _P, _P]),
    "evac_get_env_params": (C.c_int, [_P, _P]),
    "evac_policy_default_config": (C.c_int, [C.POINTER(EvacPolicyConfig), C.c_int32, C.c_int32]),
    "evac_policy_default_linear_config": (C.c_int, [C.POINTER(EvacPolicyConfig), C.c_int32]),
    "evac_policy_create": (C.c_int, [C.POINTER(EvacPolicyConfig), C.c_int32, C.POINTER(_P)]),
    "evac_policy_destroy": (C.c_int, [_P]),
    "evac_policy_num_weights": (C.c_int64, [_P]),
    "evac_policy_load_weights": (C.c_int, [_P, _P, C.c_int64]),
    "evac_policy_reserve": (C.c_int, [_P, C.c_int32]),
    "evac_policy_forward": (C.c_int, [_P, C.POINTER(EvacPolicyIO), _P]),
    "evac_policy_launch_count": (C.c_int64, [_P]),
    "evac_normalize_reward": (C.c_int, [C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_float, C.c_float, C.c_float, _P]),
    "evac_rollout_policy": (C.c_int, [_P, _P, C.c_int32, C.POINTER(EvacPolicyRolloutIO), _P]),
    "evac_probe_fma": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_double)]),
    "evac_probe_pairwise": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_double)]),
}

_lib = None


def build_id() -> str:
    """Build id of the LOADED library (== evacuation_b200.build.source_hash() of the tree it was built from)."""
    return load().evac_build_id().decode()


class EvacNativeError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the in-tree CUDA library; raise (never fall back) if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    want = _build.source_hash()
    if _build.library_build_id() != want and not os.environ.get("EVAC_B200_LIB"):
        # missing, or built from other sources than the tree holds (content hash, not mtime): rebuild or fail -- never run it
        try:
            _build.build(force=True)
        except Exception as exc:
            raise EvacNativeError(
                f"{LIB_PATH} is missing or stale (build id {_build.library_build_id()} != source hash {want}) and could not be "
                f"rebuilt: {exc}.  Build it with `python -m evacuation_b200.build`; evacuation_b200 has no CPU fallback.") from exc
    if not os.path.exists(LIB_PATH):
        raise EvacNativeError(f"{LIB_PATH} is missing: build it with `python -m evacuation_b200.build`.  evacuation_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    if lib.evac_abi_version() != EVAC_ABI_VERSION:
        raise EvacNativeError("libevac_b200.so ABI version mismatch; rebuild")
    got = lib.evac_build_id().decode()
    if got != want and not os.environ.get("EVAC_B200_LIB"):  # (EVAC_B200_LIB: an explicitly chosen library built elsewhere)
        raise EvacNativeError(f"{LIB_PATH} was built from other sources (build id {got}, tree {want}); rebuild")
    _lib = lib
    return lib


def check(rc: int) -> None:
    """Map C error codes onto the exception types the reference raises for the same mistakes."""
    if rc == 0:
        return
    msg = load().evac_last_error().decode()
    if rc == -3:
        raise NotImplementedError(msg)
    if rc == -1:
        raise ValueError(msg)
    raise EvacNativeError(f"evac error {rc}: {msg}")
