"""ctypes binding of libdrl_b200.so (the C ABI declared in include/drl_b200.h).

There is no CPU fallback: if the CUDA library cannot be loaded, `lib()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import build as _build

_LIB = None

u8p, i32p, u32p, u64p, f32p, f64p = (C.c_void_p,) * 6  # device pointers travel as raw addresses


class EnvT(C.Structure):
    _fields_ = [("kind", C.c_int32), ("num_envs", C.c_int32), ("seed", C.c_uint64), ("env_gid0", C.c_uint32),
                ("max_episode_steps", C.c_int32), ("state", C.c_void_p), ("elapsed", C.c_void_p),
                ("ep_ret", C.c_void_p), ("ep_len", C.c_void_p)]


class EpLogT(C.Structure):
    _fields_ = [("count", C.c_void_p), ("sum_ret", C.c_void_p), ("sum_len", C.c_void_p), ("entries", C.c_void_p),
                ("cap", C.c_uint32)]


class NetT(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("hidden", C.c_int32), ("num_actions", C.c_int32), ("obs_stride", C.c_int32)]


class RolloutBufT(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("act", C.c_void_p), ("logp", C.c_void_p), ("val", C.c_void_p),
                ("rew", C.c_void_p), ("done", C.c_void_p), ("logits", C.c_void_p)]


class EvalTraceT(C.Structure):
    _fields_ = [("state", C.c_void_p), ("obs", C.c_void_p), ("logits", C.c_void_p), ("act", C.c_void_p)]


class CommT(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("peer", C.c_void_p * 8), ("seq", C.c_uint32),
                ("error_flag", C.c_void_p)]


class CtrlT(C.Structure):
    _fields_ = [("env_step", C.c_uint64), ("epoch_ctr", C.c_uint32), ("comm_seq", C.c_uint32), ("adam_step", C.c_int64),
                ("neg_step_size", C.c_float * 64), ("bc2_sqrt", C.c_float * 64)]


class PpoCoefT(C.Structure):
    _fields_ = [("clip_coef", C.c_float), ("ent_coef", C.c_float), ("vf_coef", C.c_float)]


# name -> (restype, argtypes); every symbol include/drl_b200.h declares
SIGNATURES = {
    "drl_abi_version": (C.c_int, []),
    "drl_last_error": (C.c_char_p, []),
    "drl_env_obs_dim": (C.c_int, [C.c_int32]),
    "drl_env_num_actions": (C.c_int, [C.c_int32]),
    "drl_env_obs_stride": (C.c_int, [C.c_int32]),
    "drl_param_count": (C.c_int64, [C.POINTER(NetT)]),
    "drl_packed_count": (C.c_int64, [C.POINTER(NetT)]),
    "drl_record_width": (C.c_int, [C.POINTER(NetT)]),
    "drl_workspace_bytes": (C.c_size_t, [C.POINTER(NetT)]),
    "drl_env_reset": (C.c_int, [C.POINTER(EnvT), f32p, C.c_void_p]),
    "drl_env_observe": (C.c_int, [C.POINTER(EnvT), f32p, C.c_void_p]),
    "drl_env_step": (C.c_int, [C.POINTER(EnvT), C.c_uint64, i32p, f32p, f32p, u8p, C.POINTER(EpLogT), C.c_void_p]),
    "drl_pack_params": (C.c_int, [C.POINTER(NetT), f32p, f32p, C.c_void_p]),
    "drl_policy_forward": (C.c_int, [C.POINTER(NetT), f32p, f32p, C.c_int64, f32p, f32p, C.c_void_p]),
    "drl_sample": (C.c_int, [f32p, C.c_int64, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint64, i32p, f32p, C.c_void_p]),
    "drl_rollout": (C.c_int, [C.POINTER(EnvT), C.POINTER(NetT), f32p, C.c_int32, C.c_uint64, C.POINTER(RolloutBufT),
                              C.POINTER(EpLogT), C.c_uint32, C.c_void_p]),
    "drl_evaluate": (C.c_int, [C.POINTER(EnvT), C.POINTER(NetT), f32p, C.c_int32, C.c_uint32, C.POINTER(EpLogT),
                               C.POINTER(EvalTraceT), C.c_void_p]),
    "drl_evaluate_tc": (C.c_int, [C.POINTER(EnvT), C.POINTER(NetT), f32p, C.c_int32, C.c_uint32, C.POINTER(EpLogT),
                                  C.POINTER(EvalTraceT), C.c_void_p]),
    "drl_gae": (C.c_int, [C.POINTER(RolloutBufT), C.POINTER(NetT), C.c_int32, C.c_int32, C.c_float, C.c_float, f32p,
                          f32p, f32p, C.c_void_p]),
    "drl_explained_variance": (C.c_int, [f32p, f32p, C.c_int64, f32p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "drl_permutation": (C.c_int, [u32p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]),
    "drl_adv_stats": (C.c_int, [C.POINTER(NetT), f32p, u32p, C.c_uint32, C.c_uint32, f32p, C.c_void_p, C.c_size_t,
                                C.c_void_p]),
    "drl_adv_stats_perm": (C.c_int, [C.POINTER(NetT), f32p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, f32p,
                                     C.c_void_p, C.c_size_t, C.c_void_p]),
    "drl_ppo_minibatch_grad": (C.c_int, [C.POINTER(NetT), f32p, f32p, u32p, C.c_uint32, C.c_uint32, f32p,
                                         C.POINTER(PpoCoefT), f32p, f32p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]),
    "drl_ppo_minibatch_update": (C.c_int, [C.POINTER(NetT), f32p, f32p, u32p, C.c_uint32, C.c_uint32, f32p, C.POINTER(PpoCoefT),
                                           f32p, f32p, f32p, f32p, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double,
                                           C.c_double, f32p, f32p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_int32, C.c_void_p]),
    "drl_ppo_minibatch_update_dist": (C.c_int, [C.POINTER(NetT), f32p, f32p, u32p, C.c_uint32, C.c_uint32, f32p, C.POINTER(PpoCoefT),
                                                f32p, f32p, f32p, f32p, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double,
                                                C.c_double, f32p, f32p, C.c_void_p, C.c_size_t, C.c_uint32, C.POINTER(CommT),
                                                C.c_int32, C.c_void_p]),
    "drl_ctrl_set": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int64, C.c_int32, C.c_double, C.c_double, C.c_double,
                               C.c_void_p]),
    "drl_rollout_ctl": (C.c_int, [C.POINTER(EnvT), C.POINTER(NetT), f32p, C.c_int32, C.c_void_p, C.POINTER(RolloutBufT),
                                  C.POINTER(EpLogT), C.c_uint32, C.c_void_p]),
    "drl_permutation_ctl": (C.c_int, [u32p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "drl_adv_stats_perm_ctl": (C.c_int, [C.POINTER(NetT), f32p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32,
                                         f32p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "drl_ppo_minibatch_update_ctl": (C.c_int, [C.POINTER(NetT), f32p, f32p, u32p, C.c_uint32, C.c_uint32, f32p, C.POINTER(PpoCoefT),
                                               f32p, f32p, f32p, f32p, C.c_void_p, C.c_int32, C.c_double, C.c_double, C.c_double,
                                               C.c_double, f32p, f32p, C.c_void_p, C.c_size_t, C.c_uint32, C.POINTER(CommT),
                                               C.c_int32, C.c_void_p]),
    "drl_comm_bytes": (C.c_size_t, [C.POINTER(NetT)]),
    "drl_comm_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p), C.c_void_p]),
    "drl_comm_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "drl_comm_close": (C.c_int, [C.c_void_p]),
    "drl_comm_free": (C.c_int, [C.c_void_p]),
    "drl_replay_sample_uniform": (C.c_int, [u32p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p]),
    "drl_replay_gather": (C.c_int, [f32p, i32p, f32p, u8p, u32p, C.c_uint32, C.c_int32, f32p, f32p, i32p, f32p, u8p, C.c_void_p]),
    "drl_replay_scratch_bytes": (C.c_size_t, [C.c_uint32]),
    "drl_replay_sample_priority": (C.c_int, [f32p, C.c_uint32, C.c_float, C.c_uint32, C.c_uint64, C.c_uint64, u32p, f32p, C.c_void_p,
                                             C.c_size_t, C.c_void_p]),
    "drl_replay_update_priorities": (C.c_int, [f32p, u32p, f32p, C.c_uint32, f32p, C.c_void_p]),
    "drl_reinforce_param_count": (C.c_int, []),
    "drl_reinforce_episodes": (C.c_int, [C.POINTER(EnvT), f32p, C.c_int32, C.c_uint64, f32p, u8p, f32p, u8p, i32p, u32p, C.POINTER(EpLogT),
                                         C.c_void_p]),
    "drl_reinforce_grad": (C.c_int, [f32p, f32p, u8p, f32p, i32p, u32p, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint64, C.c_float, f32p, f32p,
                                     f32p, f32p, C.c_void_p]),
    "drl_adam_step": (C.c_int, [f32p, f32p, f32p, f32p, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_void_p]),
    "drl_selftest_umma": (C.c_int, [C.c_int32, C.c_int32, f32p, f32p, f32p, C.c_void_p]),
    "drl_selftest_tanh": (C.c_int, [f32p, f32p, C.c_int64, C.c_void_p]),
    "drl_clip_adam": (C.c_int, [C.POINTER(NetT), f32p, f32p, f32p, f32p, C.c_int64, C.c_double, C.c_double, C.c_double,
                                C.c_double, C.c_double, C.c_double, f32p, f32p, C.c_void_p]),
}


class DrlError(RuntimeError):
    pass


def lib_path() -> str:
    return _build.SO


ABI_VERSION = 2


def lib() -> C.CDLL:
    """Load the CUDA library, (re)building it first when it is absent or older than its sources and a compiler is
    available (under an inter-process file lock, so that the ranks of one torchrun job do not race).  Raises if the
    library can neither be found nor built."""
    global _LIB
    if _LIB is None:
        path = _build.build_locked()
        L = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)   # AttributeError here = header/library mismatch: fail loudly
            fn.restype, fn.argtypes = res, args
        if L.drl_abi_version() != ABI_VERSION:
            raise DrlError(f"libdrl_b200 ABI version {L.drl_abi_version()} != {ABI_VERSION}")
        _LIB = L
    return _LIB


def check(rc: int) -> None:
    if rc != 0:
        raise DrlError(f"libdrl_b200 error {rc}: {lib().drl_last_error().decode()}")


def require_cuda() -> None:
    if not torch.cuda.is_available():
        raise DrlError("deep_rl_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def ptr(t) -> int:
    """Raw device address of a tensor (None -> NULL)."""
    return 0 if t is None else t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream
