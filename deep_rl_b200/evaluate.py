"""Policy evaluation on fresh episodes: N envs x K whole episodes of a frozen policy in ONE kernel launch (drl_evaluate for
64-wide nets, fp32 CUDA cores; drl_evaluate_tc for 256-wide nets, tcgen05 with the training rollout's bf16 numerics).

The counterpart of CleanRL's eval scripts and SB3's `evaluate_policy`: unlike `PPOTrainer.metrics()["mean_return"]` (the
training episodes that happened to finish inside one rollout window, produced by several successive policies, always
sampled), every env here starts a fresh episode from the reset draw of the evaluation key and plays exactly
`episodes_per_env` episodes with the current parameters, greedy (argmax) or sampled.  Results depend on (parameters,
env_id, seed, global env ids, greedy) only: the same call gives the same numbers bit for bit, and ranks that evaluate
disjoint global env ids (env_gid0 = rank * num_envs) play disjoint episodes, whose results the caller may gather.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _lib
from .envs import MAX_EPISODE_STEPS, VecEnv

DRL_EVAL_GREEDY = 1


@dataclass
class EvalResult:
    returns: np.ndarray          # [N, K] float32: episode k of env n, in the order the env played them
    lengths: np.ndarray          # [N, K] int32
    mean_return: float
    std_return: float            # population standard deviation over the N * K episodes (like SB3's evaluate_policy)
    mean_length: float
    env_steps: int               # sum of the lengths: env steps the launch took
    greedy: bool
    # trace=True only ([S][N] rows, S = K * max_episode_steps; rows after an env's quota have act == 0xFF):
    state: Optional[torch.Tensor] = None     # [S, N, 4] float64: the state each action was chosen in
    obs: Optional[torch.Tensor] = None       # [S, N, OP] float32
    logits: Optional[torch.Tensor] = None    # [S, N, A] float32
    act: Optional[torch.Tensor] = None       # [S, N] uint8

    @property
    def episodes(self) -> int:
        return int(self.returns.size)


def evaluate(agent, env_id: str, num_envs: int, episodes_per_env: int = 1, greedy: bool = True, seed: int = 0,
             env_gid0: int = 0, trace: bool = False) -> EvalResult:
    """Play `episodes_per_env` episodes on each of `num_envs` fresh envs with `agent`'s current parameters: fp32 forward for
    hidden = 64 (drl_evaluate), the tensor-core forward of the training rollout for hidden = 256 (drl_evaluate_tc).  `seed` is the evaluation key of the env resets and of the sampled actions; `env_gid0` the global id of
    env 0.  Synchronises the current stream once, to read the episode log.  `trace=True` also returns the per-step planes
    (tests; S * N * (32 + 4 * OP + 4 * A + 1) bytes)."""
    _lib.require_cuda()
    N, K = int(num_envs), int(episodes_per_env)
    if N < 1 or K < 1:
        raise ValueError(f"num_envs={N} and episodes_per_env={K} must be >= 1")
    env = VecEnv(env_id, N, seed=seed, env_gid0=env_gid0, device=agent.device, log_capacity=N * K)
    agent._ensure_packed()
    tr = None
    out = {}
    if trace:
        S = K * MAX_EPISODE_STEPS[env_id]
        dev = agent.device
        out = {"state": torch.zeros((S, N, 4), dtype=torch.float64, device=dev),
               "obs": torch.zeros((S, N, env.obs_stride), dtype=torch.float32, device=dev),
               "logits": torch.zeros((S, N, env.num_actions), dtype=torch.float32, device=dev),
               "act": torch.zeros((S, N), dtype=torch.uint8, device=dev)}
        tr = _lib.EvalTraceT(*(out[k].data_ptr() for k in ("state", "obs", "logits", "act")))
    name = "drl_evaluate_tc" if agent.hidden == 256 else "drl_evaluate"
    _lib.check(getattr(env.L, name)(C.byref(env.struct), C.byref(agent.net), agent.packed.data_ptr(), K,
                                    DRL_EVAL_GREEDY if greedy else 0, C.byref(env.log.struct),
                                    C.byref(tr) if tr is not None else None, _lib.stream_ptr()))
    n, _, _, e = env.log.drain_arrays()
    if n != N * K:
        raise _lib.DrlError(f"{name} logged {n} episodes, expected {N * K}")
    order = np.lexsort((e["step"], e["env"]))          # by env, then by the step the episode ended at
    returns = np.ascontiguousarray(e["ret"][order]).reshape(N, K).copy()
    lengths = np.ascontiguousarray(e["len"][order]).reshape(N, K).astype(np.int32)
    return EvalResult(returns=returns, lengths=lengths, mean_return=float(returns.mean(dtype=np.float64)),
                      std_return=float(returns.std(dtype=np.float64)), mean_length=float(lengths.mean(dtype=np.float64)),
                      env_steps=int(lengths.sum(dtype=np.int64)), greedy=bool(greedy), **out)
