"""deep_rl_b200 -- B200-native (sm_100a) PPO rollout-and-update hot path of qgallouedec/deep_rl.

Public surface (mirrors deep_rl/ppo.py):
    make(env_id, num_envs, seed)   -> VecEnv      (gym.make + RecordEpisodeStatistics + TorchWrapper)
    ActorCritic(env)               -> agent       (get_value / get_action_distribution / get_action)
    PPOConfig, PPOTrainer, train   -> the loop of ppo.py:105-192 as CUDA kernels behind a C ABI
    ReplayBuffer                   -> storage, index samplers and batch gather of dqn.py / per.py (SURVEY.md 8f-4)
    evaluate(agent, env_id, N, K)  -> EvalResult  (N fresh envs x K episodes of a frozen policy, greedy or sampled, one launch)
Importing the package does not need a GPU; constructing any of the above does (no CPU fallback).
"""
from .agent import ActorCritic, layer_init  # noqa: F401
from .envs import VecEnv, make  # noqa: F401
from .evaluate import EvalResult, evaluate  # noqa: F401
from .ppo import PPOConfig, PPOTrainer, train  # noqa: F401
from .replay import ReplayBuffer  # noqa: F401

__all__ = ["ActorCritic", "layer_init", "VecEnv", "make", "EvalResult", "evaluate", "PPOConfig", "PPOTrainer", "train",
           "ReplayBuffer"]
