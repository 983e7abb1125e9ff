"""drl_evaluate on CartPole-v1, greedy, N = 4,096 and 65,536 envs x 1 episode, for two policies: the initial one and one this
script trains first (4,096 envs x 128 steps x 40 updates).  Reports, per (policy, N):

  * useful env-steps/s = sum of episode lengths / kernel time (CUDA events around each launch, after a warm-up);
  * lane utilisation = sum of lengths / (EPW x sum over warps of the longest episode run in the warp): the share of the lane
    slots of the launch that stepped an env, i.e. the cost of ragged episode lengths inside a warp (EPW = envs per warp,
    the choice of pick_envs_per_warp in rollout.cu, mirrored below);
  * for comparison, the fp32 CUDA-core drl_rollout (flags 0) at the same N and T = 500 with the same parameters, timed in
    the same run: env-steps/s = N x T / kernel time;

plus the GPU name and power limit.

    python profiles/tools/eval_probe.py [--out FILE.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import deep_rl_b200 as drl  # noqa: E402
from deep_rl_b200 import _lib  # noqa: E402
from deep_rl_b200.envs import VecEnv  # noqa: E402

ENV_ID = "CartPole-v1"
EVAL_SEED = 77
REPS = 10


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def envs_per_warp(N: int) -> int:
    """pick_envs_per_warp (rollout.cu), for the utilisation ratio."""
    ov = os.environ.get("DRL_ROLLOUT_EPW")
    if ov in ("4", "8", "16", "32"):
        return int(ov)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if N <= sms * 8 * 4:
        return 4
    w8 = (N + 7) // 8
    return 8 if w8 <= sms * 24 else 16 if w8 <= sms * 48 else 32


def time_ms(call, reps=REPS, before=None):
    """Mean device time of `call` over `reps` launches (each bracketed by its own events), after two warm-up launches."""
    for _ in range(2):
        if before:
            before()
        call()
    ms = []
    for _ in range(reps):
        if before:
            before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.mean(ms)), float(np.std(ms))


def probe_eval(agent, N):
    env = VecEnv(ENV_ID, N, seed=EVAL_SEED, log_capacity=N)
    agent._ensure_packed()
    call = lambda: _lib.check(env.L.drl_evaluate(C.byref(env.struct), C.byref(agent.net), agent.packed.data_ptr(), 1, 1,
                                                 C.byref(env.log.struct), None, _lib.stream_ptr()))
    ms, sd = time_ms(call, before=env.log.clear)
    res = drl.evaluate(agent, ENV_ID, N, episodes_per_env=1, greedy=True, seed=EVAL_SEED)     # the lengths of that launch
    total = res.lengths.sum(axis=1).astype(np.int64)
    epw = envs_per_warp(N)
    pad = (-N) % epw
    per_warp_max = np.concatenate([total, np.zeros(pad, np.int64)]).reshape(-1, epw).max(axis=1)
    steps = int(total.sum())
    return {"N": N, "eval_ms": ms, "eval_ms_std": sd, "env_steps": steps, "mean_return": res.mean_return,
            "mean_length": res.mean_length, "max_length": int(total.max()), "envs_per_warp": epw,
            "useful_env_steps_per_s": steps / (ms * 1e-3), "lane_utilisation": steps / float(epw * per_warp_max.sum())}


def probe_rollout(agent, N, T=500):
    env = VecEnv(ENV_ID, N, seed=EVAL_SEED, log_capacity=1 << 16)
    env.reset()
    dev, OP = env.device, env.obs_stride
    planes = [torch.zeros((T + 1, N, OP), dtype=torch.float32, device=dev), torch.zeros((T + 1, N), dtype=torch.uint8, device=dev)]
    planes += [torch.zeros((T + 1, N), dtype=torch.float32, device=dev) for _ in range(3)]
    planes.append(torch.zeros((T + 1, N), dtype=torch.uint8, device=dev))
    obs, act, logp, val, rew, done = planes
    buf = _lib.RolloutBufT(obs.data_ptr(), act.data_ptr(), logp.data_ptr(), val.data_ptr(), rew.data_ptr(), done.data_ptr(), None)
    agent._ensure_packed()
    k = [0]

    def call():
        _lib.check(env.L.drl_rollout(C.byref(env.struct), C.byref(agent.net), agent.packed.data_ptr(), T, k[0] * T, C.byref(buf),
                                     C.byref(env.log.struct), 0, _lib.stream_ptr()))
        k[0] += 1
    ms, sd = time_ms(call, before=env.log.clear)
    return {"N": N, "T": T, "rollout_fp32_ms": ms, "rollout_fp32_ms_std": sd, "rollout_fp32_env_steps_per_s": N * T / (ms * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    _lib.require_cuda()
    torch.cuda.set_device(0)
    gpu = {"name": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    print(f"GPU: {gpu['name']}, power limit {gpu['power_limit']}")
    init = drl.PPOTrainer(drl.PPOConfig(num_envs=64, seed=1)).agent
    cfg = drl.PPOConfig(num_envs=4096, num_steps=128, total_timesteps=4096 * 128 * 40, seed=1)
    tr = drl.PPOTrainer(cfg)
    for _ in range(cfg.num_updates()):
        tr.update()
    torch.cuda.synchronize()
    rows = []
    for name, agent in (("initial", init), ("trained", tr.agent)):
        for N in (4096, 65536):
            r = {"policy": name, **probe_eval(agent, N), **probe_rollout(agent, N)}
            r["eval_over_rollout_per_env_step"] = r["useful_env_steps_per_s"] / r["rollout_fp32_env_steps_per_s"]
            rows.append(r)
            print(f"{name:8s} N={N:6d}: eval {r['eval_ms']:.3f} ms, mean length {r['mean_length']:.1f} (max {r['max_length']}), "
                  f"{r['useful_env_steps_per_s'] / 1e9:.3f} G useful env-steps/s, lane utilisation {r['lane_utilisation']:.3f} "
                  f"(EPW {r['envs_per_warp']}) | fp32 rollout T=500 {r['rollout_fp32_ms']:.3f} ms, "
                  f"{r['rollout_fp32_env_steps_per_s'] / 1e9:.3f} G env-steps/s | eval/rollout {r['eval_over_rollout_per_env_step']:.2f}")
    out = {"gpu": gpu, "rows": rows}
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
