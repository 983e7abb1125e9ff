"""drl_evaluate_tc (evaluate256_kernel) on CartPole-v1, greedy, N = 4,096 and 65,536 envs x 1 episode, for two 256-wide
policies: the initial one and one this script trains first (the configuration of test_h256_trainer_learns_and_keeps_ratio_one:
1,024 envs x 64 steps x 40 updates, seed 1).  Reports, per (policy, N):

  * useful env-steps/s = sum of episode lengths / kernel time (CUDA events around each launch, after a warm-up);
  * tile utilisation = sum of lengths / (128 x sum over CTAs of the CTA's longest env): the share of the row slots of the
    launch that stepped an env, i.e. the cost of ragged episode lengths inside a 128-env CTA, which steps in lock-step;
  * for comparison, drl_rollout with DRL_ROLLOUT_TENSOR_CORES at the same N and T = 500 with the same parameters, timed in
    the same run: the whole call (rollout256_kernel + the batched critic pass) with CUDA events, and the actor kernel alone
    (rollout256_kernel's device time from a torch.profiler pass over the same calls);

plus the GPU name and power limit.

    python profiles/tools/eval256_probe.py [--out FILE.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
import deep_rl_b200 as drl  # noqa: E402
from deep_rl_b200 import _lib  # noqa: E402
from deep_rl_b200.envs import VecEnv  # noqa: E402
from eval_probe import ENV_ID, EVAL_SEED, power_limit, time_ms  # noqa: E402

TILE = 128


def probe_eval(agent, N):
    env = VecEnv(ENV_ID, N, seed=EVAL_SEED, log_capacity=N)
    agent._ensure_packed()
    call = lambda: _lib.check(env.L.drl_evaluate_tc(C.byref(env.struct), C.byref(agent.net), agent.packed.data_ptr(), 1, 1,
                                                    C.byref(env.log.struct), None, _lib.stream_ptr()))
    ms, sd = time_ms(call, before=env.log.clear)
    res = drl.evaluate(agent, ENV_ID, N, episodes_per_env=1, greedy=True, seed=EVAL_SEED)     # the lengths of that launch
    total = res.lengths.sum(axis=1).astype(np.int64)
    per_cta_max = np.concatenate([total, np.zeros((-N) % TILE, np.int64)]).reshape(-1, TILE).max(axis=1)
    steps = int(total.sum())
    return {"N": N, "eval_ms": ms, "eval_ms_std": sd, "env_steps": steps, "mean_return": res.mean_return,
            "mean_length": res.mean_length, "max_length": int(total.max()), "cta_steps": int(per_cta_max.sum()),
            "useful_env_steps_per_s": steps / (ms * 1e-3), "tile_utilisation": steps / float(TILE * per_cta_max.sum())}


def probe_rollout(agent, N, T=500):
    env = VecEnv(ENV_ID, N, seed=EVAL_SEED, log_capacity=1 << 20)
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
                                     C.byref(env.log.struct), 1, _lib.stream_ptr()))
        k[0] += 1
    ms, sd = time_ms(call, before=env.log.clear)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            env.log.clear()
            call()
        torch.cuda.synchronize()
    actor = [e.time_range.elapsed_us() for e in prof.events()
             if e.device_type == torch.autograd.DeviceType.CUDA and "rollout256_kernel" in e.name]
    actor_ms = float(np.mean(actor)) * 1e-3 if actor else float("nan")     # profiler times are in microseconds
    return {"T": T, "rollout_tc_ms": ms, "rollout_tc_ms_std": sd, "rollout_tc_env_steps_per_s": N * T / (ms * 1e-3),
            "rollout256_kernel_ms": actor_ms, "rollout256_kernel_env_steps_per_s": N * T / (actor_ms * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    _lib.require_cuda()
    torch.cuda.set_device(0)
    gpu = {"name": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    print(f"GPU: {gpu['name']}, power limit {gpu['power_limit']}")
    init = drl.PPOTrainer(drl.PPOConfig(num_envs=64, hidden=256, seed=1)).agent
    cfg = drl.PPOConfig(num_envs=1024, num_steps=64, hidden=256, seed=1, total_timesteps=1024 * 64 * 40)
    tr = drl.PPOTrainer(cfg)
    for _ in range(cfg.num_updates()):
        tr.update()
    torch.cuda.synchronize()
    rows = []
    for name, agent in (("initial", init), ("trained", tr.agent)):
        for N in (4096, 65536):
            r = {"policy": name, **probe_eval(agent, N), **probe_rollout(agent, N)}
            r["eval_over_rollout_per_env_step"] = r["useful_env_steps_per_s"] / r["rollout_tc_env_steps_per_s"]
            rows.append(r)
            print(f"{name:8s} N={N:6d}: eval {r['eval_ms']:.3f} ms, mean length {r['mean_length']:.1f} (max {r['max_length']}), "
                  f"{r['useful_env_steps_per_s'] / 1e9:.3f} G useful env-steps/s, tile utilisation {r['tile_utilisation']:.3f} | "
                  f"tc rollout T=500 {r['rollout_tc_ms']:.3f} ms ({r['rollout_tc_env_steps_per_s'] / 1e9:.3f} G env-steps/s), "
                  f"actor kernel {r['rollout256_kernel_ms']:.3f} ms ({r['rollout256_kernel_env_steps_per_s'] / 1e9:.3f} G env-steps/s) "
                  f"| eval/rollout {r['eval_over_rollout_per_env_step']:.2f}")
    out = {"gpu": gpu, "rows": rows}
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
