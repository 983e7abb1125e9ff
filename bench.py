#!/usr/bin/env python
"""bench.py -- PPO env-steps/sec (rollout + update) on CartPole-v1, the metric BASELINE.json names.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...             # the reference's CPU implementation (port)

A "step" is one PPO update = one rollout of T env steps on every env, GAE, and 4 epochs x 4 minibatch
optimizer steps (deep_rl/ppo.py:105-192).  Workloads (BASELINE.json configs):
    N = 1 : C2  CartPole-v1, 4096 envs x 128 steps, 64-wide MLP
    N > 1 : C3  CartPole-v1, 65,536 envs per GPU x 128 steps, env-sharded, NCCL gradient all-reduce
`value` times the K updates with everything resident in HBM (per-update CUDA events, L2 flushed between
updates outside the events, max over ranks); `e2e` drives the same K updates through the public API with
a host round trip every update (metrics read back device->host, host-side logging logic).  Rank 0 prints
ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_FWD = {("CartPole-v1", 64): 17_792, ("Acrobot-v1", 64): 18_432, ("MountainCar-v0", 64): 17_408}   # forward FLOPs per sample (SURVEY.md 8d)
BYTES_PER_ENV_STEP = {"CartPole-v1": 195, "Acrobot-v1": 235, "MountainCar-v0": 155}
GRAD_BYTES_PER_SAMPLE = {"CartPole-v1": 37, "Acrobot-v1": 45, "MountainCar-v0": 29}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled in-process every millisecond (the timed
    region of the default run is only tens of milliseconds long, too short for `nvidia-smi -lms`), with nvidia-smi as the
    fallback when pynvml is not importable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake"}

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.nvml, self.handle, self.stop_flag = None, None, False
        self.sm, self.reasons, self.sm_max = [], set(), None

    def _nvml_sample(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        try:
            mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            for bit, name in self.BITS.items():
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _nvml_loop(self):
        while not self.stop_flag:
            try:
                self._nvml_sample()
            except Exception:
                break
            time.sleep(0.001)

    def start(self):
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                self.handle = torch.cuda._get_pynvml_handler(self.gpu)      # maps the CUDA ordinal to the NVML device
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nvml = pynvml
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return self
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            try:
                self._nvml_sample()          # the GPU is still draining the timed work when this is called
            except Exception:
                pass
            self.stop_flag = True
            self.t.join(timeout=2)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.sm_max,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the path on THIS arm's configuration.  /root/reference and gym do
# not exist on the GPU box, so it is the oracle port: the N-env port (oracle/ppo_vector_port.py: batched PyTorch CPU ops on
# all host threads + the C env/sampler/GAE) on the benchmarked workload, and -- for information -- the faithful single-env
# port of the script (oracle/ppo_port.py), one process per host core.
# ------------------------------------------------------------------------------------------------
def _port_worker(seed: int, updates: int, warm: int, q):
    import torch
    torch.set_num_threads(1)
    from oracle import ppo_port as pp
    cfg = pp.PortConfig(seed=seed)
    pp.run(cfg, max_updates=max(1, warm))
    t0 = time.perf_counter()
    tr = pp.run(cfg, max_updates=updates)
    q.put((tr.env_steps, time.perf_counter() - t0))


def _single_env_processes(updates: int, warm: int):
    """One faithful single-env port process per host core -> (env-steps/s summed, processes)."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    procs_n = max(1, min(cores, 64))
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_port_worker, args=(i + 1, updates, warm, q)) for i in range(procs_n)]
    for p in procs:
        p.start()
    res = [q.get() for _ in procs]
    for p in procs:
        p.join()
    return sum(r[0] for r in res) / max(r[1] for r in res), procs_n


def _workload_name(world: int, envs: int, T: int, env_id: str, hidden: int = 64) -> str:
    if world == 1 and envs == 4096 and T == 128 and env_id == "CartPole-v1" and hidden == 64:
        return "C2: PPO CartPole-v1, 4096 envs x 128 steps, 64-wide MLP, 1xB200"
    if envs == 65_536 and T == 128 and env_id == "CartPole-v1" and hidden == 64:
        return (f"C3: PPO CartPole-v1, 65,536 envs/GPU x 128 steps env-sharded across {world} B200, one gradient all-reduce per minibatch "
                f"(in-kernel over NVLink peer memory; NCCL with --grad-allreduce nccl)")
    return f"custom: {env_id}, {envs} envs/GPU x {T} steps, {hidden}-wide MLP"


def _vector_port_sample(env_id: str, envs: int, T: int, updates: int, warm: int, budget_s: float):
    """Times `updates` updates of the N-env CPU port on all host threads.  The env count is reduced (power of two) when the
    full workload would not fit the time budget.  Returns (env-steps/s, seconds per update, envs used, threads)."""
    import torch
    from oracle import ppo_vector_port as vp
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    probe_envs = min(envs, 512)
    probe = vp.VectorPort(env_id, probe_envs, T)
    probe.update()
    t0 = time.perf_counter()
    probe.update()
    per_env_update = (time.perf_counter() - t0) / probe_envs          # pessimistic: larger batches are more efficient
    total = updates + max(1, warm)
    use = envs
    while use > 256 and per_env_update * use * total > budget_s:
        use //= 2
    port = vp.VectorPort(env_id, use, T)
    for _ in range(max(1, warm)):
        port.update()
    secs = []
    for _ in range(updates):
        t0 = time.perf_counter()
        port.update()
        secs.append(time.perf_counter() - t0)
    return use * T * updates / sum(secs), sum(secs) / updates, use, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = args.gpus
    envs = args.envs_per_gpu if args.envs_per_gpu else (4096 if world == 1 else 65_536)
    T = args.num_steps
    t_all = time.perf_counter()
    value, per_update, used, threads = _vector_port_sample(args.env_id, envs, T, args.steps, args.warmup, budget_s=150.0)
    single, procs_n = _single_env_processes(min(args.steps, 5), 1)
    wall = time.perf_counter() - t_all
    B = used * T
    sample = (f"{args.steps} updates of the N-env CPU port (oracle/ppo_vector_port.py: batched PyTorch CPU ops + C env/sampler/GAE) with "
              f"{used} envs x {T} steps on {threads} host threads after {max(1, args.warmup)} warm-up update(s), {per_update:.2f} s per update"
              + ("" if used == envs else f"; bounded sample: {used} of the {envs} envs per GPU, same per-env-step work")
              + f"; for information, the faithful single-env port of ppo.py as {procs_n} independent processes: {single:.0f} env-steps/s; wall {wall:.0f}s")
    line = {
        "impl": "reference", "metric": "PPO env-steps/sec (rollout+update) CartPole-v1", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * per_update,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": _workload_name(world, envs, T, args.env_id) + ("" if used == envs else
                                                                              f" -- CPU arm bounded to {used} of the {envs} envs per GPU"),
                   "precision": "fp32 (PyTorch CPU)", "env_id": args.env_id,
                   "envs_per_gpu": used, "envs_per_gpu_of_the_gpu_arm": envs, "num_steps": T, "hidden": 64, "minibatch_size": (B + 3) // 4, "update_epochs": 4,
                   "optimizer_steps_per_update": 16, "parallelism": f"host CPU, {threads} threads (no GPU)"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample},
        "single_env_reference_shape": {"value": single, "unit": "env-steps/s", "processes": procs_n},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
GAE_BYTES = {"CartPole-v1": 17 + 21 + 32, "Acrobot-v1": 17 + 29 + 64, "MountainCar-v0": 17 + 21 + 32}   # planes + record packing
ROLLOUT_BYTES = {"CartPole-v1": 30, "Acrobot-v1": 38, "MountainCar-v0": 30}
ENV_STEP_BYTES = {"CartPole-v1": 62 + 32, "Acrobot-v1": 70 + 32, "MountainCar-v0": 62 + 32}             # SURVEY 8d + fp64 state r/w


def _timed_updates(tr, nu, steps, flush, dist, dev, instrument=False):
    """`steps` updates, each bracketed by CUDA events on the launching stream with the L2 flushed before it (outside the
    events).  instrument=False is the measured configuration (the trainer replays its captured CUDA graph on the tcgen05
    path); instrument=True additionally brackets every kernel call with CUDA events (eager launches: events cannot be read
    from inside a replayed graph) and feeds the per-kernel rooflines."""
    import torch
    tr.timing = bool(instrument)
    tr.phase_events.clear()
    launches0 = tr.kernel_launches
    evs = []
    dist.barrier()
    torch.cuda.synchronize()
    for _ in range(steps):
        flush.zero_()
        tr.env.log.clear()      # as a caller that reads the episode records after every update leaves it (the e2e leg does read them)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tr.update(nu)
        e1.record()
        evs.append((e0, e1))
    return evs, launches0


def _finish_timed(tr, evs, launches0, dist, dev):
    import torch
    torch.cuda.synchronize()
    dist.barrier()
    launches = tr.kernel_launches - launches0
    phases = tr.phase_ms()
    tr.timing = False
    local_ms = sum(a.elapsed_time(b) for a, b in evs)
    return dist.all_reduce_max(local_ms, dev), local_ms, phases, launches


def _grad_roofline(env_id, hidden, M, phases, total_ms, value, world, tc, peaks, traffic=None):
    F = flops_fwd(env_id, hidden)
    g = phases.get("minibatch_grad", {"mean_ms": float("nan"), "total_ms": 0.0})
    flops_per_launch = 3 * F * M
    achieved_tf = flops_per_launch / (g["mean_ms"] * 1e-3) / 1e12
    return {"kernel": ("ppo_grad_tc_kernel" if tc else "ppo_grad_kernel (+grad_reduce_kernel)") if hidden == 64 else
            "mlp256_kernel + dw2_gemm256_kernel + grad_reduce256_kernel (one drl_ppo_minibatch_grad call)",
            "bound": "tensor", "achieved": achieved_tf, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
            "frac": achieved_tf / peaks["bf16_tflops_sustained"], "traffic": traffic,
            "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
            "flops_per_launch": flops_per_launch, "launch_ms": g["mean_ms"],
            "hbm": {"achieved_gbs": GRAD_BYTES_PER_SAMPLE[env_id] * M / (g["mean_ms"] * 1e-3) / 1e9, "peak_gbs": peaks["hbm_gbs"]},
            "end_to_end": {"hbm_frac": value * BYTES_PER_ENV_STEP[env_id] / world / 1e9 / peaks["hbm_gbs"],
                           "tensor_frac": value * 13 * F / world / 1e12 / peaks["bf16_tflops_sustained"]},
            "share_of_step": g["total_ms"] / max(1e-9, total_ms)}


def flops_fwd(env_id, hidden):
    O, A = {"CartPole-v1": (4, 2), "Acrobot-v1": (6, 3), "MountainCar-v0": (2, 3)}[env_id]
    return 2 * (O * hidden + hidden * hidden + hidden * A) + 2 * (O * hidden + hidden * hidden + hidden)      # SURVEY.md 8d


def _hbm_rooflines(env_id, envs, T, E, phases, peaks):
    """HBM fractions of the bandwidth-bound kernels from the CUDA events recorded around each call inside the timed region
    (algorithmic bytes per sample: SURVEY.md 8d / DESIGN.md section 3)."""
    B = envs * T
    out = []
    for name, kernel, nbytes, per in (("gae", "gae_kernel", GAE_BYTES[env_id] * B, "update"),
                                      ("rollout", "rollout kernel", ROLLOUT_BYTES[env_id] * B, "update"),
                                      ("permutation", "permutation_kernel", 4 * B, "epoch"),
                                      ("adv_stats", "adv_stats_perm_kernel", 4 * B, "epoch")):
        ph = phases.get(name)
        if not ph or not ph["mean_ms"]:
            continue
        gbs = nbytes / (ph["mean_ms"] * 1e-3) / 1e9
        out.append({"kernel": kernel, "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": gbs / peaks["hbm_gbs"], "bytes_per_launch": nbytes, "launch_ms": ph["mean_ms"], "per": per})
    return out


def _env_step_roofline(env_id, dev, peaks, n_envs=1 << 22, steps=20):
    """One-off timing of the stand-alone env_step_kernel (drl_env_step: state in HBM) on n_envs environments."""
    import torch
    import deep_rl_b200 as drl
    env = drl.make(env_id, num_envs=n_envs, seed=3, device=dev, log_capacity=1 << 22)   # ~200 k episodes end per step
    env.reset()
    act = torch.randint(0, env.num_actions, (n_envs,), dtype=torch.int32, device=dev)
    import ctypes as C
    from deep_rl_b200 import _lib
    call = lambda k: _lib.check(env.L.drl_env_step(C.byref(env.struct), k, act.data_ptr(), env._obs.data_ptr(), env._rew.data_ptr(),
                                                   env._done.data_ptr(), C.byref(env.log.struct), _lib.stream_ptr()))
    for k in range(3):
        call(k)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        call(3 + k)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    nbytes = ENV_STEP_BYTES[env_id] * n_envs
    gbs = nbytes / (ms * 1e-3) / 1e9
    return {"kernel": "env_step_kernel", "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
            "bytes_per_launch": nbytes, "launch_ms": ms, "per": "env step", "envs": n_envs,
            "note": "stand-alone drl_env_step (fp64 state read + written in HBM every step; 4 Mi envs = 394 MB per launch, larger than "
                    "the L2; random actions); the training loop uses the fused rollout, whose state lives in registers"}


def _run_config(name, env_id, envs, T, hidden, steps, warm, rank, world, dev, flush, dist, peaks, precision="auto", grad_allreduce="peer"):
    """One extra workload (BASELINE.json configs C4 / C5 / C3-on-one-GPU) timed like the headline one."""
    import torch
    from deep_rl_b200 import PPOConfig, PPOTrainer
    total_updates = warm + steps + 4
    cfg = PPOConfig(env_id=env_id, num_envs=envs, num_steps=T, hidden=hidden, total_timesteps=envs * T * world * total_updates, seed=1,
                    update_precision=precision, grad_allreduce=grad_allreduce)
    tr = PPOTrainer(cfg, rank=rank, world=world, device=dev)
    nu = cfg.num_updates(world)
    for _ in range(warm):
        tr.update(nu)
    torch.cuda.synchronize()
    evs, l0 = _timed_updates(tr, nu, steps, flush, dist, dev)
    dev_ms, _, _, launches = _finish_timed(tr, evs, l0, dist, dev)
    evs, l0 = _timed_updates(tr, nu, max(2, steps // 2), flush, dist, dev, instrument=True)
    _, local_ms, phases, _ = _finish_timed(tr, evs, l0, dist, dev)
    inst_steps = max(2, steps // 2)
    m = tr.metrics(with_episode_log=False)
    value = envs * T * world * steps / (dev_ms * 1e-3)
    tc = tr.update_precision == "bf16"
    rec = {"name": name, "workload": f"{env_id}, {envs} envs/GPU x {T} steps, {hidden}-wide MLP, {world} GPU(s)", "value": value,
           "unit": "env-steps/s", "ms_per_step": dev_ms / steps, "steps": steps, "warmup": warm, "n_gpus": world,
           "dtype": "bf16" if tc else "f32", "episodes_dropped": m["episodes_dropped"],
           "roofline": _grad_roofline(env_id, hidden, cfg.minibatch_size * tr.mb_per_launch, phases, local_ms, value, world, tc, peaks),
           "minibatches_per_launch": tr.mb_per_launch,
           "rooflines": _hbm_rooflines(env_id, envs, T, cfg.update_epochs, phases, peaks),
           "phases_ms_per_update": {k: v["total_ms"] / inst_steps for k, v in phases.items()}, "gpu_launches": launches,
           "cuda_graph": tr._graph is not None}
    if hidden == 256:      # SURVEY 8d C5: gather-only split = one pass of the keyed-permutation gather over the packed records
        import ctypes as C
        from deep_rl_b200 import _lib
        net = C.byref(tr.net)
        B, M = cfg.batch_size, cfg.minibatch_size
        call = lambda: _lib.check(tr.L.drl_adv_stats(net, tr.records.data_ptr(), tr.idx[0].data_ptr(), B, M, tr.adv_stats[0].data_ptr(),
                                                    tr.workspace.data_ptr(), tr.ws_bytes, _lib.stream_ptr()))
        call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); call(); e1.record()
        torch.cuda.synchronize()
        gms = e0.elapsed_time(e1)
        rec["splits_ms_per_update"] = {"gae_only": rec["phases_ms_per_update"].get("gae"), "update_only": rec["phases_ms_per_update"].get("minibatch_grad", 0.0)
                                       + rec["phases_ms_per_update"].get("clip_adam", 0.0) + rec["phases_ms_per_update"].get("allreduce", 0.0),
                                       "rollout_only": rec["phases_ms_per_update"].get("rollout"),
                                       "gather_only_one_epoch": gms, "gather_only_gbs": 36.0 * B / (gms * 1e-3) / 1e9,
                                       "gather_note": "random 32-byte record + 4-byte index per sample (drl_adv_stats, gather form), one epoch"}
    if tr.peer is not None:
        tr.peer.close()
    del tr
    torch.cuda.empty_cache()
    return rec


def _params_checksum(tr):
    """64-bit checksum of the parameters and the second Adam moment (exact integer sums of the raw bit patterns)."""
    import torch
    a = tr.agent.flat_params.view(torch.int32).to(torch.int64)
    b = tr.exp_avg_sq.view(torch.int32).to(torch.int64)
    w = torch.arange(1, a.numel() + 1, device=a.device, dtype=torch.int64)
    return int(((a * w).sum() + 31 * (b * w).sum()).item())


DUMP_BYTES = 64 << 20


def _dump_outputs(tr, out_dir):
    """Writes what the last timed update left for its caller as out_dir/<name>.npy (float32, or float64 for the episode log):
    parameters, Adam moments, loss terms, gradient norm, the rollout planes, advantages / returns and the finished-episode log.
    When the [T+1][N] planes of all envs would pass half of DUMP_BYTES, they are kept for a fixed, seeded sample of env
    columns (`env_index`) and the episode log for those envs only.  Reads the episode log, which clears it."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    T1, N = tr.rewards.shape
    O = tr.env.obs_dim
    per_env = T1 * (O + 7) * 4                      # observations + 7 one-value planes, float32
    cols = np.arange(N)
    if N * per_env > DUMP_BYTES // 2:
        cols = np.sort(np.random.default_rng(0).choice(N, (DUMP_BYTES // 2) // per_env, replace=False))
    sel = torch.from_numpy(cols).to(tr.device)
    planes = {"observations": tr.observations[:, :, :O], "actions": tr.actions, "log_probs": tr.log_probs, "values": tr.values,
              "rewards": tr.rewards, "dones": tr.dones, "advantages": tr.advantages, "returns": tr.returns}
    out = {k: v.index_select(1, sel).float().cpu().numpy() for k, v in planes.items()}
    out.update({"params": tr.agent.flat_params, "exp_avg": tr.exp_avg, "exp_avg_sq": tr.exp_avg_sq, "loss_terms": tr.loss_terms,
                "grad_norm": tr.grad_norm})
    out = {k: (v.float().cpu().numpy() if torch.is_tensor(v) else v) for k, v in out.items()}
    out["env_index"] = cols.astype(np.float64)
    ep = tr.metrics(with_episode_log="arrays")["episode_log"]
    ep = {k: np.asarray(ep[k], dtype=np.float64) for k in ("step", "env", "ret", "len")}
    keep = np.isin(ep["env"], cols)
    order = np.lexsort((ep["env"][keep], ep["step"][keep]))       # the device appends in completion order: sort by (step, env)
    out.update({f"episode_{k}": v[keep][order] for k, v in ep.items()})
    total = sum(v.nbytes for v in out.values())
    assert total <= DUMP_BYTES, f"dump of {total} bytes exceeds {DUMP_BYTES}"
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v)
    return {"dir": out_dir, "arrays": sorted(out), "bytes": total, "envs": len(cols)}


def _multi_gpu_checks(tr, nu, dev, world):
    """Driver-visible multi-GPU correctness (GPUTEST runs on one GPU): (1) every rank holds bit-identical parameters and Adam
    moments after the timed updates; (2) two more updates from the same state through the in-kernel peer all-reduce and
    through NCCL (drl_ppo_minibatch_grad -> torch.distributed.all_reduce -> drl_clip_adam) agree to fp32 rounding."""
    import torch
    import torch.distributed as td
    out = {}
    torch.cuda.synchronize()
    mine = torch.tensor([_params_checksum(tr)], dtype=torch.int64, device=dev)
    allc = [torch.zeros_like(mine) for _ in range(world)]
    td.all_gather(allc, mine)
    out["ranks_bit_identical"] = bool(all(int(c.item()) == int(allc[0].item()) for c in allc))
    if tr.peer is not None:
        sd = tr.state_dict()
        tr.update(nu); tr.update(nu)
        torch.cuda.synchronize()
        p_peer = tr.agent.flat_params.clone()
        tr.load_state_dict(sd)
        peer, tr.peer = tr.peer, None                # same trainer, NCCL exchange between the kernels
        tr.update(nu); tr.update(nu)
        torch.cuda.synchronize()
        p_nccl = tr.agent.flat_params.clone()
        tr.peer = peer
        tr.load_state_dict(sd)
        diff = torch.tensor([float((p_peer - p_nccl).abs().max().item())], dtype=torch.float64, device=dev)
        td.all_reduce(diff, op=td.ReduceOp.MAX)
        out["peer_vs_nccl_max_abs"] = float(diff.item())
        out["peer_vs_nccl_param_scale"] = float(p_nccl.abs().max().item())
        c2 = torch.tensor([_params_checksum(tr)], dtype=torch.int64, device=dev)
        alld = [torch.zeros_like(c2) for _ in range(world)]
        td.all_gather(alld, c2)
        out["ranks_bit_identical"] = out["ranks_bit_identical"] and bool(all(int(c.item()) == int(alld[0].item()) for c in alld))
    return out


def run_b200(args):
    import torch
    from deep_rl_b200 import PPOConfig, PPOTrainer, dist

    rank, world = dist.init_from_env()
    if world != args.gpus and rank == 0:
        print(f"[bench] warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    peaks = load_peaks()

    envs = args.envs_per_gpu if args.envs_per_gpu else (4096 if world == 1 else 65_536)
    T = args.num_steps
    hidden = args.hidden
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    headline = envs in (4096, 65_536) and T == 128 and args.env_id == "CartPole-v1" and hidden == 64

    # ---- N > 1: the per-GPU workload on ONE GPU first (every rank runs its own world-1 trainer), so that the scaling
    # efficiency can be read off like for like in the same run ----
    single = None
    if world > 1 and not args.no_scaling_reference:
        single = _run_config("per-GPU workload on one GPU", args.env_id, envs, T, hidden, args.steps, max(3, args.warmup), 0, 1, dev, flush,
                             _SoloDist(), peaks, precision=args.precision)
        single_ms = dist.all_reduce_max(single["ms_per_step"], dev)
        single["ms_per_step_max_over_ranks"] = single_ms

    workload = _workload_name(world, envs, T, args.env_id, hidden)
    total_updates = args.warmup + 2 * args.steps + 16
    cfg = PPOConfig(env_id=args.env_id, num_envs=envs, num_steps=T, hidden=hidden, total_timesteps=envs * T * world * total_updates, seed=1,
                    update_precision=args.precision, grad_allreduce=args.grad_allreduce)
    tr = PPOTrainer(cfg, rank=rank, world=world, device=dev)
    nu = cfg.num_updates(world)
    n_mb = tr.n_mb
    tr_peer = tr.peer is not None
    tc = tr.update_precision == "bf16"

    for _ in range(max(3, args.warmup)):
        tr.update(nu)
    tr.metrics()
    torch.cuda.synchronize()

    # ---- device-resident timing: per-update CUDA events, L2 flushed between updates ----
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    evs, l0 = _timed_updates(tr, nu, args.steps, flush, dist, dev)
    clocks = sampler.stop() if sampler else None      # last sample while the queued updates are still running
    dev_ms, _, _, launches = _finish_timed(tr, evs, l0, dist, dev)
    dumped = _dump_outputs(tr, args.dump_outputs) if args.dump_outputs and rank == 0 else None
    steps_per_update = envs * T * world
    value = steps_per_update * args.steps / (dev_ms * 1e-3)
    graphed = tr._graph is not None
    # the same updates once more with CUDA events around every kernel call (eager launches): per-kernel rooflines
    evs, l0 = _timed_updates(tr, nu, args.steps, flush, dist, dev, instrument=True)
    inst_ms, local_ms, phases, _ = _finish_timed(tr, evs, l0, dist, dev)

    # ---- end to end through the public API: update + host round trip every update ----
    tr.metrics()
    dist.barrier()
    torch.cuda.synchronize()
    d2h, dropped = 0, 0
    t0 = time.perf_counter()
    pending = None
    for _ in range(args.steps):
        tr.update(nu)
        # D2H every update, like the reference's prints: loss terms + grad norm (36 B), episode count + sums (32 B) and the
        # (step, env, return, length) record of every finished episode (24 B each).  The read of update k is enqueued right
        # behind it and consumed on the host while update k+1 runs (metrics_async); every record is read inside this region.
        h = tr.metrics_async()
        d2h += h.d2h_bytes
        if pending is not None:
            m = pending.result()
            dropped += m["episodes_dropped"]
            _ = (m["mean_return"], m["loss"], len(m["episode_log"]["ret"]))
        pending = h
    m = pending.result()
    dropped += m["episodes_dropped"]
    _ = (m["mean_return"], m["loss"], len(m["episode_log"]["ret"]))
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_s = dist.all_reduce_max(e2e_s, dev)
    e2e_value = steps_per_update * args.steps / e2e_s
    assert dropped == 0, f"{dropped} finished episodes did not fit the episode log: e2e would not read what the reference prints"

    # ---- roofline of the dominant kernel + the bandwidth-bound kernels ----
    M = cfg.minibatch_size
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            kname = 'ppo_grad_tc_kernel' if tc else 'ppo_grad_kernel'
            traffic = tj.get(f"{kname}@{M}x{tr.mb_per_launch}") if tr.mb_per_launch > 1 else tj.get(f"{kname}@{M}")
        except Exception:
            traffic = None
    mb_per_launch = tr.mb_per_launch
    roofline = _grad_roofline(args.env_id, hidden, M * mb_per_launch, phases, local_ms, value, world, tc, peaks, traffic)
    roofline.update({
        "minibatches_per_launch": mb_per_launch,
        "kernel_launch_includes": (f"{mb_per_launch} consecutive minibatch steps (one epoch), each = gradient + fold of the per-SM partials + clip + Adam, "
                                   "in ONE cooperative launch") if tc else "gradient kernel only",
        "limiter": ("the shared-memory data pipe: operand fetch of the small-N tcgen05 GEMMs (35 % of its peak at C3) + the compute warps' "
                    "bf16 tile stores and broadcast weight loads (53 %), ncu l1tex__data_pipe_{tc,lsu}_wavefronts_mem_shared in "
                    "profiles/r2_grad_tc_c3_full.txt; then issue slots (57 %) and the XU pipe (tanh + bf16 packs, 35 %); at this "
                    "minibatch size a third of the launch is the per-minibatch tail (fold, three grid barriers, clip, Adam, weight reload) "
                    "-- DESIGN.md section 3" if tc else "FP32 FMA issue"),
        "note": ("tcgen05 path: every GEMM of the two MLPs (layers 1-2 forward, dh1, all weight-gradient reductions) runs on the "
                 "tensor pipe (bf16 operands, fp32 TMEM accumulators); FLOPs counted are the algorithmic 3F per sample; launch_ms is the "
                 "whole minibatch-step call (the gradient kernel carries the fold + clip + Adam tail)" if tc else
                 "FP32 CUDA-core (FFMA) path; the tensor-pipe peak is the roof the tcgen05 path is held to")})
    rooflines = _hbm_rooflines(args.env_id, envs, T, cfg.update_epochs, phases, peaks)

    multi = _multi_gpu_checks(tr, nu, dev, world) if world > 1 else None
    if tr_peer:
        tr.peer.close()
    del tr
    torch.cuda.empty_cache()

    # ---- the other BASELINE.json configurations, timed the same way (the driver only runs the default command line) ----
    extra, fp32_path, scaling_ref = [], None, None
    if headline and not args.no_extra_configs:
        xs = max(3, min(args.steps, 10))
        if world == 1:
            rooflines.append(_env_step_roofline(args.env_id, dev, peaks))
            scaling_ref = _run_config("C3 on one GPU (the per-GPU work of the N>1 runs)", "CartPole-v1", 65_536, 128, 64, args.steps, 3,
                                      0, 1, dev, flush, dist, peaks)
            extra.append(_run_config("C4: PPO Acrobot-v1, 16,384 envs x 256 steps, 1xB200", "Acrobot-v1", 16_384, 256, 64, xs, 3, 0, 1, dev,
                                     flush, dist, peaks))
            f32 = _run_config("strict fp32 path (CUDA cores) on the headline workload", args.env_id, envs, T, 64, 3, 3, 0, 1, dev, flush, dist,
                              peaks, precision="fp32")
            fp32_path = {"value": f32["value"], "unit": "env-steps/s", "ms_per_step": f32["ms_per_step"], "workload": workload}
            if args.hidden256:
                extra.append(_run_config("C5: synthetic stress, 1M envs x 256 steps, 256-wide MLP, 1xB200", "CartPole-v1", 1 << 20, 256, 256,
                                         2, 1, 0, 1, dev, flush, dist, peaks, grad_allreduce="nccl"))
        else:
            per = 16_384 // world
            extra.append(_run_config(f"C4 strong scaling: Acrobot-v1, 16,384 envs total ({per}/GPU) x 256 steps", "Acrobot-v1", per, 256, 64, xs, 3,
                                     rank, world, dev, flush, dist, peaks))
            extra.append(_run_config("C4 weak scaling: Acrobot-v1, 16,384 envs/GPU x 256 steps", "Acrobot-v1", 16_384, 256, 64, xs, 3,
                                     rank, world, dev, flush, dist, peaks))
            if args.hidden256:
                extra.append(_run_config(f"C5: synthetic stress, 1M envs total ({(1 << 20) // world}/GPU) x 256 steps, 256-wide MLP",
                                         "CartPole-v1", (1 << 20) // world, 256, 256, 3, 1, rank, world, dev, flush, dist, peaks, grad_allreduce="nccl"))

    if rank != 0:
        dist.shutdown()
        return

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        # the same workload on the host cores: N-env CPU port on all threads (bounded to ~cpu_seconds), plus the faithful
        # single-env port of the script on one core for information
        from oracle import ppo_port as pp
        import torch as _t
        v, per_update, used, threads = _vector_port_sample(args.env_id, envs, T, 2, 1, budget_s=args.cpu_seconds)
        _t.set_num_threads(1)
        r = pp.time_port(min(5.0, args.cpu_seconds))
        cpu_baseline = {"value": v, "unit": "env-steps/s", "cores": threads, "kind": "port",
                        "sample": f"2 updates of the N-env CPU port (oracle/ppo_vector_port.py) with {used} envs x {T} steps on {threads} host "
                                  f"threads, {per_update:.2f} s per update" + ("" if used == envs else f" (bounded sample of the {envs} envs)")
                                  + f"; the faithful single-env port of ppo.py on one core: {r['steps_per_s']:.0f} env-steps/s "
                                  f"({r['updates']} updates x 128 env-steps)",
                        "single_env_one_core": r["steps_per_s"]}

    line = {
        "metric": "PPO env-steps/sec (rollout+update) CartPole-v1", "value": value, "unit": "env-steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if tc else "f32", "data": "synthetic",
        "config": {"workload": workload, "precision": ("rollout + update GEMMs bf16 x bf16 -> fp32 on tcgen05; env fp64; GAE, loss, Adam fp32" if tc else "fp32"),
                   "env_id": args.env_id, "envs_per_gpu": envs, "num_steps": T, "hidden": hidden,
                   "minibatch_size": M, "update_epochs": cfg.update_epochs, "optimizer_steps_per_update": cfg.update_epochs * n_mb,
                   "parallelism": f"env-sharded x{world}" + ("" if world == 1 else (", gradient all-reduce inside the gradient kernel over NVLink peer memory"
                                                                                  if tr_peer else ", NCCL gradient all-reduce per minibatch")), "l2": "flushed between updates (256 MiB memset outside the timed events); "
                   "every update regenerates its own rollout data",
                   "launch": ("one captured CUDA graph per update (26 kernel nodes) + one drl_ctrl_set launch" if graphed else "eager launches")},
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": d2h / args.steps,
                "episodes_dropped": dropped,
                "note": "public API PPOTrainer.update() + metrics_async().result(): every update is followed by a device->host read of "
                        "its loss terms, gradient norm, episode statistics and per-episode records (what the reference prints) into "
                        "pinned memory; the host consumes update k's read while update k+1 runs; wall clock around the whole loop; "
                        "the environments live on the device, so the only per-update host inputs are kernel arguments (no tensor H2D)"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "rooflines": rooflines, "cpu_baseline": cpu_baseline,
        "phases_ms_per_update": {k: v["total_ms"] / args.steps for k, v in phases.items()},
        "cuda_graph": graphed, "ms_per_step_eager_instrumented": inst_ms / args.steps,
        "scaling_reference": scaling_ref, "extra_configs": extra, "fp32_path": fp32_path, "dumped_outputs": dumped,
    }
    if world > 1:
        line.update(multi)
        if single is not None:
            line["single_gpu_same_workload"] = {"value": single["value"], "ms_per_step": single["ms_per_step_max_over_ranks"],
                                                "steps": single["steps"], "unit": "env-steps/s"}
            line["scaling_efficiency_like_for_like"] = single["ms_per_step_max_over_ranks"] / (dev_ms / args.steps)
    print(json.dumps(line), flush=True)
    dist.shutdown()


class _SoloDist:
    """dist-shaped no-ops for a world-1 trainer that runs inside a multi-rank job (every rank times its own copy)."""
    @staticmethod
    def barrier():
        pass

    @staticmethod
    def all_reduce_max(x, dev):
        return x


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=0)
    ap.add_argument("--num-steps", type=int, default=128)
    ap.add_argument("--env-id", default="CartPole-v1")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-scaling-reference", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip C3-on-one-GPU / C4 / C5 / fp32 / env-step records")
    ap.add_argument("--hidden", type=int, default=64)
    ap.add_argument("--no-hidden256", dest="hidden256", action="store_false", default=True,
                    help="skip the C5 (1M envs x 256 steps, 256-wide MLP) record of extra_configs")
    ap.add_argument("--grad-allreduce", default="peer", choices=["peer", "nccl"],
                    help="multi-GPU gradient exchange: in-kernel NVLink peer-memory all-reduce, or NCCL between kernels")
    ap.add_argument("--precision", default="auto", choices=["auto", "bf16", "fp32"],
                    help="update GEMMs: bf16 = tcgen05 tensor cores (bf16 operands, fp32 accumulate), fp32 = CUDA cores")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed updates, write what the last one computed (parameters, Adam moments, loss terms, rollout "
                         "planes, advantages, returns, finished episodes) as DIR/<name>.npy, at most 64 MiB; rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
