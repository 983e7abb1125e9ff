"""PPO rollout-and-update loop on the GPU -- the B200 counterpart of the script deep_rl/ppo.py.

Hyper-parameter names and defaults are the reference's (ppo.py:62-76,83); `num_envs` and `hidden`
are the two additions (SURVEY.md D1/D5).  The loop keeps the shape of ppo.py:105-192:

    for update in range(num_updates):
        lr anneal                          ppo.py:107-108   (host scalar)
        rollout of num_steps               ppo.py:110-141   drl_rollout        (1 launch)
        GAE + returns (+ record packing)   ppo.py:144-151   drl_gae            (1 launch)
        permutations of all epochs         ppo.py:155       drl_permutation      (side stream, during the rollout)
        advantage statistics per epoch     ppo.py:169       drl_adv_stats_perm   (side stream, one epoch ahead)
        for epoch in range(update_epochs):
            for each minibatch:            ppo.py:156-192   drl_ppo_minibatch_update[_dist]: gather + loss + backward + fold +
                                                            [in-kernel NVLink all-reduce] + clip + Adam, ONE cooperative launch
                                           (fp32 / NCCL variant: drl_ppo_minibatch_grad, NCCL all-reduce, drl_clip_adam)

Precision: `update_precision="auto"` runs the tcgen05 (bf16 operands, fp32 accumulate) kernels from 2,048 envs per rank and
the strict fp32 CUDA-core kernels below (the reference shape, N = 1, is fp32 end to end); the rollout always follows the
update so that the log-probs and values it records are re-evaluated with the same numerics (ratio = 1, approx_kl = 0 at
the first minibatch of an update).

Run as a script:  python -m deep_rl_b200.ppo [--num-envs N] [--total-timesteps K] ...
"""
from __future__ import annotations

import argparse
import contextlib
import ctypes as C
from dataclasses import dataclass
from typing import Dict, Optional

import torch

from . import _lib, dist as _dist
from .agent import ActorCritic
from .envs import VecEnv
from .evaluate import EvalResult, evaluate as _evaluate

EVAL_SEED_OFFSET = 0x9E3779B97F4A7C15     # default evaluation key = (cfg.seed + this) mod 2^64: never a training key


def eval_seed(seed: int) -> int:
    """The default evaluation key of a trainer keyed `seed`."""
    return (int(seed) + EVAL_SEED_OFFSET) % (1 << 64)


@dataclass
class PPOConfig:
    env_id: str = "CartPole-v1"
    total_timesteps: int = 20_000
    num_steps: int = 128
    update_epochs: int = 4
    gamma: float = 0.99
    gae_lambda: float = 0.95
    learning_rate: float = 2.5e-4
    clip_coef: float = 0.2
    ent_coef: float = 0.01
    vf_coef: float = 0.5
    max_grad_norm: float = 0.5
    seed: int = 1
    # additions over the reference script
    num_envs: int = 1            # environments per rank
    hidden: int = 64
    num_minibatches: int = 4     # reference: minibatch_size = num_steps // 4
    anneal_lr: bool = True
    rollout_precision: str = "auto"  # "bf16": tcgen05 rollout (32-128 envs per CTA); "fp32": CUDA-core rollout; "auto": the
                                     # precision of the update (same numerics when log-probs / values are re-evaluated)
    overlap_streams: bool = True     # permutations (during the rollout) and advantage statistics of later epochs (during the
                                     # minibatch steps of earlier ones) run on a second CUDA stream
    global_adv_stats: bool = False   # multi-GPU: normalise advantages with the statistics of the GLOBAL minibatch (one extra
                                     # all-reduce of 3 numbers per minibatch, once per update) instead of per-rank ones
    grad_allreduce: str = "peer"     # multi-GPU gradient exchange: "peer" = one-shot all-reduce over NVLink peer memory inside
                                     # the gradient kernel (bf16 update only), "nccl" = NCCL all-reduce between kernels
    update_precision: str = "auto"   # "bf16": tcgen05 tensor-core update (bf16 operands, fp32 accumulate); "fp32": CUDA-core
                                     # update; "auto": bf16 from 2048 envs per rank (minibatches of >= 64k samples), else fp32
    debug_logits: bool = False       # record the logits every action was sampled from ([T][N][A] plane, parity tests)
    steps_per_launch: int = 0        # tcgen05 fused step: minibatches per kernel launch (0 = auto: a whole epoch when its minibatches
                                     # are equally sized, at most 8 and of at most 2^19 samples -- where the per-launch fixed costs
                                     # matter -- else 1)
    cuda_graph: bool = True          # tcgen05 path: capture the launches of one update in a CUDA graph (counters live in a
                                     # device-resident drl_ctrl_t) and replay it; results are bit-identical to the eager path
    eval_every: int = 0              # train(): greedy evaluation after every eval_every-th update (0 = off)
    eval_episodes: int = 1024        # envs of that evaluation, one fresh episode each

    def resolved_update_precision(self) -> str:
        if self.update_precision == "auto":
            return "bf16" if (self.num_envs >= 2048 or self.hidden != 64) else "fp32"
        return self.update_precision

    def resolved_rollout_precision(self) -> str:
        return self.resolved_update_precision() if self.rollout_precision == "auto" else self.rollout_precision

    @property
    def batch_size(self) -> int:             # samples per rank per update
        return self.num_envs * self.num_steps

    @property
    def minibatch_size(self) -> int:
        return self.batch_size // self.num_minibatches

    def num_updates(self, world: int = 1) -> int:
        return self.total_timesteps // (self.batch_size * world)


class _Phase:
    """CUDA-event bracket around one phase of the update (only when trainer.timing is on)."""

    def __init__(self, tr: "PPOTrainer", name: str):
        self.tr, self.name = tr, name

    def __enter__(self):
        if self.tr.timing:
            self.t0 = torch.cuda.Event(enable_timing=True)
            self.t1 = torch.cuda.Event(enable_timing=True)
            self.t0.record()
        return self

    def __exit__(self, *exc):
        if self.tr.timing:
            self.t1.record()
            self.tr.phase_events.setdefault(self.name, []).append((self.t0, self.t1))
        return False


class MetricsRead:
    """Handle of PPOTrainer.metrics_async()."""

    def __init__(self, tr: "PPOTrainer", host_terms: torch.Tensor, log_read):
        self.tr, self.host_terms, self.log_read = tr, host_terms, log_read
        self.d2h_bytes = 36 + tr.env.log.last_d2h_bytes

    def result(self) -> Dict[str, object]:
        n, sum_ret, sum_len, e, lost = self.log_read.result()      # waits for the copies (both precede the event)
        lt = self.host_terms.tolist()
        return {"loss": lt[0], "pg_loss": lt[1], "v_loss": lt[2], "entropy": lt[3], "approx_kl": lt[4], "clipfrac": lt[5],
                "grad_norm": lt[8], "episodes": n, "episodes_dropped": max(0, n - self.tr.env.log.cap) + max(0, min(n, self.tr.env.log.cap) - len(e)),
                "mean_return": (sum_ret / n) if n else float("nan"), "mean_length": (sum_len / n) if n else float("nan"),
                "episode_log": {"step": e["step"], "env": e["env"], "ret": e["ret"], "len": e["len"]}}


class PPOTrainer:
    """Owns the device buffers of one rank and issues the kernels of one update."""

    def __init__(self, cfg: PPOConfig, rank: int = 0, world: int = 1, device: Optional[torch.device] = None,
                 agent: Optional[ActorCritic] = None):
        _lib.require_cuda()
        self.cfg, self.rank, self.world = cfg, int(rank), int(world)
        self.L = _lib.lib()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        N, T = cfg.num_envs, cfg.num_steps
        self.env = VecEnv(cfg.env_id, num_envs=N, seed=cfg.seed, env_gid0=self.rank * N, device=self.device)
        if agent is None:
            torch.manual_seed(cfg.seed)      # same init draws on every rank (ppo.py:86,89)
            agent = ActorCritic(self.env, hidden=cfg.hidden, device=self.device, sample_seed=cfg.seed)
        self.agent = agent
        self.net = agent.net
        OP = self.env.obs_stride
        dev = self.device
        f32, u8 = torch.float32, torch.uint8
        # storage, ppo.py:93-98, SoA [T+1][N]
        self.observations = torch.zeros((T + 1, N, OP), dtype=f32, device=dev)
        self.actions = torch.zeros((T + 1, N), dtype=u8, device=dev)
        self.log_probs = torch.zeros((T + 1, N), dtype=f32, device=dev)
        self.values = torch.zeros((T + 1, N), dtype=f32, device=dev)
        self.rewards = torch.zeros((T + 1, N), dtype=f32, device=dev)
        self.dones = torch.zeros((T + 1, N), dtype=u8, device=dev)
        self.advantages = torch.zeros((T + 1, N), dtype=f32, device=dev)
        self.returns = torch.zeros((T + 1, N), dtype=f32, device=dev)
        self.logits = torch.zeros((T, N, self.env.num_actions), dtype=f32, device=dev) if cfg.debug_logits else None
        self.buf = _lib.RolloutBufT(self.observations.data_ptr(), self.actions.data_ptr(), self.log_probs.data_ptr(),
                                    self.values.data_ptr(), self.rewards.data_ptr(), self.dones.data_ptr(),
                                    _lib.ptr(self.logits))
        B = cfg.batch_size
        self.RW = self.L.drl_record_width(C.byref(self.net))
        self.records = torch.zeros((B, self.RW), dtype=f32, device=dev)
        self.n_mb = (B + cfg.minibatch_size - 1) // cfg.minibatch_size
        # one index array and one statistics block per epoch: they are produced ahead of the epoch that consumes them
        self.idx = torch.zeros((cfg.update_epochs, B), dtype=torch.int32, device=dev)
        self.adv_stats = torch.zeros((cfg.update_epochs, self.n_mb, 2), dtype=f32, device=dev)
        self.side = torch.cuda.Stream(device=dev) if cfg.overlap_streams else None
        self._ev_gae = torch.cuda.Event()
        self._ev_stats = [torch.cuda.Event() for _ in range(cfg.update_epochs)]
        self._perms_scheduled = False
        self._merge_stats = bool(cfg.global_adv_stats and self.world > 1 and torch.distributed.is_available()
                                 and torch.distributed.is_initialized())
        M_ = cfg.minibatch_size
        self._mb_counts = torch.tensor([[min(M_, B - k * M_) for k in range(self.n_mb)]] * cfg.update_epochs, dtype=torch.float64, device=dev)
        P = agent.flat_params.numel()
        self.grad = torch.zeros(P, dtype=f32, device=dev)
        self.exp_avg = torch.zeros(P, dtype=f32, device=dev)
        self.exp_avg_sq = torch.zeros(P, dtype=f32, device=dev)
        n_rows = cfg.update_epochs * self.n_mb
        self._terms_and_norm = torch.zeros(n_rows * 8 + 1, dtype=f32, device=dev)
        self.loss_terms = self._terms_and_norm[: n_rows * 8].view(n_rows, 8)
        self.grad_norm = self._terms_and_norm[n_rows * 8:]
        self._h_terms = torch.zeros(9, dtype=f32).pin_memory()
        self._h_terms_ring = [torch.zeros(9, dtype=f32).pin_memory() for _ in range(2)]
        self._h_flip = 0
        self.ws_bytes = int(self.L.drl_workspace_bytes(C.byref(self.net)))
        self.workspace = torch.zeros(self.ws_bytes, dtype=u8, device=dev)
        self.coef = _lib.PpoCoefT(cfg.clip_coef, cfg.ent_coef, cfg.vf_coef)
        if cfg.hidden != 64 and "fp32" in (cfg.resolved_update_precision(), cfg.resolved_rollout_precision()):
            raise ValueError(f"hidden={cfg.hidden} exists on the tensor-core (bf16) path only")
        if cfg.update_precision not in ("auto", "bf16", "fp32"):
            raise ValueError(f"update_precision={cfg.update_precision!r}")
        if cfg.rollout_precision not in ("auto", "bf16", "fp32"):
            raise ValueError(f"rollout_precision={cfg.rollout_precision!r}")
        self.update_precision = cfg.resolved_update_precision()
        self.rollout_precision = cfg.resolved_rollout_precision()
        self.grad_flags = 1 if self.update_precision == "bf16" else 0
        self.rollout_flags = 1 if self.rollout_precision == "bf16" else 0
        self._ev_out = torch.zeros(1, dtype=f32, device=dev)
        self.adam_step = 0
        self.update_idx = 0
        self.global_step = 0       # env steps taken on this rank's envs x world (reference counter at N=1)
        self.env.reset()           # ppo.py:101
        self.kernel_launches = 0
        self.fused_step = cfg.hidden == 64     # single GPU: fold + clip + Adam inside the gradient kernel's launch (64-wide nets)
        self.peer = None
        if (self.world > 1 and cfg.grad_allreduce == "peer" and self.grad_flags == 1 and cfg.hidden == 64
                and torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.peer = _dist.PeerComm(self.net, self.rank, self.world, dev)
        # minibatches per launch of the fused tensor-core step (a whole epoch when possible)
        equal = B % cfg.minibatch_size == 0
        self.mb_per_launch = 1
        if self.grad_flags == 1 and cfg.hidden == 64 and equal and (self.world == 1 or self.peer is not None):
            want = cfg.steps_per_launch if cfg.steps_per_launch > 0 else (self.n_mb if cfg.minibatch_size <= (1 << 19) else 1)
            self.mb_per_launch = max(1, min(want, self.n_mb, 8))
            while self.n_mb % self.mb_per_launch:
                self.mb_per_launch -= 1
        self.timing = False        # record CUDA events around each phase (bench.py)
        self.phase_events: Dict[str, list] = {}
        # graph-replayable update: device-resident counters + one captured graph (tcgen05 fused step only)
        self.ctrl = torch.zeros(C.sizeof(_lib.CtrlT), dtype=u8, device=dev)
        self._graph = None
        self._graph_launches = 0
        self._graph_warm = 0
        n_opt = cfg.update_epochs * self.n_mb
        self.graph_ok = bool(cfg.cuda_graph and self.grad_flags == 1 and cfg.hidden == 64 and self.n_mb <= 8 and n_opt <= 64 and not self._merge_stats
                             and (self.world == 1 or self.peer is not None))

    def phase_ms(self) -> Dict[str, Dict[str, float]]:
        """Per-phase device time from the recorded events: {phase: {calls, total_ms, mean_ms}} (synchronises)."""
        torch.cuda.synchronize()
        out = {}
        for name, evs in self.phase_events.items():
            ms = [a.elapsed_time(b) for a, b in evs]
            out[name] = {"calls": len(ms), "total_ms": float(sum(ms)), "mean_ms": float(sum(ms) / max(1, len(ms)))}
        return out

    # ------------------------------------------------------------------------------------------
    def learning_rate(self, update: int, num_updates: int) -> float:
        if not self.cfg.anneal_lr:
            return self.cfg.learning_rate
        return (1.0 - update / num_updates) * self.cfg.learning_rate      # ppo.py:107-108

    def rollout(self, ctl: bool = False) -> None:
        """ppo.py:110-141 for all envs: one kernel launch."""
        cfg = self.cfg
        with _Phase(self, "rollout"):
            if ctl:
                _lib.check(self.L.drl_rollout_ctl(C.byref(self.env.struct), C.byref(self.net), self.agent.packed.data_ptr(),
                                                  cfg.num_steps, self.ctrl.data_ptr(), C.byref(self.buf),
                                                  C.byref(self.env.log.struct), self.rollout_flags, _lib.stream_ptr()))
            else:
                _lib.check(self.L.drl_rollout(C.byref(self.env.struct), C.byref(self.net), self.agent.packed.data_ptr(),
                                              cfg.num_steps, self.env.step_count, C.byref(self.buf),
                                              C.byref(self.env.log.struct), self.rollout_flags, _lib.stream_ptr()))
        self.env.step_count += cfg.num_steps
        self.global_step += cfg.num_steps * cfg.num_envs * self.world
        self.kernel_launches += 1

    def compute_gae(self) -> None:
        """ppo.py:144-151 (+ packs the per-sample records the update gathers)."""
        cfg = self.cfg
        with _Phase(self, "gae"):
            _lib.check(self.L.drl_gae(C.byref(self.buf), C.byref(self.net), cfg.num_steps, cfg.num_envs, cfg.gamma,
                                      cfg.gae_lambda, self.advantages.data_ptr(), self.returns.data_ptr(),
                                      self.records.data_ptr(), _lib.stream_ptr()))
        self.kernel_launches += 1

    def _side(self):
        return torch.cuda.stream(self.side) if self.side is not None else contextlib.nullcontext()

    def schedule_permutations(self, ctl: bool = False) -> None:
        """ppo.py:155 for every epoch of the coming update.  The keyed permutation depends on counters only, so with
        `overlap_streams` it runs on the side stream while the rollout kernel runs on the main one."""
        cfg = self.cfg
        if self.side is not None:
            self.side.wait_stream(torch.cuda.current_stream())     # the previous update has finished reading idx / adv_stats
        with self._side():
            st = _lib.stream_ptr()
            for epoch in range(cfg.update_epochs):
                epoch_ctr = self.update_idx * cfg.update_epochs + epoch
                with _Phase(self, "permutation"):
                    if ctl:
                        _lib.check(self.L.drl_permutation_ctl(self.idx[epoch].data_ptr(), cfg.batch_size, cfg.seed, self.ctrl.data_ptr(),
                                                              epoch, self.rank, st))
                    else:
                        _lib.check(self.L.drl_permutation(self.idx[epoch].data_ptr(), cfg.batch_size, cfg.seed, epoch_ctr, self.rank, st))
        self.kernel_launches += cfg.update_epochs
        self._perms_scheduled = True

    def schedule_adv_stats(self, ctl: bool = False) -> None:
        """ppo.py:169 statistics of every (epoch, minibatch): needs the advantages, i.e. runs after GAE; epoch e + 1's pass
        overlaps epoch e's minibatch steps on the side stream."""
        cfg = self.cfg
        B, M = cfg.batch_size, cfg.minibatch_size
        net = C.byref(self.net)
        if self.side is not None:
            self._ev_gae.record()
            self.side.wait_event(self._ev_gae)
        with self._side():
            st = _lib.stream_ptr()
            for epoch in range(cfg.update_epochs):
                epoch_ctr = self.update_idx * cfg.update_epochs + epoch
                with _Phase(self, "adv_stats"):
                    if ctl:
                        _lib.check(self.L.drl_adv_stats_perm_ctl(net, self.advantages.data_ptr(), B, M, cfg.seed, self.ctrl.data_ptr(), epoch,
                                                                 self.rank, self.adv_stats[epoch].data_ptr(), self.workspace.data_ptr(),
                                                                 self.ws_bytes, st))
                    elif self.n_mb <= 8:   # no gather: natural-order pass over the advantage plane + inverse permutation
                        _lib.check(self.L.drl_adv_stats_perm(net, self.advantages.data_ptr(), B, M, cfg.seed, epoch_ctr, self.rank,
                                                             self.adv_stats[epoch].data_ptr(), self.workspace.data_ptr(),
                                                             self.ws_bytes, st))
                    else:
                        _lib.check(self.L.drl_adv_stats(net, self.records.data_ptr(), self.idx[epoch].data_ptr(), B, M,
                                                        self.adv_stats[epoch].data_ptr(), self.workspace.data_ptr(),
                                                        self.ws_bytes, st))
                if self.side is not None and not self._merge_stats:
                    self._ev_stats[epoch].record()
            if self._merge_stats:     # all epochs' statistics first, then one exchange for the whole update
                _dist.merge_minibatch_stats(self.adv_stats, self._mb_counts)
                if self.side is not None:
                    for ev in self._ev_stats:
                        ev.record()
        self.kernel_launches += cfg.update_epochs

    def optimize(self, lr: float, ctl: bool = False) -> None:
        """ppo.py:154-192."""
        cfg = self.cfg
        B, M = cfg.batch_size, cfg.minibatch_size
        net = C.byref(self.net)
        if self.world > 1 and self.peer is None and not (torch.distributed.is_available() and torch.distributed.is_initialized()):
            raise _lib.DrlError("world > 1 needs an initialised torch.distributed process group for the gradient all-reduce "
                                "(deep_rl_b200.dist.init_from_env); without it the gradient would only be scaled by 1/world")
        if not self._perms_scheduled:
            self.schedule_permutations(ctl)
        self._perms_scheduled = False
        self.schedule_adv_stats(ctl)
        st = _lib.stream_ptr()
        for epoch in range(cfg.update_epochs):
            if self.side is not None:
                torch.cuda.current_stream().wait_event(self._ev_stats[epoch])
            idx_ptr = self.idx[epoch].data_ptr()
            stats_ptr = self.adv_stats[epoch].data_ptr()
            for k in range(0, self.n_mb, self.mb_per_launch):
                start = k * M
                count = min(M, B - start)
                row = epoch * self.n_mb + k
                ns = self.mb_per_launch     # minibatches of this launch (equally sized when > 1)
                if ctl:     # counters from the device control block: the launch is identical from update to update
                    self.adam_step += ns
                    if self.peer is not None:
                        for _ in range(ns):
                            self.peer.next()
                    with _Phase(self, "minibatch_grad"):
                        _lib.check(self.L.drl_ppo_minibatch_update_ctl(
                            net, self.agent.packed.data_ptr(), self.records.data_ptr(), idx_ptr, start, count,
                            stats_ptr + 8 * k, C.byref(self.coef), self.agent.flat_params.data_ptr(),
                            self.grad.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), self.ctrl.data_ptr(), row,
                            0.9, 0.999, 1e-5, cfg.max_grad_norm, self.loss_terms.data_ptr() + 32 * row,
                            self.grad_norm.data_ptr(), self.workspace.data_ptr(), self.ws_bytes, self.grad_flags,
                            C.byref(self.peer.struct) if self.peer is not None else None, ns, st))
                    self.kernel_launches += 1
                    continue
                if self.peer is not None:
                    first_step = self.adam_step + 1
                    self.adam_step += ns
                    comm = self.peer.next()          # sequence number of the launch's first minibatch step
                    for _ in range(ns - 1):
                        self.peer.next()
                    comm.seq = self.peer.seq - ns + 1
                    with _Phase(self, "minibatch_grad"):    # gradient + fold + NVLink all-reduce + clip + Adam: one launch
                        _lib.check(self.L.drl_ppo_minibatch_update_dist(
                            net, self.agent.packed.data_ptr(), self.records.data_ptr(), idx_ptr, start, count,
                            stats_ptr + 8 * k, C.byref(self.coef), self.agent.flat_params.data_ptr(),
                            self.grad.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), first_step, lr,
                            0.9, 0.999, 1e-5, cfg.max_grad_norm, self.loss_terms.data_ptr() + 32 * row,
                            self.grad_norm.data_ptr(), self.workspace.data_ptr(), self.ws_bytes, self.grad_flags,
                            C.byref(comm), ns, st))
                    comm.seq = self.peer.seq
                    self.kernel_launches += 1
                    continue
                if self.world == 1 and self.fused_step:
                    first_step = self.adam_step + 1
                    self.adam_step += ns
                    with _Phase(self, "minibatch_grad"):    # gradient kernel + fused fold/clip/Adam kernel
                        _lib.check(self.L.drl_ppo_minibatch_update(
                            net, self.agent.packed.data_ptr(), self.records.data_ptr(), idx_ptr, start, count,
                            stats_ptr + 8 * k, C.byref(self.coef), self.agent.flat_params.data_ptr(),
                            self.grad.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), first_step, lr,
                            0.9, 0.999, 1e-5, cfg.max_grad_norm, self.loss_terms.data_ptr() + 32 * row,
                            self.grad_norm.data_ptr(), self.workspace.data_ptr(), self.ws_bytes, self.grad_flags, ns, st))
                    self.kernel_launches += 1 if self.grad_flags == 1 else 2
                    continue
                with _Phase(self, "minibatch_grad"):
                    _lib.check(self.L.drl_ppo_minibatch_grad(
                        net, self.agent.packed.data_ptr(), self.records.data_ptr(), idx_ptr, start, count,
                        stats_ptr + 8 * k, C.byref(self.coef), self.grad.data_ptr(),
                        self.loss_terms.data_ptr() + 32 * row, self.workspace.data_ptr(), self.ws_bytes, self.grad_flags, st))
                if self.world > 1:
                    with _Phase(self, "allreduce"):
                        _dist.all_reduce_sum(self.grad)       # the only collective: NCCL over NVLink
                self.adam_step += 1
                with _Phase(self, "clip_adam"):
                    _lib.check(self.L.drl_clip_adam(net, self.agent.flat_params.data_ptr(), self.grad.data_ptr(),
                                                    self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), self.adam_step, lr,
                                                    0.9, 0.999, 1e-5, cfg.max_grad_norm, 1.0 / self.world,
                                                    self.agent.packed.data_ptr(), self.grad_norm.data_ptr(), st))
                self.kernel_launches += 3

    def _issue_update(self, lr: float, ctl: bool) -> None:
        self.schedule_permutations(ctl)
        self.rollout(ctl)
        self.compute_gae()
        self.optimize(lr, ctl)

    def update(self, num_updates: Optional[int] = None) -> None:
        """One full update (rollout + GAE + epochs), asynchronous: no host synchronisation.  On the tcgen05 path the launches
        are captured once in a CUDA graph (third update onwards) and replayed; per update the host then issues one tiny
        drl_ctrl_set launch (step / epoch / Adam counters, learning rate) and one graph launch."""
        nu = num_updates if num_updates is not None else max(1, self.cfg.num_updates(self.world))
        lr = self.learning_rate(self.update_idx, nu)
        use_ctl = self.graph_ok and not self.timing
        if not use_ctl:
            self._issue_update(lr, False)
        else:
            cfg = self.cfg
            n_opt = cfg.update_epochs * self.n_mb
            _lib.check(self.L.drl_ctrl_set(self.ctrl.data_ptr(), self.env.step_count, self.update_idx * cfg.update_epochs,
                                           self.peer.seq if self.peer is not None else 0, self.adam_step, n_opt, lr, 0.9, 0.999,
                                           _lib.stream_ptr()))
            if self._graph is None and self._graph_warm >= 2:
                self._capture_graph(lr)
            if self._graph is not None:
                self._graph.replay()
                self._advance_host_counters(n_opt)
                self.kernel_launches += self._graph_launches
            else:
                self._graph_warm += 1
                self._issue_update(lr, True)
            self.kernel_launches += 1       # drl_ctrl_set
        self.update_idx += 1
        self.agent.mark_packed_current()

    def _advance_host_counters(self, n_opt: int) -> None:
        """Host mirrors of the counters the replayed kernels read from the control block."""
        cfg = self.cfg
        self.env.step_count += cfg.num_steps
        self.global_step += cfg.num_steps * cfg.num_envs * self.world
        self.adam_step += n_opt
        if self.peer is not None:
            self.peer.seq += n_opt

    def _capture_graph(self, lr: float) -> None:
        """Stream-capture one update issued through the *_ctl entry points.  Nothing executes during capture, so the host
        counters are restored afterwards; the side-stream fork / join (permutations, statistics) becomes part of the graph."""
        snap = (self.env.step_count, self.global_step, self.adam_step, self.kernel_launches, self.peer.seq if self.peer is not None else 0,
                self._perms_scheduled)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._issue_update(lr, True)
        self._graph_launches = self.kernel_launches - snap[3]
        self.env.step_count, self.global_step, self.adam_step, self.kernel_launches = snap[0], snap[1], snap[2], snap[3]
        if self.peer is not None:
            self.peer.seq = snap[4]
        self._perms_scheduled = False
        self._graph = g

    def metrics(self, with_episode_log: bool = True) -> Dict[str, float]:
        """Device->host read of the last update's loss terms, gradient norm and finished-episode statistics
        (synchronises).  `with_episode_log=False` skips the per-episode entries (36 + 24 bytes are read instead of
        20 more bytes per finished episode); `"arrays"` returns them as numpy arrays {"step","env","ret","len"} instead of
        a sorted list of tuples."""
        self._h_terms.copy_(self._d_terms_src(), non_blocking=True)
        if with_episode_log == "arrays":     # every finished episode as numpy arrays (no per-entry Python objects)
            n, sum_ret, sum_len, entries = self.env.log.drain_arrays()
        else:
            n, sum_ret, sum_len, entries = self.env.log.drain(with_entries=with_episode_log)
        lt = self._h_terms.tolist()
        self.check_peers()
        return {"loss": lt[0], "pg_loss": lt[1], "v_loss": lt[2], "entropy": lt[3], "approx_kl": lt[4],
                "clipfrac": lt[5], "grad_norm": lt[8], "episodes": n, "episodes_dropped": max(0, n - self.env.log.cap),
                "mean_return": (sum_ret / n) if n else float("nan"), "mean_length": (sum_len / n) if n else float("nan"),
                "episode_log": entries}

    def metrics_async(self) -> "MetricsRead":
        """Enqueue the device->host read of this update's loss terms, gradient norm, episode statistics and finished-episode
        records (one 36-byte and one header + records copy into pinned memory, then the clear of the log) and return a handle;
        `handle.result()` waits for the copies only.  Lets a training loop read update k's metrics while update k+1 runs:

            tr.update(); h = tr.metrics_async(); tr.update(); m = h.result(); ...
        """
        host = self._h_terms_ring[self._h_flip]
        self._h_flip ^= 1
        host.copy_(self._d_terms_src(), non_blocking=True)
        return MetricsRead(self, host, self.env.log.read_async())

    def check_peers(self) -> None:
        """Raises if a peer rank missed the in-kernel all-reduce (the kernels skip the optimizer step from then on).
        Synchronises: called from metrics() and state_dict(), which synchronise anyway."""
        if self.peer is not None and int(self.peer.error_flag.item()) != 0:
            raise _lib.DrlError("a peer rank did not arrive at the in-kernel all-reduce within the timeout; "
                                "optimizer steps have been skipped since")

    def _d_terms_src(self) -> torch.Tensor:
        # loss terms of the last minibatch (8 floats) followed by the pre-clip gradient norm: rows are contiguous
        return self._terms_and_norm[-9:]

    # ------------------------------------------------------------------------------------------
    def state_dict(self) -> Dict[str, object]:
        """Everything needed to resume bit-identically: model + optimizer (ppo.py:86-90), counters, env state and the carried
        reward / done slot of the one-slot-shifted storage (ppo.py:93-98).  Tensors are CPU copies (synchronises)."""
        e = self.env
        self.check_peers()
        return {"model": {k: v.detach().cpu().clone() for k, v in self.agent.state_dict().items()},
                "exp_avg": self.exp_avg.cpu().clone(), "exp_avg_sq": self.exp_avg_sq.cpu().clone(),
                "adam_step": self.adam_step, "update_idx": self.update_idx, "global_step": self.global_step,
                "env": {"state": e.state.cpu().clone(), "elapsed": e.elapsed.cpu().clone(), "ep_ret": e.ep_ret.cpu().clone(),
                        "ep_len": e.ep_len.cpu().clone(), "step_count": e.step_count},
                "carry": {"rewards0": self.rewards[0].cpu().clone(), "dones0": self.dones[0].cpu().clone()},
                "config": self._resume_key()}

    def _resume_key(self) -> Dict[str, object]:
        """Everything a bit-identical resume depends on besides the tensors: shapes, Philox key / counters' owner, numerics."""
        c = self.cfg
        return {"env_id": c.env_id, "num_envs": c.num_envs, "num_steps": c.num_steps, "seed": c.seed, "hidden": c.hidden,
                "rank": self.rank, "world": self.world, "update_precision": self.update_precision,
                "rollout_precision": self.rollout_precision}

    def load_state_dict(self, sd: Dict[str, object]) -> None:
        c, mine = sd["config"], self._resume_key()
        diff = {k: (c.get(k), v) for k, v in mine.items() if c.get(k) != v}
        if diff:
            raise ValueError(f"checkpoint does not match this trainer (checkpoint, trainer): {diff}")
        self.agent.load_state_dict(sd["model"])
        self.agent.sync()
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.adam_step, self.update_idx, self.global_step = int(sd["adam_step"]), int(sd["update_idx"]), int(sd["global_step"])
        e, se = self.env, sd["env"]
        e.state.copy_(se["state"]); e.elapsed.copy_(se["elapsed"]); e.ep_ret.copy_(se["ep_ret"]); e.ep_len.copy_(se["ep_len"])
        e.step_count = int(se["step_count"])
        self.rewards[0].copy_(sd["carry"]["rewards0"])
        self.dones[0].copy_(sd["carry"]["dones0"])
        self._perms_scheduled = False

    def explained_variance(self) -> float:
        """ppo.py:194-195 over all T+1 slots like the reference: drl_explained_variance (one launch, synchronises for the read)."""
        _lib.check(self.L.drl_explained_variance(self.values.data_ptr(), self.returns.data_ptr(), self.values.numel(),
                                                 self._ev_out.data_ptr(), self.workspace.data_ptr(), self.ws_bytes,
                                                 _lib.stream_ptr()))
        return float(self._ev_out.item())

    def evaluate(self, num_envs: int = 1024, episodes_per_env: int = 1, greedy: bool = True,
                 seed: Optional[int] = None) -> EvalResult:
        """Evaluate the current policy on `num_envs` fresh envs x `episodes_per_env` episodes (one drl_evaluate launch, or
        drl_evaluate_tc for a 256-wide net, on private envs and log; synchronises).  Touches no trainer state: training
        continues bit-identically.  The key
        defaults to eval_seed(cfg.seed); rank r plays global env ids [r * num_envs, (r + 1) * num_envs), so ranks play
        disjoint episodes -- pooling them across ranks (e.g. torch.distributed.all_gather of `returns`) is the caller's."""
        return _evaluate(self.agent, self.cfg.env_id, num_envs, episodes_per_env, greedy,
                         eval_seed(self.cfg.seed) if seed is None else seed, env_gid0=self.rank * int(num_envs))


def train(cfg: PPOConfig, quiet: bool = False, rank: int = 0, world: int = 1) -> PPOTrainer:
    """The training loop of the reference script; prints its `global_step=..., episodic_return=...` lines.  With
    cfg.eval_every > 0, after every eval_every-th update a greedy evaluation over cfg.eval_episodes fresh episodes follows,
    printed by rank 0 as `global_step=..., eval_return=<mean>±<std> (greedy, <n> episodes)` (rank 0's episodes)."""
    tr = PPOTrainer(cfg, rank=rank, world=world)
    nu = cfg.num_updates(world)
    per_vec_step = cfg.num_envs * world
    for u in range(nu):
        tr.update(nu)
        m = tr.metrics()
        if not quiet and rank == 0:
            if cfg.num_envs * world <= 16:
                for step, env_gid, ret, _len in m["episode_log"]:
                    print(f"global_step={step * per_vec_step + env_gid}, episodic_return={ret:.2f}")
            elif m["episodes"]:
                print(f"global_step={tr.global_step}, episodic_return={m['mean_return']:.2f} "
                      f"(mean of {m['episodes']} episodes)")
        if cfg.eval_every > 0 and (u + 1) % cfg.eval_every == 0:
            ev = tr.evaluate(num_envs=cfg.eval_episodes, episodes_per_env=1, greedy=True)
            if not quiet and rank == 0:
                print(f"global_step={tr.global_step}, eval_return={ev.mean_return:.2f}±{ev.std_return:.2f} "
                      f"(greedy, {ev.episodes} episodes)")
    return tr


def main(argv=None) -> None:
    p = argparse.ArgumentParser(description="PPO on device-resident classic-control envs (B200)")
    d = PPOConfig()
    p.add_argument("--env-id", default=d.env_id)
    p.add_argument("--total-timesteps", type=int, default=d.total_timesteps)
    p.add_argument("--num-steps", type=int, default=d.num_steps)
    p.add_argument("--num-envs", type=int, default=d.num_envs)
    p.add_argument("--update-epochs", type=int, default=d.update_epochs)
    p.add_argument("--learning-rate", type=float, default=d.learning_rate)
    p.add_argument("--seed", type=int, default=d.seed)
    p.add_argument("--eval-every", type=int, default=d.eval_every, help="greedy evaluation every N updates (0 = off)")
    p.add_argument("--eval-episodes", type=int, default=d.eval_episodes)
    p.add_argument("--hidden", type=int, default=d.hidden, choices=(64, 256), help="width of both hidden layers")
    a = p.parse_args(argv)
    rank, world = _dist.init_from_env()
    cfg = PPOConfig(env_id=a.env_id, total_timesteps=a.total_timesteps, num_steps=a.num_steps, num_envs=a.num_envs,
                    update_epochs=a.update_epochs, learning_rate=a.learning_rate, seed=a.seed, eval_every=a.eval_every,
                    eval_episodes=a.eval_episodes, hidden=a.hidden)
    train(cfg, rank=rank, world=world)
    _dist.shutdown()


if __name__ == "__main__":
    main()
