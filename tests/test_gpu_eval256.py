"""Tensor-core policy evaluation of 256-wide nets (drl_evaluate_tc / deep_rl_b200.evaluate / PPOTrainer.evaluate with
hidden = 256): teacher-forced parity against the bf16-emulating oracle, bit-identity with the training rollout, invariances,
non-interference with training, learning signal, and the C ABI's argument validation (CPU)."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

from oracle import clib, ppo_oracle as po

EVAL_SEED = 0x123456789ABCDEF1       # both key words non-zero
HID = 256


def _gpu_tanh(x: torch.Tensor) -> torch.Tensor:
    """tanh.approx.f32 evaluated by the device (the activation of the tensor-core kernels) for the bf16-emulating oracle."""
    from deep_rl_b200 import _lib as L
    xd = x.detach().to("cuda:0", torch.float32).contiguous()
    yd = torch.empty_like(xd)
    L.check(L.lib().drl_selftest_tanh(xd.data_ptr(), yd.data_ptr(), xd.numel(), L.stream_ptr()))
    return yd.cpu().reshape(x.shape)


_AGENTS = {}


def _agent(env_id, trained):
    """The initial 256-wide agent of a fresh trainer, or one after two bf16 updates (cached per module)."""
    import deep_rl_b200 as drl
    key = (env_id, trained)
    if key not in _AGENTS:
        tr = drl.PPOTrainer(drl.PPOConfig(env_id=env_id, num_envs=256, num_steps=32, hidden=HID, seed=3,
                                          total_timesteps=256 * 32 * 10))
        if trained:
            tr.update(); tr.update()
            torch.cuda.synchronize()
        _AGENTS[key] = tr.agent
    return _AGENTS[key]


def _check_eval256(env_id, N, K, greedy, trained):
    import deep_rl_b200 as drl
    agent = _agent(env_id, trained)
    res = drl.evaluate(agent, env_id, N, episodes_per_env=K, greedy=greedy, seed=EVAL_SEED, trace=True)
    assert res.returns.shape == (N, K) and res.lengths.shape == (N, K)
    assert (res.lengths >= 1).all() and res.env_steps == int(res.lengths.sum())
    S = K * clib.MAX_EPISODE_STEPS[env_id]
    assert res.act.shape == (S, N)
    # every env plays exactly its K episodes back to back from t = 0, then its trace rows say 0xFF
    total = res.lengths.sum(axis=1)
    act_all = res.act.cpu().numpy()
    live_all = act_all != 0xFF
    assert np.array_equal(live_all, np.arange(S)[:, None] < total[None, :]), "act rows vs episode quota"
    R = int(total.max())
    state = res.state[:R].cpu().numpy()
    obs = res.obs[:R].cpu().numpy()
    klog = res.logits[:R].cpu().numpy()
    act = act_all[:R].astype(np.int32)
    live = live_all[:R]
    ends = np.cumsum(res.lengths, axis=1) - 1          # step at which each logged episode ended

    O, A = agent.obs_dim, agent.num_actions
    flat = agent.flat_params.cpu().numpy()
    el = po.mlp_forward_bf16_emulated(flat, obs[:, :, :O].reshape(-1, O), O, HID, A, tanh_fn=_gpu_tanh)[0]
    el = el.numpy().reshape(R, N, A)
    # one flipped bf16 rounding moves a 256-wide output by up to ~1e-3 (the tolerance of test_rollout_h256_vs_oracle)
    np.testing.assert_allclose(klog[live], el[live], rtol=0, atol=3e-3, err_msg="logits vs bf16-emulating oracle")
    ora = clib.OracleVecEnv(env_id, N, seed=EVAL_SEED)
    np.testing.assert_allclose(obs[0, :, :O], ora.reset(), rtol=0, atol=1e-7)
    fin = []
    for t in range(R):
        m = live[t]
        want = np.argmax(klog[t], axis=1) if greedy else clib.sample(klog[t], EVAL_SEED, 0, t)[0]
        assert np.array_equal(act[t][m], want[m]), f"actions t={t}: envs {np.nonzero(m & (act[t] != want))[0]}"
        a = np.where(m, act[t], 0).astype(np.int32)
        ora.set_state(state[t])                       # teacher forcing: the kernel's fp64 state of step t
        o, _, d, info = ora.step(a)
        if t + 1 < R:                                 # next observation (reset draw included) of the envs still playing
            nxt = live[t + 1]
            np.testing.assert_allclose(obs[t + 1, :, :O][nxt], o[nxt], rtol=0, atol=1e-6, err_msg=f"obs t={t + 1}")
        for i in np.nonzero(m & d.astype(bool))[0]:
            fin.append((t, int(i), float(info["final_return"][i]), int(info["final_length"][i])))
    got = sorted((int(ends[i, k]), i, float(res.returns[i, k]), int(res.lengths[i, k])) for i in range(N) for k in range(K))
    assert got == sorted(fin), "episode log vs episodes rebuilt by the oracle env"
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,N", [("CartPole-v1", 1), ("CartPole-v1", 100), ("CartPole-v1", 128), ("CartPole-v1", 300),
                                      ("Acrobot-v1", 130), ("MountainCar-v0", 96)])
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("greedy", [True, False])
@pytest.mark.parametrize("trained", [False, True])
def test_evaluate256_vs_oracle(env_id, N, K, greedy, trained):
    _check_eval256(env_id, N, K, greedy, trained)


@pytest.mark.gpu
def test_evaluate256_replays_the_training_rollout():
    """A sampled evaluation is the training rollout started from the evaluation key: drl_rollout (tensor cores, step0 = 0)
    on VecEnv(seed=key).reset() gives bit-identical obs, logits and actions in every row an env plays, and its first K logged
    episodes per env are the evaluation's."""
    import deep_rl_b200 as drl
    from deep_rl_b200 import _lib
    from deep_rl_b200.envs import VecEnv
    agent = _agent("CartPole-v1", True)
    N, K = 256, 2
    T = K * 500
    env = VecEnv("CartPole-v1", N, seed=EVAL_SEED, log_capacity=N * T)
    env.reset()
    dev, OP, A = env.device, env.obs_stride, env.num_actions
    obs = torch.zeros((T + 1, N, OP), dtype=torch.float32, device=dev)
    act = torch.zeros((T + 1, N), dtype=torch.uint8, device=dev)
    logp, val, rew = (torch.zeros((T + 1, N), dtype=torch.float32, device=dev) for _ in range(3))
    done = torch.zeros((T + 1, N), dtype=torch.uint8, device=dev)
    logits = torch.zeros((T, N, A), dtype=torch.float32, device=dev)
    buf = _lib.RolloutBufT(*(x.data_ptr() for x in (obs, act, logp, val, rew, done, logits)))
    agent._ensure_packed()
    _lib.check(env.L.drl_rollout(C.byref(env.struct), C.byref(agent.net), agent.packed.data_ptr(), T, 0, C.byref(buf),
                                 C.byref(env.log.struct), 1, _lib.stream_ptr()))
    n, _, _, e = env.log.drain_arrays()
    assert n <= N * T
    res = drl.evaluate(agent, "CartPole-v1", N, episodes_per_env=K, greedy=False, seed=EVAL_SEED, trace=True)
    total = torch.as_tensor(res.lengths.sum(axis=1), device=dev)
    rows = torch.arange(T, device=dev)[:, None] < total[None, :]
    assert torch.equal(res.obs.view(torch.int32)[rows], obs[:T].view(torch.int32)[rows]), "obs rows differ"
    assert torch.equal(res.logits.view(torch.int32)[rows], logits.view(torch.int32)[rows]), "logits rows differ"
    assert torch.equal(res.act[rows], act[:T][rows]), "actions differ"
    for i in range(N):
        sel = np.nonzero(e["env"] == i)[0]
        sel = sel[np.argsort(e["step"][sel])][:K]
        assert np.array_equal(e["ret"][sel], res.returns[i]) and np.array_equal(e["len"][sel], res.lengths[i]), f"env {i}"


@pytest.mark.gpu
def test_evaluate256_invariances():
    import deep_rl_b200 as drl
    agent = _agent("CartPole-v1", True)

    def run(N, gid0=0, seed=EVAL_SEED):
        r = drl.evaluate(agent, "CartPole-v1", N, episodes_per_env=2, greedy=False, seed=seed, env_gid0=gid0)
        return r.returns, r.lengths

    a, b = run(300), run(300)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), "same call, different result"
    lo, hi = run(100, 0), run(200, 100)
    assert np.array_equal(a[0], np.concatenate([lo[0], hi[0]])) and np.array_equal(a[1], np.concatenate([lo[1], hi[1]])), \
        "the tiling of envs into CTAs changed the episodes"
    c = run(300, seed=EVAL_SEED + 1)
    assert not np.array_equal(a[1], c[1]), "a different key played the same episodes"


def _train(cfg, n_updates, with_eval):
    import deep_rl_b200 as drl
    tr = drl.PPOTrainer(cfg)
    logs, evals = [], []
    for _ in range(n_updates):
        tr.update(10)
        if with_eval:
            evals.append(tr.evaluate(num_envs=64))
        m = tr.metrics(with_episode_log="arrays")
        logs.append({k: np.array(v) for k, v in m["episode_log"].items()})
    torch.cuda.synchronize()
    return tr, logs, evals


@pytest.mark.gpu
def test_evaluate256_does_not_touch_training():
    """Training a 256-wide net with an evaluation after every update is bit-identical to training without; evaluation
    results survive state_dict() / load_state_dict() into a fresh trainer."""
    import deep_rl_b200 as drl
    cfg = drl.PPOConfig(num_envs=256, num_steps=32, hidden=HID, seed=2, total_timesteps=256 * 32 * 10)
    a, la, _ = _train(cfg, 4, False)
    b, lb, evals = _train(cfg, 4, True)
    assert len(evals) == 4 and all(e.episodes == 64 for e in evals)
    assert torch.equal(a.agent.flat_params, b.agent.flat_params)
    assert torch.equal(a.exp_avg, b.exp_avg) and torch.equal(a.exp_avg_sq, b.exp_avg_sq)
    assert torch.equal(a.env.state, b.env.state) and a.env.step_count == b.env.step_count
    for x, y in zip(la, lb):
        for k in ("step", "env", "ret", "len"):
            assert np.array_equal(np.sort(x[k]), np.sort(y[k])), k
    before = b.evaluate(num_envs=128, episodes_per_env=2, greedy=False)
    c = drl.PPOTrainer(cfg)
    c.load_state_dict(b.state_dict())
    after = c.evaluate(num_envs=128, episodes_per_env=2, greedy=False)
    assert np.array_equal(before.returns, after.returns) and np.array_equal(before.lengths, after.lengths)


_EVAL_LINE = re.compile(r"global_step=\d+, eval_return=-?\d+\.\d\d±\d+\.\d\d \(greedy, 64 episodes\)")
_REF_LINE = re.compile(r"global_step=\d+, episodic_return=-?\d+\.\d\d( \(mean of \d+ episodes\))?")


@pytest.mark.gpu
def test_train_prints_eval_lines_h256(capsys):
    import deep_rl_b200 as drl
    base = dict(num_envs=32, num_steps=32, total_timesteps=32 * 32 * 4, seed=1, hidden=HID)
    drl.train(drl.PPOConfig(**base, eval_every=2, eval_episodes=64))
    with_eval = capsys.readouterr().out.strip().splitlines()
    drl.train(drl.PPOConfig(**base))
    plain = capsys.readouterr().out.strip().splitlines()
    evals = [ln for ln in with_eval if "eval_return" in ln]
    assert len(evals) == 2 and all(_EVAL_LINE.fullmatch(ln) for ln in evals), evals
    assert all(_REF_LINE.fullmatch(ln) for ln in plain), plain
    assert [ln for ln in with_eval if "eval_return" not in ln] == plain      # evaluation changes no training output


@pytest.mark.gpu
def test_cli_hidden_256_with_evaluation(capsys):
    from deep_rl_b200.ppo import main
    main(["--hidden", "256", "--num-envs", "32", "--num-steps", "32", "--total-timesteps", str(32 * 32 * 2), "--eval-every", "1",
          "--eval-episodes", "64"])
    evals = [ln for ln in capsys.readouterr().out.strip().splitlines() if "eval_return" in ln]
    assert len(evals) == 2 and all(_EVAL_LINE.fullmatch(ln) for ln in evals), evals


@pytest.mark.gpu
def test_h256_evaluation_learning_signal():
    """The configuration of test_h256_trainer_learns_and_keeps_ratio_one (1,024 envs x 64 steps x 40 updates, seed 1): the
    greedy policy over 1,024 fresh episodes.  The initial policy, sampled, scores like a random one (< 60)."""
    import deep_rl_b200 as drl
    init = drl.PPOTrainer(drl.PPOConfig(num_envs=64, hidden=HID, seed=1)).evaluate(num_envs=1024, greedy=False)
    assert init.episodes == 1024 and init.mean_return < 60, init.mean_return
    cfg = drl.PPOConfig(num_envs=1024, num_steps=64, hidden=HID, seed=1, total_timesteps=1024 * 64 * 40)
    tr = drl.PPOTrainer(cfg)
    for _ in range(cfg.num_updates()):
        tr.update()
    ev = tr.evaluate(num_envs=1024)
    print(f"h256 learning signal: initial sampled {init.mean_return:.2f}, trained greedy {ev.mean_return:.2f}±{ev.std_return:.2f}")
    assert ev.episodes == 1024 and ev.mean_return > 100, (ev.mean_return, ev.std_return)


# ---------------------------------------------------------------- CPU: argument validation
def _abi():
    from deep_rl_b200 import _lib
    return _lib, _lib.lib()


def _args(L, kind=0, N=8, max_steps=500, net=(4, HID, 2, 4), K=2, cap=None, flags=1, log=True, packed=0x1000):
    env = L.EnvT(kind, N, 1, 0, max_steps, 0x1000, 0x2000, 0x3000, 0x4000)     # never dereferenced: validation fails first
    lg = L.EpLogT(0x5000, 0x5008, 0x5010, 0x5020, N * K if cap is None else cap)
    return (C.byref(env), C.byref(L.NetT(*net)), packed, K, flags, C.byref(lg) if log else None, None, None)


@pytest.mark.parametrize("case,msg", [
    (dict(kind=7), b"unknown env kind"),
    (dict(N=0), b"num_envs=0"),
    (dict(net=(4, 128, 2, 4)), b"hidden=128"),
    (dict(net=(6, HID, 3, 8)), b"does not match env kind"),
    (dict(packed=None), b"packed is NULL"),
    (dict(K=0), b"episodes_per_env=0"),
    (dict(K=(1 << 31) // 500 + 1), b"exceeds int32"),
    (dict(log=False), b"log (count and entries) is required"),
    (dict(cap=15), b"log cap 15"),
    (dict(flags=2), b"unknown flags"),
])
def test_evaluate_tc_rejects_bad_arguments(case, msg):
    L, lib = _abi()
    assert lib.drl_evaluate_tc(*_args(L, **case)) == -1
    assert msg in lib.drl_last_error(), lib.drl_last_error()


def test_evaluate_tc_rejects_null_env():
    L, lib = _abi()
    assert lib.drl_evaluate_tc(None, C.byref(L.NetT(4, HID, 2, 4)), 0x1000, 1, 1, None, None, None) == -1
    assert b"env is NULL" in lib.drl_last_error()


def test_evaluate_tc_sends_64_wide_nets_to_drl_evaluate():
    L, lib = _abi()
    assert lib.drl_evaluate_tc(*_args(L, net=(4, 64, 2, 4))) == -2          # DRL_ERR_UNSUPPORTED
    assert b"use drl_evaluate" in lib.drl_last_error(), lib.drl_last_error()
