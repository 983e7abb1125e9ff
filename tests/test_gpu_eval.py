"""Policy evaluation (drl_evaluate / deep_rl_b200.evaluate / PPOTrainer.evaluate): teacher-forced parity against the CPU
oracle, free-running agreement with a CPU reference, invariances, non-interference with training, learning signal, and the
C ABI's argument validation (CPU)."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

from oracle import clib, ppo_oracle as po

EVAL_SEED = 0x123456789ABCDEF1       # both key words non-zero


def _reference_evaluate(flat_np, env_id, N, K, seed, greedy, H=64, env_gid0=0):
    """Free-running CPU reference of drl_evaluate built from the oracle pieces: OracleVecEnv reset with the evaluation key,
    steps t = 0, 1, ... with the argmax (first max) or the oracle sampler at step t; each env counted until its K-th finished
    episode.  Returns (returns [N, K] float32, lengths [N, K] int32)."""
    env = clib.OracleVecEnv(env_id, N, seed=seed, env_gid0=env_gid0)
    O, A = env.obs_dim, env.num_actions
    flat = torch.tensor(np.asarray(flat_np, dtype=np.float32))
    rets, lens = np.zeros((N, K), np.float32), np.zeros((N, K), np.int32)
    count = np.zeros(N, np.int64)
    obs = env.reset()
    for t in range(K * env.max_steps):
        if (count >= K).all():
            break
        with torch.no_grad():
            logits = po.mlp_forward(flat, torch.from_numpy(obs), O, H, A)[0].numpy()
        a = np.argmax(logits, axis=1).astype(np.int32) if greedy else clib.sample(logits, seed, env_gid0, t)[0]
        obs, _, done, info = env.step(a)
        for i in np.nonzero(done.astype(bool) & (count < K))[0]:
            rets[i, count[i]], lens[i, count[i]] = info["final_return"][i], info["final_length"][i]
            count[i] += 1
    return rets, lens


_AGENTS = {}


def _agent(env_id, trained):
    """The initial agent of a fresh trainer, or one after two fp32 updates (cached per module)."""
    import deep_rl_b200 as drl
    key = (env_id, trained)
    if key not in _AGENTS:
        tr = drl.PPOTrainer(drl.PPOConfig(env_id=env_id, num_envs=32, num_steps=64, seed=3, total_timesteps=32 * 64 * 10,
                                          update_precision="fp32"))
        if trained:
            tr.update(); tr.update()
            torch.cuda.synchronize()
        _AGENTS[key] = tr.agent
    return _AGENTS[key]


def _check_eval(env_id, N, K, greedy, trained, gid0=0):
    import deep_rl_b200 as drl
    agent = _agent(env_id, trained)
    res = drl.evaluate(agent, env_id, N, episodes_per_env=K, greedy=greedy, seed=EVAL_SEED, env_gid0=gid0, trace=True)
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
    flat = agent.flat_params.cpu()
    ora = clib.OracleVecEnv(env_id, N, seed=EVAL_SEED, env_gid0=gid0)
    np.testing.assert_allclose(obs[0, :, :O], ora.reset(), rtol=0, atol=1e-7)
    free = clib.OracleVecEnv(env_id, N, seed=EVAL_SEED, env_gid0=gid0) if env_id == "CartPole-v1" else None
    if free is not None:
        free.reset()
    fin, fin_free = [], []
    for t in range(R):
        m = live[t]
        with torch.no_grad():
            logits = po.mlp_forward(flat, torch.from_numpy(np.ascontiguousarray(obs[t, :, :O])), O, 64, A)[0].numpy()
        np.testing.assert_allclose(klog[t][m], logits[m], rtol=0, atol=2e-5, err_msg=f"logits t={t}")
        want = np.argmax(klog[t], axis=1) if greedy else clib.sample(klog[t], EVAL_SEED, gid0, t)[0]
        assert np.array_equal(act[t][m], want[m]), f"actions t={t}: envs {np.nonzero(m & (act[t] != want))[0]}"
        a = np.where(m, act[t], 0).astype(np.int32)
        ora.set_state(state[t])                       # teacher forcing: the kernel's fp64 state of step t
        o, _, d, info = ora.step(a)
        if t + 1 < R:                                 # next observation (reset draw included) of the envs still playing
            nxt = live[t + 1]
            np.testing.assert_allclose(obs[t + 1, :, :O][nxt], o[nxt], rtol=0, atol=1e-6, err_msg=f"obs t={t + 1}")
        for i in np.nonzero(m & d.astype(bool))[0]:
            fin.append((t, int(i), float(info["final_return"][i]), int(info["final_length"][i])))
        if free is not None:                          # CartPole is not chaotic: the oracle env also runs free
            fo, _, fd, finfo = free.step(a)
            if t + 1 < R:
                np.testing.assert_allclose(obs[t + 1, :, :O][nxt], fo[nxt], rtol=0, atol=1e-6, err_msg=f"free-running obs t={t + 1}")
            for i in np.nonzero(m & fd.astype(bool))[0]:
                fin_free.append((t, int(i), float(finfo["final_return"][i]), int(finfo["final_length"][i])))
    got = sorted((int(ends[i, k]), i, float(res.returns[i, k]), int(res.lengths[i, k])) for i in range(N) for k in range(K))
    assert got == sorted(fin), "episode log vs episodes rebuilt by the oracle env"
    if free is not None:
        assert got == sorted(fin_free), "episode log vs free-running oracle env"
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,N", [("CartPole-v1", 1), ("CartPole-v1", 13), ("CartPole-v1", 256), ("CartPole-v1", 4096),
                                      ("Acrobot-v1", 40), ("MountainCar-v0", 45)])
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("greedy", [True, False])
@pytest.mark.parametrize("trained", [False, True])
def test_evaluate_vs_oracle(env_id, N, K, greedy, trained):
    _check_eval(env_id, N, K, greedy, trained)


@pytest.mark.gpu
def test_evaluate_vs_oracle_offset_gids():
    _check_eval("CartPole-v1", 37, 2, False, True, gid0=1000)


@pytest.mark.gpu
@pytest.mark.parametrize("greedy", [True, False])
def test_evaluate_free_running_vs_reference(greedy):
    """Logits agree with the CPU forward to ~2e-5, so a flipped argmax or sample edge is rare but possible: at least 62 of
    the 64 envs must play identical episodes."""
    import deep_rl_b200 as drl
    agent = _agent("CartPole-v1", True)
    res = drl.evaluate(agent, "CartPole-v1", 64, episodes_per_env=2, greedy=greedy, seed=EVAL_SEED)
    rr, rl = _reference_evaluate(agent.flat_params.cpu().numpy(), "CartPole-v1", 64, 2, EVAL_SEED, greedy)
    same = (res.returns == rr).all(axis=1) & (res.lengths == rl).all(axis=1)
    assert same.sum() >= 62, np.nonzero(~same)[0]


@pytest.mark.gpu
def test_evaluate_invariances(monkeypatch):
    import deep_rl_b200 as drl
    agent = _agent("CartPole-v1", True)

    def run(N, gid0=0, greedy=False):
        r = drl.evaluate(agent, "CartPole-v1", N, episodes_per_env=2, greedy=greedy, seed=EVAL_SEED, env_gid0=gid0)
        return r.returns, r.lengths

    a, b = run(256), run(256)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), "same call, different result"
    lo, hi = run(128, 0), run(128, 128)
    assert np.array_equal(a[0], np.concatenate([lo[0], hi[0]])) and np.array_equal(a[1], np.concatenate([lo[1], hi[1]]))
    for greedy in (True, False):
        ref = None
        for epw in (4, 8, 16, 32):
            monkeypatch.setenv("DRL_ROLLOUT_EPW", str(epw))
            got = run(300, greedy=greedy)
            if ref is None:
                ref = got
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), f"epw={epw} greedy={greedy}"


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
@pytest.mark.parametrize("prec,N,T,n_updates", [("fp32", 64, 32, 3), ("bf16", 256, 16, 6)])
def test_evaluate_does_not_touch_training(prec, N, T, n_updates):
    """Training with an evaluation after every update is bit-identical to training without (the bf16 case captures and
    replays the update's CUDA graph); evaluation results survive state_dict() / load_state_dict() into a fresh trainer."""
    import deep_rl_b200 as drl
    cfg = drl.PPOConfig(num_envs=N, num_steps=T, seed=2, total_timesteps=N * T * 10, update_precision=prec)
    a, la, _ = _train(cfg, n_updates, False)
    b, lb, evals = _train(cfg, n_updates, True)
    assert len(evals) == n_updates and all(e.episodes == 64 for e in evals)
    if prec == "bf16":
        assert b._graph is not None, "the CUDA graph was never captured"
    assert torch.equal(a.agent.flat_params, b.agent.flat_params)
    assert torch.equal(a.exp_avg, b.exp_avg) and torch.equal(a.exp_avg_sq, b.exp_avg_sq)
    assert torch.equal(a.env.state, b.env.state) and a.env.step_count == b.env.step_count
    for x, y in zip(la, lb):
        for k in ("step", "env", "ret", "len"):
            assert np.array_equal(np.sort(x[k]), np.sort(y[k])), k
    before = b.evaluate(num_envs=128, episodes_per_env=2, greedy=False)
    sd = b.state_dict()
    c = drl.PPOTrainer(cfg)
    c.load_state_dict(sd)
    after = c.evaluate(num_envs=128, episodes_per_env=2, greedy=False)
    assert np.array_equal(before.returns, after.returns) and np.array_equal(before.lengths, after.lengths)


@pytest.mark.gpu
def test_default_eval_key_differs_from_training_key():
    import deep_rl_b200 as drl
    from deep_rl_b200.ppo import eval_seed
    tr = drl.PPOTrainer(drl.PPOConfig(num_envs=64, seed=5))
    assert eval_seed(5) != 5
    d = tr.evaluate(num_envs=64, greedy=False)
    e = drl.evaluate(tr.agent, "CartPole-v1", 64, greedy=False, seed=eval_seed(5))
    assert np.array_equal(d.returns, e.returns)


@pytest.mark.gpu
def test_initial_policy_scores_low():
    """The untrained policy, sampled, scores like a random one (~22).  Its greedy score is no such baseline: the near-zero
    head makes argmax a fixed linear controller, which scores anywhere from ~9 to 500 depending on the init seed."""
    import deep_rl_b200 as drl
    tr = drl.PPOTrainer(drl.PPOConfig(num_envs=64, seed=1))
    ev = tr.evaluate(num_envs=1024, greedy=False)
    assert ev.mean_return < 60, ev.mean_return


@pytest.mark.gpu
def test_trained_policy_scores_high():
    """The configuration of test_many_envs_learns_cartpole: the greedy policy over 1,024 fresh episodes."""
    import deep_rl_b200 as drl
    cfg = drl.PPOConfig(num_envs=512, num_steps=128, total_timesteps=512 * 128 * 100, seed=1, update_precision="bf16")
    tr = drl.PPOTrainer(cfg)
    for _ in range(cfg.num_updates()):
        tr.update()
    ev = tr.evaluate(num_envs=1024)
    assert ev.episodes == 1024 and ev.mean_return > 150, (ev.mean_return, ev.std_return)


_EVAL_LINE = re.compile(r"global_step=\d+, eval_return=-?\d+\.\d\d±\d+\.\d\d \(greedy, 64 episodes\)")
_REF_LINE = re.compile(r"global_step=\d+, episodic_return=-?\d+\.\d\d( \(mean of \d+ episodes\))?")


@pytest.mark.gpu
def test_train_prints_eval_lines(capsys):
    import deep_rl_b200 as drl
    base = dict(num_envs=32, num_steps=32, total_timesteps=32 * 32 * 4, seed=1)
    drl.train(drl.PPOConfig(**base, eval_every=2, eval_episodes=64))
    with_eval = capsys.readouterr().out.strip().splitlines()
    drl.train(drl.PPOConfig(**base))
    plain = capsys.readouterr().out.strip().splitlines()
    evals = [ln for ln in with_eval if "eval_return" in ln]
    assert len(evals) == 2 and all(_EVAL_LINE.fullmatch(ln) for ln in evals), evals
    assert all(_REF_LINE.fullmatch(ln) for ln in plain), plain
    assert [ln for ln in with_eval if "eval_return" not in ln] == plain      # evaluation changes no training output


# ---------------------------------------------------------------- CPU: argument validation, no CPU fallback
def _abi():
    from deep_rl_b200 import _lib
    return _lib, _lib.lib()


def _args(L, kind=0, N=8, max_steps=500, net=(4, 64, 2, 4), K=2, cap=None, flags=1, log=True, packed=0x1000):
    env = L.EnvT(kind, N, 1, 0, max_steps, 0x1000, 0x2000, 0x3000, 0x4000)     # never dereferenced: validation fails first
    lg = L.EpLogT(0x5000, 0x5008, 0x5010, 0x5020, N * K if cap is None else cap)
    return (C.byref(env), C.byref(L.NetT(*net)), packed, K, flags, C.byref(lg) if log else None, None, None)


@pytest.mark.parametrize("case,msg", [
    (dict(kind=7), b"unknown env kind"),
    (dict(N=0), b"num_envs=0"),
    (dict(net=(4, 128, 2, 4)), b"hidden=128"),
    (dict(net=(6, 64, 3, 8)), b"does not match env kind"),
    (dict(net=(4, 256, 2, 4)), b"hidden=256"),
    (dict(packed=None), b"packed is NULL"),
    (dict(K=0), b"episodes_per_env=0"),
    (dict(K=(1 << 31) // 500 + 1), b"exceeds int32"),
    (dict(log=False), b"log (count and entries) is required"),
    (dict(cap=15), b"log cap 15"),
    (dict(flags=2), b"unknown flags"),
])
def test_evaluate_rejects_bad_arguments(case, msg):
    L, lib = _abi()
    assert lib.drl_evaluate(*_args(L, **case)) == -1
    assert msg in lib.drl_last_error(), lib.drl_last_error()


def test_evaluate_rejects_null_env():
    L, lib = _abi()
    assert lib.drl_evaluate(None, C.byref(L.NetT(4, 64, 2, 4)), 0x1000, 1, 1, None, None, None) == -1
    assert b"env is NULL" in lib.drl_last_error()


def test_evaluate_has_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import deep_rl_b200 as drl
    with pytest.raises(Exception, match="no CPU fallback"):
        drl.evaluate(None, "CartPole-v1", 4)
