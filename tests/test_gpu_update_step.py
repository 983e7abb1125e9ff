"""GPU tests of the optimizer-step entry points against teacher-forced references.

test_gpu_kernels.py pins the gradient kernels.  This file pins what consumes their output: the fold of the per-CTA partials,
the global-norm clip, Adam and the packed-weight refresh of drl_ppo_minibatch_update[_ctl] (tcgen05 fused step and fp32 fused
tail), the Adam scalars of drl_ctrl_set, drl_clip_adam at hidden = 256, the chunk loop of the 256-wide gradient, and the
trainer's wiring of all of them.  Each optimizer step is compared with drl_ppo_minibatch_grad on the same packed weights
followed by the CPU oracle's clip + Adam (oracle.ppo_oracle.clip_adam), and exp_avg / exp_avg_sq are compared as well as the
parameters: Adam normalises away a wrong clip coefficient in the parameter change, but not in the moments.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import ppo_oracle as po  # noqa: E402

BETA1, BETA2, EPS = 0.9, 0.999, 1e-5
COEF = (0.2, 0.01, 0.5)
DRL_ERR_ARG = -1
CHUNK_256 = 4096 * 128          # samples per launch of the 256-wide gradient kernels (STAGE_TILES x TC_TILE, update256.cu)
C_BAR = 1e-3                    # per-tensor relative L2, full multi-chunk call vs the weighted single-chunk pieces
REPLAY_BARS = {"params abs": 1e-5, "m rel": 1e-3, "v rel": 1e-3, "terms rel": 1e-4}


def _L():
    from deep_rl_b200 import _lib
    return _lib


def _dev():
    return torch.device("cuda:0")


def _net(O, A, H=64):
    return _L().NetT(O, H, A, 4 if O <= 4 else 8)


def _nan(n):
    return torch.full((n,), float("nan"), dtype=torch.float32, device=_dev())


def _workspace(net):
    n = int(_L().lib().drl_workspace_bytes(C.byref(net)))
    return torch.zeros(n, dtype=torch.uint8, device=_dev()), n


def _pack(net, params):
    """A fresh drl_pack_params of the device tensor `params` into a zeroed buffer."""
    L = _L()
    packed = torch.zeros(int(L.lib().drl_packed_count(C.byref(net))), dtype=torch.float32, device=_dev())
    L.check(L.lib().drl_pack_params(C.byref(net), params.data_ptr(), packed.data_ptr(), L.stream_ptr()))
    return packed


def _perm(B, seed):
    """The keyed Feistel permutation of drl_permutation (int32 on the device)."""
    L = _L()
    idx = torch.empty(B, dtype=torch.int32, device=_dev())
    L.check(L.lib().drl_permutation(idx.data_ptr(), B, seed, 1, 0, L.stream_ptr()))
    return idx


def _gpu_tanh(x):
    """The device's tanh.approx.f32, for the bf16-emulating oracle."""
    L = _L()
    xd = x.detach().to(_dev(), torch.float32).contiguous()
    yd = torch.empty_like(xd)
    L.check(L.lib().drl_selftest_tanh(xd.data_ptr(), yd.data_ptr(), xd.numel(), L.stream_ptr()))
    return yd.cpu().reshape(x.shape)


def _opt_state(O, A, H, seed):
    """Random parameters and non-zero Adam moments (numpy float32)."""
    P = po.param_count(O, H, A)
    params = (po.init_params(O, H, A, seed) + (0.05 if H == 64 else 0.02) * torch.randn(P)).numpy()
    rng = np.random.default_rng(seed)
    m = (rng.normal(size=P) * 3e-3).astype(np.float32)
    v = (rng.uniform(size=P) * 1e-5).astype(np.float32)
    return params, m, v


class _State:
    """params, exp_avg, exp_avg_sq and the packed weights of one optimizer, on the device."""

    def __init__(self, net, params, m, v):
        d = _dev()
        self.net = net
        self.p = torch.tensor(params, device=d)
        self.m = torch.tensor(m, device=d)
        self.v = torch.tensor(v, device=d)
        self.packed = _pack(net, self.p)

    def host(self):
        return self.p.cpu().numpy(), self.m.cpu().numpy(), self.v.cpu().numpy()


def _records(net, O, A, params, B, seed, heavy=None):
    """Sample records [B][RW] on the device, built as in test_tc_minibatch_grad_vs_torch_oracle: log-probs and values of
    the current policy plus noise (ratios on both sides of the clip), advantages ~ N(0.3, 2).  `heavy` (sample ids): an
    advantage of 100 sigma and a log-prob without noise, so that the ratio stays inside the clip.
    Returns (records, advantages as numpy)."""
    L = _L()
    rng = np.random.default_rng(seed)
    RW = 8 if O <= 4 else 16
    obs = np.zeros((B, net.obs_stride), np.float32)
    obs[:, :O] = rng.normal(size=(B, O))
    act = rng.integers(0, A, size=B)
    od = torch.from_numpy(obs).to(_dev())
    logits = torch.empty((B, A), dtype=torch.float32, device=_dev())
    value = torch.empty(B, dtype=torch.float32, device=_dev())
    packed = _pack(net, torch.tensor(params, device=_dev()))
    L.check(L.lib().drl_policy_forward(C.byref(net), packed.data_ptr(), od.data_ptr(), B, logits.data_ptr(), value.data_ptr(),
                                       L.stream_ptr()))
    logp = torch.log_softmax(logits, -1).cpu().numpy()[np.arange(B), act]
    noise = rng.normal(scale=0.15, size=B)
    adv = rng.normal(size=B) * 2 + 0.3
    if heavy is not None:
        noise[heavy] = 0.0
        adv[heavy] = 0.3 + 100 * 2.0
    rec = np.zeros((B, RW), np.float32)
    rec[:, :O] = obs[:, :O]
    rec[:, RW - 4] = logp + noise
    rec[:, RW - 3] = adv
    rec[:, RW - 2] = value.cpu().numpy() + rng.normal(scale=0.3, size=B)
    rec[:, RW - 1] = act.astype(np.int32).view(np.float32)
    return torch.from_numpy(rec).to(_dev()), rec[:, RW - 3].copy()


def _stats(adv, idx, start, M, S):
    """[S][2] (mean, unbiased std) of S consecutive minibatches of M samples from position `start` of idx."""
    order = idx.cpu().numpy().astype(np.int64) if idx is not None else np.arange(len(adv))
    st = []
    for s in range(S):
        a = adv[order[start + s * M:start + (s + 1) * M]].astype(np.float64)
        st.append([a.mean(), a.std(ddof=1)])
    return torch.tensor(np.asarray(st, np.float32), device=_dev())


def _grad(net, packed, rec, idx, start, count, stats, ws, flags):
    L = _L()
    P = int(L.lib().drl_param_count(C.byref(net)))
    grad, terms = _nan(P), _nan(8)
    cf = L.PpoCoefT(*COEF)
    L.check(L.lib().drl_ppo_minibatch_grad(C.byref(net), packed.data_ptr(), rec.data_ptr(), L.ptr(idx), start, count,
                                           stats.data_ptr(), C.byref(cf), grad.data_ptr(), terms.data_ptr(), ws[0].data_ptr(),
                                           ws[1], flags, L.stream_ptr()))
    return grad, terms


def _update(net, st, rec, idx, start, count, stats, ws, flags, step, lr, mgn, nsteps=1, ctrl=None, ordinal=0):
    """drl_ppo_minibatch_update (ctrl None) or _ctl on the state `st`; returns (grad_out, loss-term rows, norm_out)."""
    L = _L()
    P = int(L.lib().drl_param_count(C.byref(net)))
    grad, terms, norm = _nan(P), _nan(8 * nsteps), _nan(1)
    cf = L.PpoCoefT(*COEF)
    if ctrl is None:
        rc = L.lib().drl_ppo_minibatch_update(C.byref(net), st.packed.data_ptr(), rec.data_ptr(), L.ptr(idx), start, count,
                                              stats.data_ptr(), C.byref(cf), st.p.data_ptr(), grad.data_ptr(), st.m.data_ptr(),
                                              st.v.data_ptr(), step, lr, BETA1, BETA2, EPS, mgn, terms.data_ptr(), norm.data_ptr(),
                                              ws[0].data_ptr(), ws[1], flags, nsteps, L.stream_ptr())
    else:
        rc = L.lib().drl_ppo_minibatch_update_ctl(C.byref(net), st.packed.data_ptr(), rec.data_ptr(), L.ptr(idx), start, count,
                                                  stats.data_ptr(), C.byref(cf), st.p.data_ptr(), grad.data_ptr(), st.m.data_ptr(),
                                                  st.v.data_ptr(), ctrl.data_ptr(), ordinal, BETA1, BETA2, EPS, mgn,
                                                  terms.data_ptr(), norm.data_ptr(), ws[0].data_ptr(), ws[1], flags, None, nsteps,
                                                  L.stream_ptr())
    L.check(rc)
    return grad, terms.view(nsteps, 8), norm


def _norm64(x):
    return float(np.linalg.norm(np.asarray(x, np.float64)))


def _per_tensor(got, want, O, A, H, floor=1e-3):
    """Worst relative L2 error over the twelve gradient tensors, the denominator floored at `floor` x the whole norm."""
    off, worst = 0, ("", 0.0)
    total = _norm64(want)
    for name, shp in zip(po.PARAM_NAMES, po.param_shapes(O, H, A)):
        n = int(np.prod(shp))
        e = _norm64(got[off:off + n] - want[off:off + n]) / max(_norm64(want[off:off + n]), floor * total)
        worst = max(worst, (name, e), key=lambda t: t[1])
        off += n
    return worst


class _Worst:
    """Running maxima of the measured deviations of one test, printed at its end."""

    def __init__(self):
        self.d = {}

    def add(self, key, val):
        self.d[key] = max(self.d.get(key, 0.0), float(val))

    def __str__(self):
        return ", ".join(f"{k} {v:.2e}" for k, v in self.d.items())


def _check_adam(w, st, params0, m0, v0, grad, step, lr, mgn, grad_scale=1.0):
    """params / exp_avg / exp_avg_sq of `st` against clip_grad_norm_ + the oracle's Adam step on grad * grad_scale.
    torch's clip_grad_norm_ sums the squares in fp32: at 135k parameters its norm is ~9e-6 (relative) off the float64 value,
    which moves exp_avg by more than fp32 rounding, while the kernels sum in fp64 (norm_out is checked against float64 to
    1e-6).  So the clip coefficient is clip_grad_norm_'s fp32 formula on the float64 norm rounded to fp32, and
    po.clip_adam applies the Adam step to the clipped gradient with the clip itself switched off."""
    gs = (np.asarray(grad, np.float32) * np.float32(grad_scale)).astype(np.float32)
    coef = np.float32(mgn) / (np.float32(_norm64(gs)) + np.float32(1e-6))
    gc = (gs * min(coef, np.float32(1.0))).astype(np.float32)
    wp, wm, wv, _ = po.clip_adam(params0, gc, m0, v0, step, lr, math.inf)
    p, m, v = st.host() if isinstance(st, _State) else st
    w.add("params abs", np.abs(p - wp).max())
    w.add("m rel", (np.abs(m - wm) / (np.abs(wm) + 1e-9)).max())
    w.add("v rel", (np.abs(v - wv) / (np.abs(wv) + 1e-12)).max())
    # only fp32 rounding differs: the association of addcdiv / addcmul
    np.testing.assert_allclose(p, wp, rtol=0, atol=3e-7)
    np.testing.assert_allclose(m, wm, rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(v, wv, rtol=1e-6, atol=1e-12)


# ------------------------------------------------------------------------------------------------
# A. drl_ppo_minibatch_update at hidden = 64, teacher-forced by drl_ppo_minibatch_grad + the oracle's clip / Adam
# ------------------------------------------------------------------------------------------------
def _check_fused_single(O, A, M, flags):
    net = _net(O, A)
    mb_start = 97
    B = mb_start + M + 31
    params0, m0, v0 = _opt_state(O, A, 64, seed=M % 1000 + O)
    rec, adv = _records(net, O, A, params0, B, seed=M + O)
    idx = _perm(B, seed=M)
    stats = _stats(adv, idx, mb_start, M, 1)
    ws = _workspace(net)            # one zeroed workspace for every call: the grid-barrier counters must re-arm
    lr = 1e-3
    w = _Worst()
    for step in (1, 37):
        for clip in (True, False):
            st = _State(net, params0, m0, v0)
            g_ref, t_ref = _grad(net, st.packed, rec, idx, mb_start, M, stats, ws, flags)
            g_ref, t_ref = g_ref.cpu().numpy(), t_ref.cpu().numpy()
            mgn = (0.25 if clip else 4.0) * _norm64(g_ref)
            grad, terms, norm = _update(net, st, rec, idx, mb_start, M, stats, ws, flags, step, lr, mgn)
            g = grad.cpu().numpy()
            # same kernel on the same grid, and the tail folds the partials with grad_reduce_kernel's association
            assert np.array_equal(g, g_ref), f"step {step} clip {clip}: grad_out differs from drl_ppo_minibatch_grad"
            n64 = _norm64(g)
            w.add("norm rel", abs(float(norm.item()) - n64) / n64)
            assert abs(float(norm.item()) - n64) <= 1e-6 * n64
            _check_adam(w, st, params0, m0, v0, g, step, lr, mgn)
            assert torch.equal(st.packed, _pack(net, st.p)), "packed weights are not a fresh pack of the new parameters"
            t = terms[0].cpu().numpy()
            w.add("loss terms abs", np.abs(t[:6] - t_ref[:6]).max())
            np.testing.assert_allclose(t[:6], t_ref[:6], rtol=1e-6, atol=1e-6)
    print(f"O={O} A={A} M={M} flags={flags}: worst {w}")


A1_CASES = [(O, A, M) for O, A in ((4, 2), (6, 3), (2, 3)) for M in (70, 129, 4096, 131_072)] + [(4, 2, 2_097_152)]


@pytest.mark.parametrize("O,A,M", A1_CASES)
def test_fused_tc_step_vs_grad_and_oracle_adam(O, A, M):
    """One minibatch per launch on the tcgen05 path; step 1 and 37, clip on (0.25 x the norm) and off (4 x)."""
    _check_fused_single(O, A, M, flags=1)


@pytest.mark.parametrize("O,A,M", [(O, A, M) for O, A in ((4, 2), (6, 3)) for M in (32, 1000, 4096)])
def test_fused_fp32_tail_vs_grad_and_oracle_adam(O, A, M):
    """reduce_clip_adam_kernel (flags = 0): the same checks; its fold is grad_reduce_kernel's, so grad_out is bitwise equal."""
    _check_fused_single(O, A, M, flags=0)


@pytest.mark.parametrize("O,A,M,S", [(4, 2, 4096, 2), (4, 2, 4096, 4), (4, 2, 4096, 8), (6, 3, 131_072, 4), (2, 3, 70, 8)])
def test_fused_multi_step_launch_equals_chain_of_single_steps(O, A, M, S):
    """num_steps = S consecutive minibatches in one launch == S single-step launches, each teacher-forced as above."""
    net = _net(O, A)
    mb_start = 211
    B = mb_start + S * M + 17
    params0, m0, v0 = _opt_state(O, A, 64, seed=S + O)
    rec, adv = _records(net, O, A, params0, B, seed=S * 7 + M)
    idx = _perm(B, seed=S + M)
    stats = _stats(adv, idx, mb_start, M, S)
    ws = _workspace(net)
    lr = 1e-3
    step0 = 1 if S != 4 else 37
    chain, multi = _State(net, params0, m0, v0), _State(net, params0, m0, v0)
    mgn = None
    rows, w = [], _Worst()
    for s in range(S):
        g_ref, _ = _grad(net, chain.packed, rec, idx, mb_start + s * M, M, stats[s], ws, 1)
        if mgn is None:
            mgn = 0.5 * _norm64(g_ref.cpu().numpy())       # the clip acts at least on the first step
        p0, m_0, v_0 = chain.host()
        g, t, n = _update(net, chain, rec, idx, mb_start + s * M, M, stats[s], ws, 1, step0 + s, lr, mgn)
        assert torch.equal(g, g_ref)
        _check_adam(w, chain, p0, m_0, v_0, g.cpu().numpy(), step0 + s, lr, mgn)
        rows.append(t[0].clone())
    gm, tm, nm = _update(net, multi, rec, idx, mb_start, M, stats, ws, 1, step0, lr, mgn, nsteps=S)
    for name, a, b in (("params", multi.p, chain.p), ("exp_avg", multi.m, chain.m), ("exp_avg_sq", multi.v, chain.v),
                       ("packed", multi.packed, chain.packed), ("grad_out", gm, g), ("norm_out", nm, n)):
        assert torch.equal(a, b), f"{name}: {S}-step launch differs from the chain of single steps"
    for s in range(S):
        assert torch.equal(tm[s], rows[s]), f"loss terms row {s}"
    print(f"O={O} A={A} M={M} S={S}: bitwise equal to the chain; chain vs oracle Adam worst {w}")


def _ctrl_read(ctrl):
    return _L().CtrlT.from_buffer_copy(ctrl.cpu().numpy().tobytes())


def test_ctrl_set_scalars_read_back_exactly():
    """drl_ctrl_set's Adam scalars are the host's fp64 arithmetic cast to float32, bit for bit; slots >= n_steps are 0."""
    L = _L()
    ctrl = torch.empty(C.sizeof(L.CtrlT), dtype=torch.uint8, device=_dev())
    for k0, n, lr in ((0, 64, 2.5e-4), (37, 8, 1e-3), (1000, 5, 7.5e-5), (56, 1, 2.5e-4), (5, 0, 1e-3)):
        ctrl.fill_(0xFF)
        L.check(L.lib().drl_ctrl_set(ctrl.data_ptr(), 123_456_789_012, 7, 99, k0, n, lr, BETA1, BETA2, L.stream_ptr()))
        c = _ctrl_read(ctrl)
        assert (c.env_step, c.epoch_ctr, c.comm_seq, c.adam_step) == (123_456_789_012, 7, 99, k0)
        want_s = np.zeros(64, np.float32)
        want_b = np.zeros(64, np.float32)
        for k in range(n):
            want_s[k] = np.float32(-(lr / (1 - BETA1 ** (k0 + k + 1))))
            want_b[k] = np.float32(math.sqrt(1 - BETA2 ** (k0 + k + 1)))
        got_s = np.array(c.neg_step_size[:], np.float32)
        got_b = np.array(c.bc2_sqrt[:], np.float32)
        assert np.array_equal(got_s.view(np.uint32), want_s.view(np.uint32)), (k0, n, got_s[:4], want_s[:4])
        assert np.array_equal(got_b.view(np.uint32), want_b.view(np.uint32)), (k0, n, got_b[:4], want_b[:4])
    assert L.lib().drl_ctrl_set(ctrl.data_ptr(), 0, 0, 0, 0, 65, 1e-3, BETA1, BETA2, L.stream_ptr()) == DRL_ERR_ARG


def test_ctl_update_equals_by_value_update():
    """drl_ppo_minibatch_update_ctl(ordinal o, num_steps s) == drl_ppo_minibatch_update(step k0 + o + 1, lr, s), bitwise,
    up to the last slots of the control block; o + s > 64 is rejected before anything runs."""
    L = _L()
    O, A, M = 4, 2, 4096
    net = _net(O, A)
    mb_start = 4096 + 5
    B = mb_start + 8 * M
    params0, m0, v0 = _opt_state(O, A, 64, seed=11)
    rec, adv = _records(net, O, A, params0, B, seed=12)
    idx = _perm(B, seed=13)
    stats = _stats(adv, idx, mb_start, M, 8)
    ws = _workspace(net)
    k0, lr, mgn = 100, 1e-3, 0.05
    ctrl = torch.zeros(C.sizeof(L.CtrlT), dtype=torch.uint8, device=_dev())
    L.check(L.lib().drl_ctrl_set(ctrl.data_ptr(), 0, 0, 0, k0, 64, lr, BETA1, BETA2, L.stream_ptr()))
    for o, s in ((0, 1), (3, 2), (21, 4), (56, 8)):
        a, b = _State(net, params0, m0, v0), _State(net, params0, m0, v0)
        ga, ta, na = _update(net, a, rec, idx, mb_start, M, stats, ws, 1, k0 + o + 1, lr, mgn, nsteps=s)
        gb, tb, nb = _update(net, b, rec, idx, mb_start, M, stats, ws, 1, 1, 0.0, mgn, nsteps=s, ctrl=ctrl, ordinal=o)
        for name, x, y in (("params", a.p, b.p), ("exp_avg", a.m, b.m), ("exp_avg_sq", a.v, b.v), ("packed", a.packed, b.packed),
                           ("grad_out", ga, gb), ("loss terms", ta, tb), ("norm_out", na, nb)):
            assert torch.equal(x, y), f"ordinal {o} steps {s}: {name}"
        assert not torch.equal(a.p, torch.tensor(params0, device=_dev()))
    st = _State(net, params0, m0, v0)
    cf = L.PpoCoefT(*COEF)
    grad, terms, norm = _nan(po.param_count(O, 64, A)), _nan(64), _nan(1)
    for o, s in ((57, 8), (63, 2)):
        rc = L.lib().drl_ppo_minibatch_update_ctl(C.byref(net), st.packed.data_ptr(), rec.data_ptr(), idx.data_ptr(), mb_start, M,
                                                  stats.data_ptr(), C.byref(cf), st.p.data_ptr(), grad.data_ptr(), st.m.data_ptr(),
                                                  st.v.data_ptr(), ctrl.data_ptr(), o, BETA1, BETA2, EPS, mgn, terms.data_ptr(),
                                                  norm.data_ptr(), ws[0].data_ptr(), ws[1], 1, None, s, L.stream_ptr())
        assert rc == DRL_ERR_ARG, (o, s, rc)
    torch.cuda.synchronize()
    assert torch.equal(st.p, torch.tensor(params0, device=_dev())) and bool(torch.isnan(grad).all())


# ------------------------------------------------------------------------------------------------
# B. drl_clip_adam at hidden = 256 (the trainer's optimizer step for 256-wide nets)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("O,A", [(4, 2), (6, 3), (2, 3)])
def test_clip_adam_h256_vs_oracle_and_fresh_pack(O, A):
    """params / m / v against the oracle, norm_out against float64, and packed_out (refreshed by packed_store256 from the
    packed image of the old parameters) bitwise equal to a fresh pack of the new parameters."""
    L = _L()
    H = 256
    net = _net(O, A, H)
    P = po.param_count(O, H, A)
    params0, m0, v0 = _opt_state(O, A, H, seed=21 + O)
    rng = np.random.default_rng(O)
    grad = (rng.normal(size=P) * 10.0 ** rng.uniform(-4, -1, size=P)).astype(np.float32)
    gdev = torch.tensor(grad, device=_dev())
    packed0 = _pack(net, torch.tensor(params0, device=_dev()))
    lr = 1e-3
    w = _Worst()
    for step in (1, 37):
        for clip in (True, False):
            for grad_scale in (1.0, 0.25):
                st = _State(net, params0, m0, v0)
                packed = packed0.clone()
                norm = _nan(1)
                gn = _norm64(grad * np.float32(grad_scale))
                mgn = (0.25 if clip else 4.0) * gn
                L.check(L.lib().drl_clip_adam(C.byref(net), st.p.data_ptr(), gdev.data_ptr(), st.m.data_ptr(), st.v.data_ptr(), step, lr,
                                              BETA1, BETA2, EPS, mgn, grad_scale, packed.data_ptr(), norm.data_ptr(), L.stream_ptr()))
                w.add("norm rel", abs(float(norm.item()) - gn) / gn)
                assert abs(float(norm.item()) - gn) <= 1e-6 * gn
                _check_adam(w, st, params0, m0, v0, grad, step, lr, mgn, grad_scale)
                assert torch.equal(packed, _pack(net, st.p)), f"step {step} clip {clip} scale {grad_scale}: packed_out is stale"
    print(f"H=256 O={O} A={A}: worst {w}")


# ------------------------------------------------------------------------------------------------
# C. The 256-wide gradient over several 524,288-sample chunks: exact decomposition into single-chunk pieces
# ------------------------------------------------------------------------------------------------
# With the advantage statistics passed explicitly, the gradient is a mean of per-sample terms, and M enters a sample's
# bf16-rounded values only through inv_m = 1 / M (update256.cu).  A piece of n = M / 2^j samples has fl(1 / n) = 2^j fl(1 / M),
# so every per-sample rounding is the same and the full call F equals sum_i (n_i / M) P_i up to the order of fp32 sums.
C_CASES = [
    # O, A, M, piece denominators, permuted idx, index of a piece without heavy samples to compare with the oracle (or None)
    (4, 2, 8 * 65_545, (2, 4, 8, 8), True, 2),          # 2 chunks, the second 72 samples: one partial tile, fewer tiles than CTAs
    (4, 2, 16 * 65_545, (4, 4, 4, 4), True, None),      # 3 chunks, the last 144 samples
    (4, 2, 8 * 65_545, (2, 4, 8, 8), False, None),      # idx = NULL
    (6, 3, 8 * 65_545, (2, 4, 8, 8), True, 2),          # RW = 16
]


@pytest.mark.parametrize("O,A,M,pieces,with_idx,oracle_piece", C_CASES)
def test_grad_h256_multi_chunk_equals_weighted_single_chunk_pieces(O, A, M, pieces, with_idx, oracle_piece):
    H = 256
    net = _net(O, A, H)
    mb_start = 1234
    B = mb_start + M + 99
    params, _, _ = _opt_state(O, A, H, seed=31)
    idx = _perm(B, seed=M + O) if with_idx else None
    order = idx.cpu().numpy().astype(np.int64) if with_idx else np.arange(B)
    last = (M - 1) // CHUNK_256 * CHUNK_256           # first position of the last chunk
    tail = order[mb_start + last:mb_start + M]
    rec, _ = _records(net, O, A, params, B, seed=M + 3 * O, heavy=tail)   # the ragged last chunk dominates the gradient
    stats = torch.tensor([[0.3, 2.0]], device=_dev())
    ws = _workspace(net)
    packed = _pack(net, torch.tensor(params, device=_dev()))
    gF, tF = _grad(net, packed, rec, idx, mb_start, M, stats, ws, 1)
    gF2, tF2 = _grad(net, packed, rec, idx, mb_start, M, stats, ws, 1)
    assert torch.equal(gF, gF2) and torch.equal(tF, tF2), "the multi-chunk gradient is not deterministic"
    gF, tF = gF.cpu().numpy(), tF.cpu().numpy()
    combo = np.zeros(gF.shape, np.float64)
    tcombo = np.zeros(6, np.float64)
    off, piece_grads = 0, []
    for d in pieces:
        n = M // d
        assert n * d == M and n <= CHUNK_256
        g, t = _grad(net, packed, rec, idx, mb_start + off, n, stats, ws, 1)
        g, t = g.cpu().numpy(), t.cpu().numpy()
        combo += g.astype(np.float64) / d
        tcombo += t[:6].astype(np.float64) / d
        piece_grads.append((off, n, g, t))
        off += n
    assert off == M
    name, err = _per_tensor(gF, combo, O, A, H)
    # what losing the last chunk would do (its share of the mean, from a call over the tail alone)
    gT, _ = _grad(net, packed, rec, idx, mb_start + last, M - last, stats, ws, 1)
    lost = _per_tensor(combo - gT.cpu().numpy().astype(np.float64) * ((M - last) / M), combo, O, A, H)
    terr = np.abs(tF[:6] - tcombo) / (np.abs(tcombo) + 1e-6)
    print(f"H=256 O={O} M={M} pieces={pieces} idx={'perm' if with_idx else 'NULL'}: full vs weighted pieces worst tensor "
          f"{name} {err:.2e}; loss terms rel {terr.max():.2e}; a lost last chunk would give {lost[1]:.2e} ({lost[0]})")
    assert err < C_BAR, (name, err)
    assert lost[1] > 100 * C_BAR, lost
    np.testing.assert_allclose(tF[:6], tcombo, rtol=1e-4, atol=1e-6)
    if oracle_piece is not None:          # close the chain back to the reference maths
        off, n, g, t = piece_grads[oracle_piece]
        sel = order[mb_start + off:mb_start + off + n]
        assert not np.isin(sel, tail).any()
        r = rec.cpu().numpy()[sel]
        RW = r.shape[1]
        wt, wg = po.minibatch_grad_bf16_emulated(params, r[:, :O], r[:, RW - 1].view(np.int32), r[:, RW - 4], r[:, RW - 3],
                                                 r[:, RW - 2], O, H, A, 0.3, 2.0, tanh_fn=_gpu_tanh)
        worst = _per_tensor(g, wg, O, A, H)
        print(f"   piece {oracle_piece} ({n} samples) vs the bf16-emulating oracle: worst tensor {worst}")
        assert worst[1] < 2e-3, worst
        np.testing.assert_allclose(t[:6], wt, rtol=1e-4, atol=2e-5)


# ------------------------------------------------------------------------------------------------
# D. Trainer-level replay: learning rate, step numbering, statistics rows and loss-term rows of a whole update
# ------------------------------------------------------------------------------------------------
def _replay(tr, params0, m0, v0, step0, lr, stats_shift=0):
    """The update's optimizer steps, one by one: drl_ppo_minibatch_grad on a fresh pack of the replay's parameters (the
    trainer's records, permutations and statistics rows), then the oracle's clip + Adam.  Returns (params, m, v, terms)."""
    cfg = tr.cfg
    net = tr.net
    M = cfg.minibatch_size
    ws = _workspace(net)
    p, m, v = params0, m0, v0
    terms = []
    for e in range(cfg.update_epochs):
        for j in range(tr.n_mb):
            k = (j + stats_shift) % tr.n_mb
            packed = _pack(net, torch.tensor(p, device=_dev()))
            g, t = _grad(net, packed, tr.records, tr.idx[e], j * M, M, tr.adv_stats[e, k], ws, 1)
            p, m, v, _ = po.clip_adam(p, g.cpu().numpy(), m, v, step0 + e * tr.n_mb + j + 1, lr, cfg.max_grad_norm)
            terms.append(t.cpu().numpy())
    return p, m, v, np.stack(terms)


def _replay_errors(tr, got, want):
    p, m, v, terms = got
    wp, wm, wv, wt = want
    # loss terms: per term (column), the worst deviation over the update's rows relative to the term's largest magnitude
    scale = np.maximum(np.abs(wt[:, :6]).max(0), 1e-3)
    return {"params abs": float(np.abs(p - wp).max()),
            "m rel": _norm64(m - wm) / _norm64(wm),
            "v rel": _norm64(v - wv) / _norm64(wv),
            "terms rel": float((np.abs(terms[:, :6] - wt[:, :6]).max(0) / scale).max())}


def _trainer_replay_check(tr, nu, bars):
    torch.cuda.synchronize()
    params0 = tr.agent.flat_params.cpu().numpy()
    m0, v0 = tr.exp_avg.cpu().numpy(), tr.exp_avg_sq.cpu().numpy()
    step0, u = tr.adam_step, tr.update_idx
    tr.update(nu)
    torch.cuda.synchronize()
    got = (tr.agent.flat_params.cpu().numpy(), tr.exp_avg.cpu().numpy(), tr.exp_avg_sq.cpu().numpy(), tr.loss_terms.cpu().numpy())
    lr = (1.0 - u / nu) * tr.cfg.learning_rate
    err = _replay_errors(tr, got, _replay(tr, params0, m0, v0, step0, lr))
    # the same replay with the learning rate of the previous update, and with the statistics rows shifted by one
    lr_off = _replay_errors(tr, got, _replay(tr, params0, m0, v0, step0, (1.0 - (u - 1) / nu) * tr.cfg.learning_rate))
    row_off = _replay_errors(tr, got, _replay(tr, params0, m0, v0, step0, lr, stats_shift=1)) if tr.n_mb > 1 else None
    print(f"update {u} (lr {lr:.3e}, Adam steps {step0 + 1}..{tr.adam_step}) vs replay: {err}")
    print(f"   replay with the lr of update {u - 1}: {lr_off}")
    if row_off is not None:
        print(f"   replay with the statistics rows shifted by one: {row_off}")
    for key, bar in bars.items():
        assert err[key] < bar, (key, err[key], bar)
    assert lr_off["params abs"] > 10 * bars["params abs"]
    if row_off is not None:
        assert row_off["terms rel"] > 10 * bars["terms rel"]


def test_trainer_h64_graph_replayed_update_vs_step_by_step_replay():
    """PPOTrainer at hidden = 64 on the tcgen05 path, 4 minibatches per launch, updates 2 and 3 replayed from a CUDA graph:
    update 3 equals its 16 optimizer steps replayed one by one with the lr of update 3 and Adam steps 49..64."""
    import deep_rl_b200 as drl
    cfg = drl.PPOConfig(num_envs=256, num_steps=32, update_precision="bf16", cuda_graph=True)
    tr = drl.PPOTrainer(cfg)
    assert tr.mb_per_launch == 4 and tr.n_mb == 4
    nu = 8
    for _ in range(3):
        tr.update(nu)
    assert tr._graph is not None and tr.adam_step == 48
    _trainer_replay_check(tr, nu, REPLAY_BARS)


def test_trainer_h256_multi_chunk_update_vs_step_by_step_replay():
    """PPOTrainer at hidden = 256 with one 524,416-sample minibatch (two chunks of the 256-wide gradient): its 4 optimizer
    steps (drl_ppo_minibatch_grad + drl_clip_adam with the packed refresh) equal the step-by-step replay."""
    import deep_rl_b200 as drl
    cfg = drl.PPOConfig(hidden=256, num_envs=4097, num_steps=128, num_minibatches=1)
    tr = drl.PPOTrainer(cfg)
    assert cfg.minibatch_size == 524_416 > CHUNK_256 and tr.n_mb == 1
    nu = 4
    tr.update(nu)                 # update 0 ...
    _trainer_replay_check(tr, nu, REPLAY_BARS)   # ... update 1 replayed
