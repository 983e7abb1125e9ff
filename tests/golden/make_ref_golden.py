"""Generate tests/golden/ref_ppo_seed1.npz from the UNMODIFIED reference script.

Run once, in the authoring container (needs /root/reference; the GPU box never runs this):

    python tests/golden/make_ref_golden.py

How: `runpy.run_path('/root/reference/deep_rl/ppo.py')` with oracle/gym_shim on sys.path as `gym`
(gym 0.21 itself is not installable here, SURVEY.md 8c).  The script is not edited; values are
observed by wrapping three library entry points it calls -- `np.random.permutation` (ppo.py:155),
`torch.nn.utils.clip_grad_norm_` (ppo.py:191) and `torch.optim.Adam.step` (ppo.py:192) -- and
reading the script's module globals from the calling frame at those moments.
"""
import contextlib
import io
import os
import re
import runpy
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = "/root/reference/deep_rl/ppo.py"
sys.path.insert(0, os.path.join(ROOT, "oracle", "gym_shim"))
sys.path.insert(0, ROOT)

GAE_UPDATES = (0, 1, 2, 50, 155)   # updates whose GAE inputs/outputs are stored
DETAIL_UPDATE = 0                   # update whose 16 optimizer steps are stored in full

rec = {"perms": [], "mb": [], "gae": {}}
state = {"adam_calls": 0}


def _script_globals():
    f = sys._getframe(1)
    while f is not None:
        g = f.f_globals
        if "num_updates" in g and "agent" in g and "observations" in g and g.get("__name__") == "__main__":
            return g
        f = f.f_back
    raise RuntimeError("reference frame not found")


def _flat(params, grad=False):
    return torch.cat([(p.grad if grad else p.detach()).reshape(-1) for p in params]).numpy().copy()


_orig_perm = np.random.permutation
_orig_clip = torch.nn.utils.clip_grad_norm_
_orig_step = torch.optim.Adam.step


def perm_spy(x):
    out = _orig_perm(x)
    g = _script_globals()
    if g["update"] == DETAIL_UPDATE:
        rec["perms"].append(np.array(out, dtype=np.int64))
    return out


def clip_spy(parameters, max_norm, *a, **k):
    parameters = list(parameters)
    g = _script_globals()
    if g["update"] == DETAIL_UPDATE:
        state["pre"] = _flat(parameters, grad=True)
    norm = _orig_clip(parameters, max_norm, *a, **k)
    state["norm"] = float(norm)
    return norm


def step_spy(self, *a, **k):
    g = _script_globals()
    upd = g["update"]
    call = state["adam_calls"]
    state["adam_calls"] += 1
    params = list(g["agent"].parameters())
    if call % 16 == 0 and upd in GAE_UPDATES:
        rec["gae"][upd] = {k2: g[k2].detach().numpy().copy() for k2 in
                           ("observations", "values", "actions", "log_probs", "rewards", "dones", "advantages", "returns")}
    if upd == DETAIL_UPDATE:
        if call == 0:
            rec["init_params"] = _flat(params)
        entry = {
            "lr": float(self.param_groups[0]["lr"]),
            "terms": np.array([float(g["loss"]), float(g["pg_loss"]), float(g["v_loss"]), float(g["entropy_loss"])], np.float64),
            "grad_pre": state["pre"], "norm": state["norm"],
        }
        out = _orig_step(self, *a, **k)
        entry["params_after"] = _flat(params)
        rec["mb"].append(entry)
        return out
    return _orig_step(self, *a, **k)


def main():
    np.random.permutation = perm_spy
    torch.nn.utils.clip_grad_norm_ = clip_spy
    torch.optim.Adam.step = step_spy
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        g = runpy.run_path(REF, run_name="__main__")
    np.random.permutation = _orig_perm
    torch.nn.utils.clip_grad_norm_ = _orig_clip
    torch.optim.Adam.step = _orig_step

    eps = np.array([(int(m.group(1)), float(m.group(2))) for m in
                    re.finditer(r"global_step=(\d+), episodic_return=([0-9.]+)", buf.getvalue())], dtype=np.float64)
    out = {
        "init_params": rec["init_params"],
        "perms": np.stack(rec["perms"]),
        "episodes": eps,
        "final_params": _flat(list(g["agent"].parameters())),
        "hyper": np.array([g["gamma"], g["gae_lambda"], g["learning_rate"], g["clip_coef"], g["ent_coef"],
                           g["vf_coef"], g["max_grad_norm"], g["num_steps"], g["num_updates"], g["minibatch_size"],
                           g["update_epochs"], g["seed"]], dtype=np.float64),
        # ppo.py:194-195 as the script leaves it after the last update (values / returns of update 155 are stored below)
        "explained_var": np.array(float(g["explained_var"]), dtype=np.float64),
    }
    for upd, d in rec["gae"].items():
        for k, v in d.items():
            out[f"u{upd}_{k}"] = v
    for key in ("lr", "terms", "grad_pre", "norm", "params_after"):
        out[f"mb_{key}"] = np.stack([np.asarray(e[key]) for e in rec["mb"]])
    # the 16 pre-clip gradients go to a file of their own, so that neither file is larger than 1 MB
    path = os.path.join(ROOT, "tests", "golden", "ref_ppo_seed1.npz")
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "ref_ppo_seed1_grads.npz"), mb_grad_pre=out.pop("mb_grad_pre"))
    np.savez_compressed(path, **out)
    print(f"wrote {path} (+ _grads): {len(eps)} episodes, adam calls {state['adam_calls']}, "
          f"first/last-20 mean return {eps[:20, 1].mean():.1f} / {eps[-20:, 1].mean():.1f}")
    print({k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
