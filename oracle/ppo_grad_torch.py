"""TEST INFRASTRUCTURE ONLY (see oracle/kbot_oracle.py header): reference gradients of the PPO minibatch loss.

The forward pass restates _ppo_scan_fn (train.py:1435-1508: actor log-prob / entropy of the stored action, critic value,
carries reset where done) with torch float64 ops, the loss is kbot_oracle.ppo_loss (ksim.compute_ppo_loss [U]), and the
gradients come from torch autograd -- an implementation independent of the hand-derived backward kernels it checks.
Parity unpinned (DESIGN.md section 2): the reference itself cannot be run here."""
from __future__ import annotations

import math

import numpy as np
import torch

import kbot_oracle as O


def _t(x):
    return torch.tensor(np.asarray(x, np.float64), dtype=torch.float64)


def weights_to_torch(w: dict, requires_grad=True) -> dict:
    out = {"w_in": _t(w["w_in"]), "b_in": _t(w["b_in"]), "w_out": _t(w["w_out"]), "b_out": _t(w["b_out"]),
           "layers": [{k: _t(l[k]) for k in ("w_ih", "w_hh", "b")} for l in w["layers"]]}
    if requires_grad:
        for v in [out["w_in"], out["b_in"], out["w_out"], out["b_out"]] + [l[k] for l in out["layers"] for k in l]:
            v.requires_grad_(True)
    return out


def trunk(w, obs, carry):
    """carry: [N, depth, 2, H] -> (out, new_carry); eqx Linear / LSTMCell (kbot_oracle.trunk_forward)."""
    x = obs @ w["w_in"].T + w["b_in"]
    new = []
    for l, lw in enumerate(w["layers"]):
        h, c = carry[:, l, 0], carry[:, l, 1]
        lin = x @ lw["w_ih"].T + h @ lw["w_hh"].T + lw["b"]
        H = h.shape[-1]
        i, f, g, o = lin[:, :H], lin[:, H:2 * H], lin[:, 2 * H:3 * H], lin[:, 3 * H:]
        c2 = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
        h2 = torch.sigmoid(o) * torch.tanh(c2)
        new.append(torch.stack([h2, c2], dim=1))
        x = h2
    return x @ w["w_out"].T + w["b_out"], torch.stack(new, dim=1)


def ppo_minibatch_loss(wa, wc, actor_obs, critic_obs, action, done, old_log_probs, advantages, value_targets, old_values,
                       p: O.OracleParams, hyper: dict, carry0: dict | None = None):
    """All inputs numpy [T, N, ...].  carry0: the carries at the first step, {"actor", "critic": [N, depth, 2, H],
    "lpf_params": [N, 20]} (None = zeros, get_initial_model_carry).
    Returns (loss, (mean policy, mean value, mean entropy), log_probs, values)."""
    T, N = done.shape
    H, depth = p.hidden_size, p.depth
    a_obs, c_obs, act = _t(actor_obs), _t(critic_obs), _t(action)
    keep = _t(1.0 - done.astype(np.float64))
    if carry0 is None:
        ca = torch.zeros((N, depth, 2, H), dtype=torch.float64)
        cc = torch.zeros((N, depth, 2, H), dtype=torch.float64)
        lpf = torch.zeros((N, O.NUM_JOINTS), dtype=torch.float64)
    else:
        ca, cc, lpf = _t(carry0["actor"]), _t(carry0["critic"]), _t(carry0["lpf_params"])
        assert ca.shape == cc.shape == (N, depth, 2, H) and lpf.shape == (N, O.NUM_JOINTS)
    jb = _t(O.joint_biases(np.float64))
    lps, ents, vals = [], [], []
    for t in range(T):
        out, ca = trunk(wa, a_obs[t], ca)
        mean_raw = out[:, :20] + jb + torch.cat([torch.zeros((N, 10), dtype=torch.float64), a_obs[t][:, -10:]], dim=1)
        std = torch.clamp((torch.nn.functional.softplus(out[:, 20:]) + p.min_std) * p.var_scale, max=p.max_std)
        lpf = lpf + p.lpf_alpha * (mean_raw - lpf)
        z = (act[t] - lpf) / std
        lps.append((-0.5 * z * z - 0.5 * math.log(2 * math.pi)).sum(-1) - torch.log(std).sum(-1))
        ents.append(torch.log(std).sum(-1) + 20 * (0.5 + 0.5 * math.log(2 * math.pi)))
        v, cc = trunk(wc, c_obs[t], cc)
        vals.append(v[:, 0])
        k = keep[t]
        ca, cc, lpf = ca * k[:, None, None, None], cc * k[:, None, None, None], lpf * k[:, None]
    lp, ent, val = torch.stack(lps), torch.stack(ents), torch.stack(vals)
    eps, lcv = hyper.get("clip_param", 0.2), hyper.get("log_clip_value", 10.0)
    ratio = torch.exp(torch.clamp(lp - _t(old_log_probs), -lcv, lcv))
    adv = _t(advantages)
    pol = torch.minimum(ratio * adv, torch.clamp(ratio, 1 - eps, 1 + eps) * adv)
    err = _t(value_targets) - val
    vl = 0.5 * err * err
    if hyper.get("use_clipped_value_loss", True):
        vo = _t(old_values)
        errc = _t(value_targets) - (vo + torch.clamp(val - vo, -eps, eps))
        vl = 0.5 * torch.maximum(err * err, errc * errc)
    obj = pol - hyper.get("value_loss_coef", 0.5) * vl + hyper.get("entropy_coef", 0.004) * ent
    return -obj.mean(), (pol.mean(), vl.mean(), ent.mean()), lp, val


def ppo_minibatch_grads(w_actor: dict, w_critic: dict, batch: dict, p: O.OracleParams, hyper: dict | None = None,
                        carry0: dict | None = None):
    """batch: actor_obs [T,N,65], critic_obs [T,N,475], action [T,N,20], done [T,N] bool, old_log_probs, advantages,
    value_targets, old_values [T,N]; carry0 as in ppo_minibatch_loss.  Returns (loss, stats, grads_actor, grads_critic,
    log_probs, values) with grads in the eqx layout."""
    hyper = hyper or {}
    wa, wc = weights_to_torch(w_actor), weights_to_torch(w_critic)
    loss, stats, lp, val = ppo_minibatch_loss(wa, wc, batch["actor_obs"], batch["critic_obs"], batch["action"], batch["done"],
                                              batch["old_log_probs"], batch["advantages"], batch["value_targets"],
                                              batch["old_values"], p, hyper, carry0)
    loss.backward()

    def grads(w):
        z = lambda v: (v.grad if v.grad is not None else torch.zeros_like(v)).numpy()
        return {"w_in": z(w["w_in"]), "b_in": z(w["b_in"]), "w_out": z(w["w_out"]), "b_out": z(w["b_out"]),
                "layers": [{k: z(l[k]) for k in ("w_ih", "w_hh", "b")} for l in w["layers"]]}

    return (float(loss.detach()), tuple(float(s.detach()) for s in stats), grads(wa), grads(wc), lp.detach().numpy(), val.detach().numpy())
