"""TEST INFRASTRUCTURE ONLY: get_ppo_variables in float64 for the VJP tests (tests/test_gpu_ppo_vjp.py).

The forward restates _ppo_scan_fn (train.py:1435-1508) step by step with the oracle's torch pieces
(oracle/ppo_grad_torch.py: weights_to_torch, trunk) exactly as ppo_grad_torch.ppo_minibatch_loss does, but returns the four
PPO variables themselves as tensors of the autograd graph, so that torch.autograd.grad takes arbitrary cotangents."""
from __future__ import annotations

import math

import numpy as np
import torch

import kbot_oracle as O
from ppo_grad_torch import trunk


def _t(x):
    return torch.tensor(np.asarray(x, np.float64), dtype=torch.float64)


def ppo_variables_torch(wa, wc, actor_obs, critic_obs, action, done, p: O.OracleParams, carry0: dict | None = None) -> dict:
    """Torch weights wa / wc (ppo_grad_torch.weights_to_torch), numpy inputs [T, N, ...] and carry0 as in
    ppo_grad_torch.ppo_minibatch_loss.  Returns {"log_probs", "values", "entropy": [T, N], "action_std": [T, N, 20]}."""
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
    jb = _t(O.joint_biases(np.float64))
    lps, ents, vals, stds = [], [], [], []
    for t in range(T):
        out, ca = trunk(wa, a_obs[t], ca)
        mean_raw = out[:, :20] + jb + torch.cat([torch.zeros((N, 10), dtype=torch.float64), a_obs[t][:, -10:]], dim=1)
        std = torch.clamp((torch.nn.functional.softplus(out[:, 20:]) + p.min_std) * p.var_scale, max=p.max_std)
        lpf = lpf + p.lpf_alpha * (mean_raw - lpf)
        z = (act[t] - lpf) / std
        lps.append((-0.5 * z * z - 0.5 * math.log(2 * math.pi)).sum(-1) - torch.log(std).sum(-1))
        ents.append(torch.log(std).sum(-1) + 20 * (0.5 + 0.5 * math.log(2 * math.pi)))
        stds.append(std)
        v, cc = trunk(wc, c_obs[t], cc)
        vals.append(v[:, 0])
        k = keep[t]
        ca, cc, lpf = ca * k[:, None, None, None], cc * k[:, None, None, None], lpf * k[:, None]
    return {"log_probs": torch.stack(lps), "values": torch.stack(vals), "entropy": torch.stack(ents),
            "action_std": torch.stack(stds)}
