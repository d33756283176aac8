"""Host-side pieces of kbs_ppo_variables_vjp that need no GPU: the float64 reference forward, the ctypes mirror of
kbs_ppo_cotangents, and the XLA-FFI target with its jax_ffi wrapper."""

import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest
import torch

import kbot_oracle as O
import ppo_grad_torch as G
from ppo_variables_ref import ppo_variables_torch
from kbot_joystick_b200 import synth

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("warm", [False, True], ids=["zero-start", "warm-start"])
def test_ppo_variables_torch_matches_the_loss_forward(warm):
    """ppo_variables_torch is the forward of ppo_minibatch_loss: the same log-probs and values, bitwise (same float64 ops),
    from zero and from non-zero start carries, with done-resets; entropy and action_std agree with their definitions."""
    T, N, H, depth = 4, 6, 32, 2
    p = O.OracleParams(hidden_size=H, depth=depth)
    wa, wc = synth.make_weights(3, 65, 40, H, depth), synth.make_weights(4, 475, 1, H, depth)
    rng = np.random.default_rng(0)
    b = {"actor_obs": rng.normal(0, 0.7, (T, N, 65)), "critic_obs": rng.normal(0, 0.7, (T, N, 475)),
         "action": 0.3 * rng.normal(size=(T, N, 20)), "done": rng.random((T, N)) < 0.3}
    carry0 = None
    if warm:
        carry0 = {"actor": rng.normal(0, 0.5, (N, depth, 2, H)), "critic": rng.normal(0, 0.5, (N, depth, 2, H)),
                  "lpf_params": rng.normal(0, 0.3, (N, 20))}
    ta, tc = G.weights_to_torch(wa, False), G.weights_to_torch(wc, False)
    v = ppo_variables_torch(ta, tc, b["actor_obs"], b["critic_obs"], b["action"], b["done"], p, carry0)
    z = np.zeros((T, N))
    _, _, lp, val = G.ppo_minibatch_loss(ta, tc, b["actor_obs"], b["critic_obs"], b["action"], b["done"], z, z, z, z, p, {},
                                         carry0)
    assert v["log_probs"].shape == (T, N) and v["values"].shape == (T, N) and v["action_std"].shape == (T, N, 20)
    assert torch.equal(v["log_probs"], lp) and torch.equal(v["values"], val)
    ent = torch.log(v["action_std"]).sum(-1) + 20 * (0.5 + 0.5 * np.log(2 * np.pi))
    assert torch.allclose(v["entropy"], ent, rtol=0, atol=1e-12)
    assert (v["action_std"] <= p.max_std).all()


def test_ppo_variables_torch_is_differentiable():
    """Arbitrary cotangents reach every weight tensor of both networks through torch.autograd.grad."""
    T, N, H = 3, 4, 16
    p = O.OracleParams(hidden_size=H, depth=1)
    wa, wc = synth.make_weights(5, 65, 40, H, 1), synth.make_weights(6, 475, 1, H, 1)
    rng = np.random.default_rng(1)
    ta, tc = G.weights_to_torch(wa), G.weights_to_torch(wc)
    v = ppo_variables_torch(ta, tc, rng.normal(size=(T, N, 65)), rng.normal(size=(T, N, 475)), rng.normal(size=(T, N, 20)),
                            np.zeros((T, N), bool), p)
    loss = sum((torch.tensor(rng.normal(size=t.shape)) * t).sum() for t in v.values())
    leaves = [ta["w_in"], ta["w_out"], tc["w_in"], tc["w_out"]] + [l[k] for w in (ta, tc) for l in w["layers"] for k in l]
    for g in torch.autograd.grad(loss, leaves):
        assert torch.isfinite(g).all() and g.abs().max() > 0


def test_cotangent_struct_mirror_matches_header():
    from kbot_joystick_b200 import _lib as L

    hdr = (ROOT / "include" / "kbotstep.h").read_text()
    body = re.search(r"typedef struct kbs_ppo_cotangents \{(.*?)\} kbs_ppo_cotangents;", hdr, flags=re.S).group(1)
    names = re.findall(r"const float\*\s*(\w+);", body)
    assert names == [f[0] for f in L.KbsPpoCotangents._fields_] == ["log_probs", "values", "entropy", "action_std"]
    assert C.sizeof(L.KbsPpoCotangents) == 4 * 8
    assert "kbs_ppo_variables_vjp" in L.EXPORTS
    decl = re.search(r"^int kbs_ppo_variables_vjp\((.*?)\);", hdr, flags=re.M | re.S).group(1)
    assert decl.count(",") + 1 == 10                       # the ctypes argtypes set in _lib.load()


def test_ffi_target_and_wrapper():
    """kbs_ppo_variables_vjp has an XLA-FFI handler bound to 11 buffers in and 5 out, forwarding to the entry point, and a
    jax_ffi wrapper registered under the same target (importable without jax)."""
    import kbot_joystick_b200.jax_ffi as kf

    assert kf._TARGETS["kbs_ppo_variables_vjp"] == "KbsPpoVariablesVjp"
    assert callable(kf.ppo_variables_vjp)
    cc = (ROOT / "kbot-joystick_b200" / "csrc" / "kbs_xla_ffi.cc").read_text()
    m = re.search(r"XLA_FFI_DEFINE_HANDLER_SYMBOL\(KbsPpoVariablesVjp, PpoVariablesVjpImpl,(.*?)\);", cc, flags=re.S)
    assert m, "no KbsPpoVariablesVjp handler"
    assert m.group(1).count(".Arg<") == 11 and m.group(1).count(".Ret<") == 5
    assert "kbs_ppo_variables_vjp(H(handle)" in cc
    # the flat gradient buffers have the size the handler's views walk (net_param_count)
    assert kf.net_param_count(65, 40, 256, 2) == 256 * 65 + 256 + 2 * (8 * 256 * 256 + 4 * 256) + 40 * 256 + 40
