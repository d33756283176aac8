"""Shared helpers of the GPU parity tests: one seeded batch presented to both sides -- AoS numpy for the oracle,
SoA CUDA tensors for the library -- and the comparison rules.

Tolerances (BASELINE.json north_star): bit-exact for termination codes / done / success / indices; 1e-5 relative
for fp32 outputs.  A pure relative bound is meaningless at zero crossings, so every float comparison is
|gpu - oracle| <= RTOL * |oracle| + ATOL with ATOL = 1e-6 x the natural scale of the quantity (stated per call).
"""

from __future__ import annotations

import numpy as np
import torch

import kbot_oracle as O
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200 import synth
from kbot_joystick_b200.engine import KbotStep

RTOL = 1e-5
P = O.OracleParams()


def close(gpu, ref, name, rtol=RTOL, atol=1e-6):
    gpu = np.asarray(gpu)
    ref = np.asarray(ref)
    assert gpu.shape == ref.shape, f"{name}: shape {gpu.shape} vs {ref.shape}"
    err = np.abs(gpu.astype(np.float64) - ref.astype(np.float64))
    bound = rtol * np.abs(ref.astype(np.float64)) + atol
    bad = err > bound
    if bad.any():
        i = np.unravel_index(np.argmax(err - bound), err.shape)
        raise AssertionError(f"{name}: {bad.sum()}/{bad.size} outside rtol={rtol} atol={atol}; worst at {i}: "
                             f"gpu={gpu[i]!r} oracle={ref[i]!r} err={err[i]:.3e}")


def exact(gpu, ref, name):
    gpu = np.asarray(gpu)
    ref = np.asarray(ref)
    assert gpu.shape == ref.shape, f"{name}: shape {gpu.shape} vs {ref.shape}"
    if not np.array_equal(gpu, ref):
        bad = gpu != ref
        i = np.unravel_index(np.argmax(bad), bad.shape)
        raise AssertionError(f"{name}: {bad.sum()}/{bad.size} differ (bit-exact required); first at {i}: "
                             f"gpu={gpu[i]!r} oracle={ref[i]!r}")


class Batch:
    """T steps x N envs of synthetic state in both representations."""

    def __init__(self, seed: int, T: int, N: int, device):
        self.T, self.N, self.dev = T, N, device
        self.ld = (N + 3) // 4 * 4
        self.np = synth.make_batch(seed, T, N)
        b = self.np
        self.state = {k: synth.to_soa(v, 1, device) for k, v in b["state"].items()}
        self.noise = {k: synth.to_soa(v, 1, device) for k, v in b["noise"].items()}
        self.episode = {k: synth.to_soa(v, 0, device) for k, v in b["episode"].items()}
        self.cmd_rand = {k: synth.to_soa(v, 1, device) for k, v in b["cmd_rand"].items()}
        r0 = b["cmd0_rand"]
        self.cmd0_np = O.initial_command(r0["mode"], r0["u6"], r0["u_arms"], P)
        self.cmd0 = synth.to_soa(self.cmd0_np, 0, device)

    def state_at(self, t):
        return {k: v[t] for k, v in self.state.items()}

    def noise_at(self, t):
        return {k: v[t] for k, v in self.noise.items() if k != "eps_action"}

    def np_state_at(self, t):
        return {k: v[t] for k, v in self.np["state"].items()}

    def np_noise_at(self, t):
        return {k: v[t] for k, v in self.np["noise"].items()}


def make_engine(hidden=256, depth=2, gemm_path=L.GEMM_SIMT_FP32, seed=77, device=None, **overrides):
    """Engine + eqx-layout weights (numpy for the oracle, packed on the device for the library)."""
    eng = KbotStep(hidden_size=hidden, depth=depth, gemm_path=gemm_path, overrides=overrides)
    wa = synth.make_weights(seed, 65, 40, hidden, depth)
    wc = synth.make_weights(seed + 1, 475, 1, hidden, depth)
    eng.pack_weights(L.NET_ACTOR, synth.weights_to_device(wa, device))
    eng.pack_weights(L.NET_CRITIC, synth.weights_to_device(wc, device))
    return eng, wa, wc


def carry_to_np(c: torch.Tensor, n: int) -> np.ndarray:
    """library AoS [depth, 2, n, H] -> oracle [n, depth, 2, H]."""
    return np.moveaxis(c.detach().cpu().numpy(), 2, 0)[:n]


def carry_from_np(c: np.ndarray, device) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(np.moveaxis(c, 0, 2))).to(device)


def scaled_err(gpu, ref, rtol=RTOL, atol=1e-6) -> float:
    """max |gpu-ref| / (rtol |ref| + atol): <= 1 passes the north_star tolerance."""
    gpu = np.asarray(gpu, np.float64)
    ref = np.asarray(ref, np.float64)
    assert gpu.shape == ref.shape, (gpu.shape, ref.shape)
    if gpu.size == 0:
        return 0.0
    return float(np.max(np.abs(gpu - ref) / (rtol * np.abs(ref) + atol)))


def rollout_buffers(b: "Batch", hidden: int, depth: int, with_critic: bool = True, start: dict | None = None) -> dict:
    """Device buffers of kbs_rollout_io for batch b: zero-initialised carries (= get_initial_model_carry), or the
    mid-episode state `start` {"actor", "critic" [N, depth, 2, H], "lpf_params" [N, 20], "pg_carry" [N, 3], "command" [N, 16]}
    (oracle layout)."""
    T, N, ld, dev = b.T, b.N, b.ld, b.dev
    f = dict(device=dev, dtype=torch.float32)
    command = torch.zeros((T + 1, 16, ld), **f)
    command[0] = b.cmd0
    io = {
        "state": b.state, "noise": {k: v for k, v in b.noise.items() if k != "eps_action"}, "episode": b.episode,
        "eps_action": b.noise["eps_action"], "u_switch": b.cmd_rand["u_switch"], "cmd_mode": b.cmd_rand["mode"],
        "cmd_u6": b.cmd_rand["u6"], "cmd_u_arms": b.cmd_rand["u_arms"], "command": command,
        "pg_carry": torch.zeros((3, ld), **f),
        "actor_carry": torch.zeros((depth, 2, N, hidden), **f),
        "critic_carry": torch.zeros((depth, 2, N, hidden), **f) if with_critic else None,
        "lpf": torch.zeros((20, ld), **f),
        "actor_obs": torch.zeros((T, 65, ld), **f), "action": torch.zeros((T, 20, ld), **f),
        "log_prob": torch.zeros((T, ld), **f), "ctrl": torch.zeros((T, 20, ld), **f),
        "term_codes": torch.zeros((T, 3, ld), device=dev, dtype=torch.int32),
        "done": torch.zeros((T, ld), device=dev, dtype=torch.uint8),
        "success": torch.zeros((T, ld), device=dev, dtype=torch.uint8),
        "value": torch.zeros((T, ld), **f) if with_critic else None, "T": T,
    }
    if start is not None:
        command[0] = synth.to_soa(start["command"], 0, dev)
        io["pg_carry"] = synth.to_soa(start["pg_carry"], 0, dev)
        io["lpf"] = synth.to_soa(start["lpf_params"], 0, dev)
        io["actor_carry"] = carry_from_np(start["actor"], dev)
        if with_critic:
            io["critic_carry"] = carry_from_np(start["critic"], dev)
    return io


def oracle_rollout(b: "Batch", wa, wc, hidden: int, depth: int, with_critic: bool = True, p=None, start: dict | None = None) -> dict:
    """O.rollout_control_steps over batch b from zero carries, or from `start` (as in rollout_buffers)."""
    p = p or O.OracleParams(hidden_size=hidden, depth=depth)
    N = b.N
    if start is None:
        carry = {"actor": np.zeros((N, depth, 2, hidden), np.float32), "critic": np.zeros((N, depth, 2, hidden), np.float32),
                 "lpf_params": np.zeros((N, 20), np.float32)}
        cmd0, pg = b.cmd0_np, np.zeros((N, 3), np.float32)
    else:
        carry = {k: start[k] for k in ("actor", "critic", "lpf_params")}
        cmd0, pg = start["command"], start["pg_carry"]
    return O.rollout_control_steps(wa, wc, b.np["state"], b.np["noise"], b.np["episode"], b.np["cmd_rand"], cmd0,
                                   carry, pg, p, with_critic=with_critic)


def compare_rollout(io: dict, ref: dict, N: int, with_critic: bool = True) -> dict:
    """scaled errors (<= 1 passes) of every float output; integer outputs must be bit-exact (raises otherwise)."""
    s = synth.from_soa
    exact(s(io["term_codes"], N, (3,)), ref["codes"], "term_codes")
    exact(s(io["done"], N).astype(bool), ref["done"], "done")
    exact(s(io["success"], N).astype(bool), ref["success"], "success")
    e = {
        "actor_obs": scaled_err(s(io["actor_obs"], N, (65,)), ref["actor_obs"]),
        "action": scaled_err(s(io["action"], N, (20,)), ref["action"]),
        "log_prob": scaled_err(s(io["log_prob"], N), ref["log_prob"], atol=1e-5),   # |log_prob| ~ 10-60
        "ctrl": scaled_err(s(io["ctrl"], N, (20,)), ref["ctrl"], atol=1e-4),         # torques ~ 10-100 N m
        "command": scaled_err(s(io["command"][:-1], N, (16,)), ref["command"]),
        "command_next": scaled_err(s(io["command"][-1], N, (16,)), ref["command_next"]),
        "actor_carry": scaled_err(carry_to_np(io["actor_carry"], N), ref["carry"]["actor"]),
        "lpf": scaled_err(s(io["lpf"], N, (20,)), ref["carry"]["lpf_params"]),
        "pg_carry": scaled_err(s(io["pg_carry"], N, (3,)), ref["pg_carry"], atol=1e-5),
    }
    if with_critic:
        # critic inputs reach |x| ~ 50 (raw touch force, train.py:1413-1414): the fp32 rounding floor of its 475-term
        # input projection is ~475 eps |w x| ~ 3e-6 for ANY summation order, hence the 1e-5 absolute floor here.
        e["value"] = scaled_err(s(io["value"], N), ref["value"], atol=1e-5)
        e["critic_carry"] = scaled_err(carry_to_np(io["critic_carry"], N), ref["carry"]["critic"], atol=1e-5)
    return e


def run_rollout_case(seed: int, T: int, N: int, hidden: int, device, gemm_path=L.GEMM_SIMT_FP32, depth: int = 2,
                     with_critic: bool = True) -> dict:
    b = Batch(seed, T, N, device)
    eng, wa, wc = make_engine(hidden=hidden, depth=depth, gemm_path=gemm_path, device=device)
    io = rollout_buffers(b, hidden, depth, with_critic)
    l0 = eng.launches
    eng.rollout(io, N)
    torch.cuda.synchronize()
    assert eng.device_status() == 0, "persistent rollout kernel: a dependency wait timed out"
    ref = oracle_rollout(b, wa, wc, hidden, depth, with_critic)
    errs = compare_rollout(io, ref, N, with_critic)
    out = {"errors": errs, "launches": eng.launches - l0, "done_count": ref["done"].sum()}
    eng.close()
    return out


def ppo_batch(rng, T, N, H, p, wa, wc, carry0=None):
    """A stored minibatch with old log-probs / values taken near the current policy (so both clip branches occur).
    carry0 (oracle layout, see ppo_grad_torch.ppo_minibatch_loss): the start state the minibatch is evaluated from -- the
    old log-probs / values must come from the same one, or every ratio lands far from 1 and the policy gradient clips to 0."""
    import ppo_grad_torch as G

    f = np.float32
    b = {"actor_obs": rng.normal(0, 0.7, (T, N, 65)).astype(f), "critic_obs": rng.normal(0, 0.7, (T, N, 475)).astype(f),
         "action": (0.3 * rng.normal(size=(T, N, 20))).astype(f), "done": rng.random((T, N)) < 0.12,
         "advantages": rng.normal(size=(T, N)).astype(f), "value_targets": rng.normal(0, 0.5, (T, N)).astype(f),
         "old_log_probs": np.zeros((T, N), f), "old_values": np.zeros((T, N), f)}
    _, _, _, _, lp, val = G.ppo_minibatch_grads(wa, wc, b, p, carry0=carry0)
    b["old_log_probs"] = (lp + rng.normal(0, 0.15, (T, N))).astype(f)
    b["old_values"] = (val + rng.normal(0, 0.25, (T, N))).astype(f)
    return b


GATES = "ifgo"


def grad_blocks(net: str, key: str, H: int) -> list:
    """(label, row slice) blocks of one gradient tensor that the block-wise check bounds on their own scale: the i / f / g / o
    rows of an LSTM matrix or bias, the mean rows 0..19 and std rows 20..39 of the actor's output layer."""
    if key in ("w_ih", "w_hh", "b"):
        return [(g, slice(k * H, (k + 1) * H)) for k, g in enumerate(GATES)]
    if net == "actor" and key in ("w_out", "b_out"):
        return [("mean", slice(0, 20)), ("std", slice(20, 40))]
    return [("all", slice(None))]


def block_bound(ref_block: np.ndarray, ref_tensor: np.ndarray) -> float:
    """Rows of a weight-gradient GEMM each accumulate their own rows of dG, so their rounding scales with their own block."""
    return 3e-4 * float(np.abs(ref_block).max()) + 1e-6 * float(np.abs(ref_tensor).max()) + 1e-12


def grad_tensors(g: dict, depth: int):
    """(name, key, layer, array) over every tensor of an eqx-layout gradient dict (numpy or torch)."""
    a = lambda x: x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
    for k in ("w_in", "b_in", "w_out", "b_out"):
        yield k, k, a(g[k])
    for l in range(depth):
        for k in ("w_ih", "w_hh", "b"):
            yield f"layers[{l}].{k}", k, a(g["layers"][l][k])


def compare_grads_blockwise(got: dict, ref: dict, net: str, H: int, depth: int) -> list:
    """Every gradient tensor within 3e-4 of its scale (+1e-9), and every block of it within block_bound.  Returns the
    failures as strings."""
    bad = []
    for (name, key, g), (_, _, r) in zip(grad_tensors(got, depth), grad_tensors(ref, depth)):
        if not np.isfinite(g).all():
            bad.append(f"{net}.{name}: non-finite")
            continue
        err, scale = np.abs(g - r).max(), np.abs(r).max()
        if not err <= 3e-4 * scale + 1e-9:
            bad.append(f"{net}.{name}: max err {err:.3e} vs scale {scale:.3e}")
        for lab, rows in grad_blocks(net, key, H):
            e, bound = np.abs(g[rows] - r[rows]).max(), block_bound(r[rows], r)
            if not e <= bound:
                bad.append(f"{net}.{name}[{lab}]: max err {e:.3e} vs bound {bound:.3e} (block scale {np.abs(r[rows]).max():.3e})")
    return bad


def grad_block_ratios(got: dict, ref: dict, net: str, H: int, depth: int) -> dict:
    """{"net.tensor": its largest block error over that block's block_bound}: <= 1 passes the block check; the margin."""
    out = {}
    for (name, key, g), (_, _, r) in zip(grad_tensors(got, depth), grad_tensors(ref, depth)):
        out[f"{net}.{name}"] = max(float(np.abs(g[rows] - r[rows]).max()) / block_bound(r[rows], r)
                                   for _, rows in grad_blocks(net, key, H))
    return out


def ppo_device_batch(b: dict, dev, carry0=None) -> dict:
    """The library's form of a ppo_batch minibatch: SoA arrays, carries at the first step in the ABI layout."""
    d = lambda a, dt=None: synth.to_soa(a if dt is None else a.astype(dt), 1, dev)
    batch = {"actor_obs": d(b["actor_obs"]), "critic_obs": d(b["critic_obs"]), "action": d(b["action"]),
             "done": d(b["done"], np.uint8), "old_log_probs": d(b["old_log_probs"]), "advantages": d(b["advantages"]),
             "value_targets": d(b["value_targets"]), "old_values": d(b["old_values"])}
    if carry0 is not None:
        batch["actor_carry0"] = carry_from_np(carry0["actor"], dev)
        batch["critic_carry0"] = carry_from_np(carry0["critic"], dev)
        batch["lpf0"] = synth.to_soa(carry0["lpf_params"], 0, dev)
    return batch


def ppo_grad_compare(e, wa, wc, b: dict, p, dev, N: int, carry0=None, hyper=None, ratios: dict | None = None) -> tuple:
    """kbs_ppo_grad on minibatch b (from carry0, with loss hyper-parameters hyper) against torch.autograd in float64
    (oracle/ppo_grad_torch.py): asserts log-probs, values and loss statistics; returns (the list of gradient tensors /
    blocks outside their bound, the reference (loss, stats, grads_actor, grads_critic, log_probs, values)).  ratios, when
    given, receives grad_block_ratios of both nets."""
    import ppo_grad_torch as G

    S = synth.from_soa
    hyper = hyper or {}
    ref = G.ppo_minibatch_grads(wa, wc, b, p, hyper=hyper, carry0=carry0)
    loss, stats, ga_ref, gc_ref, lp_ref, val_ref = ref

    def nan_like_w(w):
        z = lambda a: torch.full(a.shape, float("nan"), device=dev)
        return {"w_in": z(w["w_in"]), "b_in": z(w["b_in"]), "w_out": z(w["w_out"]), "b_out": z(w["b_out"]),
                "layers": [{k: z(l[k]) for k in ("w_ih", "w_hh", "b")} for l in w["layers"]]}

    ga, gc = nan_like_w(wa), nan_like_w(wc)
    out = e.ppo_grad(ppo_device_batch(b, dev, carry0), ga, gc, n_envs=N, **hyper)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    close(S(out["log_probs"], N), lp_ref, "log_probs", atol=1e-4)
    close(S(out["values"], N), val_ref, "values", atol=1e-5)
    close(out["stats"].cpu().numpy(), np.array((loss,) + stats, np.float32), "loss stats", rtol=2e-5, atol=1e-5)
    bad = (compare_grads_blockwise(ga, ga_ref, "actor", p.hidden_size, p.depth) +
           compare_grads_blockwise(gc, gc_ref, "critic", p.hidden_size, p.depth))
    if ratios is not None:
        ratios.update(grad_block_ratios(ga, ga_ref, "actor", p.hidden_size, p.depth))
        ratios.update(grad_block_ratios(gc, gc_ref, "critic", p.hidden_size, p.depth))
    return bad, ref


def run_ppo_grad_case(dev, T, N, hidden, path, carry0=None, hyper=None, depth=2) -> list:
    """kbs_ppo_grad on a seeded minibatch against torch.autograd in float64 (ppo_grad_compare): asserts log-probs, values
    and loss statistics, returns the list of gradient tensors (or gate / mean / std blocks of them) outside their bound."""
    e, wa, wc = make_engine(hidden=hidden, depth=depth, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=hidden, depth=depth)
    rng = np.random.default_rng(90 + N)
    b = ppo_batch(rng, T, N, hidden, p, wa, wc, carry0=carry0)
    try:
        return ppo_grad_compare(e, wa, wc, b, p, dev, N, carry0=carry0, hyper=hyper)[0]
    finally:
        e.close()
