"""The fused entry points from a non-zero start state, and the loss branches of the PPO gradient.

Production never starts from zero: a rollout continues from the previous rollout's carries, a PPO minibatch starts from the
carries stored at its trajectories' first step.  From a zero start every gradient term that involves h0 or c0 is exactly zero
(step 0's dG0^T h0 in dW_hh, dc c0 sigma'(f) in the forget gate), so a kernel that ignored, swapped or mis-indexed the start
state would pass every zero-start test.  Here each env gets its own start state -- the final state of a warm-up rollout of
the oracle, or random carries with an unbounded cell state -- and the reference is the float64 autograd oracle
(oracle/ppo_grad_torch.py) or the NumPy oracle from the same carries."""

import numpy as np
import pytest
import torch

import harness as Hn
import kbot_oracle as O
import ppo_grad_torch as G
from harness import Batch, close
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200 import spec, synth

pytestmark = pytest.mark.gpu

S = synth.from_soa
SIMT = pytest.param(L.GEMM_SIMT_FP32, id="simt")
TF32 = pytest.param(L.GEMM_TC_3XTF32, id="tc3xtf32")
F16 = pytest.param(L.GEMM_TC_2XF16, id="tc2xf16")
PATHS = [SIMT, TF32, F16]
# the PPO gradient's forms: the FP16-split datapath runs the persistent update unless KBS_PPO_PER_STEP=1
GRAD_FORMS = [pytest.param(L.GEMM_SIMT_FP32, False, id="simt"), pytest.param(L.GEMM_TC_3XTF32, False, id="tc3xtf32"),
              pytest.param(L.GEMM_TC_2XF16, False, id="tc2xf16"), pytest.param(L.GEMM_TC_2XF16, True, id="tc2xf16-per-step")]


@pytest.fixture(scope="module")
def dev(cuda_device, lib_built):
    return cuda_device


# ---- start states ----------------------------------------------------------------------------------------------------------


def warm_start(wa, wc, N, H, depth, seed, steps=12):
    """The state a rollout leaves behind: the oracle's rollout of `steps` steps from zero on batch `seed` (envs done at
    the last step are back at zero, the others are mid-episode)."""
    p = O.OracleParams(hidden_size=H, depth=depth)
    b = synth.make_batch(seed, steps, N)
    r0 = b["cmd0_rand"]
    cmd0 = O.initial_command(r0["mode"], r0["u6"], r0["u_arms"], p)
    z = np.zeros((N, depth, 2, H), np.float32)
    ref = O.rollout_control_steps(wa, wc, b["state"], b["noise"], b["episode"], b["cmd_rand"], cmd0,
                                  {"actor": z, "critic": z.copy(), "lpf_params": np.zeros((N, 20), np.float32)},
                                  np.zeros((N, 3), np.float32), p)
    c = ref["carry"]
    return {"actor": c["actor"], "critic": c["critic"], "lpf_params": c["lpf_params"], "pg_carry": ref["pg_carry"],
            "command": ref["command_next"]}


def weights(H, depth):
    """The weights Hn.make_engine packs (seed 77), for the oracle side of a case that needs them before its engine."""
    return synth.make_weights(77, 65, 40, H, depth), synth.make_weights(78, 475, 1, H, depth)


def random_carry(rng, N, depth, H):
    c = np.empty((N, depth, 2, H), np.float32)
    c[:, :, 0] = rng.uniform(-0.95, 0.95, (N, depth, H))
    c[:, :, 1] = rng.normal(0, 2.0, (N, depth, H))            # the cell state is unbounded
    return c


def random_start(seed, N, depth, H):
    rng = np.random.default_rng(seed)
    return {"actor": random_carry(rng, N, depth, H), "critic": random_carry(rng, N, depth, H),
            "lpf_params": rng.normal(0, 0.3, (N, 20)).astype(np.float32)}


def start_state(kind, wa, wc, N, H, depth, seed):
    return warm_start(wa, wc, N, H, depth, seed) if kind == "warm" else random_start(seed, N, depth, H)


# ---- PPO gradient ------------------------------------------------------------------------------------------------------------


def clear_kinks(b, lp, val, hyper):
    """Move the stored old log-probs / values / targets off the kinks of the clipped loss (ratio at 1 +- eps, value change at
    +-eps, the two value errors equal): an entry within fp32 rounding of a kink could take the other branch on the GPU and
    change the gradient by a whole term."""
    eps = hyper.get("clip_param", 0.2)
    for _ in range(3):
        lr = lp - b["old_log_probs"]
        near = np.minimum(np.abs(lr - np.log1p(eps)), np.abs(lr - np.log1p(-eps))) < 3e-3
        b["old_log_probs"] = np.where(near, b["old_log_probs"] - 8e-3, b["old_log_probs"]).astype(np.float32)
        d = val - b["old_values"]
        near = np.abs(np.abs(d) - eps) < 1e-3
        b["old_values"] = np.where(near, b["old_values"] - 3e-3 * np.sign(d), b["old_values"]).astype(np.float32)
        err = b["value_targets"] - val
        errc = b["value_targets"] - (b["old_values"] + np.clip(val - b["old_values"], -eps, eps))
        near = np.abs(err * err - errc * errc) < 1e-4
        b["value_targets"] = np.where(near, b["value_targets"] + 5e-3, b["value_targets"]).astype(np.float32)
    return b


def make_ppo_batch(seed, T, N, p, wa, wc, carry0, hyper=None, edit=None):
    """Hn.ppo_batch from carry0; edit(b) changes it before the old log-probs / values are taken (done pattern)."""
    rng = np.random.default_rng(seed)
    b = Hn.ppo_batch(rng, T, N, p.hidden_size, p, wa, wc, carry0=carry0)
    if edit is not None:
        edit(b)
        _, _, _, _, lp, val = G.ppo_minibatch_grads(wa, wc, b, p, carry0=carry0)
        b["old_log_probs"] = (lp + rng.normal(0, 0.15, (T, N))).astype(np.float32)
        b["old_values"] = (val + rng.normal(0, 0.25, (T, N))).astype(np.float32)
    _, _, _, _, lp, val = G.ppo_minibatch_grads(wa, wc, b, p, carry0=carry0)
    return clear_kinks(b, lp, val, hyper or {})


def assert_start_state_matters(ref, ref0, depth):
    """Non-vacuous: from carry0 the reference gradients of every layer's w_hh and forget-gate bias rows, in both nets, differ
    from the zero-start ones by more than 100x the bound they are checked to."""
    H = ref[2]["layers"][0]["w_hh"].shape[1]
    f = slice(H, 2 * H)
    for net, g, g0 in (("actor", ref[2], ref0[2]), ("critic", ref[3], ref0[3])):
        for l in range(depth):
            for key, rows in (("w_hh", slice(None)), ("b", f)):
                r, r0 = g["layers"][l][key], g0["layers"][l][key]
                diff = np.abs(r[rows] - r0[rows]).max()
                assert diff > 100 * Hn.block_bound(r[rows], r), (net, l, key, diff, Hn.block_bound(r[rows], r))


def run_grad(dev, e, wa, wc, b, p, N, carry0, hyper, per_step, path, monkeypatch):
    monkeypatch.setenv("KBS_PPO_PER_STEP", "1" if per_step else "0")
    e.profile(True)
    bad, ref = Hn.ppo_grad_compare(e, wa, wc, b, p, dev, N, carry0=carry0, hyper=hyper)
    prof = e.profile_read()
    e.profile(False)
    persistent = prof.get("bptt_persist_kernel", (0, 0))[1]
    if path == L.GEMM_TC_2XF16 and not per_step:
        assert persistent > 0, "the persistent update did not run"
    else:
        assert persistent == 0
    assert not bad, bad
    return ref


START_CASES = [pytest.param(7, 70, 256, 2, None, id="7x70"),
               pytest.param(1, 64, 256, 2, None, id="T1"),              # dW_hh and the step-0 forget-gate term: all from carry0
               pytest.param(2, 96, 256, 2, "done0", id="T2-done0"),     # carry0 used at step 0, then reset for some envs
               pytest.param(6, 130, 128, 2, None, id="H128"),
               pytest.param(3, 5, 256, 2, None, id="N5"),
               pytest.param(4, 129, 256, 2, None, id="N129")]


@pytest.mark.parametrize("path,per_step", GRAD_FORMS)
@pytest.mark.parametrize("kind", ["warm", "random"])
@pytest.mark.parametrize("T,N,H,depth,pattern", START_CASES)
def test_ppo_grad_from_start_state(dev, T, N, H, depth, pattern, kind, path, per_step, monkeypatch):
    """kbs_ppo_grad with actor_carry0 / critic_carry0 / lpf0 (the run_net_k copy, the F.carry0 conversion of the persistent
    forward pass, lpf0 in the actor-head kernels) against float64 autograd from the same carries."""
    e, wa, wc = Hn.make_engine(hidden=H, depth=depth, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H, depth=depth)
    carry0 = start_state(kind, wa, wc, N, H, depth, seed=3000 + N)

    def done0(b):
        b["done"][0] = np.arange(N) % 3 == 0

    b = make_ppo_batch(2000 + T + N, T, N, p, wa, wc, carry0, edit=done0 if pattern == "done0" else None)
    try:
        ref = run_grad(dev, e, wa, wc, b, p, N, carry0, {}, per_step, path, monkeypatch)
    finally:
        e.close()
    assert_start_state_matters(ref, G.ppo_minibatch_grads(wa, wc, b, p), depth)


@pytest.mark.parametrize("path,per_step", [GRAD_FORMS[0], GRAD_FORMS[2], GRAD_FORMS[3]])
@pytest.mark.parametrize("kind", ["warm", "random"])
def test_ppo_grad_from_start_state_depth1(dev, kind, path, per_step, monkeypatch):
    """One LSTM layer: the persistent update accepts depth <= 2 and had never run at depth 1."""
    test_ppo_grad_from_start_state(dev, 7, 70, 256, 1, None, kind, path, per_step, monkeypatch)


@pytest.mark.parametrize("path,per_step", [GRAD_FORMS[2], GRAD_FORMS[3]])
def test_ppo_grad_from_start_state_long(dev, path, per_step, monkeypatch):
    """T = 130: above T = 127 the block actor head's shared memory exceeds 48 KB and the persistent update uses
    actor_head_fwd_bwd_warp_kernel instead (also reading lpf0)."""
    test_ppo_grad_from_start_state(dev, 130, 40, 256, 2, None, "random", path, per_step, monkeypatch)


def actor_std(wa, b, p, carry0=None):
    """The action std of every (t, env, joint) of minibatch b (float64 forward of the reference)."""
    T, N = b["done"].shape
    w = G.weights_to_torch(wa, requires_grad=False)
    ca = G._t(carry0["actor"]) if carry0 is not None else torch.zeros((N, p.depth, 2, p.hidden_size), dtype=torch.float64)
    a_obs, keep = G._t(b["actor_obs"]), G._t(1.0 - b["done"])
    out = []
    for t in range(T):
        o, ca = G.trunk(w, a_obs[t], ca)
        out.append(torch.clamp((torch.nn.functional.softplus(o[:, 20:]) + p.min_std) * p.var_scale, max=p.max_std))
        ca = ca * keep[t][:, None, None, None]
    return torch.stack(out).numpy()


BRANCHES = {
    "unclipped_value": {"use_clipped_value_loss": 0},
    "coefs": {"clip_param": 0.1, "value_loss_coef": 1.0, "entropy_coef": 0.01},
    "log_ratio_saturated": {},
    "std_clamped": {},
}


@pytest.mark.parametrize("path,per_step", GRAD_FORMS)
@pytest.mark.parametrize("branch", list(BRANCHES))
def test_ppo_grad_loss_branches(dev, branch, path, per_step, monkeypatch):
    """The gradient branches the default hyper-parameters and near-policy batches never take, in every head kernel
    (actor_head_fwd_bwd_{block,warp}, actor_head_bwd_warp, critic_{value_head,head_fwd_bwd,head_bwd}): the unclipped value
    loss, non-default clip / loss coefficients, log-ratios beyond log_clip_value (zero policy gradient) and the max_std clamp
    (zero std gradient).  The same hyper dict goes to the library and to the reference, and each branch is asserted to occur
    in the reference batch."""
    T, N, H = 6, 96, 256
    hyper = BRANCHES[branch]
    e, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H)
    if branch == "std_clamped":
        wa["b_out"] = wa["b_out"].copy()
        wa["b_out"][20:25] += 4.0
        e.pack_weights(L.NET_ACTOR, synth.weights_to_device(wa, dev))
    b = make_ppo_batch(4000 + len(branch), T, N, p, wa, wc, None, hyper=hyper)
    if branch == "log_ratio_saturated":
        rng = np.random.default_rng(5)
        shift = np.where(rng.random((T, N)) < 0.15, rng.choice([-15.0, 15.0], (T, N)), 0.0)
        b["old_log_probs"] = (b["old_log_probs"] + shift).astype(np.float32)
    _, _, _, _, lp, val = G.ppo_minibatch_grads(wa, wc, b, p, hyper=hyper)
    eps, lcv = hyper.get("clip_param", 0.2), hyper.get("log_clip_value", 10.0)
    lr = lp - b["old_log_probs"]
    ratio, adv = np.exp(np.clip(lr, -lcv, lcv)), b["advantages"]
    assert ((ratio > 1 + eps) & (adv > 0)).any() and ((ratio < 1 - eps) & (adv < 0)).any(), "the ratio clips on both sides"
    if hyper.get("use_clipped_value_loss", 1):
        d = val - b["old_values"]
        err2 = (b["value_targets"] - val) ** 2
        errc2 = (b["value_targets"] - b["old_values"] - np.clip(d, -eps, eps)) ** 2
        assert ((d > eps) & (errc2 > err2)).any() and ((d < -eps) & (errc2 > err2)).any(), "the value clip goes both ways"
    if branch == "log_ratio_saturated":
        assert (np.abs(lr) > lcv).any() and (np.abs(lr) < lcv).any()
    if branch == "std_clamped":
        std = actor_std(wa, b, p)
        assert (std >= p.max_std).any() and (std < p.max_std).any()
    try:
        run_grad(dev, e, wa, wc, b, p, N, None, hyper, per_step, path, monkeypatch)
    finally:
        e.close()


# ---- rollout ------------------------------------------------------------------------------------------------------------------


def rollout(dev, b, path, H, depth, with_critic, start, per_step=None, monkeypatch=None):
    if per_step is not None:
        monkeypatch.setenv("KBS_TC_PER_STEP", "1" if per_step else "0")
    e, _, _ = Hn.make_engine(hidden=H, depth=depth, gemm_path=path, device=dev)
    io = Hn.rollout_buffers(b, H, depth, with_critic, start=start)
    e.rollout(io, b.N)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    e.close()
    return io


def assert_scaled(errs):
    bad = {k: v for k, v in errs.items() if not v <= 1.0}
    assert not bad, f"scaled errors > 1: {bad} (all: {errs})"


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("T,N,H,depth,with_critic", [(6, 130, 256, 2, True), (5, 77, 128, 2, True), (5, 140, 256, 1, True),
                                                     (5, 200, 256, 2, False), (8, 2048, 256, 2, True)])
def test_rollout_from_mid_episode_state(dev, path, T, N, H, depth, with_critic):
    """kbs_rollout from non-zero actor / critic carries, lpf, pg_carry and command[0] (carry_convert_kernel's ABI -> split
    SB / FB modes, the lag state of the observations) against O.rollout_control_steps from the same state."""
    wa, wc = weights(H, depth)
    start = warm_start(wa, wc, N, H, depth, seed=6000 + N)
    b = Batch(6100 + N, T, N, dev)
    io = rollout(dev, b, path, H, depth, with_critic, start)
    ref = Hn.oracle_rollout(b, wa, wc, H, depth, with_critic, start=start)
    assert_scaled(Hn.compare_rollout(io, ref, N, with_critic))
    zero = Hn.oracle_rollout(b, wa, wc, H, depth, with_critic)
    assert np.abs(zero["carry"]["actor"] - ref["carry"]["actor"]).max() > 1e-3 and np.abs(zero["log_prob"][0] - ref["log_prob"][0]).max() > 1e-2


def test_rollout_from_mid_episode_state_persistent_vs_per_step(dev, monkeypatch):
    """The persistent recurrence kernel and the per-step launches from the same mid-episode state agree to rounding level
    (as from zero, test_rollout_persistent_vs_per_step_launches)."""
    T, N = 12, 2048
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=6500)
    b = Batch(6501, T, N, dev)
    a = rollout(dev, b, L.GEMM_TC_2XF16, 256, 2, True, start, per_step=False, monkeypatch=monkeypatch)
    c = rollout(dev, b, L.GEMM_TC_2XF16, 256, 2, True, start, per_step=True, monkeypatch=monkeypatch)
    close(a["actor_carry"].cpu().numpy(), c["actor_carry"].cpu().numpy(), "actor carry", atol=2e-6)
    close(a["critic_carry"].cpu().numpy(), c["critic_carry"].cpu().numpy(), "critic carry", atol=2e-6)
    close(S(a["action"], N, (20,)), S(c["action"], N, (20,)), "action")
    close(S(a["log_prob"], N), S(c["log_prob"], N), "log_prob", atol=1e-5)
    close(S(a["value"], N), S(c["value"], N), "value", atol=1e-5)
    close(S(a["lpf"], N, (20,)), S(c["lpf"], N, (20,)), "lpf")


def healthy_at(b: Batch, t: int):
    """No episode ends at step t: a call's first step has no done of the step before it, so the lag state of the projected
    gravity observation restarts only inside a call.  Splitting a rollout where no episode ends keeps the split exact."""
    st = b.np["state"]
    st["time"][t] = np.minimum(st["time"][t], 11.0)
    st["xpos"][t, :, spec.BODY_BASE, 2] = st["qpos"][t, :, 2]
    st["qpos"][t, :, 3:7] = np.array([1, 0, 0, 0], np.float32)
    st["xquat"][t, :, spec.BODY_BASE] = st["qpos"][t, :, 3:7]
    b.state = {k: synth.to_soa(v, 1, b.dev) for k, v in st.items()}


@pytest.mark.parametrize("path", PATHS)
def test_rollout_continuation_split_in_two_calls(dev, path):
    """One call over T1 + T2 steps against two calls of T1 and T2, the second starting from the first's carries, pg_carry,
    lpf and command[T1]: h crosses the call boundary as fp32 and is re-split by the same conversion, c stays fp32, so the
    two must be bit-identical -- and both match the oracle from a mid-episode start."""
    T1, T2, N = 21, 19, 2048                                   # T1 not a multiple of the 32-step scan chunks
    T = T1 + T2
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=7000)
    b = Batch(7001, T, N, dev)
    healthy_at(b, T1 - 1)
    whole = rollout(dev, b, path, 256, 2, True, start)
    ref = Hn.oracle_rollout(b, wa, wc, 256, 2, start=start)
    assert not ref["done"][T1 - 1].any() and ref["done"].sum() > 0
    assert_scaled(Hn.compare_rollout(whole, ref, N))

    def part(t0, t1):
        bb = Batch.__new__(Batch)
        bb.T, bb.N, bb.dev, bb.ld, bb.cmd0 = t1 - t0, N, dev, b.ld, b.cmd0
        bb.state = {k: v[t0:t1].contiguous() for k, v in b.state.items()}
        bb.noise = {k: v[t0:t1].contiguous() for k, v in b.noise.items()}
        bb.cmd_rand = {k: v[t0:t1].contiguous() for k, v in b.cmd_rand.items()}
        bb.episode = b.episode
        return bb

    e, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    first = Hn.rollout_buffers(part(0, T1), 256, 2, start=start)
    e.rollout(first, N)
    second = Hn.rollout_buffers(part(T1, T), 256, 2)
    second["command"][0] = first["command"][T1]
    for k in ("actor_carry", "critic_carry", "lpf", "pg_carry"):
        second[k] = first[k].clone()
    e.rollout(second, N)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    e.close()
    for k in ("actor_obs", "action", "log_prob", "ctrl", "term_codes", "done", "success", "value"):
        assert torch.equal(torch.cat([first[k], second[k]]), whole[k]), k
    assert torch.equal(torch.cat([first["command"][:T1], second["command"]]), whole["command"]), "command"
    for k in ("actor_carry", "critic_carry", "lpf", "pg_carry"):
        assert torch.equal(second[k], whole[k]), k


# ---- PPO variables ------------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("T,N,H", [(8, 50, 256), (5, 130, 128)])
def test_ppo_variables_from_start_state(dev, path, T, N, H):
    """kbs_ppo_variables from non-zero carries, the mirror carries included, against O.get_ppo_variables from the same
    carries; and the same trajectory in two calls (carries in / out between them) gives the same results."""
    e, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H, actor_mirror_loss_scale=1.0, critic_mirror_loss_scale=0.01)
    b = Batch(8000 + N, T, N, dev)
    rng = np.random.default_rng(8)
    obs = [O.get_observations(b.np_state_at(t), b.np_noise_at(t), b.np["episode"], None, Hn.P)[0] for t in range(T)]
    cmd = np.stack([b.cmd0_np] * T)
    done = rng.random((T, N)) < 0.15
    act = (np.stack([o["joint_position"] for o in obs]) + 0.2 * rng.standard_normal((T, N, 20))).astype(np.float32)
    w = warm_start(wa, wc, N, H, 2, seed=8100 + N)
    m = random_start(8200 + N, N, 2, H)
    carry0 = {"actor": w["actor"], "critic": w["critic"], "lpf_params": w["lpf_params"], "actor_mirror": m["actor"],
              "critic_mirror": m["critic"], "lpf_params_mirror": m["lpf_params"]}
    ref, c_end = O.get_ppo_variables(wa, wc, obs, cmd, act, done, dict(carry0), p, mirror=True)
    zero, _ = O.get_ppo_variables(wa, wc, obs, cmd, act, done, O.initial_model_carry((N,), p), p, mirror=True)
    assert np.abs(zero["log_probs"][0] - ref["log_probs"][0]).max() > 1e-2
    assert np.abs(zero["value_mirror_loss"][0] - ref["value_mirror_loss"][0]).max() > 1e-6
    m_obs = [O.mirror_obs(o) for o in obs]
    m_cmd = np.stack([O.mirror_cmd(c) for c in cmd])
    d = lambda a: synth.to_soa(a, 1, dev)
    arrays = {"a_obs": d(np.stack([O.actor_obs_from_dict(o, c) for o, c in zip(obs, cmd)])),
              "c_obs": d(np.stack([O.critic_obs_from_dict(o, c) for o, c in zip(obs, cmd)])),
              "am_obs": d(np.stack([O.actor_obs_from_dict(o, c) for o, c in zip(m_obs, m_cmd)])),
              "cm_obs": d(np.stack([O.critic_obs_from_dict(o, c) for o, c in zip(m_obs, m_cmd)])),
              "act": d(act), "done": d(done.astype(np.uint8))}

    def carries():
        return {"ac": Hn.carry_from_np(carry0["actor"], dev), "cc": Hn.carry_from_np(carry0["critic"], dev),
                "lpf": synth.to_soa(carry0["lpf_params"], 0, dev), "acm": Hn.carry_from_np(carry0["actor_mirror"], dev),
                "ccm": Hn.carry_from_np(carry0["critic_mirror"], dev), "lpfm": synth.to_soa(carry0["lpf_params_mirror"], 0, dev)}

    def run(c, t0, t1):
        a = {k: v[t0:t1].contiguous() for k, v in arrays.items()}
        mir = {"actor_obs": a["am_obs"], "critic_obs": a["cm_obs"], "actor_carry": c["acm"], "critic_carry": c["ccm"],
               "lpf": c["lpfm"], "actor_scale": p.actor_mirror_loss_scale, "critic_scale": p.critic_mirror_loss_scale}
        out = e.ppo_variables(a["a_obs"], a["act"], a["done"], c["ac"], c["lpf"], a["c_obs"], c["cc"], n_envs=N, mirror=mir)
        torch.cuda.synchronize()
        assert e.device_status() == 0
        return out

    c = carries()
    out = run(c, 0, T)
    close(S(out["log_probs"], N), ref["log_probs"][..., 0], "log_probs", atol=1e-4)
    close(S(out["entropy"], N), ref["entropy"][..., 0], "entropy", atol=1e-5)
    close(S(out["values"], N), ref["values"], "values", atol=1e-5)
    close(S(out["action_std"], N, (20,)), ref["action_std"], "action_std")
    close(S(out["action_mirror_loss"], N), ref["action_mirror_loss"], "action_mirror_loss", rtol=1e-4, atol=1e-6)
    close(S(out["value_mirror_loss"], N), ref["value_mirror_loss"], "value_mirror_loss", rtol=1e-4, atol=2e-7)
    close(Hn.carry_to_np(c["ac"], N), c_end["actor"], "actor carry")
    close(Hn.carry_to_np(c["cc"], N), c_end["critic"], "critic carry", atol=1e-5)
    close(S(c["lpf"], N, (20,)), c_end["lpf_params"], "lpf")
    close(Hn.carry_to_np(c["acm"], N), c_end["actor_mirror"], "actor_mirror carry")
    close(Hn.carry_to_np(c["ccm"], N), c_end["critic_mirror"], "critic_mirror carry", atol=1e-5)
    close(S(c["lpfm"], N, (20,)), c_end["lpf_params_mirror"], "lpf_params_mirror")
    # the same trajectory in two calls: the second continues from the carries the first left
    T1 = T // 2 + 1
    c2 = carries()
    o1, o2 = run(c2, 0, T1), run(c2, T1, T)
    for k in ("log_probs", "entropy", "values", "action_std", "action_mirror_loss", "value_mirror_loss"):
        assert torch.equal(torch.cat([o1[k], o2[k]])[..., :N], out[k][..., :N]), k      # lanes N..ld are padding
    for k in c:
        assert torch.equal(c2[k][..., :N], c[k][..., :N]), k
    e.close()
