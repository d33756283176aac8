"""Every network depth kbs_create accepts (1 to KBS_MAX_DEPTH = 4) through every entry point, against the references the
depth-2 tests use: the NumPy oracle in fp32 at the harness tolerances, and float64 autograd (oracle/ppo_grad_torch.py) with
the block-wise gradient bounds.

Depth is a task setting.  At depth 2 a layer loop that reads the wrong ping-pong slot, or converts the carries of the first
two layers only, still gives the right answer.  The persistent tensor-core kernels hold at most two layers, so above depth 2
the tensor-core datapaths run the per-step launches: the rollout's layer loop over the xmid slots (l - 1) & 1, the ABI-carry
fallback (pack_rows + fb_convert, taken when nets x depth x 2 > 8: depth >= 3 with the critic), kbs_tc_lstm_stack's
x_sb[l & 1] ping-pong (actor / critic / policy step), and the per-step PPO gradient on 3xTF32 and FP16-split.  Depth 1 runs
the persistent kernels with one layer.  Where a tensor-core entry point has no per-step form above depth 2 (dist.mean(), the
mirror pass, the online step), it refuses with KBS_E_SHAPE before it launches anything.

The worst scaled errors of the rollouts and the gradient block margins (block error / harness.block_bound, per layer) are
printed, so `pytest -s` puts the precision margin of each datapath and depth on record."""

import ctypes as C

import numpy as np
import pytest
import torch

import harness as Hn
import kbot_oracle as O
import ppo_grad_torch as G
from harness import Batch, P, close
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200 import checkpoint, synth
from kbot_joystick_b200.engine import KbotStep
from kbot_joystick_b200.ppo import PpoUpdater
from test_gpu_ppo_epoch import assert_same, epoch_with_pass_states, make_rollout, reference_epoch, state
from test_gpu_ppo_epoch import refill as refill_rollout
from test_gpu_ppo_iteration import assert_iteration_equal, ending_at, reward_carry
from test_gpu_ppo_update import assert_repacked, check_update, clip_limit, minibatch, refill, snapshot, weights_at
from test_gpu_rollout_step import (TRAJ, assert_steps_equal_record, hand_loop, online_loop, rc_of, step_inputs, stored,
                                   traj_buffers)
from test_gpu_start_state import assert_start_state_matters, make_ppo_batch, warm_start, weights

pytestmark = pytest.mark.gpu

S = synth.from_soa
SIMT, TF32, F16 = L.GEMM_SIMT_FP32, L.GEMM_TC_3XTF32, L.GEMM_TC_2XF16
NAMES = {SIMT: "simt", TF32: "tc3xtf32", F16: "tc2xf16"}
PATHS = list(NAMES)
L_SHAPE = -2                                   # KBS_E_SHAPE


@pytest.fixture(scope="module")
def dev(cuda_device, lib_built):
    return cuda_device


def assert_scaled(errs: dict, what: str):
    worst = max(errs, key=errs.get)
    print(f"\n[depths] {what}: worst scaled error {errs[worst]:.3f} ({worst})")
    bad = {k: v for k, v in errs.items() if not v <= 1.0}
    assert not bad, f"{what}: scaled errors > 1: {bad} (all: {errs})"


def start_of(wa, wc, N, H, depth, seed) -> dict:
    """warm_start, asserted non-zero in every layer's h and c of both nets (a layer whose carry were dropped would show)."""
    st = warm_start(wa, wc, N, H, depth, seed)
    for net in ("actor", "critic"):
        for l in range(depth):
            assert np.abs(st[net][:, l, 0]).max() > 1e-2 and np.abs(st[net][:, l, 1]).max() > 1e-2, (net, l)
    return st


# ---- kbs_create / pack_weights ------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("path", PATHS, ids=NAMES.get)
def test_create_and_pack_every_depth(dev, path):
    """Depth 0, 5 and -1 are refused with KBS_E_SHAPE; 1 to KBS_MAX_DEPTH create a handle and pack both networks."""
    lib = L.load()
    for depth in (0, L.MAX_DEPTH + 1, -1):
        p = L.default_params()
        p.depth, p.gemm_path = depth, path
        h = C.c_void_p()
        assert lib.kbs_create(C.byref(p), C.byref(h)) == L_SHAPE, depth
    for depth in range(1, L.MAX_DEPTH + 1):
        e, _, _ = Hn.make_engine(depth=depth, gemm_path=path, device=dev)
        got = L.KbsParams()
        assert lib.kbs_get_params(e._h, C.byref(got)) == 0 and got.depth == depth
        e.close()


# ---- kbs_rollout ------------------------------------------------------------------------------------------------------------------

# per depth, one (T, N, H) for each (critic, start) combination: ragged env counts, a panel + 1 / + 2, one multi-panel case, T = 1
ROLLOUT_SHAPES = {3: [(5, 77, 256), (1, 130, 256), (6, 1100, 256), (8, 129, 128)],
                  4: [(7, 129, 256), (1, 5, 256), (5, 130, 256), (6, 1100, 256)]}
COMBOS = [(True, "mid"), (False, "zero"), (True, "zero"), (False, "mid")]
ROLLOUT_CASES = [pytest.param(path, d, c, s, *ROLLOUT_SHAPES[d][i],
                              id=f"{NAMES[path]}-d{d}-{'critic' if c else 'nocritic'}-{s}-T{ROLLOUT_SHAPES[d][i][0]}"
                                 f"xN{ROLLOUT_SHAPES[d][i][1]}xH{ROLLOUT_SHAPES[d][i][2]}")
                 for path in PATHS for d in (3, 4) for i, (c, s) in enumerate(COMBOS)]


@pytest.mark.parametrize("path,depth,with_critic,start,T,N,H", ROLLOUT_CASES)
def test_rollout(dev, path, depth, with_critic, start, T, N, H):
    """kbs_rollout at depth 3 and 4 from zero carries and from a mid-episode state (carries of every layer, lpf, pg_carry,
    command) against O.rollout_control_steps: every float output within the harness tolerance, integer outputs bit-exact.
    Depth 3 or 4 with the critic on a tensor-core datapath converts the carries through pack_rows / fb_convert."""
    wa, wc = weights(H, depth)
    st = start_of(wa, wc, N, H, depth, seed=6000 + N + depth) if start == "mid" else None
    b = Batch(6100 + N + depth, T, N, dev)
    e, _, _ = Hn.make_engine(hidden=H, depth=depth, gemm_path=path, device=dev)
    io = Hn.rollout_buffers(b, H, depth, with_critic, start=st)
    e.rollout(io, N)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    e.close()
    ref = Hn.oracle_rollout(b, wa, wc, H, depth, with_critic, start=st)
    assert_scaled(Hn.compare_rollout(io, ref, N, with_critic),
                  f"rollout {NAMES[path]} depth {depth} {'critic' if with_critic else 'nocritic'} {start} T{T}xN{N}xH{H}")
    if st is not None:      # non-vacuous: the start state changes the result
        zero = Hn.oracle_rollout(b, wa, wc, H, depth, with_critic)
        assert np.abs(zero["carry"]["actor"] - ref["carry"]["actor"]).max() > 1e-3


# ---- kbs_actor_step / kbs_critic_step ------------------------------------------------------------------------------------------


@pytest.mark.parametrize("path", PATHS, ids=NAMES.get)
@pytest.mark.parametrize("depth,H,N", [(3, 256, 200), (3, 128, 77), (4, 256, 130)])
def test_actor_and_critic_step(dev, path, depth, H, N):
    """Three actor / critic steps from a mid-episode state with done resets (on the tensor-core datapaths: kbs_tc_lstm_stack
    over 3 or 4 layers) against O.sample_action / O.critic_forward: mean, std, action, log-prob, entropy, value, carries and
    lpf; then the stored-action path (log-prob of a given action, argmax mode)."""
    e, wa, wc = Hn.make_engine(hidden=H, depth=depth, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H, depth=depth)
    st = start_of(wa, wc, N, H, depth, seed=310 + N)
    b = Batch(300 + N, 3, N, dev)
    ac_np, cc_np, lpf_np = st["actor"], st["critic"], st["lpf_params"]
    ac, cc, lpf = Hn.carry_from_np(ac_np, dev), Hn.carry_from_np(cc_np, dev), synth.to_soa(lpf_np, 0, dev)
    rng = np.random.default_rng(9)
    for t in range(3):
        o, _ = O.get_observations(b.np_state_at(t), b.np_noise_at(t), b.np["episode"], None, P)
        a_obs, c_obs = O.actor_obs_from_dict(o, b.cmd0_np), O.critic_obs_from_dict(o, b.cmd0_np)
        done_np = rng.random(N) < 0.3
        done = synth.to_soa(done_np.astype(np.uint8), 0, dev)
        out = e.actor_step(synth.to_soa(a_obs, 0, dev), ac, lpf, eps=b.noise["eps_action"][t], done=done, n_envs=N)
        act, mean, std, ac_np, lpf_np = O.sample_action(wa, a_obs, ac_np, lpf_np, b.np["noise"]["eps_action"][t], False, p)
        close(S(out["mean"], N, (20,)), mean, f"mean t={t}")
        close(S(out["std"], N, (20,)), std, f"std t={t}")
        close(S(out["action"], N, (20,)), act, f"action t={t}")
        close(S(out["log_prob"], N), O.mvn_log_prob(mean, std, act), f"log_prob t={t}", atol=1e-5)
        close(S(out["entropy"], N), O.mvn_entropy(std), f"entropy t={t}", atol=1e-5)
        ac_np = np.where(done_np[:, None, None, None], 0, ac_np).astype(np.float32)
        lpf_np = np.where(done_np[:, None], 0, lpf_np).astype(np.float32)
        close(Hn.carry_to_np(ac, N), ac_np, f"actor carry t={t}")
        close(S(lpf, N, (20,)), lpf_np, f"lpf t={t}")
        val = e.critic_step(synth.to_soa(c_obs, 0, dev), cc, done=done, n_envs=N)
        v_np, cc_np = O.critic_forward(wc, c_obs, cc_np)
        close(S(val, N), v_np[:, 0], f"value t={t}", atol=1e-5)         # see harness.compare_rollout on the floor
        cc_np = np.where(done_np[:, None, None, None], 0, cc_np).astype(np.float32)
        close(Hn.carry_to_np(cc, N), cc_np, f"critic carry t={t}", atol=1e-5)
    a_in = (mean + 0.3 * rng.standard_normal(mean.shape)).astype(np.float32)
    out = e.actor_step(synth.to_soa(a_obs, 0, dev), ac.clone(), lpf.clone(), eps=None, action_in=synth.to_soa(a_in, 0, dev),
                       n_envs=N)
    _, mean2, std2, _, _ = O.sample_action(wa, a_obs, ac_np, lpf_np, None, True, p)
    close(S(out["action"], N, (20,)), mean2, "mode()")
    close(S(out["log_prob"], N), O.mvn_log_prob(mean2, std2, a_in), "log_prob(action_in)", atol=1e-5)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    e.close()


# ---- kbs_policy_step from a checkpoint -----------------------------------------------------------------------------------------


@pytest.mark.parametrize("path", PATHS, ids=NAMES.get)
@pytest.mark.parametrize("depth,N", [(1, 33), (3, 300), (4, 130)])
def test_checkpoint_to_policy_step(dev, path, depth, N, tmp_path):
    """An eqx leaf stream of a depth-d model -> checkpoint.load_policy(depth=d) -> kbs_policy_step with the flat carry
    [n, depth*2*H + 20], three steps from init_fn()'s zero carry, against O.policy_step.  At depth 1 the tensor-core
    datapaths run the persistent kernel; at depth 3 and 4 the per-step stack."""
    H = 256
    wa, wc = synth.make_weights(510 + depth, 65, 40, H, depth), synth.make_weights(520 + depth, 475, 1, H, depth)
    static = (np.asarray(65), np.asarray(40), np.asarray(0.01, np.float32))
    path_ckpt = tmp_path / "model.eqx"
    checkpoint.write_leaves(checkpoint.weights_to_leaves(wa, wc, static, static[:2]), path_ckpt)
    la, lc = checkpoint.load_policy(path_ckpt, hidden=H, depth=depth)
    assert len(la["layers"]) == depth and len(lc["layers"]) == depth
    e = KbotStep(hidden_size=H, depth=depth, gemm_path=path)
    e.pack_weights(L.NET_ACTOR, synth.weights_to_device(la, dev))
    e.pack_weights(L.NET_CRITIC, synth.weights_to_device(lc, dev))
    p = O.OracleParams(depth=depth)
    b = Batch(17 + depth, 3, N, dev)
    flat = np.zeros((N, depth * 2 * H + 20), np.float32)
    flat_d = torch.from_numpy(flat).to(dev)
    for t in range(3):
        o, _ = O.get_observations(b.np_state_at(t), b.np_noise_at(t), b.np["episode"], None, P)
        args = (o["noisy_biased_joint_position"], o["noisy_joint_velocity"], o["noisy_imu_projected_gravity"],
                o["noisy_imu_gyro"], b.cmd0_np)
        act, flat = O.policy_step(wa, *args, flat, p)
        act_d, flat_d = e.policy_step(*(torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in args), flat_d)
        close(act_d.cpu().numpy(), act, f"policy action t={t}")
        close(flat_d.cpu().numpy(), flat, f"policy carry t={t}")
    assert np.abs(flat[:, (depth - 1) * 2 * H:depth * 2 * H]).max() > 1e-2        # the top layer's carry took part
    e.close()


# ---- kbs_ppo_variables ----------------------------------------------------------------------------------------------------------

VARS_CASES = [pytest.param(SIMT, 1, 8, 50, 256, True, id="simt-d1-mirror"),
              pytest.param(SIMT, 3, 5, 130, 128, True, id="simt-d3-mirror"),
              pytest.param(SIMT, 4, 6, 129, 256, True, id="simt-d4-mirror"),
              pytest.param(TF32, 1, 8, 50, 256, True, id="tc3xtf32-d1-mirror"),
              pytest.param(F16, 1, 5, 130, 256, True, id="tc2xf16-d1-mirror"),
              pytest.param(TF32, 3, 5, 77, 256, False, id="tc3xtf32-d3"),
              pytest.param(F16, 3, 6, 130, 128, False, id="tc2xf16-d3"),
              pytest.param(TF32, 4, 8, 129, 256, False, id="tc3xtf32-d4"),
              pytest.param(F16, 4, 5, 50, 256, False, id="tc2xf16-d4")]


@pytest.mark.parametrize("path,depth,T,N,H,mirror", VARS_CASES)
def test_ppo_variables(dev, path, depth, T, N, H, mirror):
    """kbs_ppo_variables from mid-episode carries with done resets against O.get_ppo_variables: log-probs, entropy, values,
    action std and every final carry; with the mirror pass, the aux losses and the mirror carries too; the same trajectory in
    two calls is bitwise one call.  On a tensor-core datapath above depth 2, dist.mean() and the mirror pass have no per-step
    form: both are refused with KBS_E_SHAPE before anything is launched, the carries untouched and the health word clear."""
    e, wa, wc = Hn.make_engine(hidden=H, depth=depth, gemm_path=path, device=dev)
    # a 4-layer critic's mirrored values differ by ~1e-2 here: at the default critic scale 0.01 the value mirror loss would sit
    # at the check's absolute floor, so depth 4 weighs it 1.0
    p = O.OracleParams(hidden_size=H, depth=depth, actor_mirror_loss_scale=1.0,
                       critic_mirror_loss_scale=1.0 if depth == 4 else 0.01)
    b = Batch(8300 + N + depth, T, N, dev)
    rng = np.random.default_rng(8 + depth)
    obs = [O.get_observations(b.np_state_at(t), b.np_noise_at(t), b.np["episode"], None, Hn.P)[0] for t in range(T)]
    cmd = np.stack([b.cmd0_np] * T)
    done = rng.random((T, N)) < 0.15
    act = (np.stack([o["joint_position"] for o in obs]) + 0.2 * rng.standard_normal((T, N, 20))).astype(np.float32)
    w = start_of(wa, wc, N, H, depth, seed=8400 + N)
    m = start_of(wa, wc, N, H, depth, seed=8500 + N)
    carry0 = {"actor": w["actor"], "critic": w["critic"], "lpf_params": w["lpf_params"], "actor_mirror": m["actor"],
              "critic_mirror": m["critic"], "lpf_params_mirror": m["lpf_params"]}
    ref, c_end = O.get_ppo_variables(wa, wc, obs, cmd, act, done, dict(carry0), p, mirror=True)
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

    def run(c, t0, t1, with_mirror, want_mean=False):
        a = {k: v[t0:t1].contiguous() for k, v in arrays.items()}
        mir = {"actor_obs": a["am_obs"], "critic_obs": a["cm_obs"], "actor_carry": c["acm"], "critic_carry": c["ccm"],
               "lpf": c["lpfm"], "actor_scale": p.actor_mirror_loss_scale, "critic_scale": p.critic_mirror_loss_scale}
        return e.ppo_variables(a["a_obs"], a["act"], a["done"], c["ac"], c["lpf"], a["c_obs"], c["cc"], n_envs=N,
                               want_mean=want_mean, mirror=mir if with_mirror else None)

    c = carries()
    out = run(c, 0, T, mirror)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    close(S(out["log_probs"], N), ref["log_probs"][..., 0], "log_probs", atol=1e-4)
    close(S(out["entropy"], N), ref["entropy"][..., 0], "entropy", atol=1e-5)
    close(S(out["values"], N), ref["values"], "values", atol=1e-5)
    close(S(out["action_std"], N, (20,)), ref["action_std"], "action_std")
    close(Hn.carry_to_np(c["ac"], N), c_end["actor"], "actor carry")
    close(Hn.carry_to_np(c["cc"], N), c_end["critic"], "critic carry", atol=1e-5)
    close(S(c["lpf"], N, (20,)), c_end["lpf_params"], "lpf")
    if mirror:
        close(S(out["action_mirror_loss"], N), ref["action_mirror_loss"], "action_mirror_loss", rtol=1e-4, atol=1e-6)
        close(S(out["value_mirror_loss"], N), ref["value_mirror_loss"], "value_mirror_loss", rtol=1e-4, atol=2e-7)
        assert float(np.abs(ref["action_mirror_loss"]).max()) > 1e-3 and float(np.abs(ref["value_mirror_loss"]).max()) > 1e-6
        close(Hn.carry_to_np(c["acm"], N), c_end["actor_mirror"], "actor_mirror carry")
        close(Hn.carry_to_np(c["ccm"], N), c_end["critic_mirror"], "critic_mirror carry", atol=1e-5)
        close(S(c["lpfm"], N, (20,)), c_end["lpf_params_mirror"], "lpf_params_mirror")
    # the same trajectory in two calls
    T1 = T // 2 + 1
    c2 = carries()
    o1, o2 = run(c2, 0, T1, mirror), run(c2, T1, T, mirror)
    keys = ("log_probs", "entropy", "values", "action_std") + (("action_mirror_loss", "value_mirror_loss") if mirror else ())
    for k in keys:
        assert torch.equal(torch.cat([o1[k], o2[k]])[..., :N], out[k][..., :N]), k
    for k in (c if mirror else ("ac", "cc", "lpf")):
        assert torch.equal(c2[k][..., :N], c[k][..., :N]), k
    if path != SIMT and depth > 2:
        c3 = carries()
        before = {k: v.clone() for k, v in c3.items()}
        l0 = e.launches
        with pytest.raises(RuntimeError, match=r"kbs_ppo_variables failed: \[-2\]"):
            run(c3, 0, T, False, want_mean=True)
        with pytest.raises(RuntimeError, match=r"kbs_ppo_variables failed: \[-2\]"):
            run(c3, 0, T, True)
        torch.cuda.synchronize()
        assert e.launches == l0, "a refused call launched kernels"
        for k in c3:
            assert torch.equal(c3[k], before[k]), f"a refused call wrote {k}"
        assert e.device_status() == 0
    e.close()


# ---- kbs_ppo_grad -------------------------------------------------------------------------------------------------------------

# (path, per_step, depth, T, N, H, start); FP16-split at depth 1 runs the persistent update unless KBS_PPO_PER_STEP=1; above
# depth 2 it always runs the per-step launches.  The lower layers of a deeper stack have the smallest dG: at depth 4, T = 1,
# n = 5 the critic's layer 0 sits deep below fp16's normal range in the FP16 split.
GRAD_CASES = []
for _d, _shapes in ((1, {"zero": (7, 70, 256), "warm": (6, 77, 256)}), (3, {"zero": (6, 129, 256), "warm": (5, 130, 128)}),
                    (4, {"zero": (7, 77, 256), "warm": (1, 5, 256)})):
    for _path, _per_step in ((SIMT, False), (TF32, False), (F16, False)) + (((F16, True),) if _d == 1 else ()):
        for _start, (_T, _N, _H) in _shapes.items():
            GRAD_CASES.append(pytest.param(_path, _per_step, _d, _T, _N, _H, _start,
                                           id=f"{NAMES[_path]}{'-per-step' if _per_step else ''}-d{_d}-{_start}-T{_T}xN{_N}xH{_H}"))
for _path in (TF32, F16):
    GRAD_CASES.append(pytest.param(_path, False, 4, 33, 300, 256, "warm", id=f"{NAMES[_path]}-d4-warm-T33xN300xH256"))


@pytest.mark.parametrize("path,per_step,depth,T,N,H,start", GRAD_CASES)
def test_ppo_grad(dev, path, per_step, depth, T, N, H, start, monkeypatch):
    """kbs_ppo_grad at depth 1, 3 and 4 against float64 autograd, from zero and from warm-start carries: log-probs, values,
    loss statistics, and every gradient tensor and gate / mean / std block of it within the bounds the depth-2 tests use
    (harness.compare_grads_blockwise).  The margin of every layer is printed: the lower layers' gradients of a deeper stack
    are orders of magnitude smaller than the top layer's."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "1" if per_step else "0")
    e, wa, wc = Hn.make_engine(hidden=H, depth=depth, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H, depth=depth)
    carry0 = None
    if start == "warm":
        w = start_of(wa, wc, N, H, depth, seed=3100 + N)
        carry0 = {k: w[k] for k in ("actor", "critic", "lpf_params")}
    b = make_ppo_batch(2100 + T + N + depth, T, N, p, wa, wc, carry0)
    ratios = {}
    try:
        e.profile(True)
        bad, ref = Hn.ppo_grad_compare(e, wa, wc, b, p, dev, N, carry0=carry0, ratios=ratios)
        prof = e.profile_read()
    finally:
        e.close()
    persistent = prof.get("bptt_persist_kernel", (0, 0))[1]
    assert (persistent > 0) == (path == F16 and not per_step and depth <= 2), persistent
    layer = lambda net, l: max(v for k, v in ratios.items() if k.startswith(f"{net}.layers[{l}]."))
    other = max(v for k, v in ratios.items() if ".layers[" not in k)
    print(f"\n[depths] ppo_grad {NAMES[path]}{'-per-step' if per_step else ''} depth {depth} {start} T{T}xN{N}xH{H}: "
          f"block error / bound per layer: actor {[round(layer('actor', l), 3) for l in range(depth)]} "
          f"critic {[round(layer('critic', l), 3) for l in range(depth)]}; projections / heads {other:.3f}")
    assert not bad, bad
    if carry0 is not None:
        assert_start_state_matters(ref, G.ppo_minibatch_grads(wa, wc, b, p), depth)


# ---- PpoUpdater.update / epoch ---------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("path,depth,H", [pytest.param(TF32, 3, 128, id="tc3xtf32-d3"), pytest.param(TF32, 4, 256, id="tc3xtf32-d4"),
                                          pytest.param(F16, 1, 256, id="tc2xf16-d1-persistent"),
                                          pytest.param(F16, 4, 256, id="tc2xf16-d4")])
def test_ppo_update_against_float64_each_update(dev, path, depth, H, monkeypatch):
    """PpoUpdater with 1, 3 or 4 layers (its flat parameter vector, AdamW, the re-pack of every layer) update by update, each
    from the state the updater had before it, as test_gpu_ppo_update.test_ppo_update_against_float64_each_update; minibatches
    alternate x1 / x8 so both clip branches occur; a fresh handle packed from the final parameters gives the same gradient."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, updates = 6, 48, 4
    e, wa, wc = Hn.make_engine(hidden=H, depth=depth, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H, depth=depth)
    seed = 9700 + 10 * depth + H
    first = minibatch(seed + 1, T, N, p, wa, wc, None, 1.0)
    limit = clip_limit(wa, wc, first, minibatch(seed + 1, T, N, p, wa, wc, None, 8.0), p, None, {})
    up = PpoUpdater(e, wa, wc, max_grad_norm=limit)
    assert up.pa.depth == depth and up.pc.depth == depth
    clipped = []
    try:
        e.profile(True)
        for k in range(1, updates + 1):
            snap = snapshot(up)
            b = first if k == 1 else minibatch(seed + k, T, N, p, *weights_at(up, snap["param"]), None, 8.0 if k % 2 == 0 else 1.0)
            db = Hn.ppo_device_batch(b, dev)
            out = up.update(db, N)
            clipped.append(check_update(up, snap, out, b, p, k, limit) > limit)
        persistent = e.profile_read().get("bptt_persist_kernel", (0, 0))[1]
        e.profile(False)
        assert (persistent > 0) == (path == F16 and depth <= 2), persistent
        assert any(clipped) and not all(clipped), ("both clip branches", clipped)
        assert_repacked(up, H, path, db, N)
    finally:
        e.close()


def test_epoch_depth3_composition_and_replay(dev, monkeypatch):
    """3xTF32 with 3 layers (the per-step update, shuffle_carry_kernel over 6 carry rows): PpoUpdater.epoch is bitwise the
    hand-built epoch of tested parts after every pass, from warm-start carries; then capture_epoch changes nothing and a
    replay on a refilled rollout is bitwise an eager epoch on another updater from the same state."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, H, depth, bs, passes, seed = 5, 256, 256, 3, 64, 2, 2025
    ea, wa, wc = Hn.make_engine(hidden=H, depth=depth, gemm_path=TF32, device=dev)
    eb, _, _ = Hn.make_engine(hidden=H, depth=depth, gemm_path=TF32, device=dev)
    try:
        carry0 = start_of(wa, wc, N, H, depth, seed=9310)
        ro = make_rollout(T, N, dev, seed=63, H=H, depth=depth, carry0=carry0)
        assert int(ro["done"][:, :N].sum()) > 0
        up, ref = PpoUpdater(ea, wa, wc), PpoUpdater(eb, wa, wc)
        got_states, out = epoch_with_pass_states(up, ro, N, bs, passes, seed)
        out = {k: t.clone() for k, t in out.items()}
        ref_states, stats, norms, perms = reference_epoch(ref, ro, N, bs, passes, seed, pass0=0)
        torch.cuda.synchronize()
        assert ea.device_status() == 0 and eb.device_status() == 0
        np.testing.assert_array_equal(out["perm"].cpu().numpy(), perms)
        for p, (g, r) in enumerate(zip(got_states, ref_states)):
            for k in g:
                assert torch.equal(g[k], r[k]), f"after pass {p}: {k} differs"
        assert torch.equal(out["stats"], stats) and torch.equal(out["norms"], norms)
        assert torch.isfinite(norms).all()
        ref.pass_dev.copy_(up.pass_dev)            # the hand-built epoch draws its permutations on the host
        before = state(up)
        up.capture_epoch(ro, N, bs, passes, seed)
        torch.cuda.synchronize()
        for k, t in before.items():
            assert torch.equal(t, state(up)[k]), f"capture changed {k}"
        refill_rollout(ro, make_rollout(T, N, dev, seed=64, H=H, depth=depth, carry0=start_of(wa, wc, N, H, depth, seed=9311)))
        oa = up.epoch(ro, N, bs, passes, seed)
        assert up._epoch_graph is not None and oa is up._epoch_out
        oa = {k: t.clone() for k, t in oa.items()}
        ob = ref.epoch(ro, N, bs, passes, seed)
        torch.cuda.synchronize()
        assert ea.device_status() == 0 and eb.device_status() == 0
        assert_same(up, ref, oa, ob, "replayed epoch")
        assert torch.isfinite(oa["norms"]).all()
    finally:
        ea.close()
        eb.close()


# ---- the online step ----------------------------------------------------------------------------------------------------------


def own_io(b: Batch, start, depth: int) -> dict:
    """test_gpu_ppo_iteration.own_io with `depth` layers."""
    io = Hn.rollout_buffers(b, 256, depth, start=start)
    for k in ("state", "noise", "episode"):
        io[k] = {n: t.clone() for n, t in io[k].items()}
    for k in ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms"):
        io[k] = io[k].clone()
    return io


def record_call(dev, b, path, depth, with_critic, start, done_prev) -> dict:
    e, _, _ = Hn.make_engine(depth=depth, gemm_path=path, device=dev)
    io = Hn.rollout_buffers(b, 256, depth, with_critic, start=start)
    io["critic_obs"] = torch.full((b.T, L.CRITIC_OBS, b.ld), float("nan"), device=dev)
    io["done_prev"] = done_prev
    e.rollout(io, b.N)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    e.close()
    return io


def step_calls(dev, b, path, depth, with_critic, start, done_prev) -> tuple:
    e, _, _ = Hn.make_engine(depth=depth, gemm_path=path, device=dev)
    io = Hn.rollout_buffers(b, 256, depth, with_critic, start=start)
    st = e.step_state(b.N, with_critic, {"actor_carry": io["actor_carry"], "critic_carry": io["critic_carry"], "lpf": io["lpf"],
                                         "pg_carry": io["pg_carry"], "command": io["command"][0], "done_prev": done_prev})
    tr = traj_buffers(io, with_critic)
    for t in range(b.T):
        e.rollout_step(st, dict(step_inputs(io, t), **tr))
    fin = stored(e, st, io)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    e.close()
    return tr, fin


ONLINE_CASES = [pytest.param(path, depth, c, m, id=f"{NAMES[path]}-d{depth}-{'critic-mid' if m else 'nocritic-zero'}")
                for path, depth in ((SIMT, 1), (TF32, 1), (F16, 1), (SIMT, 3), (SIMT, 4)) for c, m in ((True, True), (False, False))]


@pytest.mark.parametrize("path,depth,with_critic,mid", ONLINE_CASES)
def test_steps_equal_one_record_call(dev, path, depth, with_critic, mid):
    """T kbs_rollout_step calls are bitwise one T-step kbs_rollout_record call (every trajectory output, the recorded state,
    the final carries, lpf, pg_carry, command, done_prev) with one layer on every datapath (rollout_persist_kernel with the
    device hsb slot word) and with 3 or 4 layers on SIMT; episodes end on steps 2 and T-1; a mid-episode start loads a
    done_prev with every third env set."""
    T, N = 7, 300
    wa, wc = weights(256, depth)
    start = start_of(wa, wc, N, 256, depth, seed=9320 + depth) if mid else None
    b = Batch(9330 + depth, T, N, dev)
    for t in (2, T - 1):
        ending_at(b, t)
    done_prev = torch.zeros(b.ld, dtype=torch.uint8, device=dev)
    if mid:
        done_prev[:N:3] = 1
    whole = record_call(dev, b, path, depth, with_critic, start, done_prev)
    assert int(whole["done"][:, :N].sum()) > N
    tr, fin = step_calls(dev, b, path, depth, with_critic, start, done_prev)
    assert_steps_equal_record(tr, fin, whole, b, with_critic, f"steps at depth {depth}")


@pytest.mark.parametrize("capture", [False, True], ids=["eager", "captured"])
def test_online_iterations_equal_record_loop_depth1(dev, capture, monkeypatch):
    """One layer, FP16-split, three closed-loop iterations: PpoUpdater.step x T + end_iteration is bitwise the loop written
    with kbs_rollout_record, kbs_rewards and epoch(), as test_gpu_rollout_step.test_online_iterations_equal_record_loop;
    captured: the step captured at t = 1 of the second iteration and every step of the third replayed."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, depth = 6, 512, 1
    wa, wc = weights(256, depth)
    start = start_of(wa, wc, N, 256, depth, seed=9640)
    b1, b2, b3 = Batch(9641, T, N, dev), Batch(9642, T, N, dev), Batch(9643, T, N, dev)
    ending_at(b1, T - 1)
    ending_at(b2, T - 1)
    ea, _, _ = Hn.make_engine(depth=depth, gemm_path=F16, device=dev)
    eb, _, _ = Hn.make_engine(depth=depth, gemm_path=F16, device=dev)
    try:
        ua, ub = PpoUpdater(ea, wa, wc), PpoUpdater(eb, wa, wc)
        ioa, iob = own_io(b1, start, depth), own_io(b1, start, depth)
        rca, rcb = reward_carry(b1.ld, dev), reward_carry(b1.ld, dev)
        io_t = step_inputs(own_io(b1, start, depth), 0)
        io_t = {k: ({n: x.clone() for n, x in v.items()} if isinstance(v, dict) else v.clone()) for k, v in io_t.items()}
        sim = {k: v.clone() for k, v in io_t["state"].items()}
        done_prev = torch.zeros(b1.ld, dtype=torch.uint8, device=dev)
        for it, b in enumerate((b1, b2, b3)):
            oa, launches = online_loop(ua, ioa, b, rca, N, capture and it == 1, io_t)
            oa = {k: v.clone() for k, v in oa.items()}
            assert (launches == 0) == (capture and it == 2), launches
            ob, done_prev = hand_loop(ub, iob, b, rcb, N, done_prev, sim)
            fin = stored(ea, ua.step_st, ioa)
            torch.cuda.synchronize()
            assert ea.device_status() == 0 and eb.device_status() == 0
            for k in ("actor_carry", "critic_carry", "lpf", "pg_carry"):
                assert torch.equal(fin[k], iob[k]), f"iteration {it + 1}: final {k}"
            assert torch.equal(fin["command"], iob["command"][0]) and torch.equal(fin["done_prev"], done_prev)
            ioa["command"][0].copy_(fin["command"])
            assert_iteration_equal(ua, ub, oa, ob, {k: ioa[k] for k in TRAJ if k in ioa}, {k: iob[k] for k in TRAJ if k in iob},
                                   f"iteration {it + 1}")
            for k in rca:
                assert torch.equal(rca[k], rcb[k]), k
            assert torch.isfinite(oa["norms"]).all()
    finally:
        ea.close()
        eb.close()


@pytest.mark.parametrize("path", [TF32, F16], ids=NAMES.get)
def test_online_step_refused_on_tensor_cores_above_depth_2(dev, path):
    """The step state holds the persistent kernel's layouts, which a tensor-core datapath does not have above depth 2:
    kbs_step_state_bytes refuses with KBS_E_SHAPE and writes no size, and PpoUpdater.begin_iteration raises that error each
    time it is called, launching nothing and leaving the caller's buffers and the updater's parameters as they were.  SIMT
    has a step state at the same depth."""
    N, depth = 64, 3
    e, wa, wc = Hn.make_engine(depth=depth, gemm_path=path, device=dev)
    try:
        for with_critic in (1, 0):
            nb = C.c_uint64(12345)
            assert e.lib.kbs_step_state_bytes(e._h, N, with_critic, C.byref(nb)) == L_SHAPE and nb.value == 12345
        assert rc_of(lambda: e.step_state(N, True)) == L_SHAPE
        up = PpoUpdater(e, wa, wc)
        io = own_io(Batch(9700, 2, N, dev), None, depth)
        before = {k: v.clone() for k, v in io.items() if torch.is_tensor(v)}
        param = up.param.clone()
        torch.cuda.synchronize()
        l0 = e.launches
        for _ in range(2):
            with pytest.raises(RuntimeError, match=r"kbs_step_state_bytes failed: \[-2\]"):
                up.begin_iteration(io, N)
        torch.cuda.synchronize()
        assert e.launches == l0
        for k, v in before.items():
            assert torch.equal(io[k], v), f"begin_iteration wrote {k}"
        assert torch.equal(up.param, param) and not hasattr(up, "step_st")
        assert e.device_status() == 0
    finally:
        e.close()
    es, _, _ = Hn.make_engine(depth=depth, gemm_path=SIMT, device=dev)
    nb = C.c_uint64(0)
    assert es.lib.kbs_step_state_bytes(es._h, N, 1, C.byref(nb)) == 0 and nb.value > 0
    es.close()
