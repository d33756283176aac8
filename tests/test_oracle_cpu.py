"""CPU suite (no GPU): pins the oracle against the golden vectors in tests/golden/ and checks its internal
invariants.  The oracle is test infrastructure; see oracle/kbot_oracle.py header ("parity unpinned")."""

from pathlib import Path

import numpy as np
import pytest

import kbot_oracle as O

G = Path(__file__).resolve().parent / "golden"
P = O.OracleParams()


def test_golden_lstm_matches_torch_lstmcell():
    g = np.load(G / "lstm.npz")
    h2, c2 = O.lstm_cell(g["w_ih"], g["w_hh"], g["b"], g["x"], g["h"], g["c"])
    np.testing.assert_allclose(h2, g["h2"], rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(c2, g["c2"], rtol=1e-12, atol=1e-13)
    f = lambda k: g[k].astype(np.float32)
    h2f, c2f = O.lstm_cell(f("w_ih"), f("w_hh"), f("b"), f("x"), f("h"), f("c"))
    assert h2f.dtype == np.float32
    np.testing.assert_allclose(h2f, g["h2"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(c2f, g["c2"], rtol=2e-5, atol=2e-6)


def test_golden_mvn_matches_torch_distributions():
    g = np.load(G / "mvn.npz")
    np.testing.assert_allclose(O.mvn_log_prob(g["mean"], g["std"], g["a"]), g["log_prob"], rtol=1e-12)
    np.testing.assert_allclose(O.mvn_entropy(g["std"]), g["entropy"], rtol=1e-12)


def test_golden_quaternions_match_scipy():
    g = np.load(G / "quat.npz")
    np.testing.assert_allclose(O.quat_to_euler(g["q"], eps=0.0), g["euler"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(O.rotate_vector_by_quat(g["v"], g["q"], eps=0.0), g["v_rot"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(O.rotate_vector_by_quat(g["v"], g["q"], inverse=True, eps=0.0), g["v_rot_inv"],
                               rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(O.euler_to_quat(g["e"]), g["q_from_e"], rtol=1e-9, atol=1e-9)
    pg = O.projected_gravity(g["q"], O.OracleParams(eps_quat=0.0))
    np.testing.assert_allclose(pg, g["g_body"], rtol=1e-9, atol=1e-9)
    # the eps the helpers add to the norm perturbs a unit quaternion by ~1e-6 relative
    np.testing.assert_allclose(O.quat_to_euler(g["q"]), g["euler"], rtol=0, atol=1e-4)


def test_golden_softplus():
    g = np.load(G / "softplus.npz")
    np.testing.assert_allclose(O.softplus(g["x"]), g["y"], rtol=1e-12, atol=1e-300)


def test_golden_gae_exact_rational_example():
    g = np.load(G / "gae.npz")
    p = O.OracleParams(gamma=float(g["gamma"]), lam=float(g["lam"]))
    for dt in (np.float32, np.float64):
        adv, tgt = O.compute_ppo_inputs(g["values"].astype(dt), g["rewards"].astype(dt), g["done"], g["success"], p)
        np.testing.assert_array_equal(adv, g["adv"].astype(dt))      # dyadic rationals: exact in fp32
        np.testing.assert_array_equal(tgt, g["targets"].astype(dt))


def test_structure_known_answers():
    g = np.load(G / "structure.npz")
    assert O.ACTOR_OBS == int(g["actor_obs"]) and O.CRITIC_OBS == int(g["critic_obs"])
    rng = np.random.default_rng(0)
    wa = O.init_net_weights(rng, 65, 40, 256, 2)
    wc = O.init_net_weights(rng, 475, 1, 256, 2)
    count = lambda w: sum(v.size for k, v in w.items() if k != "layers") + sum(v.size for l in w["layers"] for v in l.values())
    assert count(wa) == int(g["actor_params_h256"]) and count(wc) == int(g["critic_params_h256"])
    assert list(O.JOINT_NAMES[10:15]) == [n for n in O.JOINT_NAMES if "right_shoulder" in n or "right_elbow" in n or "right_wrist" in n]
    assert len(O.JOINT_NAMES) == len(O.JOINT_BIASES64) == len(O.JOINT_LIMITS64) == 20   # train.py:70


def _batch(T=6, N=9, seed=3):
    from kbot_joystick_b200 import synth

    return synth.make_batch(seed, T, N)


def _obs(b, t=0):
    st = {k: v[t] for k, v in b["state"].items()}
    nz = {k: v[t] for k, v in b["noise"].items()}
    return O.get_observations(st, nz, b["episode"], None, P)


def test_observation_shapes_and_slots():
    b = _batch()
    o, carry = _obs(b)
    cmd = O.initial_command(b["cmd0_rand"]["mode"], b["cmd0_rand"]["u6"], b["cmd0_rand"]["u_arms"], P)
    a = O.actor_obs_from_dict(o, cmd)
    c = O.critic_obs_from_dict(o, cmd)
    assert a.shape == (9, 65) and c.shape == (9, 475) and a.dtype == np.float32 and c.dtype == np.float32
    np.testing.assert_array_equal(a[:, 49:65], cmd)
    np.testing.assert_array_equal(a[:, -10:], cmd[:, 6:16])          # train.py:932 arm command = obs[-10:]
    np.testing.assert_array_equal(c[:, 474], b["state"]["xpos"][0][:, 1, 2])
    np.testing.assert_array_equal(c[:, 80:90], b["state"]["cinert"][0][:, 1, :])
    np.testing.assert_array_equal(c[:, 310:316], b["state"]["cvel"][0][:, 1, :])
    assert len([k for k in o if not k.startswith("noisy_")]) >= 18
    for k in ("noisy_biased_joint_position", "noisy_joint_velocity", "noisy_imu_gyro", "noisy_imu_projected_gravity"):
        assert k in o
    assert carry.shape == (9, 3)


def test_command_law():
    b = _batch(N=4000)
    r = b["cmd0_rand"]
    cmd = O.initial_command(r["mode"], r["u6"], r["u_arms"], P)
    assert cmd.shape == (4000, 16)                                     # train.py:765
    zc = O.zero_cmd_mask(cmd)
    np.testing.assert_array_equal(zc[(r["mode"] == 4) | (r["mode"] == 5)], True)
    assert abs(zc.mean() - 1 / 3) < 0.03                               # "2/6 standing" train.py:752
    arms = cmd[:, 6:]
    lim = O.JOINT_LIMITS64[10:].astype(np.float32)
    on = (r["mode"] == 3) | (r["mode"] == 4)
    assert np.all(arms[~on] == 0)
    # same key for uniform() and bernoulli(): an arm command is non-zero only in the lower half of its range
    mid = lim[:, 0] + 0.5 * (lim[:, 1] - lim[:, 0])
    nz = arms[on] != 0
    assert np.all((arms[on] <= mid + 1e-6) | ~nz)
    prev = np.ones_like(cmd)
    keep = O.command_step(prev, np.full(4000, 0.5, np.float32), r["mode"], r["u6"], r["u_arms"], P)
    np.testing.assert_array_equal(keep, prev)
    sw = O.command_step(prev, np.zeros(4000, np.float32), r["mode"], r["u6"], r["u_arms"], P)
    np.testing.assert_array_equal(sw, cmd)


def test_mirror_involutions():
    b = _batch()
    o, _ = _obs(b)
    mo = O.mirror_obs(O.mirror_obs(o))
    for k in mo:
        np.testing.assert_array_equal(mo[k], o[k])
    cmd = O.initial_command(b["cmd0_rand"]["mode"], b["cmd0_rand"]["u6"], b["cmd0_rand"]["u_arms"], P)
    np.testing.assert_array_equal(O.mirror_cmd(O.mirror_cmd(cmd)), cmd)
    j = np.arange(20, dtype=np.float32)
    # legs swapped, arms NOT swapped (train.py:1577-1582 as written)
    np.testing.assert_array_equal(O.mirror_joints(j), -np.array([5, 6, 7, 8, 9, 0, 1, 2, 3, 4] + list(range(10, 20)), np.float32))
    np.testing.assert_array_equal(O.mirror_cmd(cmd)[:, 6:], -cmd[:, 6:])


def test_terminations_codes():
    b = _batch(T=1, N=500)
    st = {k: v[0] for k, v in b["state"].items()}
    codes, done, succ = O.terminations(st["xpos"], st["qpos"][:, 3:7], st["time"], P)
    assert codes.dtype == np.int32 and set(np.unique(codes)) <= {-1, 0, 1}
    np.testing.assert_array_equal(done, (codes != 0).any(-1))
    np.testing.assert_array_equal(succ, done & (codes != -1).all(-1))
    assert done.any() and (~done).any() and succ.any()


def _traj(b, ctrl=None, done=None):
    st = b["state"]
    T, N = st["time"].shape
    rng = np.random.default_rng(11)
    r = b["cmd_rand"]
    cmd = np.empty((T, N, 16), np.float32)
    c = O.initial_command(b["cmd0_rand"]["mode"], b["cmd0_rand"]["u6"], b["cmd0_rand"]["u_arms"], P)
    for t in range(T):
        cmd[t] = c
        c = O.command_step(c, (r["u_switch"][t] * 0.02).astype(np.float32), r["mode"][t], r["u6"][t], r["u_arms"][t], P)
    return {"xquat": st["xquat"], "xpos": st["xpos"], "qpos": st["qpos"], "qvel": st["qvel"],
            "ctrl": (20 * rng.standard_normal((T, N, 20))).astype(np.float32) if ctrl is None else ctrl,
            "command": cmd, "touch_l": st["sensordata"][..., O.SD_TOUCH_L], "touch_r": st["sensordata"][..., O.SD_TOUCH_R],
            "com_distance": st["com_distance"], "done": (rng.random((T, N)) < 0.1) if done is None else done}


def test_rewards_ranges_and_streaming_equivalence():
    b = _batch(T=40, N=64)
    tr = _traj(b)
    c0 = O.reward_initial_carry((64,))
    comp, total, c1 = O.rewards(tr, c0, P)
    assert set(comp) == set(O.REWARD_NAMES) and total.shape == (40, 64) and total.dtype == np.float32
    for k in O.REWARD_NAMES:
        assert comp[k].shape == (40, 64), k
        if k != "feet_airtime":
            assert np.all((comp[k] >= 0) & (comp[k] <= 1)), k
    np.testing.assert_allclose(total, sum(np.float32(s) * comp[k] for k, s in zip(O.REWARD_NAMES, O.REWARD_SCALES)),
                               rtol=1e-6, atol=1e-6)
    # base_accel: first step of every rollout has zero difference (edge pad, train.py:489-490)
    np.testing.assert_array_equal(comp["base_accel"][0], 1.0)
    # stateful terms: two half-trajectories chained through the carry == the whole trajectory (Appendix E)
    h1 = {k: v[:20] for k, v in tr.items()}
    h2 = {k: v[20:] for k, v in tr.items()}
    ca, _, cm = O.rewards(h1, c0, P)
    cb, _, ce = O.rewards(h2, cm, P)
    for k in ("single_contact", "feet_airtime"):
        np.testing.assert_array_equal(np.concatenate([ca[k], cb[k]]), comp[k])
    for k in c1:
        np.testing.assert_array_equal(ce[k], c1[k])


def test_feet_orient_is_rotating_reduces_over_time_as_written():
    b = _batch(T=8, N=16)
    tr = _traj(b)
    tr["command"][..., 2] = 0.0
    c0 = O.reward_initial_carry((16,))
    a = O.rewards(tr, c0, P)[0]["feet_orient"]
    tr2 = dict(tr)
    tr2["command"] = tr["command"].copy()
    tr2["command"][7, :, 2] = 0.5            # turning only at the LAST step ...
    b2 = O.rewards(tr2, c0, P)[0]["feet_orient"]
    assert np.any(a[0] != b2[0])             # ... changes the reward of the FIRST step (train.py:455)


def test_network_forward_and_ppo_scan():
    rng = np.random.default_rng(5)
    p = O.OracleParams(hidden_size=32)
    wa = O.init_net_weights(rng, 65, 40, 32, 2)
    wc = O.init_net_weights(rng, 475, 1, 32, 2)
    b = _batch(T=5, N=7)
    carry = O.initial_model_carry((7,), p)
    cmd = O.initial_command(b["cmd0_rand"]["mode"], b["cmd0_rand"]["u6"], b["cmd0_rand"]["u_arms"], P)
    obs_list, acts = [], []
    ac, lpf = carry["actor"], carry["lpf_params"]
    for t in range(5):
        o, _ = _obs(b, t)
        obs_list.append(o)
        a, mean, std, ac, lpf = O.sample_action(wa, O.actor_obs_from_dict(o, cmd), ac, lpf, b["noise"]["eps_action"][t], False, p)
        assert np.all(std > 0) and np.all(std <= 1.0) and a.shape == (7, 20)
        acts.append(a)
    done = np.zeros((5, 7), bool)
    done[2, 3] = True
    out, c2 = O.get_ppo_variables(wa, wc, obs_list, np.stack([cmd] * 5), np.stack(acts), done, carry, p)
    assert out["log_probs"].shape == (5, 7, 1) and out["values"].shape == (5, 7)
    assert out["entropy"].shape == (5, 7, 1) and out["action_std"].shape == (5, 7, 20)
    # argmax log-prob identity: log_prob(mean) = -sum log std - 10 log 2pi
    lp = O.mvn_log_prob(out["mean"], out["action_std"], out["mean"])
    np.testing.assert_allclose(lp, -np.log(out["action_std"]).sum(-1) - 10 * np.log(2 * np.pi), rtol=1e-5)
    # policy_step (convert.py) == actor_forward mode with the flat carry
    flat = np.concatenate([carry["actor"].reshape(7, -1), carry["lpf_params"]], -1)
    o0 = obs_list[0]
    act, flat2 = O.policy_step(wa, o0["noisy_biased_joint_position"], o0["noisy_joint_velocity"],
                               o0["noisy_imu_projected_gravity"], o0["noisy_imu_gyro"], cmd, flat, p)
    m0, _, nc0, nl0 = O.actor_forward(wa, O.actor_obs_from_dict(o0, cmd), carry["actor"], carry["lpf_params"], p)
    np.testing.assert_array_equal(act, m0)
    assert flat2.shape == (7, 2 * 2 * 32 + 20)                         # convert.py:71
    np.testing.assert_array_equal(flat2[:, -20:], nl0)


def test_fp32_oracle_tracks_fp64():
    b = _batch(T=12, N=40)
    tr = _traj(b)
    tr64 = {k: (v.astype(np.float64) if v.dtype == np.float32 else v) for k, v in tr.items()}
    c32, t32, _ = O.rewards(tr, O.reward_initial_carry((40,)), P)
    c64, t64, _ = O.rewards(tr64, O.reward_initial_carry((40,), np.float64), P)
    for k in O.REWARD_NAMES:
        if k in ("roll_pitch", "feet_orient"):   # 1 - d^2 with error_scale 0.01-0.03: conditioning ~ 1e2
            np.testing.assert_allclose(c32[k], c64[k], rtol=2e-3, atol=1e-6, err_msg=k)
        else:
            np.testing.assert_allclose(c32[k], c64[k], rtol=2e-4, atol=1e-6, err_msg=k)


def test_com_distance_known_answers():
    """O12 (train.py:509-659) on hand-checkable polygons: unit square -> centroid (0.5, 0.5); a triangle -> mean of its
    vertices; interior points do not move the hull; < 3 distinct geom2 values -> -1; coincident points -> fallback mean."""
    f = np.float32
    sq = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0], [0.5, 0.5, 0], [0.25, 0.75, 0]], f)
    g1 = np.zeros((6,), np.int32)
    g2 = np.array([7, 7, 12, 12, 3, 3], np.int32)
    d = O.com_distance_observation(g1[None], g2[None], sq[None], np.array([[0.5, 0.5, 0.8]], f))
    assert abs(float(d[0])) < 1e-6
    d = O.com_distance_observation(g1[None], g2[None], sq[None], np.array([[3.5, 4.5, 0.8]], f))
    np.testing.assert_allclose(d, [5.0], rtol=1e-6)                     # 3-4-5 triangle from the centroid
    tri = np.array([[0, 0, 0], [3, 0, 0], [0, 3, 0], [1, 1, 0]], f)
    d = O.com_distance_observation(np.zeros((1, 4), np.int32), np.array([[1, 2, 3, 3]], np.int32), tri[None],
                                   np.array([[1, 1, 0]], f))
    assert abs(float(d[0])) < 1e-6                                       # centroid of the triangle = (1, 1)
    d = O.com_distance_observation(np.zeros((1, 4), np.int32), np.array([[1, 1, 2, 2]], np.int32), tri[None],
                                   np.array([[1, 1, 0]], f))
    assert float(d[0]) == -1.0                                           # 2 distinct geoms: not enough support
    same = np.tile(np.array([[0.2, -0.1, 0]], f), (5, 1))
    d = O.com_distance_observation(np.zeros((1, 5), np.int32), np.array([[1, 2, 3, 4, 5]], np.int32), same[None],
                                   np.array([[0.2, -0.1, 0]], f))
    assert abs(float(d[0])) < 1e-6                                       # degenerate hull -> mean of the vertices
    # non-floor rows collapse to the origin and stay in the point set (as written, train.py:637-638)
    g1b = np.array([0, 0, 0, 5], np.int32)
    pts = np.array([[2, 2, 0], [3, 2, 0], [2, 3, 0], [9, 9, 9]], f)
    d_with_origin = O.com_distance_observation(g1b[None], np.array([[1, 2, 3, 4]], np.int32), pts[None], np.zeros((1, 3), f))
    d_tri_only = O.com_distance_observation(np.zeros((1, 3), np.int32), np.array([[1, 2, 3]], np.int32), pts[None, :3],
                                            np.zeros((1, 3), f))
    assert float(d_with_origin[0]) < float(d_tri_only[0])               # the origin pulls the hull centroid towards it


def test_ppo_loss_known_answers():
    """PPO loss restatement: on-policy data (ratio = 1) gives policy = A; a ratio outside the clip range with a positive
    advantage is capped at (1 + eps) A; the clipped value loss takes the larger of the two squared errors."""
    f = np.float32
    one = np.ones((2, 3), f)
    lp = np.zeros((2, 3), f)
    loss, pol, val, ent, obj = O.ppo_loss(lp, lp, 2 * one, one, one, one, 3 * one, entropy_coef=0.5)
    assert pol == 2.0 and val == 0.0 and ent == 3.0 and loss == -(2.0 + 0.5 * 3.0)
    _, pol, _, _, _ = O.ppo_loss(lp + f(np.log(2.0)), lp, one, one, one, one, one)          # ratio 2, A = 1 -> 1.2
    np.testing.assert_allclose(pol, 1.2, rtol=1e-6)
    _, pol, _, _, _ = O.ppo_loss(lp + f(np.log(2.0)), lp, -one, one, one, one, one)         # ratio 2, A = -1 -> -2
    np.testing.assert_allclose(pol, -2.0, rtol=1e-6)
    # v moved 1.0 away from v_old = 0 towards the target 1: unclipped error 0, clipped value = 0.2 -> error 0.8
    _, _, val, _, _ = O.ppo_loss(lp, lp, one, one, 0 * one, one, one)
    np.testing.assert_allclose(val, 0.5 * 0.8 ** 2, rtol=1e-6)
    _, _, val, _, _ = O.ppo_loss(lp, lp, one, one, 0 * one, one, one, use_clipped_value_loss=False)
    assert val == 0.0


def test_reference_goldens_when_present():
    """tests/golden/ref_*.npz are outputs of the REAL reference packages (tools/verify_against_ref.py --dump, run wherever
    jax / ksim / xax / equinox / distrax import).  None can be produced in this image, so until someone commits them this
    test skips and parity stays UNPINNED; once present, every one of them must match the oracle's restatement."""
    import importlib.util
    from pathlib import Path

    root = Path(__file__).resolve().parent.parent
    spec = importlib.util.spec_from_file_location("verify_against_ref", root / "tools" / "verify_against_ref.py")
    V = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(V)
    rep = V.check(root / "tests" / "golden")
    pinned = {k: v for k, v in rep.items() if v["status"] != "unverified"}
    if not pinned:
        pytest.skip("no reference goldens committed: parity unpinned (oracle-defined, reference-unverified)")
    bad = {k: v for k, v in pinned.items() if v["status"] != "verified"}
    assert not bad, bad


def _random_carry(rng, N, depth, H, dtype=np.float64):
    """A mid-episode start state: h inside (-1, 1) as tanh leaves it, an unbounded cell state, a low-pass state of joint scale."""
    c = np.empty((N, depth, 2, H), dtype)
    c[:, :, 0] = rng.uniform(-0.95, 0.95, (N, depth, H))
    c[:, :, 1] = rng.normal(0, 2.0, (N, depth, H))
    return c


def test_ppo_grad_reference_from_nonzero_start_state():
    """The float64 autograd reference (oracle/ppo_grad_torch.py) from a non-zero carry0: its log-probs and values are the
    NumPy oracle's get_ppo_variables from the same carries, and a gradient entry that only a non-zero c0 / h0 makes non-zero
    matches a central finite difference of the loss."""
    import torch

    import ppo_grad_torch as G

    T, N, H, depth = 2, 3, 8, 2
    p = O.OracleParams(hidden_size=H, depth=depth)
    rng = np.random.default_rng(12)
    wa = O.init_net_weights(rng, 65, 40, H, depth, dtype=np.float64)
    wc = O.init_net_weights(rng, 475, 1, H, depth, dtype=np.float64)
    b = _batch(T, N, seed=5)
    obs = [{k: v.astype(np.float64) for k, v in _obs(b, t)[0].items()} for t in range(T)]
    cmd = np.stack([O.initial_command(b["cmd0_rand"]["mode"], b["cmd0_rand"]["u6"], b["cmd0_rand"]["u_arms"], P)] * T)
    cmd = cmd.astype(np.float64)
    carry0 = {"actor": _random_carry(rng, N, depth, H), "critic": _random_carry(rng, N, depth, H),
              "lpf_params": rng.normal(0, 0.3, (N, 20))}
    done = np.array([[True, False, False], [False, True, False]])
    action = np.stack([o["joint_position"] for o in obs]) + 0.2 * rng.standard_normal((T, N, 20))
    ref, _ = O.get_ppo_variables(wa, wc, obs, cmd, action, done, carry0, p, mirror=False)
    batch = {"actor_obs": np.stack([O.actor_obs_from_dict(o, c) for o, c in zip(obs, cmd)]),
             "critic_obs": np.stack([O.critic_obs_from_dict(o, c) for o, c in zip(obs, cmd)]),
             "action": action, "done": done, "advantages": rng.normal(size=(T, N)), "value_targets": rng.normal(0, 0.5, (T, N))}
    batch["old_log_probs"] = ref["log_probs"][..., 0] + rng.normal(0, 0.05, (T, N))
    batch["old_values"] = ref["values"] + rng.normal(0, 0.05, (T, N))
    loss, _, ga, gc, lp, val = G.ppo_minibatch_grads(wa, wc, batch, p, carry0=carry0)
    np.testing.assert_allclose(lp, ref["log_probs"][..., 0], rtol=1e-12, atol=1e-10)
    np.testing.assert_allclose(val, ref["values"], rtol=1e-12, atol=1e-12)
    _, _, ga0, gc0, lp0, _ = G.ppo_minibatch_grads(wa, wc, batch, p)
    assert np.abs(lp0 - lp).max() > 1e-3                               # carry0 reached the forward pass

    def loss_at(net, layer, key, idx, delta):
        w = {"actor": wa, "critic": wc}
        w2 = {k: {kk: (vv if kk != "layers" else [dict(l) for l in vv]) for kk, vv in x.items()} for k, x in w.items()}
        a = w2[net]["layers"][layer][key].copy()
        a[idx] += delta
        w2[net]["layers"][layer][key] = a
        args = [batch[k] for k in ("actor_obs", "critic_obs", "action", "done", "old_log_probs", "advantages",
                                   "value_targets", "old_values")]
        with torch.no_grad():
            l, _, _, _ = G.ppo_minibatch_loss(G.weights_to_torch(w2["actor"], False), G.weights_to_torch(w2["critic"], False),
                                              *args, p, {}, carry0)
        return float(l)

    # forget-gate bias of the actor's layer 0 (env 0 is reset after step 0: the gradient of the others carries dc c0 sigma'(f)),
    # w_hh of the critic's top layer (step 0's term is dG0^T h0): both exactly 0 from a zero start at T = 1
    for net, layer, key, idx, g, g0 in (("actor", 0, "b", (H + 3,), ga, ga0), ("critic", 1, "w_hh", (2 * H + 1, 5), gc, gc0)):
        eps = 1e-5
        fd = (loss_at(net, layer, key, idx, eps) - loss_at(net, layer, key, idx, -eps)) / (2 * eps)
        got = g["layers"][layer][key][idx]
        assert abs(got - fd) <= 1e-6 * abs(fd) + 1e-10, (net, key, got, fd)
        assert abs(got - g0["layers"][layer][key][idx]) > 1e-3 * abs(got), (net, key, "does not depend on carry0")
