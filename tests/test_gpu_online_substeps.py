"""The physics sub-steps of the online rollout (kbs_actuator_substep on a caller-owned actuator state beside the step state):
S one-sub-step calls after each control step are bitwise kbs_torque_substeps on the S joint states stacked, the sub-steps
apply the action of the step that just ran across iterations and rewinds, validation and the range guard, and
PpoUpdater.substep / capture_substep in a closed loop against the same loop written with kbs_torque_substeps."""

import numpy as np
import pytest
import torch

import harness as Hn
import kbot_oracle as O
from harness import Batch
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200 import engine as E
from kbot_joystick_b200 import synth
from kbot_joystick_b200.ppo import PpoUpdater
from test_gpu_ppo_iteration import assert_iteration_equal, ending_at, own_io, reward_carry
from test_gpu_rollout_step import INPUTS, TRAJ, rc_of, step_inputs, stored
from test_gpu_start_state import warm_start, weights

pytestmark = pytest.mark.gpu

L_NULL, L_SHAPE, L_ALIGN, L_PARAM, L_DEVICE = -1, -2, -3, -5, -6
SUB_DT, DROP = 0.004, 0.05


@pytest.fixture(scope="module")
def dev(cuda_device, lib_built):
    return cuda_device


def actuator_draws(g, T, ld, dev):
    """u_drop / latency [T, ld] per control step.  Latencies put the switch on every sub-step 0..3 (0, 4, 8 and 12 ms; 8 ms is
    2 sub_dt exactly in fp32, the boundary of k sub_dt >= latency), the rest U(3 ms, 10 ms); every 7th env drops its command."""
    lat = 0.003 + 0.007 * torch.rand((T, ld), generator=g, device=dev)
    for i, v in enumerate((0.0, 0.004, 0.008, 0.012)):
        lat[:, i::11] = v
    u = DROP + (1 - DROP) * torch.rand((T, ld), generator=g, device=dev)
    u[:, 3::7] = 0.5 * DROP * torch.rand((T, ld), generator=g, device=dev)[:, 3::7]
    return u.contiguous(), lat.contiguous()


def joint_state(g, ld, dev):
    return 0.5 * torch.randn((27, ld), generator=g, device=dev), 2.0 * torch.randn((26, ld), generator=g, device=dev)


def drive(e, st, ast, io, b, S, episode, g, prev_ref, steps, check_oracle=False):
    """Control steps `steps` of b (kbs_rollout_step into io's trajectories), each followed by S kbs_actuator_substep calls on
    random joint states; every ctrl_k and the stored prev_action bitwise against kbs_torque_substeps(action[t], prev_ref, ...)
    on the stacked states (prev_ref advanced in place)."""
    N, ld, dev = b.N, b.ld, b.dev
    u_drop, lat = actuator_draws(g, b.T, ld, dev)
    tr = {k: io[k] for k in TRAJ if io.get(k) is not None}
    for t in steps:
        e.rollout_step(st, dict(step_inputs(io, t), **tr))
        qs, ctrls = [], []
        for k in range(S):
            qpos, qvel = joint_state(g, ld, dev)
            ctrl = torch.full((20, ld), float("nan"), device=dev)
            e.actuator_substep(st, ast, {"action": io["action"], "u_drop": u_drop[t], "latency": lat[t], "qpos": qpos,
                                         "qvel": qvel, "episode": episode, "ctrl": ctrl, "sub_dt": SUB_DT, "drop_prob": DROP})
            qs.append((qpos, qvel))
            ctrls.append(ctrl)
        prev0 = prev_ref.clone()
        q_sub = torch.stack([q[7:27] for q, _ in qs]).contiguous()
        qd_sub = torch.stack([qd[6:26] for _, qd in qs]).contiguous()
        ref = e.torque_substeps(io["action"][t], prev_ref, u_drop[t], lat[t], q_sub, qd_sub, episode, sub_dt=SUB_DT,
                                drop_prob=DROP, n_envs=N)
        got_prev = e.actuator_state_store(ast)
        torch.cuda.synchronize()
        for k in range(S):
            assert torch.equal(ctrls[k][:, :N], ref[k][:, :N]), f"step {t}: ctrl of sub-step {k} differs"
        assert torch.equal(got_prev[:, :N], prev_ref[:, :N]), f"step {t}: prev_action differs"
        if check_oracle:
            ep = {k: synth.from_soa(v, N, (20,)) for k, v in (episode or {}).items() if k in ("kp", "kd", "tau_limit",
                                                                                              "action_bias", "torque_bias")}
            want, applied = O.position_actuator_substeps(
                synth.from_soa(io["action"][t], N, (20,)), synth.from_soa(prev0, N, (20,)), synth.from_soa(u_drop[t], N),
                synth.from_soa(lat[t], N), synth.from_soa(q_sub, N, (20,)), synth.from_soa(qd_sub, N, (20,)), sub_dt=SUB_DT,
                drop_prob=DROP, **ep)
            Hn.close(synth.from_soa(torch.stack(ctrls), N, (20,)), want, f"step {t}: sub-step torques vs oracle", atol=1e-4)
            Hn.exact(synth.from_soa(got_prev, N, (20,)), applied, f"step {t}: applied action vs oracle")
    # the latency cases put the switch on sub-steps 0..3, and some commands were dropped
    if S == 5:
        f = np.float32
        k_sw = (np.arange(S, dtype=f)[:, None] * f(SUB_DT) >= synth.from_soa(lat, N)[:, None, :]).argmax(1)
        assert set(np.unique(k_sw).tolist()) >= {0, 1, 2, 3}
    assert int((u_drop[:, :N] < DROP).sum()) > 0


def full_episode(b: Batch, g) -> dict:
    ep = dict(b.episode)
    ep["torque_bias"] = (torch.rand(ep["torque_bias"].shape, generator=g, device=b.dev) - 0.5).contiguous()
    return ep


# ---- 1. online sub-steps == kbs_torque_substeps ---------------------------------------------------------------------------------


@pytest.mark.parametrize("S,N,gains", [(5, 601, "all"), (5, 512, "null"), (1, 601, "all"), (1, 64, "null")],
                         ids=["S5-601-all", "S5-512-null", "S1-601-all", "S1-64-null"])
def test_substeps_equal_torque_substeps(dev, S, N, gains):
    """FP16-split step state loaded mid-episode, T control steps, S sub-steps after each: bitwise kbs_torque_substeps (every
    ctrl_k, prev_action), with every gain / bias field of the episode view set (torque_bias nonzero) or all of them NULL; the
    oracle at the torque tolerance."""
    T = 4
    g = torch.Generator(device=dev).manual_seed(7000 + N + S)
    wa, wc = weights(256, 2)
    b = Batch(7001 + N, T, N, dev)
    e, _, _ = Hn.make_engine(gemm_path=L.GEMM_TC_2XF16, device=dev)
    try:
        io = Hn.rollout_buffers(b, 256, 2, start=warm_start(wa, wc, N, 256, 2, seed=7002))
        st = e.step_state(N, True, {"actor_carry": io["actor_carry"], "critic_carry": io["critic_carry"], "lpf": io["lpf"],
                                    "pg_carry": io["pg_carry"], "command": io["command"][0]})
        prev = (0.3 * torch.randn((20, b.ld), generator=g, device=dev)).contiguous()
        ast = e.actuator_state(N, S, prev)
        episode = full_episode(b, g) if gains == "all" else None
        drive(e, st, ast, io, b, S, episode, g, prev.clone(), range(T), check_oracle=True)
        torch.cuda.synchronize()
        assert e.device_status() == 0
    finally:
        e.close()


# ---- 2. the slot and the index across iterations ----------------------------------------------------------------------------


def test_substeps_follow_the_step_across_rewinds(dev):
    """Two iterations of T steps on one step state, rewound in between (end_iteration's rewind): the sub-steps after step t
    apply action[t] of that iteration, and prev_action carries across the rewind."""
    T, N, S = 3, 256, 5
    g = torch.Generator(device=dev).manual_seed(7100)
    b1, b2 = Batch(7101, T, N, dev), Batch(7102, T, N, dev)
    e, _, _ = Hn.make_engine(gemm_path=L.GEMM_TC_2XF16, device=dev)
    try:
        io = Hn.rollout_buffers(b1, 256, 2)
        st = e.step_state(N, True)
        ast = e.actuator_state(N, S)
        prev = torch.zeros((20, b1.ld), device=dev)
        episode = full_episode(b1, g)
        drive(e, st, ast, io, b1, S, episode, g, prev, range(T))
        first = io["action"].clone()
        e.step_state_rewind(st)
        io2 = dict(Hn.rollout_buffers(b2, 256, 2), action=io["action"])       # the same trajectory, slot 0 again
        drive(e, st, ast, io2, b2, S, episode, g, prev, range(T))
        torch.cuda.synchronize()
        assert not torch.equal(first, io["action"])                            # the second iteration wrote its own actions
        assert e.device_status() == 0
    finally:
        e.close()


# ---- 3. validation -----------------------------------------------------------------------------------------------------------


def test_substep_validation(dev):
    T, N, S = 2, 64, 5
    b = Batch(7200, T, N, dev)
    ld = b.ld
    e, _, _ = Hn.make_engine(gemm_path=L.GEMM_TC_2XF16, device=dev)
    try:
        io = Hn.rollout_buffers(b, 256, 2)
        st = e.step_state(N, True)
        ast = e.actuator_state(N, S)
        qpos, qvel = b.state["qpos"][0], b.state["qvel"][0]
        ctrl = torch.full((20, ld), float("nan"), device=dev)
        base = {"action": io["action"], "u_drop": torch.ones(ld, device=dev), "latency": torch.zeros(ld, device=dev),
                "qpos": qpos, "qvel": qvel, "episode": b.episode, "ctrl": ctrl}
        sub = lambda st_=st, ast_=ast, **kw: e.actuator_substep(st_, ast_, dict(base, **kw))
        tr = {k: io[k] for k in TRAJ if io.get(k) is not None}
        for k in ("action", "u_drop", "latency", "qpos", "qvel", "ctrl"):
            assert rc_of(lambda: sub(**{k: None})) == L_NULL, k
        f = torch.zeros(20 * ld + 8, device=dev)
        assert rc_of(lambda: sub(ctrl=f[1:1 + 20 * ld].view(20, ld))) == L_ALIGN
        assert rc_of(lambda: sub(episode=dict(b.episode, kp=f[1:1 + 20 * ld].view(20, ld)))) == L_ALIGN
        for kw in ({"sub_dt": 0.0}, {"sub_dt": -0.004}, {"sub_dt": float("nan")}, {"drop_prob": -0.01}, {"drop_prob": 1.01},
                   {"drop_prob": float("nan")}):
            assert rc_of(lambda: sub(**kw)) == L_PARAM, kw
        other = e.actuator_state(N + 4, S)
        assert rc_of(lambda: sub(ast_=other)) == L_SHAPE                      # n_envs of the two states differ
        zero_s = E.ActuatorState(ast.buf, L.KbsActuatorState(ast.buf.data_ptr(), ast.desc.bytes, N, 0))
        assert rc_of(lambda: sub(ast_=zero_s)) == L_SHAPE
        assert rc_of(lambda: e.actuator_state_load(zero_s)) == L_SHAPE
        small = E.ActuatorState(ast.buf, L.KbsActuatorState(ast.buf.data_ptr(), ast.desc.bytes - 256, N, S))
        assert rc_of(lambda: sub(ast_=small)) == L_SHAPE
        off = torch.empty(int(ast.desc.bytes) + 512, dtype=torch.uint8, device=dev)
        mis = E.ActuatorState(off, L.KbsActuatorState(off.data_ptr() + 16, ast.desc.bytes, N, S))
        assert rc_of(lambda: sub(ast_=mis)) == L_ALIGN
        assert rc_of(lambda: e.actuator_state_store(mis)) == L_ALIGN
        assert rc_of(lambda: e.actuator_state_load(ast, f[1:1 + 20 * ld].view(20, ld))) == L_ALIGN
        torch.cuda.synchronize()
        assert e.device_status() == 0 and torch.isnan(ctrl).all()             # nothing above reached the device

        def refused_on_device(what):
            sub()
            torch.cuda.synchronize()
            assert torch.isnan(ctrl).all(), f"{what}: ctrl written"
            assert e.device_status() & L.STATUS_SUBSTEP_RANGE, what
            assert rc_of(lambda: sub()) == L_DEVICE, what
            assert rc_of(lambda: e.rollout_step(st, dict(step_inputs(io, 0), **tr))) == L_DEVICE, what
            e.device_status_reset()

        refused_on_device("t = 0 after load")
        e.rollout_step(st, dict(step_inputs(io, 0), **tr))
        sub()                                                                  # t = 1: applies action[0]
        torch.cuda.synchronize()
        assert e.device_status() == 0 and torch.isfinite(ctrl[:, :N]).all()
        ctrl.fill_(float("nan"))
        e.rollout_step(st, dict(step_inputs(io, 1), **tr))                     # t = 2 > T of a one-step action trajectory
        sub(action=io["action"][:1])
        torch.cuda.synchronize()
        assert torch.isnan(ctrl).all() and e.device_status() & L.STATUS_SUBSTEP_RANGE
        e.device_status_reset()
        e.step_state_rewind(st)
        refused_on_device("t = 0 after rewind")
        e.rollout_step(st, dict(step_inputs(io, 0), **tr))
        sub()
        torch.cuda.synchronize()
        assert e.device_status() == 0 and torch.isfinite(ctrl[:, :N]).all()
    finally:
        e.close()


# ---- 4. PpoUpdater: the closed loop with sub-steps -------------------------------------------------------------------------------


def integrate_substep(state: dict, ctrl):
    """A toy simulator's physics step: the joint state of sub-step k + 1 follows ctrl_k."""
    state["qpos"][7:27] += 1e-4 * ctrl
    state["qvel"][6:26].mul_(0.9).add_(1e-3 * ctrl)


def batch_inputs(b: Batch) -> dict:
    return dict(state=b.state, noise={k: v for k, v in b.noise.items() if k != "eps_action"}, eps_action=b.noise["eps_action"],
                u_switch=b.cmd_rand["u_switch"], cmd_mode=b.cmd_rand["mode"], cmd_u6=b.cmd_rand["u6"], cmd_u_arms=b.cmd_rand["u_arms"])


def online_loop(up, io, b, rc, N, capture, io_t, io_k, draws):
    """begin_iteration -> T x (step -> 5 x (substep -> physics step on ctrl_k)) -> end_iteration.  -> (its output, library
    launches enqueued from the host during the T steps and their sub-steps)."""
    u_drop, lat = draws
    up.begin_iteration(io, N)
    l0 = up.eng.launches
    for t in range(b.T):
        src = step_inputs(dict(io, **batch_inputs(b)), t)
        for n in io_t["noise"]:
            io_t["noise"][n].copy_(src["noise"][n])
        for n in io_t["state"]:
            if n not in ("qpos", "qvel") or t == 0:
                io_t["state"][n].copy_(src["state"][n])
        for k in INPUTS:
            io_t[k].copy_(src[k])
        if capture and t == 1:
            up.capture_step(io_t)
        up.step(io_t)
        io_k["u_drop"].copy_(u_drop[t])
        io_k["latency"].copy_(lat[t])
        io_k["qpos"].copy_(io_t["state"]["qpos"])
        io_k["qvel"].copy_(io_t["state"]["qvel"])
        for k in range(5):
            if capture and t == 1 and k == 0:
                up.capture_substep(io_k)
            up.substep(io_k)
            integrate_substep(io_k, io_k["ctrl"])
        io_t["state"]["qpos"].copy_(io_k["qpos"])
        io_t["state"]["qvel"].copy_(io_k["qvel"])
    launches = up.eng.launches - l0
    return up.end_iteration(rc, N, 128, 2, 13), launches


def hand_loop(up, io, b, rc, N, done_prev, sim, prev, episode, draws):
    """The same with T = 1 kbs_rollout_record calls (pointers offset to slot t), kbs_rewards, epoch(), and sub-step k's torque
    = row k of a kbs_torque_substeps call on the k + 1 joint states so far with a clone of prev_action (the call on all five
    advances prev_action)."""
    u_drop, lat = draws
    T, ld = b.T, b.ld
    c0 = {k + "0": io[k].clone() for k in ("actor_carry", "critic_carry", "lpf")}
    cobs = torch.empty((T, L.CRITIC_OBS, ld), device=b.dev)
    traj = {k: torch.empty_like(v) for k, v in b.state.items()}
    inp = batch_inputs(b)
    for t in range(T):
        for n in traj:
            if n not in ("qpos", "qvel") or t == 0:
                sim[n].copy_(b.state[n][t])
            traj[n][t].copy_(sim[n])
        one = dict(io, state={k: v[None] for k, v in sim.items()}, noise={k: v[t:t + 1] for k, v in inp["noise"].items()},
                   **{k: inp[k][t:t + 1] for k in INPUTS}, command=io["command"][t:t + 2], critic_obs=cobs[t:t + 1],
                   done_prev=done_prev, T=1,
                   **{k: io[k][t:t + 1] for k in ("actor_obs", "action", "log_prob", "ctrl", "term_codes", "done", "success", "value")})
        up.eng.rollout(one, N)
        done_prev = io["done"][t].clone()
        qs, qds = [], []
        for k in range(5):
            qs.append(sim["qpos"][7:27].clone())
            qds.append(sim["qvel"][6:26].clone())
            p = prev.clone() if k < 4 else prev
            ctrl = up.eng.torque_substeps(io["action"][t], p, u_drop[t], lat[t], torch.stack(qs), torch.stack(qds), episode,
                                          n_envs=N)[k]
            integrate_substep(sim, ctrl)
    rew = up.eng.rewards(traj, io["command"][:T], io["ctrl"], io["done"], rc, n_envs=N)
    ro = dict(c0, actor_obs=io["actor_obs"], critic_obs=cobs, action=io["action"], done=io["done"], success=io["success"], rewards=rew)
    out = dict(up.epoch(ro, N, batch_size=128, num_passes=2, seed=13), rewards=rew)
    io["command"][0].copy_(io["command"][T])
    return out, done_prev


@pytest.mark.parametrize("capture", [False, True], ids=["eager", "captured"])
def test_closed_loop_substeps_equal_hand_loop(dev, capture, monkeypatch):
    """FP16-split, three iterations, a simulator in the loop that takes five physics steps per control step on the online
    sub-step torques: bitwise the loop written by hand with kbs_torque_substeps -- parameters, optimiser state, statistics,
    trajectories, final carries, the simulator's state and prev_action.  Captured: the first iteration eager, the step and the
    sub-step captured in the second, and the third launches nothing from the host."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N = 6, 512
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=7300)
    bs = [Batch(7301 + i, T, N, dev) for i in range(3)]
    ending_at(bs[0], T - 1)
    ending_at(bs[1], 2)
    g = torch.Generator(device=dev).manual_seed(7310)
    draws = [actuator_draws(g, T, bs[0].ld, dev) for _ in bs]
    episode = full_episode(bs[0], g)
    ea, _, _ = Hn.make_engine(gemm_path=L.GEMM_TC_2XF16, device=dev)
    eb, _, _ = Hn.make_engine(gemm_path=L.GEMM_TC_2XF16, device=dev)
    try:
        ua, ub = PpoUpdater(ea, wa, wc), PpoUpdater(eb, wa, wc)
        ioa, iob = own_io(bs[0], start), own_io(bs[0], start)
        rca, rcb = reward_carry(bs[0].ld, dev), reward_carry(bs[0].ld, dev)
        io_t = step_inputs(own_io(bs[0], start), 0)
        io_t = {k: ({n: x.clone() for n, x in v.items()} if isinstance(v, dict) else v.clone()) for k, v in io_t.items()}
        io_t["episode"] = episode
        io_k = {"qpos": io_t["state"]["qpos"].clone(), "qvel": io_t["state"]["qvel"].clone(), "u_drop": draws[0][0][0].clone(),
                "latency": draws[0][1][0].clone(), "episode": episode, "ctrl": torch.empty((20, bs[0].ld), device=dev)}
        iob["episode"] = episode
        sim = {k: v.clone() for k, v in io_t["state"].items()}
        prev = torch.zeros((20, bs[0].ld), device=dev)
        done_prev = torch.zeros(bs[0].ld, dtype=torch.uint8, device=dev)
        for it, b in enumerate(bs):
            oa, launches = online_loop(ua, ioa, b, rca, N, capture and it == 1, io_t, io_k, draws[it])
            oa = {k: v.clone() for k, v in oa.items()}
            if capture and it == 2:
                assert launches == 0                                 # every step and sub-step was a replay
            else:
                assert launches > 0
            ob, done_prev = hand_loop(ub, iob, b, rcb, N, done_prev, sim, prev, episode, draws[it])
            fin = stored(ea, ua.step_st, ioa)
            got_prev = ea.actuator_state_store(ua.act_st)
            torch.cuda.synchronize()
            assert ea.device_status() == 0 and eb.device_status() == 0
            what = f"iteration {it + 1}"
            for k in ("actor_carry", "critic_carry", "lpf", "pg_carry"):
                assert torch.equal(fin[k], iob[k]), f"{what}: final {k}"
            assert torch.equal(fin["command"], iob["command"][0]) and torch.equal(fin["done_prev"], done_prev), what
            assert torch.equal(got_prev, prev), f"{what}: prev_action"
            for k in ("qpos", "qvel"):
                assert torch.equal(io_t["state"][k], sim[k]), f"{what}: simulator {k}"
            ioa["command"][0].copy_(fin["command"])
            assert_iteration_equal(ua, ub, oa, ob, {k: ioa[k] for k in TRAJ if k in ioa}, {k: iob[k] for k in TRAJ if k in iob},
                                   what)
            for k in rca:
                assert torch.equal(rca[k], rcb[k]), k
            assert torch.isfinite(oa["norms"]).all()
        assert float(prev[:, :N].abs().sum()) > 0
    finally:
        ea.close()
        eb.close()
