"""The online rollout (kbs_rollout_step on a caller-owned step state): T one-step calls are bitwise one T-step
kbs_rollout_record call on every datapath, the state's load / store round trip is exact, other entry points between steps
change nothing, a captured step replays for every t, validation, and PpoUpdater's begin_iteration / step / end_iteration
against the same loop written with kbs_rollout_record and a simulator whose next state depends on the step's ctrl."""

import pytest
import torch

import harness as Hn
from harness import Batch
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200 import engine as E
from kbot_joystick_b200.ppo import PpoUpdater
from test_gpu_ppo_iteration import assert_iteration_equal, ending_at, own_io, reward_carry, run
from test_gpu_start_state import random_carry, warm_start, weights

pytestmark = pytest.mark.gpu

PATHS = [pytest.param(L.GEMM_SIMT_FP32, id="simt"), pytest.param(L.GEMM_TC_3XTF32, id="tc3xtf32"),
         pytest.param(L.GEMM_TC_2XF16, id="tc2xf16")]
TRAJ = ("actor_obs", "critic_obs", "action", "log_prob", "ctrl", "term_codes", "done", "success", "value", "command")
INPUTS = ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms")
L_NULL, L_SHAPE, L_ALIGN, L_STATE, L_DEVICE = -1, -2, -3, -4, -6


@pytest.fixture(scope="module")
def dev(cuda_device, lib_built):
    return cuda_device


def step_inputs(io: dict, t: int) -> dict:
    """Step t's [F, ld] inputs out of a rollout_buffers io."""
    d = {"state": {k: v[t] for k, v in io["state"].items()}, "noise": {k: v[t] for k, v in io["noise"].items()},
         "episode": io["episode"]}
    d.update({k: io[k][t] for k in INPUTS})
    return d


def traj_buffers(io: dict, with_critic: bool, critic_obs: bool = True) -> dict:
    T, ld = io["T"], io["done"].shape[1]
    dev = io["done"].device
    out = {k: torch.full_like(io[k], 7) if io[k].dtype == torch.uint8 else torch.full_like(io[k], float("nan"))
           for k in ("actor_obs", "action", "log_prob", "ctrl", "done", "success")}
    out["term_codes"] = torch.full_like(io["term_codes"], -9)
    out["command"] = torch.full_like(io["command"], float("nan"))
    out["critic_obs"] = torch.full((T, L.CRITIC_OBS, ld), float("nan"), device=dev) if critic_obs else None
    out["value"] = torch.full((T, ld), float("nan"), device=dev) if with_critic else None
    out["traj_state"] = {k: torch.full_like(v, float("nan")) for k, v in io["state"].items()}
    return out


def stored(e, st, like: dict) -> dict:
    out = {k: torch.full_like(like[k], float("nan")) for k in ("actor_carry", "lpf", "pg_carry")}
    out["critic_carry"] = torch.full_like(like["critic_carry"], float("nan")) if like.get("critic_carry") is not None else None
    out["command"] = torch.full_like(like["command"][0], float("nan"))
    out["done_prev"] = torch.full_like(like["done"][0], 9)
    return e.step_state_store(st, out)


def run_steps(dev, b: Batch, path, with_critic, start, between=None, critic_obs=True, done_prev=None) -> tuple:
    """b's rollout as T kbs_rollout_step calls from a state loaded with the start carries and done_prev -> (trajectories,
    stored state)."""
    e, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    io = Hn.rollout_buffers(b, 256, 2, with_critic, start=start)
    st = e.step_state(b.N, with_critic, {"actor_carry": io["actor_carry"], "critic_carry": io["critic_carry"], "lpf": io["lpf"],
                                        "pg_carry": io["pg_carry"], "command": io["command"][0], "done_prev": done_prev})
    tr = traj_buffers(io, with_critic, critic_obs)
    for t in range(b.T):
        e.rollout_step(st, dict(step_inputs(io, t), **tr))
        if between is not None:
            between(e, io)
    fin = stored(e, st, io)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    e.close()
    return tr, fin


def assert_steps_equal_record(tr: dict, fin: dict, whole: dict, b: Batch, with_critic: bool, what: str):
    for k in TRAJ:
        if whole.get(k) is not None:
            assert torch.equal(tr[k], whole[k]), f"{what}: {k} differs"
    for k in b.state:
        assert torch.equal(tr["traj_state"][k], b.state[k]), f"{what}: traj_state {k}"
    for k in ("actor_carry", "critic_carry", "lpf", "pg_carry"):
        if whole.get(k) is not None:
            assert torch.equal(fin[k], whole[k]), f"{what}: final {k} differs"
    assert torch.equal(fin["command"], whole["command"][b.T]), f"{what}: final command"
    assert torch.equal(fin["done_prev"], whole["done"][b.T - 1]), f"{what}: done_prev"


# ---- 1. T steps == one T-step kbs_rollout_record call --------------------------------------------------------------------------


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("with_critic,mid,critic_obs", [(True, True, True), (False, False, True), (True, False, True),
                                                        (True, True, False)],
                         ids=["critic-mid", "nocritic-zero", "critic-zero", "critic-mid-nocobs"])
def test_steps_equal_one_record_call(dev, path, with_critic, mid, critic_obs):
    """Episodes end on steps 2, 5 and T-1; every trajectory output, the recorded state rows, the final carries, lpf, pg_carry,
    command and done are bitwise those of kbs_rollout_record over all T steps, with critic_obs recorded or not.  A mid-episode
    start also loads a done_prev with every third env set (their lag state restarts on step 0), which the record call gets too."""
    T, N = 9, 600
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=9300) if mid else None
    b = Batch(9301, T, N, dev)
    for t in (2, 5, T - 1):
        ending_at(b, t)
    done_prev = torch.zeros(b.ld, dtype=torch.uint8, device=dev)
    if mid:
        done_prev[:N:3] = 1
    whole = run(dev, b, path, with_critic, start, critic_obs=critic_obs, done_prev=done_prev)
    assert int(whole["done"][:, :N].sum()) > N
    if mid:      # the loaded done_prev matters: without it step 0 differs
        other = run(dev, b, path, with_critic, start, critic_obs=critic_obs, done_prev=torch.zeros_like(done_prev))
        assert not torch.equal(other["actor_obs"][0], whole["actor_obs"][0])
    tr, fin = run_steps(dev, b, path, with_critic, start, critic_obs=critic_obs, done_prev=done_prev if mid else None)
    assert_steps_equal_record(tr, fin, whole, b, with_critic, "steps")


@pytest.mark.parametrize("path", [L.GEMM_SIMT_FP32, L.GEMM_TC_2XF16], ids=["simt", "tc2xf16"])
def test_other_entry_points_between_steps(dev, path):
    """kbs_ppo_variables (which reuses the handle's scratch) between every two steps changes nothing."""
    T, N = 5, 600
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=9400)
    b = Batch(9401, T, N, dev)
    ending_at(b, 2)
    whole = run(dev, b, path, True, start, critic_obs=True, done_prev=torch.zeros(b.ld, dtype=torch.uint8, device=dev))

    def between(e, io):
        ac, cc = torch.zeros_like(io["actor_carry"]), torch.zeros_like(io["critic_carry"])
        e.ppo_variables(torch.rand_like(io["actor_obs"]), torch.rand_like(io["action"]), io["done"], ac, torch.zeros_like(io["lpf"]),
                        torch.rand((T, L.CRITIC_OBS, b.ld), device=dev), cc, n_envs=N)

    tr, fin = run_steps(dev, b, path, True, start, between=between)
    assert_steps_equal_record(tr, fin, whole, b, True, "steps with kbs_ppo_variables between")


@pytest.mark.parametrize("path", PATHS)
def test_load_store_round_trip(dev, path):
    N, H = 300, 256
    ld = E.round_up4(N)
    g = torch.Generator(device=dev).manual_seed(5)
    rng = __import__("numpy").random.default_rng(3)
    c = {"actor_carry": Hn.carry_from_np(random_carry(rng, N, 2, H), dev),
         "critic_carry": Hn.carry_from_np(random_carry(rng, N, 2, H), dev),
         "lpf": torch.randn((20, ld), generator=g, device=dev), "pg_carry": torch.randn((3, ld), generator=g, device=dev),
         "command": torch.randn((16, ld), generator=g, device=dev),
         "done_prev": (torch.rand(ld, generator=g, device=dev) < 0.5).to(torch.uint8)}
    e, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    try:
        st = e.step_state(N, True, c)
        out = e.step_state_store(st, {k: torch.full_like(v, 3) for k, v in c.items()})
        zst = e.step_state(N, True)
        zero = e.step_state_store(zst, {k: torch.full_like(v, 3) for k, v in c.items()})
        torch.cuda.synchronize()
        for k in c:
            assert torch.equal(out[k], c[k]), k
            assert not zero[k].any(), k
    finally:
        e.close()


# ---- 2. validation -------------------------------------------------------------------------------------------------------------


def rc_of(fn) -> int:
    with pytest.raises(RuntimeError) as ex:
        fn()
    return int(str(ex.value).split("[")[1].split("]")[0])


@pytest.mark.parametrize("path", [L.GEMM_SIMT_FP32, L.GEMM_TC_2XF16], ids=["simt", "tc2xf16"])
def test_rollout_step_validation(dev, path):
    T, N = 2, 64
    b = Batch(9500, T, N, dev)
    e, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    try:
        io = Hn.rollout_buffers(b, 256, 2)
        st = e.step_state(N, True)
        step = lambda **kw: e.rollout_step(st, dict(dict(step_inputs(io, 0), **{k: io[k] for k in TRAJ if k in io}), **kw))
        assert rc_of(lambda: step(action=None)) == L_NULL
        assert rc_of(lambda: step(u_switch=None)) == L_NULL
        assert rc_of(lambda: step(state={k: v for k, v in step_inputs(io, 0)["state"].items() if k != "cvel"})) == L_NULL
        assert rc_of(lambda: step(traj_state={"cvel": torch.zeros((T, 144, b.ld), device=dev)},
                                  state={k: v for k, v in step_inputs(io, 0)["state"].items() if k != "cvel"},
                                  value=None)) == L_NULL
        f = torch.zeros(T * 20 * b.ld + 8, device=dev)
        assert rc_of(lambda: step(action=f[1:1 + T * 20 * b.ld].view(T, 20, b.ld))) == L_ALIGN
        u8 = torch.zeros(T * b.ld + 8, dtype=torch.uint8, device=dev)
        assert rc_of(lambda: step(done=u8[1:1 + T * b.ld].view(T, b.ld))) == L_ALIGN
        wide = Hn.rollout_buffers(Batch(9500, T, N + 8, dev), 256, 2)        # another ld than the state's
        assert rc_of(lambda: e.rollout_step(st, dict(step_inputs(wide, 0), **{k: wide[k] for k in TRAJ if k in wide}))) == L_SHAPE
        nc = e.step_state(N, False)
        assert rc_of(lambda: e.rollout_step(nc, dict(step_inputs(io, 0), **{k: io[k] for k in TRAJ if k in io}))) == -5
        small = E.StepState(st.buf, L.KbsStepState(st.buf.data_ptr(), st.desc.bytes - 256, N, 1))
        assert rc_of(lambda: e.rollout_step(small, dict(step_inputs(io, 0), **{k: io[k] for k in TRAJ if k in io}))) == L_SHAPE
        off = torch.empty(int(st.desc.bytes) + 512, dtype=torch.uint8, device=dev)
        mis = E.StepState(off, L.KbsStepState(off.data_ptr() + 16, st.desc.bytes, N, 1))
        assert rc_of(lambda: e.step_state_load(mis, {})) == L_ALIGN
        assert rc_of(lambda: e.step_state_load(st, {"done_prev": u8[1:1 + b.ld]})) == L_ALIGN
        # weights not packed
        e2 = E.KbotStep(gemm_path=path)
        try:
            st2 = e2.step_state(N, True)
            assert rc_of(lambda: e2.rollout_step(st2, dict(step_inputs(io, 0), **{k: io[k] for k in TRAJ if k in io}))) == L_STATE
        finally:
            e2.close()
        # a step past T: recorded nothing, flagged on the device, refused by the next call
        for t in range(T):
            step()
        before = {k: io[k].clone() for k in ("action", "done", "command")}
        step()
        torch.cuda.synchronize()
        for k, v in before.items():
            assert torch.equal(io[k], v), k
        assert e.device_status() & L.STATUS_STEP_RANGE
        assert rc_of(lambda: step()) == L_DEVICE
        e.device_status_reset()
        e.step_state_rewind(st)
        step()
        torch.cuda.synchronize()
        assert e.device_status() == 0
    finally:
        e.close()


# ---- 3. PpoUpdater's online form ----------------------------------------------------------------------------------------------


def integrate(state: dict, ctrl, t: int):
    """A toy simulator: the joint positions / velocities of step t + 1 follow the ctrl of step t."""
    state["qpos"][7:27] += 1e-3 * ctrl[t]
    state["qvel"][6:26].mul_(0.5).add_(1e-2 * ctrl[t])


def online_loop(up, io, b, rc, N, capture, steps_io):
    """PpoUpdater.begin_iteration -> step x T (simulator in the loop) -> end_iteration.  -> (its output, the library launches
    the T steps enqueued from the host: 0 when every step was a graph replay)."""
    up.begin_iteration(io, N)
    l0 = up.eng.launches
    io_t = steps_io
    for t in range(b.T):
        src = step_inputs(dict(io, state=b.state, noise={k: v for k, v in b.noise.items() if k != "eps_action"},
                               eps_action=b.noise["eps_action"], u_switch=b.cmd_rand["u_switch"], cmd_mode=b.cmd_rand["mode"],
                               cmd_u6=b.cmd_rand["u6"], cmd_u_arms=b.cmd_rand["u_arms"]), t)
        for k in ("noise",):
            for n in io_t[k]:
                io_t[k][n].copy_(src[k][n])
        for n in io_t["state"]:
            if n not in ("qpos", "qvel") or t == 0:
                io_t["state"][n].copy_(src["state"][n])
        for k in INPUTS:
            io_t[k].copy_(src[k])
        if capture and t == 1:
            up.capture_step(io_t)
        up.step(io_t)
        integrate(io_t["state"], io["ctrl"], t)
    launches = up.eng.launches - l0
    return up.end_iteration(rc, N, 128, 2, 13), launches


def hand_loop(up, io, b, rc, N, done_prev, sim):
    """The same with today's kbs_rollout_record (T = 1, pointers offset to slot t), kbs_rewards and epoch()."""
    T, ld = b.T, b.ld
    c0 = {k + "0": io[k].clone() for k in ("actor_carry", "critic_carry", "lpf")}
    cobs = torch.empty((T, L.CRITIC_OBS, ld), device=b.dev)
    traj = {k: torch.empty_like(v) for k, v in b.state.items()}
    for t in range(T):
        for n in traj:
            if n not in ("qpos", "qvel") or t == 0:
                sim[n].copy_(b.state[n][t])
            traj[n][t].copy_(sim[n])
        one = dict(io, state={k: v[None] for k, v in sim.items()}, noise={k: v[t:t + 1] for k, v in b.noise.items() if k != "eps_action"},
                   eps_action=b.noise["eps_action"][t:t + 1], u_switch=b.cmd_rand["u_switch"][t:t + 1],
                   cmd_mode=b.cmd_rand["mode"][t:t + 1], cmd_u6=b.cmd_rand["u6"][t:t + 1], cmd_u_arms=b.cmd_rand["u_arms"][t:t + 1],
                   command=io["command"][t:t + 2], critic_obs=cobs[t:t + 1], done_prev=done_prev, T=1,
                   **{k: io[k][t:t + 1] for k in ("actor_obs", "action", "log_prob", "ctrl", "term_codes", "done", "success", "value")})
        up.eng.rollout(one, N)
        done_prev = io["done"][t].clone()
        integrate(sim, io["ctrl"], t)
    rew = up.eng.rewards(traj, io["command"][:T], io["ctrl"], io["done"], rc, n_envs=N)
    ro = dict(c0, actor_obs=io["actor_obs"], critic_obs=cobs, action=io["action"], done=io["done"], success=io["success"], rewards=rew)
    out = dict(up.epoch(ro, N, batch_size=128, num_passes=2, seed=13), rewards=rew)
    io["command"][0].copy_(io["command"][T])
    return out, done_prev


@pytest.mark.parametrize("capture", [False, True], ids=["eager", "captured"])
def test_online_iterations_equal_record_loop(dev, capture, monkeypatch):
    """Closed loop, FP16-split, three iterations, episodes ending on the last step of the first two: PpoUpdater.step x T +
    end_iteration is bitwise the loop written with kbs_rollout_record, kbs_rewards and epoch() -- parameters, optimiser state,
    counters, loss statistics, norms, permutations, rewards, every trajectory output and the final carries.  Eager, or
    captured: the first iteration eager (capture_step needs one), the step captured at t = 1 of the second, and every step of
    the third replayed."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N = 6, 512
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=9600)
    b1, b2, b3 = Batch(9601, T, N, dev), Batch(9602, T, N, dev), Batch(9603, T, N, dev)
    ending_at(b1, T - 1)
    ending_at(b2, T - 1)
    ea, _, _ = Hn.make_engine(gemm_path=L.GEMM_TC_2XF16, device=dev)
    eb, _, _ = Hn.make_engine(gemm_path=L.GEMM_TC_2XF16, device=dev)
    try:
        ua, ub = PpoUpdater(ea, wa, wc), PpoUpdater(eb, wa, wc)
        ioa, iob = own_io(b1, start), own_io(b1, start)
        rca, rcb = reward_carry(b1.ld, dev), reward_carry(b1.ld, dev)
        io_t = step_inputs(own_io(b1, start), 0)
        io_t = {k: ({n: x.clone() for n, x in v.items()} if isinstance(v, dict) else v.clone()) for k, v in io_t.items()}
        sim = {k: v.clone() for k, v in io_t["state"].items()}
        done_prev = torch.zeros(b1.ld, dtype=torch.uint8, device=dev)
        for it, b in enumerate((b1, b2, b3)):
            oa, launches = online_loop(ua, ioa, b, rca, N, capture and it == 1, io_t)
            oa = {k: v.clone() for k, v in oa.items()}
            if capture and it == 2:
                assert launches == 0                                 # every step of the third iteration was a replay
            else:
                assert launches > 0
            ob, done_prev = hand_loop(ub, iob, b, rcb, N, done_prev, sim)
            fin = stored(ea, ua.step_st, ioa)
            torch.cuda.synchronize()
            assert ea.device_status() == 0 and eb.device_status() == 0
            for k in ("actor_carry", "critic_carry", "lpf", "pg_carry"):
                assert torch.equal(fin[k], iob[k]), f"iteration {it + 1}: final {k}"
            assert torch.equal(fin["command"], iob["command"][0]) and torch.equal(fin["done_prev"], done_prev)
            ioa["command"][0].copy_(fin["command"])                 # the state carries it; io's row 0 is the trajectory's
            assert_iteration_equal(ua, ub, oa, ob, {k: ioa[k] for k in TRAJ if k in ioa}, {k: iob[k] for k in TRAJ if k in iob},
                                   f"iteration {it + 1}")
            for k in rca:
                assert torch.equal(rca[k], rcb[k]), k
            assert torch.isfinite(oa["norms"]).all()
            if it == 0:
                assert int(done_prev[:N].sum()) > N // 3
    finally:
        ea.close()
        eb.close()
