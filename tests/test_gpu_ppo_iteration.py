"""A PPO iteration on the rollout the library records: kbs_rollout_record's critic observations (against the oracle and
kbs_observations, and without changing any other output), its done_prev (a rollout split at an episode end, or run one step
per call, is the one-call rollout), its validation, and ppo.PpoUpdater.iteration as the composition rollout -> rewards ->
epoch, eager and replayed as one CUDA graph."""

import numpy as np
import pytest
import torch

import harness as Hn
import kbot_oracle as O
from harness import Batch
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200 import synth
from kbot_joystick_b200.ppo import PpoUpdater
from test_gpu_start_state import warm_start, weights

pytestmark = pytest.mark.gpu

S = synth.from_soa
PATHS = [pytest.param(L.GEMM_SIMT_FP32, id="simt"), pytest.param(L.GEMM_TC_3XTF32, id="tc3xtf32"),
         pytest.param(L.GEMM_TC_2XF16, id="tc2xf16")]
OUTPUTS = ("actor_obs", "action", "log_prob", "ctrl", "term_codes", "done", "success", "value", "command", "actor_carry",
           "critic_carry", "lpf", "pg_carry")
L_NULL, L_ALIGN = -1, -3          # KBS_E_NULL, KBS_E_ALIGN


@pytest.fixture(scope="module")
def dev(cuda_device, lib_built):
    return cuda_device


def run(dev, b, path, with_critic=True, start=None, critic_obs=False, done_prev=None, chunks=None, monkeypatch=None):
    """One rollout call on batch b on a fresh engine; critic_obs=True records them, done_prev is passed through."""
    if chunks is not None:
        monkeypatch.setenv("KBS_ROLLOUT_CHUNKS", str(chunks))
    e, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    io = Hn.rollout_buffers(b, 256, 2, with_critic, start=start)
    if critic_obs:
        io["critic_obs"] = torch.full((b.T, L.CRITIC_OBS, b.ld), float("nan"), device=dev)
    io["done_prev"] = done_prev
    e.rollout(io, b.N)
    torch.cuda.synchronize()
    assert e.device_status() == 0
    e.close()
    return io


def assert_outputs_equal(a: dict, b: dict, what: str):
    for k in OUTPUTS:
        if a.get(k) is not None or b.get(k) is not None:
            assert torch.equal(a[k], b[k]), f"{what}: {k} differs"


# ---- 1. recorded critic observations ------------------------------------------------------------------------------------------


NAMES = {L.GEMM_SIMT_FP32: "simt", L.GEMM_TC_3XTF32: "tc3xtf32", L.GEMM_TC_2XF16: "tc2xf16"}
CASES = [(p, c, 1, m) for p in NAMES for c, m in ((True, False), (False, True), (True, True))] + [
    (L.GEMM_TC_2XF16, True, 4, True), (L.GEMM_TC_3XTF32, False, 4, False)]
CASES = [pytest.param(*c, id=f"{NAMES[c[0]]}-{'critic' if c[1] else 'nocritic'}-chunks{c[2]}-{'mid' if c[3] else 'zero'}")
         for c in CASES]


@pytest.mark.parametrize("path,with_critic,chunks,mid", CASES)
def test_recorded_critic_obs(dev, path, with_critic, chunks, mid, monkeypatch):
    """critic_obs of every step against the oracle's critic_obs_from_dict (at the observation tolerance of the parity tests)
    and bitwise against kbs_observations(critic_obs) on the same stored state and command.  The critic concatenation holds
    the clean projected gravity, not the lagged one, so it does not depend on how a datapath computes the lag state (the
    obs kernel's inline EMA on SIMT, the scan of phase A on the tensor-core paths): every datapath must match bitwise.
    Every other output is bitwise that of the same call without critic_obs (with chunks = 4: the per-chunk scratch is
    replaced by the caller's buffer)."""
    T, N = 7, 300
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=8100) if mid else None
    b = Batch(8200 + N, T, N, dev)
    plain = run(dev, b, path, with_critic, start, chunks=chunks, monkeypatch=monkeypatch)
    rec = run(dev, b, path, with_critic, start, critic_obs=True, chunks=chunks, monkeypatch=monkeypatch)
    assert_outputs_equal(rec, plain, "with critic_obs")
    ref = Hn.oracle_rollout(b, wa, wc, 256, 2, with_critic, start=start)
    got = S(rec["critic_obs"], N, (475,))
    assert np.isfinite(got).all()
    for t in range(T):
        o, _ = O.get_observations(b.np_state_at(t), b.np_noise_at(t), b.np["episode"], None, Hn.P)
        Hn.close(got[t], O.critic_obs_from_dict(o, ref["command"][t]), f"critic_obs t={t}")
    e, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    want = torch.full_like(rec["critic_obs"], float("nan"))
    for t in range(T):
        e.observations(b.state_at(t), rec["command"][t], b.noise_at(t), b.episode, critic_obs=want[t], n_envs=N)
    torch.cuda.synchronize()
    e.close()
    assert torch.equal(rec["critic_obs"][:, :, :N], want[:, :, :N])


# ---- 2. splits at episode ends ------------------------------------------------------------------------------------------------


def ending_at(b: Batch, t: int):
    """Every other env's episode ends at step t (time past max_length_sec): the split the lag state has to cross."""
    st = b.np["state"]
    st["time"][t, ::2] = 12.5
    b.state = {k: synth.to_soa(v, 1, b.dev) for k, v in st.items()}


def part(b: Batch, t0: int, t1: int) -> Batch:
    bb = Batch.__new__(Batch)
    bb.T, bb.N, bb.dev, bb.ld, bb.cmd0 = t1 - t0, b.N, b.dev, b.ld, b.cmd0
    bb.state = {k: v[t0:t1].contiguous() for k, v in b.state.items()}
    bb.noise = {k: v[t0:t1].contiguous() for k, v in b.noise.items()}
    bb.cmd_rand = {k: v[t0:t1].contiguous() for k, v in b.cmd_rand.items()}
    bb.episode = b.episode
    return bb


def split_run(dev, b: Batch, path, bounds, start, pass_done: bool) -> dict:
    """The rollout of b as consecutive calls over [bounds[i], bounds[i+1]), each continuing from the previous one's carries,
    pg_carry, lpf and command[T]; pass_done: done_prev = the previous call's done[T-1].  -> the outputs concatenated."""
    e, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    parts, prev = [], None
    for t0, t1 in zip(bounds[:-1], bounds[1:]):
        io = Hn.rollout_buffers(part(b, t0, t1), 256, 2, start=start if prev is None else None)
        if prev is not None:
            io["command"][0] = prev["command"][-1]
            for k in ("actor_carry", "critic_carry", "lpf", "pg_carry"):
                io[k] = prev[k].clone()
            if pass_done:
                io["done_prev"] = prev["done"][-1].clone()
        e.rollout(io, b.N)
        parts.append(io)
        prev = io
    torch.cuda.synchronize()
    assert e.device_status() == 0
    e.close()
    out = {k: torch.cat([p[k] for p in parts]) for k in ("actor_obs", "action", "log_prob", "ctrl", "term_codes", "done", "success",
                                                         "value")}
    out["command"] = torch.cat([p["command"][:-1] for p in parts] + [parts[-1]["command"][-1:]])
    for k in ("actor_carry", "critic_carry", "lpf", "pg_carry"):
        out[k] = parts[-1][k]
    return out


@pytest.mark.parametrize("path", PATHS)
def test_split_at_episode_end_with_done_prev(dev, path):
    """Two calls split where episodes end (T1 - 1), the second given the first's done[T1-1], are bitwise the one-call
    rollout, which matches the oracle.  Without done_prev the lag state of the envs that ended does not restart on step T1,
    and the actor observation there differs: the case is really exercised."""
    T1, T2, N = 21, 19, 2048
    T = T1 + T2
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=8300)
    b = Batch(8301, T, N, dev)
    ending_at(b, T1 - 1)
    whole = run(dev, b, path, True, start)
    ref = Hn.oracle_rollout(b, wa, wc, 256, 2, start=start)
    ended = ref["done"][T1 - 1]
    assert ended.sum() > N // 3 and (~ended).any()
    errs = Hn.compare_rollout(whole, ref, N)
    assert all(v <= 1.0 for v in errs.values()), errs
    split = split_run(dev, b, path, (0, T1, T), start, pass_done=True)
    assert_outputs_equal(split, whole, "split with done_prev")
    bad = split_run(dev, b, path, (0, T1, T), start, pass_done=False)
    a_bad, a_whole = S(bad["actor_obs"][T1], N, (65,)), S(whole["actor_obs"][T1], N, (65,))
    assert np.array_equal(a_bad[~ended], a_whole[~ended])
    assert (a_bad[ended][:, 40:45] != a_whole[ended][:, 40:45]).any(axis=1).mean() > 0.8   # the noisy lagged-gravity encoding


@pytest.mark.parametrize("path", PATHS)
def test_one_step_calls_equal_one_call(dev, path):
    """The online form: T calls of one step each, every call given the previous call's done, are bitwise the T-step call,
    with episodes ending on several steps."""
    T, N = 12, 2048
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=8400)
    b = Batch(8401, T, N, dev)
    for t in (2, 5, 6):
        ending_at(b, t)
    whole = run(dev, b, path, True, start)
    assert int(whole["done"][:, :N].sum()) > N
    steps = split_run(dev, b, path, tuple(range(T + 1)), start, pass_done=True)
    assert_outputs_equal(steps, whole, "one-step calls")


# ---- 3. validation ------------------------------------------------------------------------------------------------------------


class _NullRecord:
    """The engine's library with kbs_rollout routed to kbs_rollout_record(rec = NULL)."""

    def __init__(self, lib):
        self._lib = lib

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def kbs_rollout(self, h, io, n, stream):
        return self._lib.kbs_rollout_record(h, io, None, n, stream)


@pytest.mark.parametrize("path", [L.GEMM_SIMT_FP32, L.GEMM_TC_2XF16], ids=["simt", "tc2xf16"])
def test_rollout_record_validation(dev, path):
    T, N = 3, 64
    b = Batch(8500, T, N, dev)
    plain = run(dev, b, path)
    e, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    try:
        e.lib = _NullRecord(e.lib)
        io = Hn.rollout_buffers(b, 256, 2)
        e.rollout(io, N)
        torch.cuda.synchronize()
        assert_outputs_equal(io, plain, "rec == NULL")
        e.lib = e.lib._lib

        def rc_of(**kw):
            io = dict(Hn.rollout_buffers(b, 256, 2), **kw)
            with pytest.raises(RuntimeError) as ex:
                e.rollout(io, N)
            return int(str(ex.value).split("[")[1].split("]")[0])

        u8 = torch.zeros(b.ld + 8, dtype=torch.uint8, device=dev)
        f = torch.zeros(T * L.CRITIC_OBS * b.ld + 8, device=dev)
        assert rc_of(done_prev=u8[1:1 + b.ld]) == L_ALIGN
        assert rc_of(critic_obs=f[1:1 + T * L.CRITIC_OBS * b.ld].view(T, L.CRITIC_OBS, b.ld)) == L_ALIGN
        cobs = torch.zeros((T, L.CRITIC_OBS, b.ld), device=dev)
        for row in ("cinert", "cvel", "actuator_force"):
            st = {k: v for k, v in b.state.items() if k != row}
            assert rc_of(state=st, value=None, critic_carry=None, critic_obs=cobs) == L_NULL, row
        # ... and without critic_obs (nor value) the same state is accepted
        st = {k: v for k, v in b.state.items() if k not in ("cinert", "cvel", "actuator_force")}
        e.rollout(dict(Hn.rollout_buffers(b, 256, 2, with_critic=False), state=st, done_prev=u8[:b.ld]), N)
        torch.cuda.synchronize()
    finally:
        e.close()


# ---- 4. the iteration -----------------------------------------------------------------------------------------------------


def own_io(b: Batch, start) -> dict:
    """rollout_buffers with inputs of its own (refilled in place between iterations)."""
    io = Hn.rollout_buffers(b, 256, 2, start=start)
    for k in ("state", "noise", "episode"):
        io[k] = {n: t.clone() for n, t in io[k].items()}
    for k in ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms"):
        io[k] = io[k].clone()
    return io


def refill_inputs(io: dict, b: Batch):
    for k in io["state"]:
        io["state"][k].copy_(b.state[k])
    for k in io["noise"]:
        io["noise"][k].copy_(b.noise[k])
    io["eps_action"].copy_(b.noise["eps_action"])
    for k, src in (("u_switch", "u_switch"), ("cmd_mode", "mode"), ("cmd_u6", "u6"), ("cmd_u_arms", "u_arms")):
        io[k].copy_(b.cmd_rand[src])


def reward_carry(ld, dev) -> dict:
    return {"t_single": torch.zeros(ld, device=dev), "airtime": torch.zeros((2, ld), device=dev),
            "prev_contact": torch.ones((2, ld), dtype=torch.uint8, device=dev)}


def updater_state(up: PpoUpdater) -> dict:
    return {k: getattr(up, k).clone() for k in ("param", "m", "v", "step_dev", "pass_dev", "norm")}


def hand_iteration(up: PpoUpdater, io: dict, rc: dict, N, bs, passes, seed, done_prev) -> tuple:
    """carry snapshot -> KbotStep.rollout with critic_obs (and done_prev) -> rewards -> epoch, called one by one."""
    T, ld = io["T"], io["done"].shape[1]
    c0 = {k + "0": io[k].clone() for k in ("actor_carry", "critic_carry", "lpf")}
    cobs = torch.empty((T, L.CRITIC_OBS, ld), device=io["done"].device)
    up.eng.rollout(dict(io, critic_obs=cobs, done_prev=done_prev), N)
    rew = up.eng.rewards(io["state"], io["command"][:T], io["ctrl"], io["done"], rc, n_envs=N)
    ro = dict(c0, actor_obs=io["actor_obs"], critic_obs=cobs, action=io["action"], done=io["done"], success=io["success"],
              rewards=rew)
    out = dict(up.epoch(ro, N, batch_size=bs, num_passes=passes, seed=seed), rewards=rew)
    io["command"][0].copy_(io["command"][T])
    return out, io["done"][T - 1].clone()


def assert_iteration_equal(ua, ub, oa, ob, ioa, iob, what):
    for k, t in updater_state(ua).items():
        assert torch.equal(t, updater_state(ub)[k]), f"{what}: {k} differs"
    for k in ("stats", "norms", "perm", "rewards"):
        assert torch.equal(oa[k], ob[k]), f"{what}: {k} differs"
    assert_outputs_equal(ioa, iob, what)


@pytest.mark.parametrize("path", [L.GEMM_TC_2XF16, L.GEMM_TC_3XTF32], ids=["tc2xf16", "tc3xtf32"])
def test_iteration_is_the_hand_composition(dev, path, monkeypatch):
    """Two consecutive iterations from a warm start, episodes ending on step T-1 of the first (so the second's done_prev
    restarts lag states): parameters, optimiser state, counters, loss statistics, norms, permutations, rewards and every
    rollout output are bitwise those of the hand-built composition."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, bs, passes, seed = 9, 512, 128, 3, 31
    wa, wc = weights(256, 2)
    start = warm_start(wa, wc, N, 256, 2, seed=8600)
    b1, b2 = Batch(8601, T, N, dev), Batch(8602, T, N, dev)
    ending_at(b1, T - 1)
    ea, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    eb, _, _ = Hn.make_engine(gemm_path=path, device=dev)
    try:
        ua, ub = PpoUpdater(ea, wa, wc), PpoUpdater(eb, wa, wc)
        ioa, iob = own_io(b1, start), own_io(b1, start)
        rca, rcb = reward_carry(b1.ld, dev), reward_carry(b1.ld, dev)
        done_prev = None
        for it, b in enumerate((b1, b2)):
            if it:
                refill_inputs(ioa, b)
                refill_inputs(iob, b)
            oa = ua.iteration(ioa, rca, N, bs, passes, seed)
            ob, done_prev = hand_iteration(ub, iob, rcb, N, bs, passes, seed, done_prev)
            torch.cuda.synchronize()
            assert ea.device_status() == 0 and eb.device_status() == 0
            assert_iteration_equal(ua, ub, oa, ob, ioa, iob, f"iteration {it + 1}")
            for k in rca:
                assert torch.equal(rca[k], rcb[k]), k
            assert torch.isfinite(oa["norms"]).all()
            if it == 0:
                assert int(done_prev[:N].sum()) > N // 3       # the second iteration restarts these lag states
        assert int(ua.step_dev.item()) == 2 * passes * N // bs
    finally:
        ea.close()
        eb.close()


def device_io(d: dict, N: int, H: int, dev) -> dict:
    T, ld = d["u_switch"].shape
    f = dict(device=dev, dtype=torch.float32)
    command = torch.zeros((T + 1, 16, ld), **f)
    io = {k: d[k] for k in ("state", "noise", "episode", "eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms")}
    io.update(command=command, pg_carry=torch.zeros((3, ld), **f), actor_carry=torch.zeros((2, 2, N, H), **f),
              critic_carry=torch.zeros((2, 2, N, H), **f), lpf=torch.zeros((20, ld), **f), actor_obs=torch.zeros((T, 65, ld), **f),
              action=torch.zeros((T, 20, ld), **f), log_prob=torch.zeros((T, ld), **f), ctrl=torch.zeros((T, 20, ld), **f),
              term_codes=None, done=torch.zeros((T, ld), dtype=torch.uint8, device=dev),
              success=torch.zeros((T, ld), dtype=torch.uint8, device=dev), value=torch.zeros((T, ld), **f), T=T)
    return io


def refill_device(io: dict, d: dict):
    for k in ("state", "noise"):
        for n in io[k]:
            io[k][n].copy_(d[k][n])
    for k in ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms"):
        io[k].copy_(d[k])


def test_iteration_graph_replay_matches_eager(dev, monkeypatch):
    """FP16-split, 4096 x 100, batch 512, 3 passes: one eager iteration, capture_iteration (changes nothing), two replays
    with the state and noise refilled in place; each bitwise equal to an eager iteration on another updater."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, H, bs, passes, seed = 100, 4096, 256, 512, 3, 5
    ea, wa, wc = Hn.make_engine(hidden=H, gemm_path=L.GEMM_TC_2XF16, device=dev)
    eb, _, _ = Hn.make_engine(hidden=H, gemm_path=L.GEMM_TC_2XF16, device=dev)
    try:
        ua, ub = PpoUpdater(ea, wa, wc), PpoUpdater(eb, wa, wc)
        d = synth.make_batch_device(9100, T, N, dev)
        ioa = device_io(d, N, H, dev)
        iob = device_io({k: ({n: t.clone() for n, t in v.items()} if isinstance(v, dict) else v.clone()) for k, v in d.items()},
                        N, H, dev)
        for io in (ioa, iob):
            io["command"][0].copy_(torch.rand((16, io["command"].shape[-1]), generator=torch.Generator(device=dev).manual_seed(1),
                                              device=dev) - 0.5)
        rca, rcb = reward_carry(ioa["done"].shape[1], dev), reward_carry(ioa["done"].shape[1], dev)
        oa = {k: t.clone() for k, t in ua.iteration(ioa, rca, N, bs, passes, seed).items()}
        ob = ub.iteration(iob, rcb, N, bs, passes, seed)
        torch.cuda.synchronize()
        assert_iteration_equal(ua, ub, oa, ob, ioa, iob, "eager iteration")
        before = updater_state(ua)
        ua.capture_iteration(ioa, rca, N, bs, passes, seed)
        torch.cuda.synchronize()
        for k, t in before.items():
            assert torch.equal(t, updater_state(ua)[k]), f"capture changed {k}"
        for r in range(2):
            d = synth.make_batch_device(9101 + r, T, N, dev)
            refill_device(ioa, d)
            refill_device(iob, d)
            oa = ua.iteration(ioa, rca, N, bs, passes, seed)
            assert oa is ua._iter_out                          # replayed, not run eagerly
            oa = {k: t.clone() for k, t in oa.items()}
            ob = ub.iteration(iob, rcb, N, bs, passes, seed)
            torch.cuda.synchronize()
            assert ea.device_status() == 0 and eb.device_status() == 0
            assert_iteration_equal(ua, ub, oa, ob, ioa, iob, f"replay {r + 1}")
            for k in rca:
                assert torch.equal(rca[k], rcb[k]), k
            assert torch.isfinite(oa["norms"]).all() and int(ioa["done"][:, :N].sum()) > 0
        assert int(ua.step_dev.item()) == 3 * passes * N // bs
    finally:
        ea.close()
        eb.close()
