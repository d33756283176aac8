"""The update phase of a PPO epoch on the device: kbs_minibatch_permutation (the permutation law, bitwise against the NumPy
restatement in test_ppo_epoch_cpu.py), kbs_shuffle_minibatches (bitwise against torch indexing), and ppo.PpoUpdater.epoch
as the composition of parts tested elsewhere (kbs_ppo_variables, kbs_gae, PpoUpdater.update), eager and replayed as one
CUDA graph."""

import os
import socket
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import scipy.stats
import torch

import harness as Hn
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200.ppo import PpoUpdater
from test_gpu_start_state import warm_start
from test_ppo_epoch_cpu import permutation

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
L_NULL, L_SHAPE, L_ALIGN = -1, -2, -3          # KBS_E_NULL, KBS_E_SHAPE, KBS_E_ALIGN


@pytest.fixture(scope="module")
def dev(cuda_device, lib_built):
    return cuda_device


@pytest.fixture(scope="module")
def eng(dev):
    e, _, _ = Hn.make_engine(hidden=256, gemm_path=L.GEMM_TC_2XF16, device=dev)
    yield e
    e.close()


def make_rollout(T, N, dev, seed, ld=None, H=256, depth=2, carry0=None) -> dict:
    """A synthetic stored rollout (what ksim's trajectory holds) with done resets; start carries random unless given
    (oracle layout, as warm_start returns them)."""
    ld = ld or N
    g = torch.Generator(device=dev).manual_seed(seed)
    rn = lambda *s, sc=1.0: torch.randn(s, generator=g, device=dev) * sc
    u8 = lambda p: (torch.rand((T, ld), generator=g, device=dev) < p).to(torch.uint8)
    done = u8(0.1)
    r = {"actor_obs": rn(T, 65, ld, sc=0.7), "critic_obs": rn(T, 475, ld, sc=0.7), "action": rn(T, 20, ld, sc=0.3),
         "done": done, "success": done & u8(0.5), "rewards": rn(T, ld, sc=0.5)}
    if carry0 is None:
        r.update(actor_carry0=rn(depth, 2, N, H, sc=0.3), critic_carry0=rn(depth, 2, N, H, sc=0.3), lpf0=rn(20, ld, sc=0.2))
    else:
        r.update(actor_carry0=Hn.carry_from_np(carry0["actor"], dev), critic_carry0=Hn.carry_from_np(carry0["critic"], dev))
        lpf = torch.zeros((20, ld), device=dev)
        lpf[:, :N] = torch.from_numpy(np.ascontiguousarray(carry0["lpf_params"].T)).to(dev)
        r["lpf0"] = lpf
    return r


def on_policy_actions(eng, ro: dict, N: int, seed: int) -> dict:
    """Replace the stored actions by samples of the policy `eng` holds, as a real rollout stores them.  Actions drawn
    independently of the policy have log-probs near -100: after one update the clipped ratio sits at exp(log_clip_value)
    and the std gradient leaves the FP16-split datapath's range (KBS_STATUS_F16_RANGE, documented in include/kbotstep.h)."""
    lpf = ro["lpf0"].clone()
    v = eng.ppo_variables(ro["actor_obs"], ro["action"], ro["done"], ro["actor_carry0"].clone(), lpf, want_std=True,
                          want_mean=True, n_envs=N)
    g = torch.Generator(device=ro["action"].device).manual_seed(seed)
    ro["action"].copy_(v["mean"] + v["action_std"] * torch.randn(v["mean"].shape, generator=g, device=ro["action"].device))
    return ro


def refill(dst: dict, src: dict):
    for k in dst:
        dst[k].copy_(src[k])


# ---- 1. the permutation law ----------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("n", [4, 64, 4096, 16384])
def test_permutation_matches_law_bitwise(eng, dev, n):
    """perm_out == argsort of (Philox key << 32) | e, for several (seed, pass, env0); the pass counter advances by one per
    call; another pass or env0 gives another permutation."""
    for seed, pass0, env0 in ((0, 0, 0), (12345, 7, 0), (2**40 + 3, 2**33 + 1, 4096), (99, 5, 3 * n)):
        pd = torch.tensor([pass0], dtype=torch.int64, device=dev)
        got = [eng.minibatch_permutation(pd, n, seed=seed, env0=env0).cpu().numpy() for _ in range(2)]
        assert int(pd.item()) == pass0 + 2
        for k in range(2):
            np.testing.assert_array_equal(got[k], permutation(seed, pass0 + k, env0, n), err_msg=f"{(seed, pass0 + k, env0)}")
        if n > 4:
            assert not np.array_equal(got[0], got[1])
            other = eng.minibatch_permutation(torch.tensor([pass0], dtype=torch.int64, device=dev), n, seed=seed, env0=env0 + n)
            assert not np.array_equal(other.cpu().numpy(), got[0])


def test_permutation_limits_and_uniformity(eng, dev):
    """n_envs above KBS_MAX_PERMUTATION_ENVS is refused; the position of element 0 over 4096 permutations of 64 passes a
    chi-square test of uniformity."""
    pd = torch.zeros(1, dtype=torch.int64, device=dev)
    with pytest.raises(RuntimeError, match=r"\[-2\]"):
        eng.minibatch_permutation(pd, L.MAX_PERMUTATION_ENVS + 4)
    assert int(pd.item()) == 0
    P = torch.empty((4096, 64), dtype=torch.int32, device=dev)
    for i in range(P.shape[0]):
        eng.minibatch_permutation(pd, 64, seed=5, out=P[i])
    assert int(pd.item()) == 4096
    pos = (P == 0).int().argmax(dim=1).cpu().numpy()
    assert scipy.stats.chisquare(np.bincount(pos, minlength=64)).pvalue > 1e-4
    assert (np.sort(P.cpu().numpy(), axis=1) == np.arange(64)).all()


# ---- 2. the shuffle -----------------------------------------------------------------------------------------------------------


def src_batch(ro: dict, g) -> dict:
    """A kbs_ppo_batch over the whole rollout: ro's fields plus [T, ld] stand-ins for the PPO variables."""
    T, _, ld = ro["actor_obs"].shape
    s = {k: ro[k] for k in ("actor_obs", "critic_obs", "action", "done", "actor_carry0", "critic_carry0", "lpf0")}
    for k in ("old_log_probs", "advantages", "value_targets", "old_values"):
        s[k] = torch.randn((T, ld), generator=g, device=ro["done"].device)
    return s


def indexed(src: dict, perm: torch.Tensor, bs: int) -> dict:
    """torch indexing x[..., perm] reshaped into minibatches: the expected kbs_shuffle_minibatches output."""
    idx = perm.long()
    nb = idx.numel() // bs
    out = {}
    for k, t in src.items():
        if t is None:
            continue
        if k.endswith("carry0"):
            x = t[:, :, idx]                                           # [depth, 2, N, H]
            out[k] = x.reshape(x.shape[0], 2, nb, bs, -1).permute(2, 0, 1, 3, 4)
        else:
            x = t[..., idx]                                            # [T, F, N] / [T, N] / [20, N]
            out[k] = x.reshape(x.shape[:-1] + (nb, bs)).movedim(-2, 0)
    return out


def assert_equal_dicts(got: dict, want: dict, what: str):
    assert got.keys() == want.keys(), what
    for k in want:
        assert torch.equal(got[k], want[k]), f"{what}: {k} differs ({int((got[k] != want[k]).sum())} entries)"


@pytest.mark.parametrize("kind", ["library", "identity", "reversal", "one-batch"])
def test_shuffle_matches_torch_indexing_bitwise(eng, dev, kind):
    """Every field, u8 done, both carries (distinct non-zero rows per env) and lpf0, at ld > n_envs."""
    T, N, H = 3, 512, 256
    ro = make_rollout(T, N, dev, seed=31, ld=N + 12)
    ro["actor_carry0"] = ro["actor_carry0"] + 1.0 + torch.arange(N, device=dev).view(1, 1, N, 1)      # distinct, non-zero
    ro["critic_carry0"] = ro["critic_carry0"] - 1.0 - torch.arange(N, device=dev).view(1, 1, N, 1)
    src = src_batch(ro, torch.Generator(device=dev).manual_seed(32))
    bs = N if kind == "one-batch" else 128
    if kind in ("library", "one-batch"):
        perm = eng.minibatch_permutation(torch.tensor([3], dtype=torch.int64, device=dev), N, seed=17)
    elif kind == "identity":
        perm = torch.arange(N, dtype=torch.int32, device=dev)
    else:
        perm = torch.arange(N - 1, -1, -1, dtype=torch.int32, device=dev)
    dst = eng.shuffle_minibatches(perm, src, N, bs)
    assert_equal_dicts(dst, indexed(src, perm, bs), kind)
    # without start carries: those destinations are left out
    src0 = {k: v for k, v in src.items() if not k.endswith("0")}
    assert_equal_dicts(eng.shuffle_minibatches(perm, src0, N, bs), indexed(src0, perm, bs), kind + " (no carries)")


def test_shuffle_validation(eng, dev):
    T, N, bs = 2, 256, 64
    ro = make_rollout(T, N, dev, seed=41, ld=N + 4)
    src = src_batch(ro, torch.Generator(device=dev).manual_seed(42))
    perm = torch.arange(N, dtype=torch.int32, device=dev)
    dst = eng.shuffle_minibatches(perm, src, N, bs)

    def rc(code, s=src, d=dst, n=N, b=bs, p=perm):
        with pytest.raises(RuntimeError, match=r"\[%d\]" % code):
            eng.shuffle_minibatches(p, s, n, b, dst=d)

    no_carry = {k: v for k, v in src.items() if k != "critic_carry0"}
    rc(L_NULL, s=no_carry)                                       # NULL source carry, non-NULL destination
    rc(L_NULL, d={k: v for k, v in dst.items() if k != "lpf0"})   # and the reverse
    rc(L_NULL, d={k: v for k, v in dst.items() if k != "done"})
    rc(L_SHAPE, n=N, b=62, d=eng.minibatch_buffers(T, 4, 62, dev))           # batch_size % 4
    rc(L_SHAPE, n=N - 8)                                          # n_envs % batch_size; num_batches != n_envs / batch_size
    rc(L_SHAPE, n=N + 64, d=eng.minibatch_buffers(T, 5, bs, dev), p=torch.arange(N + 64, dtype=torch.int32, device=dev))   # ld < n_envs
    skew = dict(dst, advantages=torch.empty(dst["advantages"].numel() + 1, device=dev)[1:].view_as(dst["advantages"]))
    rc(L_ALIGN, d=skew)
    rc(L_ALIGN, p=torch.arange(N + 1, dtype=torch.int32, device=dev)[1:])


def test_shuffle_out_of_range_index_gives_nan_columns(eng, dev):
    """Entries n_envs, -1 and n_envs + 5 of a permutation: their float columns are NaN (done 0) in their minibatch only;
    every other column is what torch indexing gives."""
    T, N, bs = 3, 512, 128
    ro = make_rollout(T, N, dev, seed=51)
    src = src_batch(ro, torch.Generator(device=dev).manual_seed(52))
    perm = eng.minibatch_permutation(torch.zeros(1, dtype=torch.int64, device=dev), N, seed=3)
    bad = perm.clone()
    cols = {1 * bs + 5: N, 1 * bs + 77: -1, 1 * bs + 127: N + 5}
    for k, v in cols.items():
        bad[k] = v
    got = eng.shuffle_minibatches(bad, src, N, bs)
    torch.cuda.synchronize()
    want = indexed(src, perm, bs)
    js = torch.tensor([k - bs for k in cols], device=dev)
    for k, t in got.items():
        w = want[k].clone()
        if k.endswith("carry0"):
            assert torch.isnan(t[1][:, :, js]).all(), k
            w[1][:, :, js] = t[1][:, :, js]
        else:
            sel = t[1][..., js]
            assert (sel == 0).all() if k == "done" else torch.isnan(sel).all(), k
            w[1][..., js] = sel
        assert torch.equal(torch.nan_to_num(t, nan=7.0) if t.is_floating_point() else t,
                           torch.nan_to_num(w, nan=7.0) if w.is_floating_point() else w), k
        others = [b for b in range(N // bs) if b != 1]
        assert not any(torch.isnan(t[b]).any() for b in others if t.is_floating_point()), k


# ---- 3. epoch == composition of tested parts, bitwise --------------------------------------------------------------------------


def state(up: PpoUpdater) -> dict:
    return {"param": up.param.clone(), "m": up.m.clone(), "v": up.v.clone(), "step": up.step_dev.clone()}


def reference_epoch(up: PpoUpdater, ro: dict, N: int, bs: int, passes: int, seed: int, pass0: int) -> tuple:
    """The epoch built by hand from tested parts: eng.ppo_variables and eng.gae called directly, minibatches by torch
    indexing with the NumPy permutation law, PpoUpdater.update.  Returns (state after each pass, stats, norms, perms)."""
    e = up.eng
    ac, cc, lpf = ro["actor_carry0"].clone(), ro["critic_carry0"].clone(), ro["lpf0"].clone()
    v = e.ppo_variables(ro["actor_obs"], ro["action"], ro["done"], ac, lpf, ro["critic_obs"], cc, want_std=False, n_envs=N)
    adv, tgt = e.gae(v["values"], ro["rewards"], ro["done"], ro["success"], n_envs=N)
    full = {"actor_obs": ro["actor_obs"], "critic_obs": ro["critic_obs"], "action": ro["action"], "done": ro["done"],
            "old_log_probs": v["log_probs"], "advantages": adv, "value_targets": tgt, "old_values": v["values"],
            "actor_carry0": ro["actor_carry0"], "critic_carry0": ro["critic_carry0"], "lpf0": ro["lpf0"]}
    states, stats, norms, perms = [], [], [], []
    for p in range(passes):
        perm = permutation(seed, pass0 + p, 0, N)
        perms.append(perm)
        for b in range(N // bs):
            idx = torch.from_numpy(perm[b * bs:(b + 1) * bs].astype(np.int64)).to(ro["done"].device)
            batch = {k: (t[:, :, idx] if k.endswith("carry0") else t[..., idx]).contiguous() for k, t in full.items()}
            stats.append(up.update(batch, bs)["stats"].clone())
            norms.append(up.norm.clone())
        states.append(state(up))
    return states, torch.stack(stats), torch.cat(norms), np.stack(perms)


def epoch_with_pass_states(up: PpoUpdater, ro: dict, N: int, bs: int, passes: int, seed: int) -> tuple:
    """up.epoch(), eager, with the updater's state cloned (stream-ordered) at the start of every pass after the first."""
    states, orig = [], up.eng.minibatch_permutation

    def spy(*a, **k):
        if k.get("out") is not None and k["out"].data_ptr() != up._ework["perm"][0].data_ptr():
            states.append(state(up))
        return orig(*a, **k)

    up.eng.minibatch_permutation = spy
    try:
        out = up.epoch(ro, N, batch_size=bs, num_passes=passes, seed=seed)
    finally:
        del up.eng.minibatch_permutation
    states.append(state(up))
    return states, out


@pytest.mark.parametrize("path", [L.GEMM_TC_2XF16, L.GEMM_TC_3XTF32], ids=["tc2xf16", "tc3xtf32"])
def test_epoch_is_the_composition_of_tested_parts(dev, path, monkeypatch):
    """Warm-start carries, done resets, T = 9, N = 512, batch 128, 3 passes: param, m, v, step counter after every pass and
    the per-update loss statistics and norms are bitwise those of the hand-built epoch.  Zero start carries change the
    result (the gathered carries are used)."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, H, bs, passes, seed = 9, 512, 256, 128, 3, 2024
    ea, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    eb, _, _ = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    ez, _, _ = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    try:
        ro = make_rollout(T, N, dev, seed=61, carry0=warm_start(wa, wc, N, H, 2, seed=9300))
        assert int(ro["done"][:, :N].sum()) > 0
        up, ref = PpoUpdater(ea, wa, wc), PpoUpdater(eb, wa, wc)
        got_states, out = epoch_with_pass_states(up, ro, N, bs, passes, seed)
        ref_states, stats, norms, perms = reference_epoch(ref, ro, N, bs, passes, seed, pass0=0)
        torch.cuda.synchronize()
        assert ea.device_status() == 0 and eb.device_status() == 0
        np.testing.assert_array_equal(out["perm"].cpu().numpy(), perms)
        assert int(up.pass_dev.item()) == passes and int(up.step_dev.item()) == passes * N // bs
        for p, (g, r) in enumerate(zip(got_states, ref_states)):
            for k in g:
                assert torch.equal(g[k], r[k]), f"after pass {p}: {k} differs"
        assert torch.equal(out["stats"], stats) and torch.equal(out["norms"], norms)
        assert torch.isfinite(norms).all()
        zero = dict(ro, actor_carry0=torch.zeros_like(ro["actor_carry0"]), critic_carry0=torch.zeros_like(ro["critic_carry0"]),
                    lpf0=torch.zeros_like(ro["lpf0"]))
        uz = PpoUpdater(ez, wa, wc)
        outz = uz.epoch(zero, N, batch_size=bs, num_passes=passes, seed=seed)
        assert not torch.equal(uz.param, up.param) and not torch.equal(outz["stats"], out["stats"])
    finally:
        for e in (ea, eb, ez):
            e.close()


# ---- 4. graph replay at the benchmarked size -------------------------------------------------------------------------------


def assert_same(a: PpoUpdater, b: PpoUpdater, oa: dict, ob: dict, what: str):
    for k in ("param", "m", "v", "step_dev", "pass_dev", "norm"):
        assert torch.equal(getattr(a, k), getattr(b, k)), f"{what}: {k} differs"
    for k in ("stats", "norms", "perm"):
        assert torch.equal(oa[k], ob[k]), f"{what}: {k} differs"


def test_epoch_graph_replay_matches_eager(dev, monkeypatch):
    """FP16-split, 4096 x 100, batch 512, 3 passes: one eager epoch, capture_epoch (changes nothing), two replays with the
    rollout refilled in place in between; each bitwise equal to an eager epoch from the same state on another updater, and
    the permutations those of the law at the same pass counter."""
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, H, bs, passes, seed = 100, 4096, 256, 512, 3, 77
    ea, wa, wc = Hn.make_engine(hidden=H, gemm_path=L.GEMM_TC_2XF16, device=dev)
    eb, _, _ = Hn.make_engine(hidden=H, gemm_path=L.GEMM_TC_2XF16, device=dev)
    try:
        ga, ref = PpoUpdater(ea, wa, wc), PpoUpdater(eb, wa, wc)
        ro = on_policy_actions(ea, make_rollout(T, N, dev, seed=71), N, seed=1)
        oa = {k: t.clone() for k, t in ga.epoch(ro, N, bs, passes, seed).items()}
        ob = ref.epoch(ro, N, bs, passes, seed)
        torch.cuda.synchronize()
        assert_same(ga, ref, oa, ob, "eager epoch")
        before = state(ga)
        ga.capture_epoch(ro, N, bs, passes, seed)
        torch.cuda.synchronize()
        for k, t in before.items():
            assert torch.equal(t, state(ga)[k]), f"capture changed {k}"
        for r in range(2):
            refill(ro, on_policy_actions(eb, make_rollout(T, N, dev, seed=72 + r), N, seed=2 + r))
            pass0 = int(ga.pass_dev.item())
            oa = ga.epoch(ro, N, bs, passes, seed)
            assert ga._epoch_graph is not None and oa is ga._epoch_out          # replayed, not run eagerly
            oa = {k: t.clone() for k, t in oa.items()}
            ob = ref.epoch(ro, N, bs, passes, seed)
            torch.cuda.synchronize()
            assert ea.device_status() == 0 and eb.device_status() == 0
            assert_same(ga, ref, oa, ob, f"replay {r + 1}")
            assert torch.isfinite(oa["norms"]).all()
            np.testing.assert_array_equal(oa["perm"].cpu().numpy(), np.stack([permutation(seed, pass0 + p, 0, N)
                                                                              for p in range(passes)]))
        assert int(ga.step_dev.item()) == 3 * passes * N // bs
    finally:
        ea.close()
        eb.close()


# ---- 5. two ranks ---------------------------------------------------------------------------------------------------------------


_NCCL_WORKER = r"""
import os, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/oracle"); sys.path.insert(0, %(root)r + "/tests")
import numpy as np, torch, torch.distributed as dist
import harness as Hn
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200.ppo import PpoUpdater
from test_gpu_ppo_epoch import make_rollout
from test_ppo_epoch_cpu import permutation
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dev = torch.device("cuda", rank)
torch.cuda.set_device(dev)
dist.init_process_group("nccl", device_id=dev)
T, N, bs = 9, 256, 128
e, wa, wc = Hn.make_engine(hidden=256, gemm_path=L.GEMM_TC_2XF16, device=dev)
up = PpoUpdater(e, wa, wc)
out = up.epoch(make_rollout(T, N, dev, seed=80 + rank), N, batch_size=bs, num_passes=2, seed=5)
perm = out["perm"].cpu().numpy()
for p in range(2):
    assert np.array_equal(perm[p], permutation(5, p, rank * N, N)), (rank, p)
allp = [torch.empty_like(up.param) for _ in range(world)]
dist.all_gather(allp, up.param)
assert all(torch.equal(x, allp[0]) for x in allp), "the replicas' parameters differ"
allq = [torch.empty_like(out["perm"]) for _ in range(world)]
dist.all_gather(allq, out["perm"])
assert not torch.equal(allq[0], allq[1]), "the ranks drew the same permutations"
e.close()
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_epoch_two_ranks_nccl(dev, tmp_path):
    """One epoch per rank on its own envs (env0 = rank * N): different permutations, bitwise identical parameters."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(_NCCL_WORKER % {"root": str(ROOT)})
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="2", OMP_NUM_THREADS="4",
               KBS_PPO_PER_STEP="0")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    try:
        outs = [p.communicate(timeout=600)[0] for p in procs]
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
                p.communicate()
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o}"
        assert f"rank {r} ok" in o
