"""ppo.PpoUpdater update by update: gradient -> all-reduce -> global norm -> AdamW (clip folded in) -> re-pack of both
networks' weight images, eager and replayed as one CUDA graph.

Two independent K-update trajectories cannot be compared element by element: Adam's first steps are close to -lr sign(g),
so a gradient entry near zero flips its parameter by 2 lr on rounding alone.  Every update k is therefore checked from the
state the updater itself had before it (param, m, v, step counter): the gradient against float64 autograd
(oracle/ppo_grad_torch.py) at those parameters -- which only holds if the previous update's re-pack reached both networks
-- the norm against the float64 norm of that gradient, and param / m / v against the float64 AdamW step
(kbot_oracle.adamw_update) from that state.  Minibatches alternate advantages and value targets scaled x1 and x8 and the
clip limit sits between their gradient norms, so both branches of the global-norm clip run."""

import os
import socket
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import harness as Hn
import kbot_oracle as O
import ppo_grad_torch as G
from harness import close
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200 import synth
from kbot_joystick_b200.engine import KbotStep
from kbot_joystick_b200.ppo import PpoUpdater
from test_gpu_start_state import clear_kinks, warm_start

pytestmark = pytest.mark.gpu

S = synth.from_soa
ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def dev(cuda_device, lib_built):
    return cuda_device


# ---- helpers ---------------------------------------------------------------------------------------------------------------


def to_np(w: dict) -> dict:
    """eqx-layout dict of device tensors (NetParams.as_dict views) -> numpy copies, the oracle's form."""
    a = lambda x: x.detach().cpu().numpy().copy()
    return {"w_in": a(w["w_in"]), "b_in": a(w["b_in"]), "w_out": a(w["w_out"]), "b_out": a(w["b_out"]),
            "layers": [{k: a(l[k]) for k in ("w_ih", "w_hh", "b")} for l in w["layers"]]}


def weights_at(up: PpoUpdater, param: torch.Tensor) -> tuple:
    """The actor's and critic's eqx-layout weights held in a flat [actor | critic] parameter vector (numpy)."""
    return to_np(up.pa.as_dict(param[:up.na])), to_np(up.pc.as_dict(param[up.na:]))


def minibatch(seed, T, N, p, wa, wc, carry0=None, scale=1.0, hyper=None) -> dict:
    """Hn.ppo_batch taken near the policy (wa, wc), advantages and value targets scaled by `scale`, moved off the kinks of
    the clipped loss at that policy."""
    rng = np.random.default_rng(seed)
    b = Hn.ppo_batch(rng, T, N, p.hidden_size, p, wa, wc, carry0=carry0)
    b["advantages"] = (b["advantages"] * scale).astype(np.float32)
    b["value_targets"] = (b["value_targets"] * scale).astype(np.float32)
    return clear_kinks(b, *forward(wa, wc, b, p, carry0), hyper or {})


def forward(wa, wc, b: dict, p, carry0=None) -> tuple:
    """The reference's log-probs and values of minibatch b under (wa, wc) (float64, no gradient)."""
    with torch.no_grad():
        _, _, lp, val = G.ppo_minibatch_loss(G.weights_to_torch(wa, False), G.weights_to_torch(wc, False), b["actor_obs"],
                                             b["critic_obs"], b["action"], b["done"], b["old_log_probs"], b["advantages"],
                                             b["value_targets"], b["old_values"], p, {}, carry0)
    return lp.numpy(), val.numpy()


def ref_norm(ref) -> float:
    """float64 global norm of a reference's [actor | critic] gradient."""
    return float(np.sqrt(sum(float((g.astype(np.float64) ** 2).sum()) for r in (ref[2], ref[3])
                             for _, _, g in Hn.grad_tensors(r, len(r["layers"])))))


def clip_limit(wa, wc, b1: dict, b8: dict, p, carry0, hyper) -> float:
    """max_grad_norm between the reference gradient norms of one minibatch at x1 and at x8 (their geometric mean)."""
    n1 = ref_norm(G.ppo_minibatch_grads(wa, wc, b1, p, hyper=hyper, carry0=carry0))
    n8 = ref_norm(G.ppo_minibatch_grads(wa, wc, b8, p, hyper=hyper, carry0=carry0))
    assert n8 > 3 * n1, (n1, n8)
    return float(np.sqrt(n1 * n8))


def snapshot(up: PpoUpdater) -> dict:
    return {"param": up.param.clone(), "m": up.m.clone(), "v": up.v.clone(), "step": up.step_count}


def assert_state_is(up: PpoUpdater, snap: dict, what: str):
    for k in ("param", "m", "v"):
        assert torch.equal(getattr(up, k), snap[k]), f"{what}: {k} changed"
    assert up.step_count == snap["step"], f"{what}: step counter {up.step_count} != {snap['step']}"


def check_update(up: PpoUpdater, snap: dict, out: dict, b: dict, p, k: int, limit: float, carry0=None, hyper=None) -> float:
    """Update k (1-based) of `up`, from the state `snap` it started from, on minibatch b (numpy).  Returns the reference
    gradient norm (which side of `limit` it is on decides the clip branch)."""
    torch.cuda.synchronize()
    assert up.eng.device_status() == 0, f"update {k}: device health word set"
    N, na = b["done"].shape[1], up.na
    wa, wc = weights_at(up, snap["param"])
    ref = G.ppo_minibatch_grads(wa, wc, b, p, hyper=hyper or {}, carry0=carry0)
    loss, stats, ga_ref, gc_ref, lp_ref, val_ref = ref
    # 1. the gradient at the parameters the update started from: the previous update re-packed both networks
    close(S(out["log_probs"], N), lp_ref, f"update {k}: log_probs", atol=1e-4)
    close(S(out["values"], N), val_ref, f"update {k}: values", atol=1e-5)
    close(out["stats"].cpu().numpy(), np.array((loss,) + stats, np.float32), f"update {k}: loss stats", rtol=2e-5, atol=1e-5)
    bad = (Hn.compare_grads_blockwise(up.pa.as_dict(up.grad[:na]), ga_ref, "actor", p.hidden_size, p.depth) +
           Hn.compare_grads_blockwise(up.pc.as_dict(up.grad[na:]), gc_ref, "critic", p.hidden_size, p.depth))
    assert not bad, (f"update {k}", bad)
    # 2. the global norm of the whole [actor | critic] gradient
    g = up.grad.double().cpu().numpy()
    gn = float(np.sqrt(np.sum(g * g)))
    assert abs(float(up.norm) - gn) <= 2e-7 * gn, (f"update {k}: norm", float(up.norm), gn)
    # 3. AdamW with the clip folded in, one step from the snapshot state (tolerances of test_adamw_and_grad_norm_against_float64)
    opt = {key: up.opt[key] for key in ("lr", "b1", "b2", "eps", "weight_decay")}
    rp, rm, rv, applied = O.adamw_update(snap["param"].cpu().numpy(), g, snap["m"].cpu().numpy(), snap["v"].cpu().numpy(), k,
                                         grad_scale=1.0, max_grad_norm=limit, **opt)
    assert applied
    close(up.param.cpu().numpy(), rp, f"update {k}: param", rtol=1e-6, atol=2e-7)
    close(up.m.cpu().numpy(), rm, f"update {k}: m", rtol=1e-5, atol=1e-9)
    close(up.v.cpu().numpy(), rv, f"update {k}: v", rtol=1e-5, atol=1e-12)
    assert up.step_count == k
    rn = ref_norm(ref)
    assert abs(np.log(rn / limit)) > 0.05, ("the clip branch is ambiguous", rn, limit)
    return rn


def refill(dst: dict, src: dict):
    """Copy a minibatch into the tensors a captured graph reads (in place: the graph holds their addresses)."""
    assert dst.keys() == src.keys()
    for k in dst:
        dst[k].copy_(src[k])


def assert_repacked(up: PpoUpdater, H: int, path: int, batch: dict, N: int):
    """The updater's engine and a fresh handle packed from up.pa / up.pc give bitwise the same kbs_ppo_grad on `batch`: the
    last update re-packed both networks' weight images from the final parameters."""
    fresh = KbotStep(hidden_size=H, depth=up.pa.depth, gemm_path=path)
    fresh.pack_weights(L.NET_ACTOR, up.pa.as_dict())
    fresh.pack_weights(L.NET_CRITIC, up.pc.as_dict())
    res = []
    for e in (up.eng, fresh):
        g = torch.full_like(up.grad, float("nan"))
        out = e.ppo_grad(batch, up.pa.as_dict(g[:up.na]), up.pc.as_dict(g[up.na:]), n_envs=N, **up.loss_hyper)
        torch.cuda.synchronize()
        assert e.device_status() == 0
        res.append((g, out))
    fresh.close()
    (ga, oa), (gb, ob) = res
    assert torch.isfinite(ga).all()
    for name, a, b in (("actor gradient", ga[:up.na], gb[:up.na]), ("critic gradient", ga[up.na:], gb[up.na:]),
                       ("log_probs", oa["log_probs"][:, :N], ob["log_probs"][:, :N]),
                       ("values", oa["values"][:, :N], ob["values"][:, :N]), ("stats", oa["stats"], ob["stats"])):
        assert torch.equal(a, b), f"re-packed weights: {name} differs from a fresh pack of the final parameters"


# ---- 1. every update against float64 at the updater's own state (+ 3. the final re-pack) --------------------------------------


FORMS = {"simt": (L.GEMM_SIMT_FP32, False), "tc3xtf32": (L.GEMM_TC_3XTF32, False), "tc2xf16": (L.GEMM_TC_2XF16, False),
         "tc2xf16-per-step": (L.GEMM_TC_2XF16, True)}
UPDATE_CASES = [pytest.param(form, 6, 48, 128, 5, None, {}, False, id=form) for form in FORMS] + [
    # whole 128-row panels: the weight-gradient GEMMs read dG / x / h in place (dw_gemm_kernel); warm-up start carries
    pytest.param("tc2xf16", 9, 256, 256, 5, "warm", {}, False, id="tc2xf16-warm-T9xN256"),
    pytest.param("tc2xf16", 6, 48, 128, 4, None, {"clip_param": 0.1, "entropy_coef": 0.01, "use_clipped_value_loss": 0},
                 False, id="tc2xf16-loss-hyper"),
    # BASELINE configs[3], the benchmarked update: one eager update, then graph replays
    pytest.param("tc2xf16", 100, 512, 256, 3, None, {}, True, id="tc2xf16-configs3-graph"),
]


@pytest.mark.parametrize("form,T,N,H,updates,start,hyper,graph", UPDATE_CASES)
def test_ppo_update_against_float64_each_update(dev, form, T, N, H, updates, start, hyper, graph, monkeypatch):
    """Each update's gradient, norm and AdamW step from the state the updater had before it; minibatches alternate x1 / x8
    so both clip branches occur; hyper-parameters go through PpoUpdater(**loss_hyper); after the last update a fresh handle
    packed from the final parameters gives bitwise the same gradient as the updater's engine."""
    path, per_step = FORMS[form]
    monkeypatch.setenv("KBS_PPO_PER_STEP", "1" if per_step else "0")
    e, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H)
    carry0 = None
    if start == "warm":
        w = warm_start(wa, wc, N, H, 2, seed=9100 + N)
        carry0 = {k: w[k] for k in ("actor", "critic", "lpf_params")}
    seed = 9000 + 10 * T + N
    first = minibatch(seed + 1, T, N, p, wa, wc, carry0, 1.0, hyper)
    limit = clip_limit(wa, wc, first, minibatch(seed + 1, T, N, p, wa, wc, carry0, 8.0, hyper), p, carry0, hyper)
    up = PpoUpdater(e, wa, wc, max_grad_norm=limit, **hyper)
    gbatch = None
    clipped = []
    try:
        for k in range(1, updates + 1):
            snap = snapshot(up)
            b = first if k == 1 else minibatch(seed + k, T, N, p, *weights_at(up, snap["param"]), carry0,
                                               8.0 if k % 2 == 0 else 1.0, hyper)
            db = Hn.ppo_device_batch(b, dev, carry0)
            if gbatch is None:
                out = up.update(db, N)
                if graph:
                    torch.cuda.synchronize()
                    gbatch = {key: t.clone() for key, t in db.items()}
                    after = snapshot(up)
                    up.capture(gbatch, N)
                    assert_state_is(up, after, "capture")
            else:
                refill(gbatch, db)
                out = up.update(gbatch, N)
            clipped.append(check_update(up, snap, out, b, p, k, limit, carry0, hyper) > limit)
        assert any(clipped) and not all(clipped), ("both clip branches", clipped)
        assert_repacked(up, H, path, db, N)
    finally:
        e.close()


# ---- 2. graph replay against eager, bitwise ----------------------------------------------------------------------------------


def assert_bitwise(a: PpoUpdater, b: PpoUpdater, sa: torch.Tensor, sb: torch.Tensor, what: str):
    for k in ("param", "m", "v", "norm", "step_dev"):
        ta, tb = getattr(a, k), getattr(b, k)
        assert torch.equal(ta, tb), f"{what}: {k} differs ({int((ta != tb).sum())} entries)"
    assert torch.equal(sa, sb), f"{what}: loss stats differ {sa.tolist()} vs {sb.tolist()}"


@pytest.mark.parametrize("form", ["tc2xf16", "tc3xtf32"])
def test_ppo_update_graph_replay_matches_eager(dev, form, monkeypatch):
    """Two updaters from identical weights on the same minibatch sequence: two eager updates each (a whole update is
    bitwise reproducible), then one captures (capturing changes nothing) and replays on its batch refilled in place while
    the other runs eagerly -- param, m, v, norm, step counter and loss stats bitwise equal after every update, also after
    an eager update on another batch object between two replays.  The replaying side passes the per-update checks."""
    path, per_step = FORMS[form]
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, H = 9, 256, 256
    ea, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    eb, _, _ = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H)
    seed = 9500 + path
    first = minibatch(seed + 1, T, N, p, wa, wc)
    limit = clip_limit(wa, wc, first, minibatch(seed + 1, T, N, p, wa, wc, scale=8.0), p, None, {})
    ga, eg = PpoUpdater(ea, wa, wc, max_grad_norm=limit), PpoUpdater(eb, wa, wc, max_grad_norm=limit)
    gbatch = None
    clipped = []
    try:
        for k in range(1, 8):
            snap = snapshot(ga)
            b = first if k == 1 else minibatch(seed + k, T, N, p, *weights_at(ga, snap["param"]), scale=8.0 if k % 2 == 0 else 1.0)
            db = Hn.ppo_device_batch(b, dev)
            if k <= 2 or k == 5:        # eager on both sides (k = 5: between two replays, on another batch object)
                out = ga.update(db, N)
                sa = out["stats"].clone()
                mode = "eager"
            else:
                refill(gbatch, db)
                out = ga.update(gbatch, N)
                sa = out["stats"].clone()
                torch.cuda.synchronize()
                assert ga.eng.device_status() == 0
                mode = "replay"
            sb = eg.update(Hn.ppo_device_batch(b, dev), N)["stats"].clone()
            torch.cuda.synchronize()
            assert_bitwise(ga, eg, sa, sb, f"update {k} ({mode})")
            clipped.append(check_update(ga, snap, out, b, p, k, limit) > limit)
            if k == 2:
                gbatch = {key: t.clone() for key, t in db.items()}
                before = snapshot(ga)
                norm = ga.norm.clone()
                ga.capture(gbatch, N)
                torch.cuda.synchronize()
                assert_state_is(ga, before, "capture")
                assert torch.equal(ga.norm, norm), "capture changed the norm"
                assert ga.eng.device_status() == 0
        assert any(clipped) and not all(clipped), ("both clip branches", clipped)
        assert_repacked(ga, H, path, db, N)
    finally:
        ea.close()
        eb.close()


# ---- 4. a non-finite minibatch ------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("form", ["tc2xf16", "tc3xtf32"])
def test_ppo_update_non_finite_minibatch_is_skipped(dev, form, monkeypatch):
    """One NaN advantage, at a transition whose ratio is clipped, eager and replayed: param, m, v and the step counter stay
    bitwise unchanged and the norm is not finite (ksim's non-finite skip).  On the FP16-split datapath the NaN reaches an FP16-split operand: the health word has
    KBS_STATUS_F16_RANGE and, as include/kbotstep.h documents, the next kbs_ppo_grad fails with KBS_E_DEVICE (changing
    nothing) until kbs_device_status_reset; on 3xTF32 no bit is set.  After that the next finite minibatch passes the
    per-update checks, eager and replayed."""
    path, per_step = FORMS[form]
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, H = 6, 128, 256
    e, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H)
    seed = 9700 + path
    up = PpoUpdater(e, wa, wc)                # default clip 10: these minibatches stay below it
    limit = up.opt["max_grad_norm"]
    k = 0

    def good(db_target=None):
        nonlocal k
        k += 1
        snap = snapshot(up)
        b = minibatch(seed + k, T, N, p, *weights_at(up, snap["param"]))
        db = Hn.ppo_device_batch(b, dev)
        if db_target is not None:
            refill(db_target, db)
            db = db_target
        out = up.update(db, N)
        assert check_update(up, snap, out, b, p, k, limit) < limit
        return db

    def non_finite(db_target=None):
        snap = snapshot(up)
        w = weights_at(up, snap["param"])
        b = minibatch(seed + 100 + k, T, N, p, *w)
        # where the clipped term is the minimum: the policy term's derivative there does not otherwise involve the advantage
        r, a = np.exp(forward(*w, b, p)[0] - b["old_log_probs"]), b["advantages"]
        t, env = np.argwhere(np.clip(r, 0.8, 1.2) * a < r * a - 1e-3)[0]
        b["advantages"][t, env] = np.nan
        db = Hn.ppo_device_batch(b, dev)
        if db_target is not None:
            refill(db_target, db)
            db = db_target
        up.update(db, N)
        torch.cuda.synchronize()
        assert not np.isfinite(float(up.norm))
        assert_state_is(up, snap, "non-finite minibatch")
        status = e.device_status()            # also what a replay needs: the graph does not check the health word itself
        if path == L.GEMM_TC_2XF16:
            assert status & L.STATUS_F16_RANGE, hex(status)
            with pytest.raises(RuntimeError, match=r"\[-6\]"):
                up.update(Hn.ppo_device_batch(minibatch(seed + 200 + k, T, N, p, wa, wc), dev), N)
            torch.cuda.synchronize()
            assert_state_is(up, snap, "refused update")
            e.device_status_reset()
            assert e.device_status() == 0
        else:
            assert status == 0, hex(status)

    try:
        good()
        non_finite()
        db = good()
        gbatch = {key: t.clone() for key, t in db.items()}
        before = snapshot(up)
        up.capture(gbatch, N)
        assert_state_is(up, before, "capture")
        non_finite(gbatch)
        good(gbatch)
        good()
        non_finite(gbatch)
        good(gbatch)
    finally:
        e.close()


# ---- 5. two ranks over NCCL ---------------------------------------------------------------------------------------------------


_NCCL_WORKER = r"""
import os, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/oracle"); sys.path.insert(0, %(root)r + "/tests")
import numpy as np, torch, torch.distributed as dist
import harness as Hn, kbot_oracle as O, ppo_grad_torch as G
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200.ppo import PpoUpdater
from test_gpu_ppo_update import check_sharded_update, clip_limit, minibatch, refill, snapshot, weights_at
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
graph = sys.argv[1] == "graph"
dev = torch.device("cuda", rank)
torch.cuda.set_device(dev)
dist.init_process_group("nccl", device_id=dev)
T, N, H = 9, 256, 256
e, wa, wc = Hn.make_engine(hidden=H, gemm_path=L.GEMM_TC_2XF16, device=dev)
p = O.OracleParams(hidden_size=H)
first = minibatch(9901, T, N, p, wa, wc)
limit = clip_limit(wa, wc, first, minibatch(9901, T, N, p, wa, wc, scale=8.0), p, None, {})
up = PpoUpdater(e, wa, wc, max_grad_norm=limit)
sl = slice(rank * N // world, (rank + 1) * N // world)      # environments shard across ranks, weights replicated
gbatch, clipped = None, []
for k in range(1, 4):
    snap = snapshot(up)
    b = first if k == 1 else minibatch(9900 + k, T, N, p, *weights_at(up, snap["param"]), scale=8.0 if k %% 2 == 0 else 1.0)
    db = Hn.ppo_device_batch({key: v[:, sl] for key, v in b.items()}, dev)
    if gbatch is None:
        up.update(db, N // world)
        if graph:
            torch.cuda.synchronize()
            gbatch = {key: t.clone() for key, t in db.items()}
            up.capture(gbatch, N // world)
    else:
        refill(gbatch, db)
        up.update(gbatch, N // world)
    clipped.append(check_sharded_update(up, snap, b, p, k, limit, world) > limit)
    allp = [torch.empty_like(up.param) for _ in range(world)]
    dist.all_gather(allp, up.param)
    assert all(torch.equal(x, allp[0]) for x in allp), f"update {k}: the replicas' parameters differ"
assert any(clipped) and not all(clipped), clipped
e.close()
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def check_sharded_update(up: PpoUpdater, snap: dict, b: dict, p, k: int, limit: float, world: int) -> float:
    """Update k of a data-parallel updater holding 1 / world of minibatch b: the summed gradient / world against float64
    autograd on the WHOLE minibatch at the snapshot parameters, the norm of the sum, AdamW with grad_scale = 1 / world."""
    torch.cuda.synchronize()
    assert up.eng.device_status() == 0
    wa, wc = weights_at(up, snap["param"])
    ref = G.ppo_minibatch_grads(wa, wc, b, p)
    mean = up.grad / world
    bad = (Hn.compare_grads_blockwise(up.pa.as_dict(mean[:up.na]), ref[2], "actor", p.hidden_size, p.depth) +
           Hn.compare_grads_blockwise(up.pc.as_dict(mean[up.na:]), ref[3], "critic", p.hidden_size, p.depth))
    assert not bad, (f"update {k}", bad)
    g = up.grad.double().cpu().numpy()
    gn = float(np.sqrt(np.sum(g * g)))
    assert abs(float(up.norm) - gn) <= 2e-7 * gn, (f"update {k}: norm", float(up.norm), gn)
    opt = {key: up.opt[key] for key in ("lr", "b1", "b2", "eps", "weight_decay")}
    rp, rm, rv, applied = O.adamw_update(snap["param"].cpu().numpy(), g, snap["m"].cpu().numpy(), snap["v"].cpu().numpy(), k,
                                         grad_scale=1.0 / world, max_grad_norm=limit, **opt)
    assert applied and up.step_count == k
    close(up.param.cpu().numpy(), rp, f"update {k}: param", rtol=1e-6, atol=2e-7)
    close(up.m.cpu().numpy(), rm, f"update {k}: m", rtol=1e-5, atol=1e-9)
    close(up.v.cpu().numpy(), rv, f"update {k}: v", rtol=1e-5, atol=1e-12)
    rn = ref_norm(ref)
    assert abs(np.log(rn / limit)) > 0.05, ("the clip branch is ambiguous", rn, limit)
    return rn


@pytest.mark.parametrize("mode", ["eager", "graph"])
def test_ppo_update_two_ranks_nccl(dev, mode, tmp_path):
    """Two NCCL ranks on one minibatch, half of its trajectories each: the critic's slice is all-reduced on the updater's
    communication stream while the actor's weight-gradient GEMMs run (kbs_ppo_grad_set_events).  Three updates, eager or
    replayed as a graph: the summed gradient / 2 matches float64 autograd on the whole minibatch, the step matches AdamW
    with grad_scale = 1/2, and both ranks hold bitwise the same parameters."""
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
    procs = [subprocess.Popen([sys.executable, str(script), mode], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    try:
        outs = [p.communicate(timeout=600)[0] for p in procs]
    finally:
        for p in procs:                        # a rank stuck in a collective is killed, not left behind
            if p.poll() is None:
                p.kill()
                p.communicate()
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o}"
        assert f"rank {r} ok" in o
