"""kbs_ppo_variables_vjp: the vector-Jacobian product of the PPO variables (log-probs, values, entropy, action std) with
respect to both networks' weights, against float64 autograd of the same forward (tests/ppo_variables_ref.py),
on every datapath of kbs_ppo_grad; its scale invariance; and PpoUpdater.update / epoch with a caller's loss_fn.

The reference is sum(ct * var) differentiated by torch autograd in float64 from the same start carries, so any cotangents
can be checked: random ones of every size, subsets with NULL members, and the library's own PPO loss formed at the VJP's
forward outputs.  Gradients are compared block-wise (harness.compare_grads_blockwise); `pytest -s` prints the largest block
error over its bound per case (1 is the limit)."""

import math

import numpy as np
import pytest
import torch

import harness as Hn
import kbot_oracle as O
import ppo_grad_torch as G
from ppo_variables_ref import ppo_variables_torch
from harness import close
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200 import synth
from kbot_joystick_b200.ppo import PpoUpdater
from test_gpu_ppo_update import minibatch, snapshot, weights_at
from test_gpu_start_state import random_start

pytestmark = pytest.mark.gpu

S = synth.from_soa
VARS = ("log_probs", "values", "entropy", "action_std")
# kbs_ppo_grad's datapaths: the FP16 split runs the persistent kernels at depth <= 2 unless KBS_PPO_PER_STEP=1
FORMS = {"simt": (L.GEMM_SIMT_FP32, False), "tc3xtf32": (L.GEMM_TC_3XTF32, False), "tc2xf16": (L.GEMM_TC_2XF16, False),
         "tc2xf16-per-step": (L.GEMM_TC_2XF16, True)}


@pytest.fixture(scope="module")
def dev(cuda_device, lib_built):
    return cuda_device


# ---- helpers ---------------------------------------------------------------------------------------------------------------


def setup(dev, form, T, N, H, depth, start, monkeypatch, seed=0):
    path, per_step = FORMS[form]
    monkeypatch.setenv("KBS_PPO_PER_STEP", "1" if per_step else "0")
    e, wa, wc = Hn.make_engine(hidden=H, depth=depth, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H, depth=depth)
    carry0 = random_start(4000 + N + seed, N, depth, H) if start == "warm" else None
    rng = np.random.default_rng(700 + 10 * T + N + seed)
    b = Hn.ppo_batch(rng, T, N, H, p, wa, wc, carry0=carry0)
    return e, wa, wc, p, carry0, b


def random_cotangents(seed, T, N, which=VARS) -> dict:
    """numpy cotangents in the oracle layout ([T, N], action_std [T, N, 20]) of a summed loss (entries of order one)."""
    rng = np.random.default_rng(seed)
    sd = {"log_probs": 1.0, "values": 3.0, "entropy": 0.5, "action_std": 1.0}
    return {k: (sd[k] * rng.normal(size=(T, N, 20) if k == "action_std" else (T, N))).astype(np.float32) for k in which}


def ct_to_device(ct: dict, dev) -> dict:
    return {k: synth.to_soa(v, 1, dev) for k, v in ct.items()}


def nan_grads(w: dict, dev) -> dict:
    z = lambda a: torch.full(a.shape, float("nan"), device=dev)
    return {"w_in": z(w["w_in"]), "b_in": z(w["b_in"]), "w_out": z(w["w_out"]), "b_out": z(w["b_out"]),
            "layers": [{k: z(l[k]) for k in ("w_ih", "w_hh", "b")} for l in w["layers"]]}


def flat(g: dict) -> torch.Tensor:
    return torch.cat([t.reshape(-1) for _, _, t in grads_t(g)])


def grads_t(g: dict):
    for k in ("w_in", "b_in", "w_out", "b_out"):
        yield k, k, g[k]
    for l, lw in enumerate(g["layers"]):
        for k in ("w_ih", "w_hh", "b"):
            yield f"layers[{l}].{k}", k, lw[k]


def run_vjp(e, wa, wc, b, ct, dev, N, carry0=None, db=None):
    """kbs_ppo_variables_vjp on minibatch b with numpy cotangents ct -> (actor grads, critic grads, forward outputs)."""
    ga, gc = nan_grads(wa, dev), nan_grads(wc, dev)
    db = db if db is not None else Hn.ppo_device_batch(b, dev, carry0)
    out = e.ppo_variables_vjp(db, ct_to_device(ct, dev), ga, gc, n_envs=N)
    torch.cuda.synchronize()
    return ga, gc, out


def ref_vjp(wa, wc, b, p, carry0, loss_of):
    """float64 autograd: (actor grads, critic grads, variables) of loss_of(variables) through ppo_variables_torch."""
    ta, tc = G.weights_to_torch(wa), G.weights_to_torch(wc)
    v = ppo_variables_torch(ta, tc, b["actor_obs"], b["critic_obs"], b["action"], b["done"], p, carry0)
    leaves = lambda w: [w["w_in"], w["b_in"], w["w_out"], w["b_out"]] + [l[k] for l in w["layers"] for k in ("w_ih", "w_hh", "b")]
    la, lc = leaves(ta), leaves(tc)
    gs = torch.autograd.grad(loss_of(v), la + lc, allow_unused=True)

    def as_dict(gl, w):
        z = [(g if g is not None else torch.zeros_like(x)).numpy() for g, x in zip(gl, leaves(w))]
        return {"w_in": z[0], "b_in": z[1], "w_out": z[2], "b_out": z[3],
                "layers": [dict(zip(("w_ih", "w_hh", "b"), z[4 + 3 * l:7 + 3 * l])) for l in range(len(w["layers"]))]}

    return as_dict(gs[:len(la)], ta), as_dict(gs[len(la):], tc), {k: t.detach().numpy() for k, t in v.items()}


def dot_loss(ct: dict):
    """sum(ct * var) over the given cotangents (oracle layout)."""
    return lambda v: sum((torch.tensor(c, dtype=torch.float64) * v[k]).sum() for k, c in ct.items())


def check_against_ref(ga, gc, ref, p, what, ratios=None):
    ga_ref, gc_ref = ref[0], ref[1]
    bad = (Hn.compare_grads_blockwise(ga, ga_ref, "actor", p.hidden_size, p.depth) +
           Hn.compare_grads_blockwise(gc, gc_ref, "critic", p.hidden_size, p.depth))
    r = {**Hn.grad_block_ratios(ga, ga_ref, "actor", p.hidden_size, p.depth),
         **Hn.grad_block_ratios(gc, gc_ref, "critic", p.hidden_size, p.depth)}
    print(f"{what}: worst block error / bound {max(r.values()):.3f} ({max(r, key=r.get)})")
    if ratios is not None:
        ratios.update(r)
    assert not bad, (what, bad)


# ---- 1. against float64 autograd: datapaths, depths, start carries, shapes, subsets of the cotangents -----------------------

CASES = [  # T, N, H, depth, start
    pytest.param(5, 70, 256, 2, "warm", id="T5xN70-warm"),          # ragged n, done-resets mid-trajectory (~12% of steps)
    pytest.param(1, 64, 128, 2, "zero", id="T1xN64-H128"),
    pytest.param(6, 48, 256, 1, "warm", id="T6xN48-depth1"),
    pytest.param(4, 40, 256, 3, "warm", id="T4xN40-depth3"),        # depth 3 / 4: the per-step launches on every datapath
    pytest.param(3, 24, 256, 4, "zero", id="T3xN24-depth4"),
]


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("T,N,H,depth,start", CASES)
def test_vjp_against_float64(dev, form, T, N, H, depth, start, monkeypatch):
    e, wa, wc, p, carry0, b = setup(dev, form, T, N, H, depth, start, monkeypatch)
    try:
        ct = random_cotangents(11 + N, T, N)
        ga, gc, out = run_vjp(e, wa, wc, b, ct, dev, N, carry0)
        assert e.device_status() == 0
        ref = ref_vjp(wa, wc, b, p, carry0, dot_loss(ct))
        close(S(out["log_probs"], N), ref[2]["log_probs"], "log_probs", atol=1e-4)
        close(S(out["values"], N), ref[2]["values"], "values", atol=1e-5)
        close(S(out["entropy"], N), ref[2]["entropy"], "entropy", atol=1e-5)
        check_against_ref(ga, gc, ref, p, f"{form} T{T} N{N} H{H} depth {depth} {start}")
    finally:
        e.close()


SUBSETS = [("log_probs",), ("values", "action_std"), ("entropy",), ("log_probs", "entropy", "action_std")]


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("which", SUBSETS, ids=["+".join(s) for s in SUBSETS])
def test_vjp_cotangent_subsets(dev, form, which, monkeypatch):
    """NULL members are zero cotangents: a network none of whose variables has a cotangent gets exactly zero gradients."""
    T, N, H = 5, 48, 256
    e, wa, wc, p, carry0, b = setup(dev, form, T, N, H, 2, "warm", monkeypatch)
    try:
        ct = random_cotangents(23, T, N, which)
        ga, gc, _ = run_vjp(e, wa, wc, b, ct, dev, N, carry0)
        if "values" not in which:
            assert torch.count_nonzero(flat(gc)) == 0
        check_against_ref(ga, gc, ref_vjp(wa, wc, b, p, carry0, dot_loss(ct)), p, f"{form} {'+'.join(which)}")
    finally:
        e.close()


def test_vjp_against_float64_configs3(dev, monkeypatch):
    """BASELINE configs[3] (512 trajectories x 100 steps), FP16-split persistent, warm start."""
    e, wa, wc, p, carry0, b = setup(dev, "tc2xf16", 100, 512, 256, 2, "warm", monkeypatch)
    try:
        ct = random_cotangents(5, 100, 512)
        ga, gc, _ = run_vjp(e, wa, wc, b, ct, dev, 512, carry0)
        assert e.device_status() == 0
        check_against_ref(ga, gc, ref_vjp(wa, wc, b, p, carry0, dot_loss(ct)), p, "configs[3] tc2xf16")
    finally:
        e.close()


# ---- 2. the forward outputs are kbs_ppo_grad's -------------------------------------------------------------------------------


@pytest.mark.parametrize("form", list(FORMS))
def test_vjp_forward_is_ppo_grads(dev, form, monkeypatch):
    T, N = 7, 128
    e, wa, wc, p, carry0, b = setup(dev, form, T, N, 256, 2, "warm", monkeypatch)
    try:
        db = Hn.ppo_device_batch(b, dev, carry0)
        _, _, out = run_vjp(e, wa, wc, b, random_cotangents(3, T, N), dev, N, db=db)
        ref = e.ppo_grad(db, nan_grads(wa, dev), nan_grads(wc, dev), n_envs=N)
        torch.cuda.synchronize()
        for k in ("log_probs", "values", "entropy"):
            assert torch.equal(out[k][:, :N], ref[k][:, :N]), k
    finally:
        e.close()


# ---- 3. the library's own loss through the VJP -------------------------------------------------------------------------------


def ppo_loss(v: dict, b: dict, clip_param=0.2, value_loss_coef=0.5, entropy_coef=0.004, log_clip_value=10.0, mean=True):
    """ksim.compute_ppo_loss as kbs_ppo_loss restates it (clipped value loss), on tensors of any dtype and layout."""
    ratio = torch.exp(torch.clamp(v["log_probs"] - b["old_log_probs"], -log_clip_value, log_clip_value))
    adv = b["advantages"]
    pol = torch.minimum(ratio * adv, torch.clamp(ratio, 1 - clip_param, 1 + clip_param) * adv)
    err = b["value_targets"] - v["values"]
    errc = b["value_targets"] - (b["old_values"] + torch.clamp(v["values"] - b["old_values"], -clip_param, clip_param))
    vl = 0.5 * torch.maximum(err * err, errc * errc)
    obj = pol - value_loss_coef * vl + entropy_coef * v["entropy"]
    return -obj.mean() if mean else -obj.sum()


def np_batch64(b: dict) -> dict:
    return {k: torch.tensor(b[k], dtype=torch.float64) for k in ("old_log_probs", "advantages", "value_targets", "old_values")}


@pytest.mark.parametrize("form", list(FORMS))
def test_library_loss_through_vjp(dev, form, monkeypatch):
    """The cotangents of the library's PPO loss, formed in float64 at the VJP's own forward outputs and rounded to fp32, give
    gradients within the block bounds of kbs_ppo_grad's; both are within them of float64 autograd of the loss."""
    T, N, H = 6, 96, 256
    path, per_step = FORMS[form]
    monkeypatch.setenv("KBS_PPO_PER_STEP", "1" if per_step else "0")
    e, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H)
    carry0 = random_start(4321, N, 2, H)
    try:
        b = minibatch(77, T, N, p, wa, wc, carry0)          # kept off the loss' kinks
        db = Hn.ppo_device_batch(b, dev, carry0)
        _, _, fwd = run_vjp(e, wa, wc, b, {}, dev, N, db=db)
        v = {k: torch.tensor(S(fwd[k], N), dtype=torch.float64, requires_grad=True) for k in ("log_probs", "values", "entropy")}
        cts = torch.autograd.grad(ppo_loss(v, np_batch64(b)), [v[k] for k in v])
        ct = {k: c.numpy().astype(np.float32) for k, c in zip(v, cts)}
        ga, gc, _ = run_vjp(e, wa, wc, b, ct, dev, N, db=db)
        pa, pc = nan_grads(wa, dev), nan_grads(wc, dev)
        e.ppo_grad(db, pa, pc, n_envs=N)
        torch.cuda.synchronize()
        assert e.device_status() == 0
        check_against_ref(ga, gc, (pa, pc), p, f"{form} VJP of the loss vs kbs_ppo_grad")
        ref = G.ppo_minibatch_grads(wa, wc, b, p, carry0=carry0)
        check_against_ref(ga, gc, (ref[2], ref[3]), p, f"{form} VJP of the loss vs float64")
        check_against_ref(pa, pc, (ref[2], ref[3]), p, f"{form} kbs_ppo_grad vs float64")
    finally:
        e.close()


# ---- 4. / 5. scale invariance, and any cotangent magnitude on the FP16 split -----------------------------------------------


@pytest.mark.parametrize("form", list(FORMS))
def test_vjp_power_of_two_scaling_is_exact(dev, form, monkeypatch):
    """VJP(2^k ct) == 2^k VJP(ct) bitwise; scaling only the value cotangent leaves the actor's gradient bitwise unchanged."""
    T, N = 5, 64
    e, wa, wc, p, carry0, b = setup(dev, form, T, N, 256, 2, "warm", monkeypatch)
    try:
        db = Hn.ppo_device_batch(b, dev, carry0)
        ct = random_cotangents(31, T, N)
        ga, gc, _ = run_vjp(e, wa, wc, b, ct, dev, N, db=db)
        base = torch.cat([flat(ga), flat(gc)])
        assert torch.isfinite(base).all()
        for k in (-30, -10, 10, 30):
            s = np.float32(2.0 ** k)
            sa, sc, _ = run_vjp(e, wa, wc, b, {n: c * s for n, c in ct.items()}, dev, N, db=db)
            assert torch.equal(torch.cat([flat(sa), flat(sc)]), base * float(s)), k
        va, vc, _ = run_vjp(e, wa, wc, b, dict(ct, values=ct["values"] * np.float32(2.0 ** 20)), dev, N, db=db)
        assert torch.equal(flat(va), flat(ga))
        assert torch.equal(flat(vc), flat(gc) * 2.0 ** 20)
    finally:
        e.close()


@pytest.mark.parametrize("per_step", [False, True], ids=["persistent", "per-step"])
def test_vjp_fp16_split_any_magnitude(dev, per_step, monkeypatch):
    """Cotangents from 1e-8 to 1e6 stay within the block bounds on the FP16 split and never set KBS_STATUS_F16_RANGE."""
    T, N = 6, 128
    e, wa, wc, p, carry0, b = setup(dev, "tc2xf16-per-step" if per_step else "tc2xf16", T, N, 256, 2, "warm", monkeypatch)
    try:
        db = Hn.ppo_device_batch(b, dev, carry0)
        ct = random_cotangents(41, T, N)
        ga_ref, gc_ref, _ = ref_vjp(wa, wc, b, p, carry0, dot_loss(ct))
        scale_tree = lambda g, s: {"w_in": g["w_in"] * s, "b_in": g["b_in"] * s, "w_out": g["w_out"] * s, "b_out": g["b_out"] * s,
                                   "layers": [{k: l[k] * s for k in l} for l in g["layers"]]}
        for m in (-8, -5, -2, 0, 3, 6):
            s = 10.0 ** m
            ga, gc, _ = run_vjp(e, wa, wc, b, {k: (c.astype(np.float64) * s).astype(np.float32) for k, c in ct.items()}, dev, N,
                                db=db)
            assert e.device_status() == 0, m
            check_against_ref(ga, gc, (scale_tree(ga_ref, s), scale_tree(gc_ref, s)), p, f"x1e{m}")
    finally:
        e.close()


# ---- 6. zero and non-finite cotangents ---------------------------------------------------------------------------------------


@pytest.mark.parametrize("form", list(FORMS))
def test_vjp_zero_and_nan(dev, form, monkeypatch):
    T, N = 4, 48
    e, wa, wc, p, carry0, b = setup(dev, form, T, N, 256, 2, "warm", monkeypatch)
    try:
        db = Hn.ppo_device_batch(b, dev, carry0)
        ga, gc, _ = run_vjp(e, wa, wc, b, {}, dev, N, db=db)
        assert torch.count_nonzero(flat(ga)) == 0 and torch.count_nonzero(flat(gc)) == 0
        ct = random_cotangents(5, T, N)
        zeros = {k: np.zeros_like(c) for k, c in ct.items()}
        ga, gc, _ = run_vjp(e, wa, wc, b, zeros, dev, N, db=db)
        assert torch.count_nonzero(flat(ga)) == 0 and torch.count_nonzero(flat(gc)) == 0
        for k, net in (("log_probs", 0), ("entropy", 0), ("action_std", 0), ("values", 1)):
            bad = {n: c.copy() for n, c in ct.items()}
            bad[k][2, 5] = np.nan                   # step 2, env 5 (every joint of it for action_std)
            ga, gc, _ = run_vjp(e, wa, wc, b, bad, dev, N, db=db)
            hit, other = (flat(ga), flat(gc)) if net == 0 else (flat(gc), flat(ga))
            assert not torch.isfinite(hit).all(), k
            assert torch.isfinite(other).all(), k
            torch.cuda.synchronize()
            e.device_status_reset()             # the FP16 split flags the NaN it was handed
    finally:
        e.close()


# ---- 7. graph capture ---------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("form", list(FORMS))
def test_vjp_graph_replay_is_eager(dev, form, monkeypatch):
    T, N = 5, 128
    e, wa, wc, p, carry0, b = setup(dev, form, T, N, 256, 2, "warm", monkeypatch)
    try:
        db = Hn.ppo_device_batch(b, dev, carry0)
        ct = ct_to_device(random_cotangents(8, T, N), dev)
        ga, gc = nan_grads(wa, dev), nan_grads(wc, dev)
        eager = e.ppo_variables_vjp(db, ct, ga, gc, n_envs=N)
        torch.cuda.synchronize()
        ref = (flat(ga).clone(), flat(gc).clone(), {k: t.clone() for k, t in eager.items()})
        ga2, gc2 = nan_grads(wa, dev), nan_grads(wc, dev)
        e.scratch_lock(True)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = e.ppo_variables_vjp(db, ct, ga2, gc2, n_envs=N)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(flat(ga2), ref[0]) and torch.equal(flat(gc2), ref[1])
        for k in out:
            assert torch.equal(out[k][:, :N], ref[2][k][:, :N]), k
        # a replay reads the cotangents in place: doubling them doubles the gradients
        for t in ct.values():
            t.mul_(2.0)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(flat(ga2), 2 * ref[0]) and torch.equal(flat(gc2), 2 * ref[1])
        e.scratch_lock(False)
    finally:
        e.close()


def test_vjp_critic_ready_event(dev, monkeypatch):
    """With critic_ready set, the event is recorded once the critic's gradients (rescaled) are final."""
    T, N = 5, 128
    e, wa, wc, p, carry0, b = setup(dev, "tc2xf16", T, N, 256, 2, "warm", monkeypatch)
    try:
        db = Hn.ppo_device_batch(b, dev, carry0)
        ct = random_cotangents(9, T, N)
        ga, gc, _ = run_vjp(e, wa, wc, b, ct, dev, N, db=db)
        ev = torch.cuda.Event()
        ev.record()
        ga2, gc2 = nan_grads(wa, dev), nan_grads(wc, dev)
        side = torch.cuda.Stream()
        copy = torch.empty_like(flat(gc))
        e.ppo_variables_vjp(db, ct_to_device(ct, dev), ga2, gc2, n_envs=N, critic_ready=ev)
        with torch.cuda.stream(side):
            side.wait_event(ev)
            copy.copy_(flat(gc2))
        torch.cuda.synchronize()
        assert torch.equal(copy, flat(gc))
        e.ppo_variables_vjp(db, ct_to_device(ct, dev), ga2, gc2, n_envs=N)   # clears the event
    finally:
        e.close()


# ---- 8. validation -------------------------------------------------------------------------------------------------------------


def test_vjp_return_codes(dev):
    """KBS_E_NULL for a missing handle, batch, cotangent struct, gradient struct, output or required batch array; KBS_E_SHAPE
    for T or n <= 0, ld < n and ld % 4 != 0; KBS_E_STATE for a handle without packed weights.  The loss' inputs of the batch
    are not read, and a cotangent struct of NULLs is valid."""
    import ctypes as C

    from kbot_joystick_b200.engine import KbotStep, _net_grads, _ppo_batch

    E_NULL, E_SHAPE, E_STATE = -1, -2, -4
    T, N, H = 2, 8, 128
    e, wa, wc = Hn.make_engine(hidden=H, gemm_path=L.GEMM_SIMT_FP32, device=dev)
    fresh = KbotStep(hidden_size=H, depth=2, gemm_path=L.GEMM_SIMT_FP32)
    try:
        b = Hn.ppo_batch(np.random.default_rng(1), T, N, H, O.OracleParams(hidden_size=H), wa, wc)
        db = Hn.ppo_device_batch(b, dev)
        for k in ("old_log_probs", "advantages", "value_targets", "old_values"):
            db.pop(k)
        bs, cs = _ppo_batch(db), L.KbsPpoCotangents()
        sa, sc = _net_grads(nan_grads(wa, dev)), _net_grads(nan_grads(wc, dev))
        out = [L.ptr(torch.empty((T, N), device=dev)) for _ in range(3)]

        def call(h=e._h, bp=C.byref(bs), cp=C.byref(cs), ga=C.byref(sa), gc=C.byref(sc), o=out, n=N):
            return e.lib.kbs_ppo_variables_vjp(h, bp, cp, ga, gc, o[0], o[1], o[2], n, None)

        assert call() == 0
        torch.cuda.synchronize()
        for kw in ({"h": None}, {"bp": None}, {"cp": None}, {"ga": None}, {"gc": None}, {"o": [None] + out[1:]},
                   {"o": out[:1] + [None] + out[2:]}, {"o": out[:2] + [None]}):
            assert call(**kw) == E_NULL, kw
        for field in ("actor_obs", "critic_obs", "action", "done"):
            saved = getattr(bs, field)
            setattr(bs, field, None)
            assert call() == E_NULL, field
            setattr(bs, field, saved)
        assert call(n=0) == E_SHAPE
        assert call(n=N + 4) == E_SHAPE                        # ld < n
        for field, bad in (("T", 0), ("ld", N + 2)):           # ld % 4 != 0
            saved = getattr(bs, field)
            setattr(bs, field, bad)
            assert call() == E_SHAPE, field
            setattr(bs, field, saved)
        assert call(h=fresh._h) == E_STATE                     # no packed weights
        assert call() == 0
        torch.cuda.synchronize()
    finally:
        fresh.close()
        e.close()


# ---- 9. PpoUpdater with a caller's loss ----------------------------------------------------------------------------------------


def fp32_lib_loss(v, b):
    return ppo_loss(v, b)


BETA = 0.05


def kl_sum_loss(v, b):
    """A different objective: the library's loss summed instead of averaged, a squared log-ratio penalty and a term on the
    action std."""
    lr = v["log_probs"] - b["old_log_probs"]
    return ppo_loss(v, b, mean=False) + BETA * (lr * lr).sum() + 1e-3 * (v["action_std"] ** 2).sum()


def check_loss_update(up, snap, b, p, k, carry0, loss_fn, limit):
    """Update k from state snap: the gradient against float64 autograd of loss_fn, the norm, and AdamW from snap."""
    torch.cuda.synchronize()
    assert up.eng.device_status() == 0
    na = up.na
    wa, wc = weights_at(up, snap["param"])
    b64 = np_batch64(b)
    ga_ref, gc_ref, _ = ref_vjp(wa, wc, b, p, carry0, lambda v: loss_fn(v, b64))
    check_against_ref(up.pa.as_dict(up.grad[:na]), up.pc.as_dict(up.grad[na:]), (ga_ref, gc_ref), p, f"update {k}")
    g = up.grad.double().cpu().numpy()
    gn = float(np.sqrt(np.sum(g * g)))
    assert abs(float(up.norm) - gn) <= 2e-7 * gn
    opt = {key: up.opt[key] for key in ("lr", "b1", "b2", "eps", "weight_decay")}
    rp, rm, rv, applied = O.adamw_update(snap["param"].cpu().numpy(), g, snap["m"].cpu().numpy(), snap["v"].cpu().numpy(), k,
                                         grad_scale=1.0, max_grad_norm=limit, **opt)
    assert applied
    close(up.param.cpu().numpy(), rp, f"update {k}: param", rtol=1e-6, atol=2e-7)
    close(up.m.cpu().numpy(), rm, f"update {k}: m", rtol=1e-5, atol=1e-9)
    close(up.v.cpu().numpy(), rv, f"update {k}: v", rtol=1e-5, atol=1e-12)
    assert up.step_count == k


LOSSES = {"library-loss-fp32": (fp32_lib_loss, 10.0), "kl-sum": (kl_sum_loss, 1e9)}


@pytest.mark.parametrize("form", ["simt", "tc2xf16", "tc2xf16-per-step"])
@pytest.mark.parametrize("loss", list(LOSSES))
def test_update_with_loss_fn_against_float64(dev, form, loss, monkeypatch):
    """update(loss_fn=...) update by update against float64 autograd of the same loss at the updater's own state; the
    minibatches are kept off the loss' kinks, so the two forwards (kbs_ppo_variables for the loss, the VJP's for the
    gradient) cannot fall on different sides of one."""
    T, N, H = 6, 48, 128
    path, per_step = FORMS[form]
    monkeypatch.setenv("KBS_PPO_PER_STEP", "1" if per_step else "0")
    loss_fn, limit = LOSSES[loss]
    e, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    p = O.OracleParams(hidden_size=H)
    carry0 = random_start(555, N, 2, H)
    up = PpoUpdater(e, wa, wc, max_grad_norm=limit)
    try:
        for k in range(1, 4):
            snap = snapshot(up)
            b = minibatch(900 + k, T, N, p, *weights_at(up, snap["param"]), carry0)
            out = up.update(Hn.ppo_device_batch(b, dev, carry0), N, loss_fn=loss_fn)
            assert torch.isfinite(out["stats"][0])
            check_loss_update(up, snap, b, p, k, carry0, loss_fn, limit)
    finally:
        e.close()


@pytest.mark.parametrize("form", ["tc2xf16", "tc3xtf32"])
def test_update_with_loss_fn_graph_replay_is_eager(dev, form, monkeypatch):
    T, N, H = 6, 128, 256
    path, per_step = FORMS[form]
    monkeypatch.setenv("KBS_PPO_PER_STEP", "1" if per_step else "0")
    p = O.OracleParams(hidden_size=H)
    ups = []
    for _ in range(2):
        e, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
        ups.append(PpoUpdater(e, wa, wc))
    a, c = ups
    try:
        batches = [Hn.ppo_device_batch(minibatch(300 + k, T, N, p, wa, wc), dev) for k in range(4)]
        for up in ups:
            up.update(batches[0], N, loss_fn=kl_sum_loss)
        gbatch = {k: t.clone() for k, t in batches[1].items()}
        a.update(gbatch, N, loss_fn=kl_sum_loss)
        c.update(batches[1], N, loss_fn=kl_sum_loss)
        a.capture(gbatch, N, loss_fn=kl_sum_loss)
        for k in (2, 3):
            for key in gbatch:
                gbatch[key].copy_(batches[k][key])
            sa = a.update(gbatch, N, loss_fn=kl_sum_loss)["stats"].clone()
            sc = c.update(batches[k], N, loss_fn=kl_sum_loss)["stats"].clone()
            torch.cuda.synchronize()
            for key in ("param", "m", "v", "norm", "step_dev"):
                assert torch.equal(getattr(a, key), getattr(c, key)), (k, key)
            assert torch.equal(sa[:1], sc[:1])
    finally:
        for up in ups:
            up.eng.close()


def test_update_with_loss_fn_non_finite_is_skipped(dev):
    T, N, H = 4, 48, 128
    e, wa, wc = Hn.make_engine(hidden=H, gemm_path=L.GEMM_TC_2XF16, device=dev)
    p = O.OracleParams(hidden_size=H)
    up = PpoUpdater(e, wa, wc)
    try:
        b = minibatch(12, T, N, p, wa, wc)
        b["advantages"][2, 5] = np.nan
        snap = snapshot(up)
        up.update(Hn.ppo_device_batch(b, dev), N, loss_fn=fp32_lib_loss)
        torch.cuda.synchronize()
        assert not math.isfinite(float(up.norm))
        for k in ("param", "m", "v"):
            assert torch.equal(getattr(up, k), snap[k]), k
        assert up.step_count == 0
        e.device_status_reset()
    finally:
        e.close()


@pytest.mark.parametrize("form", ["tc2xf16", "tc3xtf32"])
def test_epoch_with_loss_fn_is_the_composition(dev, form, monkeypatch):
    """epoch(loss_fn=...) is bitwise the epoch built by hand from kbs_ppo_variables, kbs_gae, the permutation law, torch
    indexing and update(loss_fn=...): parameters, moments, counters, norms and losses after warm-start carries and done
    resets."""
    from test_gpu_ppo_epoch import make_rollout
    from test_gpu_start_state import warm_start
    from test_ppo_epoch_cpu import permutation

    path, _ = FORMS[form]
    monkeypatch.setenv("KBS_PPO_PER_STEP", "0")
    T, N, H, bs, passes, seed = 9, 256, 256, 128, 2, 2024
    ea, wa, wc = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    eb, _, _ = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    try:
        ro = make_rollout(T, N, dev, seed=61, carry0=warm_start(wa, wc, N, H, 2, seed=9300))
        assert int(ro["done"][:, :N].sum()) > 0
        up, ref = PpoUpdater(ea, wa, wc), PpoUpdater(eb, wa, wc)
        out = up.epoch(ro, N, batch_size=bs, num_passes=passes, seed=seed, loss_fn=kl_sum_loss)
        ac, cc, lpf = ro["actor_carry0"].clone(), ro["critic_carry0"].clone(), ro["lpf0"].clone()
        v = eb.ppo_variables(ro["actor_obs"], ro["action"], ro["done"], ac, lpf, ro["critic_obs"], cc, want_std=False, n_envs=N)
        adv, tgt = eb.gae(v["values"], ro["rewards"], ro["done"], ro["success"], n_envs=N)
        full = {"actor_obs": ro["actor_obs"], "critic_obs": ro["critic_obs"], "action": ro["action"], "done": ro["done"],
                "old_log_probs": v["log_probs"], "advantages": adv, "value_targets": tgt, "old_values": v["values"],
                "actor_carry0": ro["actor_carry0"], "critic_carry0": ro["critic_carry0"], "lpf0": ro["lpf0"]}
        losses, norms = [], []
        for p in range(passes):
            perm = permutation(seed, p, 0, N)
            for b in range(N // bs):
                idx = torch.from_numpy(perm[b * bs:(b + 1) * bs].astype(np.int64)).to(dev)
                batch = {k: (t[:, :, idx] if k.endswith("carry0") else t[..., idx]).contiguous() for k, t in full.items()}
                losses.append(ref.update(batch, bs, loss_fn=kl_sum_loss)["stats"][0].clone())
                norms.append(ref.norm.clone())
        torch.cuda.synchronize()
        assert ea.device_status() == 0 and eb.device_status() == 0
        for k in ("param", "m", "v", "step_dev", "norm"):
            assert torch.equal(getattr(up, k), getattr(ref, k)), k
        assert torch.equal(out["norms"], torch.cat(norms)) and torch.isfinite(out["norms"]).all()
        assert torch.equal(out["stats"][:, 0], torch.stack(losses))
        assert int(up.step_dev.item()) == passes * N // bs
    finally:
        ea.close()
        eb.close()
