"""The FP16-split datapath below fp16's normal range, and the PPO gradient at the loss scales training reaches.

The FP16 split writes an operand element x as hi + lo / 2^11 with both planes in fp16.  fp16's normal range ends at 2^-14;
below it hi must still be exactly an fp16 value (a multiple of 2^-24), or the rounding of its fp16 conversion, up to 2^-25,
is in neither plane.  The PPO gradient's dG is pre-scaled by a power of two chosen from T n only, so it reaches that range
whenever the loss is small: small advantages, or the small value residuals (target - value) of a critic that has learned.
AdamW is scale-invariant, so the gradient's relative error is the update's error however small the gradient is.

1. The split probe: one LSTM layer's gates (kbs_debug_tc_gates) on operands whose rows sit near 2^-8 ... 2^-30, against
   float64, per element within c1 sum|x||w| + c2 sum|w| (c1 the relative accuracy test_gpu_tc holds O(1) data to, c2 the
   floor of the exact split); 3xTF32 (no such range) is the control.
2. kbs_ppo_grad on every datapath with the advantages or the value residuals scaled by 1 ... 1e-3, against float64 autograd
   at the bounds every other gradient test uses (harness.compare_grads_blockwise); below x1, of the residuals the library's
   own forward values give (run_scaled says why).
3. Scales 1e1 ... 1e4: the gradient is within those bounds, or the health word says KBS_STATUS_F16_RANGE (an FP16-split
   operand reached 65504).  A non-finite or wrong gradient with a clean health word fails.

`pytest -s` prints the probe's worst ratio per exponent and every case's block error / bound per layer."""

import functools

import numpy as np
import pytest
import torch

import harness as Hn
from harness import close
import kbot_oracle as O
import ppo_grad_torch as G
from kbot_joystick_b200 import _lib as L
from kbot_joystick_b200 import synth
from kbot_joystick_b200.engine import KbotStep
from test_gpu_ppo_update import minibatch
from test_gpu_start_state import weights
from test_gpu_tc import _gates as gates

pytestmark = pytest.mark.gpu

SIMT, TF32, F16 = L.GEMM_SIMT_FP32, L.GEMM_TC_3XTF32, L.GEMM_TC_2XF16


@pytest.fixture(scope="module")
def dev(cuda_device, lib_built):
    return cuda_device


# ---- 1. the split probe ----------------------------------------------------------------------------------------------------

C1 = 2.0 ** -20      # test_gpu_tc: max error < 8e-6 where sum|x||w| ~ 9 .. 13 (H = 256, O(1) data)
C2 = 4 * 2.0 ** -35  # the exact split: each element within 2^-36 below 2^-14, x4 for the dropped lo.lo and the accumulation
EXPONENTS = np.arange(8, 31)


def probe_engine(path: int, H: int, dev, rng):
    """Actor layer 0 with w_ih, w_hh ~ U(-1, 1) and a zero bias: the gates are the bare products."""
    wa, wc = weights(H, 2)
    lw = wa["layers"][0]
    lw["w_ih"] = rng.uniform(-1, 1, lw["w_ih"].shape).astype(np.float32)
    lw["w_hh"] = rng.uniform(-1, 1, lw["w_hh"].shape).astype(np.float32)
    lw["b"] = np.zeros_like(lw["b"])
    e = KbotStep(hidden_size=H, depth=2, gemm_path=path)
    e.pack_weights(L.NET_ACTOR, synth.weights_to_device(wa, dev))
    e.pack_weights(L.NET_CRITIC, synth.weights_to_device(wc, dev))
    return e, lw


@pytest.mark.parametrize("operand", ["x", "h"])
@pytest.mark.parametrize("path", [pytest.param(TF32, id="tc3xtf32"), pytest.param(F16, id="tc2xf16")])
def test_split_probe_small_magnitudes(dev, path, operand):
    """n = 130 rows, row r with elements of magnitude 2^-e * U[1, 2), e = 8 + r mod 23 (down to 2^-30), random signs, the
    other operand zero (operand "h" swaps them: the recurrent half).  Every gate within C1 sum|x||w| + C2 sum over the
    non-zero elements of |w| of the float64 product.  A split whose hi is rounded to 11 bits before its fp16 conversion
    misses this 37-60x for 2^-26 <= |x| < 2^-14 (B200)."""
    H, n = 256, 130
    rng = np.random.default_rng(14)
    e, lw = probe_engine(path, H, dev, rng)
    try:
        ex = EXPONENTS[np.arange(n) % len(EXPONENTS)]
        v = (np.ldexp(rng.uniform(1, 2, (n, H)), -ex[:, None]) * rng.choice([-1.0, 1.0], (n, H))).astype(np.float32)
        z = np.zeros_like(v)
        x, h = (v, z) if operand == "x" else (z, v)
        g = gates(e, L.NET_ACTOR, 0, x, h, dev)
    finally:
        e.close()
    f = np.float64
    wi, wh = np.abs(lw["w_ih"].astype(f)), np.abs(lw["w_hh"].astype(f))
    ref = x.astype(f) @ lw["w_ih"].astype(f).T + h.astype(f) @ lw["w_hh"].astype(f).T
    bound = C1 * (np.abs(x.astype(f)) @ wi.T + np.abs(h.astype(f)) @ wh.T) + C2 * ((x != 0) @ wi.T + (h != 0) @ wh.T)
    ratio = np.abs(g - ref) / bound
    worst = {int(k): float(ratio[ex == k].max()) for k in EXPONENTS}
    print(f"\n[f16-range] split probe {'tc2xf16' if path == F16 else 'tc3xtf32'} operand {operand}: error / bound per "
          f"exponent e of 2^-e: " + ", ".join(f"{k}: {r:.3g}" for k, r in worst.items()))
    assert np.isfinite(g).all()
    bad = {k: r for k, r in worst.items() if not r <= 1.0}
    assert not bad, f"rows beyond c1 sum|x||w| + c2 sum|w| (exponent: error / bound): {bad}"


# ---- 2. / 3. the PPO gradient across loss scales -----------------------------------------------------------------------------

FORMS = {"tc2xf16": (F16, False), "tc2xf16-per-step": (F16, True), "tc3xtf32": (TF32, False), "simt": (SIMT, False)}
# (T, n, H): a ragged n, whole 128-row panels (the weight-gradient GEMMs read dG in place), H = 128, a long multi-panel case
SHAPES = [(7, 70, 256), (9, 256, 256), (6, 130, 128), (33, 300, 256)]
SMALL = [1.0, 1e-1, 1e-2, 1e-3]
LARGE = [1e1, 1e2, 1e3, 1e4]


def scale_cases(scales, skip_unit=False):
    # the four datapaths innermost, so that consecutive cases share one cached minibatch and reference
    out = []
    for T, N, H in SHAPES:
        for which in ("adv", "res"):
            for s in scales:
                if skip_unit and which == "res" and s == 1.0:
                    continue        # the same minibatch as adv x1
                for form in FORMS:
                    out.append(pytest.param(form, T, N, H, which, s, id=f"{form}-T{T}xN{N}xH{H}-{which}{s:g}"))
    return out


@functools.lru_cache(maxsize=1)
def scaled_case(T: int, N: int, H: int, s_adv: float, s_res: float) -> tuple:
    """test_gpu_ppo_update.minibatch with the value residuals at s_res x N(0, 0.5) around the current value (old values
    likewise), the advantages x s_adv; and its float64 reference."""
    wa, wc = weights(H, 2)
    p = O.OracleParams(hidden_size=H)
    b = minibatch(7000 + T + N + H, T, N, p, wa, wc, residual_scale=s_res)
    b["advantages"] = (b["advantages"] * s_adv).astype(np.float32)
    return wa, wc, p, b, G.ppo_minibatch_grads(wa, wc, b, p)


def nan_grads(w: dict, dev) -> dict:
    z = lambda a: torch.full(a.shape, float("nan"), device=dev)
    return {"w_in": z(w["w_in"]), "b_in": z(w["b_in"]), "w_out": z(w["w_out"]), "b_out": z(w["b_out"]),
            "layers": [{k: z(l[k]) for k in ("w_ih", "w_hh", "b")} for l in w["layers"]]}


def run_scaled(dev, form, T, N, H, which, s, monkeypatch, range_ok):
    """kbs_ppo_grad on scaled_case against its float64 reference (as harness.ppo_grad_compare, with the loss statistics'
    absolute floor scaled with the advantages).  Value residuals below x1 are compared with the float64 gradient of the
    library's own residuals (target - its fp32 value): a residual of 5e-4 is only ~500x the ~1e-6 error of the forward's
    values (checked to 1e-5 here), which the gradient inherits whatever the backward does -- 3xTF32 measured 3x beyond
    its bound at x1e-3 against the plain reference.  This isolates the backward pass, where the FP16 split acts."""
    path, per_step = FORMS[form]
    monkeypatch.setenv("KBS_PPO_PER_STEP", "1" if per_step else "0")
    s_adv, s_res = (s, 1.0) if which == "adv" else (1.0, s)
    wa, wc, p, b, (loss, stats, ga_ref, gc_ref, lp_ref, val_ref) = scaled_case(T, N, H, s_adv, s_res)
    e, _, _ = Hn.make_engine(hidden=H, gemm_path=path, device=dev)
    ga, gc = nan_grads(wa, dev), nan_grads(wc, dev)
    try:
        e.profile(True)
        out = e.ppo_grad(Hn.ppo_device_batch(b, dev), ga, gc, n_envs=N)
        torch.cuda.synchronize()
        status = e.device_status()
        persistent = e.profile_read().get("bptt_persist_kernel", (0, 0))[1]
    finally:
        e.close()
    assert (persistent > 0) == (path == F16 and not per_step), persistent
    what = f"ppo_grad {form} T{T}xN{N}xH{H} {'advantages' if which == 'adv' else 'value residuals'} x{s:g}"
    if range_ok and status == L.STATUS_F16_RANGE:
        print(f"\n[f16-range] {what}: KBS_STATUS_F16_RANGE")
        return
    assert status == 0, hex(status)
    values = synth.from_soa(out["values"], N)
    close(synth.from_soa(out["log_probs"], N), lp_ref, "log_probs", atol=1e-4)
    close(values, val_ref, "values", atol=1e-5)
    # the mean policy term averages ratio x advantage over advantages of both signs: its rounding grows with them
    close(out["stats"].cpu().numpy(), np.array((loss,) + stats, np.float32), "loss stats", rtol=2e-5, atol=1e-5 * max(1.0, s_adv))
    if s_res < 1.0:
        assert np.abs(val_ref - b["old_values"]).max() < 0.2 - 1e-3, "a value change reaches the clip"
        own = dict(b, value_targets=b["value_targets"] + (val_ref - values.astype(np.float64)))
        ga_ref, gc_ref = G.ppo_minibatch_grads(wa, wc, own, p)[2:4]
    bad = Hn.compare_grads_blockwise(ga, ga_ref, "actor", H, 2) + Hn.compare_grads_blockwise(gc, gc_ref, "critic", H, 2)
    ratios = {**Hn.grad_block_ratios(ga, ga_ref, "actor", H, 2), **Hn.grad_block_ratios(gc, gc_ref, "critic", H, 2)}
    layer = lambda net, l: max(v for k, v in ratios.items() if k.startswith(f"{net}.layers[{l}]."))
    other = max(v for k, v in ratios.items() if ".layers[" not in k)
    print(f"\n[f16-range] {what}: block error / bound per layer: actor {[round(layer('actor', l), 3) for l in range(2)]} "
          f"critic {[round(layer('critic', l), 3) for l in range(2)]}; projections / heads {other:.3f}")
    assert not bad, bad


@pytest.mark.parametrize("form,T,N,H,which,s", scale_cases(SMALL, skip_unit=True))
def test_ppo_grad_small_loss_scales(dev, form, T, N, H, which, s, monkeypatch):
    """kbs_ppo_grad with the advantages or the value residuals x1 ... x1e-3 against float64 autograd (run_scaled): log-probs,
    values, loss statistics and every gradient block within harness.block_bound, on FP16-split (persistent and per-step),
    3xTF32 and SIMT."""
    run_scaled(dev, form, T, N, H, which, s, monkeypatch, range_ok=False)


@pytest.mark.parametrize("form,T,N,H,which,s", scale_cases(LARGE))
def test_ppo_grad_large_loss_scales(dev, form, T, N, H, which, s, monkeypatch):
    """The same x1e1 ... x1e4: within the bounds, or (FP16-split only) the health word is exactly KBS_STATUS_F16_RANGE."""
    run_scaled(dev, form, T, N, H, which, s, monkeypatch, range_ok=FORMS[form][0] == F16)
