"""kbs_ppo_variables_vjp against kbs_ppo_grad, and PpoUpdater.update(loss_fn) against update(), at BASELINE configs[3]
(512 trajectories x 100 steps, H 256, depth 2), FP16-split datapath, each replayed as a CUDA graph.

Timing: CUDA events around `--reps` back-to-back replays; `--rounds` rounds alternate the two sides of each pair, and the
median and range over the rounds are reported.  The VJP's cotangents are those of the library's PPO loss (so the two
calls back-propagate the same thing).  A separate torch.profiler pass gives the device time of the kernels the VJP adds
(ct_absmax_kernel, grad_rescale_kernel).  The card's name and power limit are read in the same run.  Prints one JSON line,
also written to --out."""
import argparse, json, statistics, subprocess, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch
import kbot_joystick_b200  # noqa: F401
from kbot_joystick_b200 import _lib as L, synth
from kbot_joystick_b200.engine import KbotStep
from kbot_joystick_b200.ppo import PpoUpdater

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=512)
ap.add_argument("--T", type=int, default=100)
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--rounds", type=int, default=7)
ap.add_argument("--out", type=str, default=None)
a = ap.parse_args()
dev = torch.device("cuda", 0)
N, T, H = a.envs, a.T, 256
wa, wc = synth.make_weights(77, 65, 40, H, 2), synth.make_weights(78, 475, 1, H, 2)
g = torch.Generator(device=dev).manual_seed(100)
rn = lambda *s, sc=1.0: torch.randn(s, generator=g, device=dev) * sc


def make_batch(eng):
    """A minibatch whose stored actions are samples of the policy and whose old log-probs / values are the current ones
    plus noise (ratios near 1, as in training)."""
    b = {"actor_obs": rn(T, 65, N, sc=0.7), "critic_obs": rn(T, 475, N, sc=0.7), "action": rn(T, 20, N, sc=0.3),
         "done": (torch.rand((T, N), generator=g, device=dev) < 0.01).to(torch.uint8), "actor_carry0": rn(2, 2, N, H, sc=0.3),
         "critic_carry0": rn(2, 2, N, H, sc=0.3), "lpf0": rn(20, N, sc=0.2)}
    pv = eng.ppo_variables(b["actor_obs"], b["action"], b["done"], b["actor_carry0"].clone(), b["lpf0"].clone(), b["critic_obs"],
                           b["critic_carry0"].clone(), want_std=True, want_mean=True, n_envs=N)
    b["action"] = pv["mean"] + pv["action_std"] * rn(T, 20, N)
    pv = eng.ppo_variables(b["actor_obs"], b["action"], b["done"], b["actor_carry0"].clone(), b["lpf0"].clone(), b["critic_obs"],
                           b["critic_carry0"].clone(), n_envs=N)
    b.update(old_log_probs=pv["log_probs"] + rn(T, N, sc=0.05), advantages=rn(T, N), value_targets=pv["values"] + rn(T, N, sc=0.3),
             old_values=pv["values"] + rn(T, N, sc=0.1))
    return b


def ppo_loss(v, b, clip_param=0.2, value_loss_coef=0.5, entropy_coef=0.004, log_clip_value=10.0):
    ratio = torch.exp(torch.clamp(v["log_probs"] - b["old_log_probs"], -log_clip_value, log_clip_value))
    adv = b["advantages"]
    pol = torch.minimum(ratio * adv, torch.clamp(ratio, 1 - clip_param, 1 + clip_param) * adv)
    err = b["value_targets"] - v["values"]
    errc = b["value_targets"] - (b["old_values"] + torch.clamp(v["values"] - b["old_values"], -clip_param, clip_param))
    obj = pol - value_loss_coef * 0.5 * torch.maximum(err * err, errc * errc) + entropy_coef * v["entropy"]
    return -obj.mean()


def replay_ms(graph, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def capture(fn):
    fn()                                   # eager first: scratch and allocations
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fn()
    graph.replay()
    torch.cuda.synchronize()
    return graph


def alternate(ga, gb):
    ra, rb = [], []
    for _ in range(a.rounds):
        ra.append(replay_ms(ga, a.reps))
        rb.append(replay_ms(gb, a.reps))
    stat = lambda r: {"median_ms": statistics.median(r), "min_ms": min(r), "max_ms": max(r)}
    return stat(ra), stat(rb)


# 1. kbs_ppo_grad against kbs_ppo_variables_vjp on one handle and one minibatch
eng = KbotStep(hidden_size=H, depth=2, gemm_path=L.GEMM_TC_2XF16)
eng.pack_weights(L.NET_ACTOR, synth.weights_to_device(wa, dev))
eng.pack_weights(L.NET_CRITIC, synth.weights_to_device(wc, dev))
batch = make_batch(eng)
zeros = lambda w: {"w_in": torch.zeros(w["w_in"].shape, device=dev), "b_in": torch.zeros(w["b_in"].shape, device=dev),
                   "w_out": torch.zeros(w["w_out"].shape, device=dev), "b_out": torch.zeros(w["b_out"].shape, device=dev),
                   "layers": [{k: torch.zeros(l[k].shape, device=dev) for k in l} for l in w["layers"]]}
ga, gc, va, vc = zeros(wa), zeros(wc), zeros(wa), zeros(wc)
fwd = eng.ppo_grad(batch, ga, gc, n_envs=N)
var = {k: fwd[k].detach().clone().requires_grad_(True) for k in ("log_probs", "values", "entropy")}
cts = dict(zip(var, torch.autograd.grad(ppo_loss(var, batch), list(var.values()))))
g_grad = capture(lambda: eng.ppo_grad(batch, ga, gc, n_envs=N))
eng.scratch_lock(True)                     # g_grad holds pointers into the scratch: the VJP must not grow it
g_vjp = capture(lambda: eng.ppo_variables_vjp(batch, cts, va, vc, n_envs=N))
torch.cuda.synchronize()
assert eng.device_status() == 0
flat = lambda d: torch.cat([d[k].reshape(-1) for k in ("w_in", "b_in", "w_out", "b_out")] +
                           [l[k].reshape(-1) for l in d["layers"] for k in ("w_ih", "w_hh", "b")])
agree = max(float((flat(x) - flat(y)).abs().max() / flat(y).abs().max()) for x, y in ((va, ga), (vc, gc)))
t_grad, t_vjp = alternate(g_grad, g_vjp)

# 2. the new kernels' device time, from a separate profiling pass over eager calls
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(a.reps):
        eng.ppo_variables_vjp(batch, cts, va, vc, n_envs=N)
    torch.cuda.synchronize()
kern = {}
for ev in prof.key_averages():
    for name in ("ct_absmax_kernel", "grad_rescale_kernel"):
        if name in ev.key:
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            kern[name] = kern.get(name, 0.0) + t / 1000.0 / a.reps          # ms per VJP call
eng.close()

# 3. a replayed update() against a replayed update(loss_fn) with the library's loss restated in torch
ups = []
for _ in range(2):
    e = KbotStep(hidden_size=H, depth=2, gemm_path=L.GEMM_TC_2XF16)
    ups.append(PpoUpdater(e, wa, wc))
b1 = make_batch(ups[0].eng)
b2 = {k: t.clone() for k, t in b1.items()}
ups[0].update(b1, N)
ups[1].update(b2, N, loss_fn=ppo_loss)
ups[0].capture(b1, N)
ups[1].capture(b2, N, loss_fn=ppo_loss)
t_upd, t_upd_fn = alternate(ups[0]._graph, ups[1]._graph)
for up in ups:
    assert up.eng.device_status() == 0
    up.eng.close()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                     text=True).stdout.strip()
res = {"config": f"BASELINE configs[3]: {N} trajectories x {T} steps, H {H}, depth 2, FP16-split, CUDA-graph replay",
       "gpu": smi or torch.cuda.get_device_name(0),
       "kbs_ppo_grad": t_grad, "kbs_ppo_variables_vjp": t_vjp,
       "vjp_over_grad_median": t_vjp["median_ms"] / t_grad["median_ms"],
       "vjp_vs_grad_max_rel_diff": agree,
       "vjp_new_kernels_device_ms": kern,
       "update": t_upd, "update_loss_fn": t_upd_fn,
       "update_loss_fn_over_update_median": t_upd_fn["median_ms"] / t_upd["median_ms"],
       "timing": f"CUDA events, {a.rounds} alternated rounds of {a.reps} replays; new kernels from torch.profiler in a separate pass"}
line = json.dumps(res)
print(line, flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(line + "\n")
