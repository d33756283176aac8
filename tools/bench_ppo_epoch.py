"""The update phase of one PPO epoch (ppo.PpoUpdater.epoch) replayed as one CUDA graph, against the sum of its parts, at the
launch configuration (train.py:1763-1766: 4096 envs x 100 steps per GPU, batch_size 512, 3 passes), FP16-split datapath.
Prints one JSON line (also written to --out): ms per replayed epoch; ms per replayed single update (PpoUpdater.capture on
one minibatch view); kbs_ppo_variables and kbs_gae (CUDA events around eager calls); the permutation and shuffle kernels
(kbs_profile_*); the bytes the shuffle moves, from shapes, and the bandwidth of a device-to-device copy of as many bytes
(the reachable baseline).  The card's name and power limit are read in the same run."""
import argparse, json, subprocess, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch
import kbot_joystick_b200  # noqa: F401
from kbot_joystick_b200 import _lib as L, synth
from kbot_joystick_b200.engine import KbotStep
from kbot_joystick_b200.ppo import PpoUpdater

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=4096)
ap.add_argument("--T", type=int, default=100)
ap.add_argument("--batch-size", type=int, default=512)
ap.add_argument("--passes", type=int, default=3)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--out", type=str, default=None)
a = ap.parse_args()
dev = torch.device("cuda", 0)
N, T, bs, P, H = a.envs, a.T, a.batch_size, a.passes, 256
B = N // bs
eng = KbotStep(hidden_size=H, depth=2, gemm_path=L.GEMM_TC_2XF16)
up = PpoUpdater(eng, synth.make_weights(77, 65, 40, H, 2), synth.make_weights(78, 475, 1, H, 2))
g = torch.Generator(device=dev).manual_seed(100)
rn = lambda *s, sc=1.0: torch.randn(s, generator=g, device=dev) * sc
done = (torch.rand((T, N), generator=g, device=dev) < 0.01).to(torch.uint8)
ro = {"actor_obs": rn(T, 65, N, sc=0.7), "critic_obs": rn(T, 475, N, sc=0.7), "action": rn(T, 20, N, sc=0.3), "done": done,
      "success": done & (torch.rand((T, N), generator=g, device=dev) < 0.5).to(torch.uint8), "rewards": rn(T, N, sc=0.5),
      "actor_carry0": rn(2, 2, N, H, sc=0.3), "critic_carry0": rn(2, 2, N, H, sc=0.3), "lpf0": rn(20, N, sc=0.2)}
# stored actions = samples of the policy, as a rollout stores them (independent draws have log-probs near -100, and the clipped
# ratio then drives the std gradient out of the FP16-split range after one update)
pv = eng.ppo_variables(ro["actor_obs"], ro["action"], ro["done"], ro["actor_carry0"].clone(), ro["lpf0"].clone(), want_std=True,
                       want_mean=True, n_envs=N)
ro["action"] = pv["mean"] + pv["action_std"] * rn(T, 20, N)
del pv


def timed(fn, reps):
    """ms per call: CUDA events around `reps` back-to-back calls, after one warm-up call."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


# 1. the epoch: one eager epoch (scratch, buffers), capture, replays
up.epoch(ro, N, bs, P, seed=1)
up.capture_epoch(ro, N, bs, P, seed=1)
epoch_ms = timed(lambda: up.epoch(ro, N, bs, P, seed=1), a.reps)
out = up.epoch(ro, N, bs, P, seed=1)
torch.cuda.synchronize()
assert torch.isfinite(out["norms"]).all() and eng.device_status() == 0
# 2. one update replayed on minibatch 0 of the shuffled buffer
view = {k: t[0] for k, t in up._ework["mb"].items()}
up.update(view, bs)
up.capture(view, bs)
update_ms = timed(lambda: up.update(view, bs), 10 * a.reps)
# 3. kbs_ppo_variables and kbs_gae, eager (the epoch's own work buffers)
w = up._ework


def variables():
    w["actor_carry"].copy_(ro["actor_carry0"]); w["critic_carry"].copy_(ro["critic_carry0"]); w["lpf"].copy_(ro["lpf0"])
    return eng.ppo_variables(ro["actor_obs"], ro["action"], ro["done"], w["actor_carry"], w["lpf"], ro["critic_obs"],
                             w["critic_carry"], want_std=False, n_envs=N)


v = variables()
variables_ms = timed(variables, a.reps)
gae_ms = timed(lambda: eng.gae(v["values"], ro["rewards"], ro["done"], ro["success"], adv=w["adv"], targets=w["targets"],
                               n_envs=N), 10 * a.reps)
# 4. permutation and shuffle kernels through the library's event profiler
src = {k: ro[k] for k in ("actor_obs", "critic_obs", "action", "done", "actor_carry0", "critic_carry0", "lpf0")}
src.update(old_log_probs=v["log_probs"], advantages=w["adv"], value_targets=w["targets"], old_values=v["values"])
pd = torch.zeros(1, dtype=torch.int64, device=dev)
perm = eng.minibatch_permutation(pd, N)
eng.shuffle_minibatches(perm, src, N, bs, dst=w["mb"])
torch.cuda.synchronize()
eng.profile(True)
R = 10 * a.reps
for _ in range(R):
    eng.minibatch_permutation(pd, N, out=perm)
    eng.shuffle_minibatches(perm, src, N, bs, dst=w["mb"])
prof = eng.profile_read()
eng.profile(False)
perm_ms = prof["minibatch_permutation_kernel"][0] / R
shuffle_ms = prof["shuffle_minibatches_kernels"][0] / R        # the row kernel + the carry kernel of one call
# 5. bytes the shuffle moves (read + write, from shapes) and a device-to-device copy of as many bytes
rows_f = T * (65 + 475 + 20 + 4) + 20                           # float rows of n_envs values
shuffle_bytes = 2 * (rows_f * N * 4 + T * N + 2 * 2 * 2 * N * H * 4)
cbuf = torch.empty(shuffle_bytes // 2, dtype=torch.uint8, device=dev)
cdst = torch.empty_like(cbuf)
copy_ms = timed(lambda: cdst.copy_(cbuf), 10 * a.reps)
copy_gbs = shuffle_bytes / (copy_ms * 1e-3) / 1e9
shuffle_gbs = shuffle_bytes / (shuffle_ms * 1e-3) / 1e9
parts_ms = P * B * update_ms + variables_ms + gae_ms + P * (shuffle_ms + perm_ms)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                     text=True).stdout.strip()
res = {"config": f"PPO epoch update phase: {N} envs x {T} steps, batch {bs}, {P} passes ({P * B} updates), FP16-split, CUDA-graph replay",
       "gpu": smi or torch.cuda.get_device_name(0), "ms_per_epoch": epoch_ms, "ms_per_update_replayed": update_ms,
       "ms_ppo_variables": variables_ms, "ms_gae": gae_ms, "ms_permutation_kernel": perm_ms, "ms_shuffle_kernels": shuffle_ms,
       "shuffle_bytes": shuffle_bytes, "shuffle_GBps": shuffle_gbs, "d2d_copy_ms_same_bytes": copy_ms, "d2d_copy_GBps": copy_gbs,
       "shuffle_over_copy_bandwidth": shuffle_gbs / copy_gbs, "sum_of_parts_ms": parts_ms, "epoch_over_parts": epoch_ms / parts_ms,
       "timing": "CUDA events; kernel times from kbs_profile_* (per-launch events)", "reps": a.reps}
line = json.dumps(res)
print(line, flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(line + "\n")
eng.close()
