"""One whole PPO iteration (ppo.PpoUpdater.iteration: rollout with value and critic_obs -> rewards -> epoch) replayed as one CUDA
graph, against the sum of its parts, at the launch configuration (4096 envs x 100 steps per GPU, batch_size 512, 3 passes),
FP16-split datapath.  Also: the rollout with against without critic_obs, alternated in the same run, and a separate
kbs_observations pass over the stored state that writes the same critic_obs (its T per-step calls replayed as one graph).
Prints one JSON line (also written to --out).  CUDA events only; the card's name and power limit are read in the same run."""
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
ap.add_argument("--envs", type=int, default=4096)
ap.add_argument("--T", type=int, default=100)
ap.add_argument("--batch-size", type=int, default=512)
ap.add_argument("--passes", type=int, default=3)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--rounds", type=int, default=7, help="alternations of the with / without critic_obs rollout comparison")
ap.add_argument("--out", type=str, default=None)
a = ap.parse_args()
dev = torch.device("cuda", 0)
N, T, bs, P, H = a.envs, a.T, a.batch_size, a.passes, 256
ld = (N + 3) // 4 * 4
eng = KbotStep(hidden_size=H, depth=2, gemm_path=L.GEMM_TC_2XF16)
up = PpoUpdater(eng, synth.make_weights(77, 65, 40, H, 2), synth.make_weights(78, 475, 1, H, 2))
d = synth.make_batch_device(1236, T, N, dev)
f32 = dict(device=dev, dtype=torch.float32)
io = {k: d[k] for k in ("state", "noise", "episode", "eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms")}
io.update(command=torch.zeros((T + 1, 16, ld), **f32), pg_carry=torch.zeros((3, ld), **f32),
          actor_carry=torch.zeros((2, 2, N, H), **f32), critic_carry=torch.zeros((2, 2, N, H), **f32),
          lpf=torch.zeros((20, ld), **f32), actor_obs=torch.zeros((T, 65, ld), **f32), action=torch.zeros((T, 20, ld), **f32),
          log_prob=torch.zeros((T, ld), **f32), ctrl=torch.zeros((T, 20, ld), **f32), term_codes=None,
          done=torch.zeros((T, ld), dtype=torch.uint8, device=dev), success=torch.zeros((T, ld), dtype=torch.uint8, device=dev),
          value=torch.zeros((T, ld), **f32), T=T)
eng.command_update(io["command"][0], d["cmd_mode"][0], d["cmd_u6"][0], d["cmd_u_arms"][0], None, N)
rcarry = {"t_single": torch.zeros(ld, **f32), "airtime": torch.zeros((2, ld), **f32),
          "prev_contact": torch.ones((2, ld), device=dev, dtype=torch.uint8)}


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


# 0. one rollout without critic_obs first: it stages the critic's observations in the handle's scratch, which must have grown
#    before capture_iteration locks it
eng.rollout(io, N)
# 1. the iteration: one eager iteration (scratch, buffers), capture, replays
up.iteration(io, rcarry, N, bs, P, seed=1)
up.capture_iteration(io, rcarry, N, bs, P, seed=1)
iteration_ms = timed(lambda: up.iteration(io, rcarry, N, bs, P, seed=1), a.reps)
out = up.iteration(io, rcarry, N, bs, P, seed=1)
torch.cuda.synchronize()
assert torch.isfinite(out["norms"]).all() and eng.device_status() == 0
# 2. its parts: the rollout with value and critic_obs, the rewards, the epoch replayed (on the iteration's own buffers)
w = up._iwork
rec = dict(io, critic_obs=w["critic_obs"], done_prev=w["done_prev"])
rollout_rec_ms = timed(lambda: eng.rollout(rec, N), a.reps)
rewards_ms = timed(lambda: eng.rewards(io["state"], io["command"][:T], io["ctrl"], io["done"], rcarry, total=w["rewards"],
                                       n_envs=N), 10 * a.reps)
ro = {"actor_obs": io["actor_obs"], "critic_obs": w["critic_obs"], "action": io["action"], "done": io["done"],
      "success": io["success"], "rewards": w["rewards"], "actor_carry0": w["actor_carry0"], "critic_carry0": w["critic_carry0"],
      "lpf0": w["lpf0"]}
up.capture_epoch(ro, N, bs, P, seed=1)
epoch_ms = timed(lambda: up.epoch(ro, N, bs, P, seed=1), a.reps)
parts_ms = rollout_rec_ms + rewards_ms + epoch_ms
# 3. the rollout with against without critic_obs, alternated
plain = dict(io, done_prev=w["done_prev"])
with_ms, without_ms = [], []
for _ in range(a.rounds):
    with_ms.append(timed(lambda: eng.rollout(rec, N), 3))
    without_ms.append(timed(lambda: eng.rollout(plain, N), 3))
# 4. the same critic_obs from a separate kbs_observations pass over the stored state (T per-step calls, replayed as one graph)
cobs = torch.empty_like(w["critic_obs"])


def obs_pass():
    for t in range(T):
        eng.observations({k: v[t] for k, v in io["state"].items()}, io["command"][t], critic_obs=cobs[t], n_envs=N)


obs_pass()
torch.cuda.synchronize()
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    obs_pass()
obs_pass_ms = timed(g.replay, 10 * a.reps)
eng.rollout(rec, N)
obs_pass()
torch.cuda.synchronize()
same = torch.equal(cobs[:, :, :N], w["critic_obs"][:, :, :N])
cobs_bytes = T * L.CRITIC_OBS * ld * 4
extra_ms = statistics.median(with_ms) - statistics.median(without_ms)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                     text=True).stdout.strip()
res = {"config": f"PPO iteration: rollout (value + critic_obs) -> rewards -> epoch ({N} envs x {T} steps, batch {bs}, {P} passes), "
                 "FP16-split, CUDA-graph replay",
       "gpu": smi or torch.cuda.get_device_name(0), "ms_per_iteration": iteration_ms, "ms_rollout_with_critic_obs": rollout_rec_ms,
       "ms_rewards": rewards_ms, "ms_epoch_replayed": epoch_ms, "sum_of_parts_ms": parts_ms,
       "iteration_over_parts": iteration_ms / parts_ms,
       "rollout_with_critic_obs_ms": with_ms, "rollout_without_critic_obs_ms": without_ms,
       "critic_obs_extra_ms_median": extra_ms, "critic_obs_bytes": cobs_bytes,
       "critic_obs_extra_GBps": cobs_bytes / (extra_ms * 1e-3) / 1e9 if extra_ms > 0 else None,
       "separate_observations_pass_ms": obs_pass_ms, "separate_pass_bitwise_equal": same,
       "in_rollout_beats_separate_pass": extra_ms < obs_pass_ms,
       "timing": "CUDA events; with / without critic_obs alternated, 3 calls per sample", "reps": a.reps}
line = json.dumps(res)
print(line, flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(line + "\n")
eng.close()
