"""The physics sub-steps of the online rollout at 4096 envs, H = 256, FP16-split: one kbs_actuator_substep replayed as a CUDA
graph, one kbs_rollout_step replayed alone, and a control step followed by its 5 replayed sub-steps, in alternated rounds;
then the device time of actuator_substep_kernel inside the replayed graphs (CUPTI through torch.profiler, a pass of its own).
The simulator's work between sub-steps is not in the window: the joint state is left as it is.  Prints one JSON line (also
written to --out).  CUDA events only; the card's name and power limit are read in the same run."""
import argparse, json, statistics, subprocess, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch
import kbot_joystick_b200  # noqa: F401
from kbot_joystick_b200 import _lib as L, synth
from kbot_joystick_b200.engine import KbotStep

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=4096)
ap.add_argument("--T", type=int, default=100)
ap.add_argument("--substeps", type=int, default=5)
ap.add_argument("--rounds", type=int, default=7, help="alternations of the three measurements")
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", type=str, default=None)
a = ap.parse_args()
dev = torch.device("cuda", 0)
N, T, H, S = a.envs, a.T, 256, a.substeps
ld = (N + 3) // 4 * 4
f32 = dict(device=dev, dtype=torch.float32)
eng = KbotStep(hidden_size=H, depth=2, gemm_path=L.GEMM_TC_2XF16)
eng.pack_weights(L.NET_ACTOR, synth.weights_to_device(synth.make_weights(77, 65, 40, H, 2), dev))
eng.pack_weights(L.NET_CRITIC, synth.weights_to_device(synth.make_weights(78, 475, 1, H, 2), dev))
d = synth.make_batch_device(1237, T, N, dev)
INPUTS = ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms")

# the trajectories one iteration of steps records (value and critic_obs included), and the simulator's one-step buffers
command = torch.zeros((T + 1, 16, ld), **f32)
eng.command_update(command[0], d["cmd_mode"][0], d["cmd_u6"][0], d["cmd_u_arms"][0], None, N)
traj = dict(command=command, actor_obs=torch.zeros((T, 65, ld), **f32), critic_obs=torch.zeros((T, L.CRITIC_OBS, ld), **f32),
            action=torch.zeros((T, 20, ld), **f32), log_prob=torch.zeros((T, ld), **f32), ctrl=torch.zeros((T, 20, ld), **f32),
            done=torch.zeros((T, ld), dtype=torch.uint8, device=dev), success=torch.zeros((T, ld), dtype=torch.uint8, device=dev),
            value=torch.zeros((T, ld), **f32),
            traj_state={k: torch.empty((T, r, ld), **f32) for k, r in (("qpos", 27), ("qvel", 26), ("sensordata", 49),
                                                                          ("xpos", 72), ("xquat", 96), ("com_distance", 1))})
io_t = {"state": {k: v[0].clone() for k, v in d["state"].items()}, "noise": {k: v[0].clone() for k, v in d["noise"].items()},
        "episode": d["episode"]}
io_t.update({k: d[k][0].clone() for k in INPUTS})
step_io = dict(io_t, **traj)
g = torch.Generator(device=dev).manual_seed(5)
io_k = {"action": traj["action"], "u_drop": torch.rand(ld, generator=g, device=dev),
        "latency": 0.003 + 0.007 * torch.rand(ld, generator=g, device=dev), "qpos": io_t["state"]["qpos"],
        "qvel": io_t["state"]["qvel"], "episode": d["episode"], "ctrl": torch.zeros((20, ld), **f32)}


def refill(t):
    for k in ("state", "noise"):
        for n, v in io_t[k].items():
            v.copy_(d[k][n][t])
    for k in INPUTS:
        io_t[k].copy_(d[k][t])


st = eng.step_state(N, True)
ast = eng.actuator_state(N, S)
# warm-up (scratch growth, the health word), then one graph of each call
eng.rollout_step(st, step_io)
for _ in range(S):
    eng.actuator_substep(st, ast, io_k)
torch.cuda.synchronize()
eng.step_state_rewind(st)
g_step, g_sub = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
with torch.cuda.graph(g_step):
    eng.rollout_step(st, step_io)
with torch.cuda.graph(g_sub):
    eng.actuator_substep(st, ast, io_k)
eng.scratch_lock(True)
torch.cuda.synchronize()


def timed(fn_t, per):
    """us per `per`: fn_t(t) bracketed by events for each step t of an iteration (inputs refilled outside the window)."""
    eng.step_state_rewind(st)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * T)]
    for t in range(T):
        refill(t)
        fn_t(t, ev[2 * t], ev[2 * t + 1])
    torch.cuda.synchronize()
    return 1e3 * sum(ev[2 * t].elapsed_time(ev[2 * t + 1]) for t in range(T)) / (T * per)


def step_alone(t, e0, e1):
    e0.record()
    g_step.replay()
    e1.record()


def step_and_subs(t, e0, e1):
    e0.record()
    g_step.replay()
    for _ in range(S):
        g_sub.replay()
    e1.record()


def subs_only(t, e0, e1):
    g_step.replay()
    e0.record()
    for _ in range(S):
        g_sub.replay()
    e1.record()


res_sub, res_step, res_both = [], [], []
for _ in range(a.rounds):
    res_sub.append(statistics.median(timed(subs_only, S) for _ in range(a.reps)))
    res_step.append(statistics.median(timed(step_alone, 1) for _ in range(a.reps)))
    res_both.append(statistics.median(timed(step_and_subs, 1) for _ in range(a.reps)))
assert eng.device_status() == 0


def device_kernels():
    """Per-kernel device time of an iteration of replayed steps, each followed by its S replayed sub-steps (CUPTI through
    torch.profiler, in a pass of its own), per control step."""
    import re
    from torch.profiler import ProfilerActivity, profile as tprofile

    def run():
        eng.step_state_rewind(st)
        for _ in range(T):
            g_step.replay()
            for _ in range(S):
                g_sub.replay()
    run()
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        low = ev.name.lower()
        if "memcpy" in low or "memset" in low:
            key = "memcpy" if "memcpy" in low else "memset"
        else:
            m = re.search(r"(\w+kernels?\w*)(<(true|false|\d)[^>]*>)?", ev.name)
            key = (m.group(1) + (m.group(2) or "")) if m else ev.name[:60]
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        o = out.setdefault(key, {"us_per_step": 0.0, "launches_per_step": 0.0})
        o["us_per_step"] += us / T
        o["launches_per_step"] += 1.0 / T
    return out


dev_k = device_kernels()
eng.scratch_lock(False)
assert eng.device_status() == 0
sub_k = dev_k.get("actuator_substep_kernel", {"us_per_step": float("nan"), "launches_per_step": 0.0})

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                     text=True).stdout.strip()
med = statistics.median
res = {"config": f"online rollout sub-steps, {N} envs, H {H}, FP16-split, {S} sub-steps per control step, value + critic_obs "
                 "recorded, CUDA-graph replay",
       "gpu": smi or torch.cuda.get_device_name(0),
       "us_per_substep_replayed": res_sub, "us_per_step_replayed_alone": res_step, "us_per_step_plus_substeps": res_both,
       "median_us_per_substep": med(res_sub), "median_us_per_step_alone": med(res_step),
       "median_us_per_step_plus_substeps": med(res_both),
       "spread_us_per_substep": max(res_sub) - min(res_sub), "spread_us_per_step_alone": max(res_step) - min(res_step),
       "spread_us_per_step_plus_substeps": max(res_both) - min(res_both),
       "actuator_substep_kernel_device_us": sub_k["us_per_step"] / max(sub_k["launches_per_step"], 1e-9),
       "kernels_step_plus_substeps_replayed_device": dev_k,
       "timing": "CUDA events; per replay of one iteration's T steps, inputs refilled outside the window; sub-step: the S "
                 "replays after a step / S; alternated rounds, median of reps per round; kernel times: CUPTI durations of the "
                 "replayed graphs per control step (memcpy = the health word's copy to the host after each call)",
       "T": T}
line = json.dumps(res)
print(line, flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(line + "\n")
eng.close()
