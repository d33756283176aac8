"""The online rollout at 4096 envs, H = 256, FP16-split: one control step as a replayed CUDA graph of kbs_rollout_step (carries
resident in a step state, recorded into slot t by one copy pass) against the same step as a T = 1 kbs_rollout_record call with
pointers offset to slot t (a graph of T such calls, per step), alternated in one run; a per-kernel breakdown of both forms
(kbs_profile_enable, eager, in a pass of its own); and a T-step iteration of PpoUpdater.step (replayed) + end_iteration
against PpoUpdater.iteration() (replayed) on the same state.  Prints one JSON line (also written to --out).  CUDA events only;
the card's name and power limit are read in the same run."""
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
ap.add_argument("--rounds", type=int, default=7, help="alternations of the step / T = 1 record comparison")
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", type=str, default=None)
a = ap.parse_args()
dev = torch.device("cuda", 0)
N, T, H = a.envs, a.T, 256
ld = (N + 3) // 4 * 4
f32 = dict(device=dev, dtype=torch.float32)
eng = KbotStep(hidden_size=H, depth=2, gemm_path=L.GEMM_TC_2XF16)
up = PpoUpdater(eng, synth.make_weights(77, 65, 40, H, 2), synth.make_weights(78, 475, 1, H, 2))
d = synth.make_batch_device(1237, T, N, dev)
INPUTS = ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms")


def make_io():
    io = {k: d[k] for k in ("state", "noise", "episode") + INPUTS}
    io.update(command=torch.zeros((T + 1, 16, ld), **f32), pg_carry=torch.zeros((3, ld), **f32),
              actor_carry=torch.zeros((2, 2, N, H), **f32), critic_carry=torch.zeros((2, 2, N, H), **f32),
              lpf=torch.zeros((20, ld), **f32), actor_obs=torch.zeros((T, 65, ld), **f32), action=torch.zeros((T, 20, ld), **f32),
              log_prob=torch.zeros((T, ld), **f32), ctrl=torch.zeros((T, 20, ld), **f32), term_codes=None,
              done=torch.zeros((T, ld), dtype=torch.uint8, device=dev), success=torch.zeros((T, ld), dtype=torch.uint8, device=dev),
              value=torch.zeros((T, ld), **f32), T=T)
    eng.command_update(io["command"][0], d["cmd_mode"][0], d["cmd_u6"][0], d["cmd_u_arms"][0], None, N)
    return io


io = make_io()
cobs = torch.empty((T, L.CRITIC_OBS, ld), **f32)
traj_state = {k: torch.empty((T, r, ld), **f32) for k, r in PpoUpdater.REWARD_STATE_ROWS.items()}
done_prev = torch.zeros(ld, dtype=torch.uint8, device=dev)
# the simulator's single-step buffers, refilled in place before every step
io_t = {"state": {k: v[0].clone() for k, v in d["state"].items()}, "noise": {k: v[0].clone() for k, v in d["noise"].items()},
        "episode": d["episode"]}
io_t.update({k: d[k][0].clone() for k in INPUTS})


def refill(t):
    for k in ("state", "noise"):
        for n, v in io_t[k].items():
            v.copy_(d[k][n][t])
    for k in INPUTS:
        io_t[k].copy_(d[k][t])


st = eng.step_state(N, True)
step_io = dict(io_t, command=io["command"], actor_obs=io["actor_obs"], critic_obs=cobs, action=io["action"],
               log_prob=io["log_prob"], ctrl=io["ctrl"], done=io["done"], success=io["success"], value=io["value"],
               traj_state=traj_state)


def record_t(t):
    """Step t as today's T = 1 kbs_rollout_record call, pointers offset to slot t."""
    eng.rollout(dict(io, state={k: v[t:t + 1] for k, v in d["state"].items()}, noise={k: v[t:t + 1] for k, v in d["noise"].items()},
                     **{k: d[k][t:t + 1] for k in INPUTS}, command=io["command"][t:t + 2], critic_obs=cobs[t:t + 1],
                     done_prev=done_prev, T=1,
                     **{k: io[k][t:t + 1] for k in ("actor_obs", "action", "log_prob", "ctrl", "done", "success", "value")}), N)


# warm-up (scratch growth) and the graphs: one step of each form; the record form is a graph of T calls (its addresses depend
# on t), the step form one graph replayed T times with the inputs refilled
eng.rollout_step(st, step_io)
record_t(0)
torch.cuda.synchronize()
eng.step_state_rewind(st)
g_step = torch.cuda.CUDAGraph()
with torch.cuda.graph(g_step):
    eng.rollout_step(st, step_io)
g_rec = torch.cuda.CUDAGraph()
with torch.cuda.graph(g_rec):
    for t in range(T):
        record_t(t)
eng.scratch_lock(True)
torch.cuda.synchronize()


def time_steps():
    """ms per step: T replays of the step graph (the simulator's refill of the inputs between steps is outside the window)."""
    eng.step_state_rewind(st)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * T)]
    for t in range(T):
        refill(t)
        ev[2 * t].record()
        g_step.replay()
        ev[2 * t + 1].record()
    torch.cuda.synchronize()
    return sum(ev[2 * t].elapsed_time(ev[2 * t + 1]) for t in range(T)) / T


def time_records():
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g_rec.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / T


step_us, rec_us = [], []
for _ in range(a.rounds):
    step_us.append(1e3 * statistics.median(time_steps() for _ in range(a.reps)))
    rec_us.append(1e3 * statistics.median(time_records() for _ in range(a.reps)))
assert eng.device_status() == 0
eng.scratch_lock(False)


def profile(fn, steps):
    eng.profile(True)
    fn()
    torch.cuda.synchronize()
    p = eng.profile_read()
    eng.profile(False)
    return {k: {"us_per_step": 1e3 * v[0] / steps, "launches_per_step": v[1] / steps} for k, v in p.items() if k != "_overflow"}


def eager_steps():
    eng.step_state_rewind(st)
    for t in range(10):
        eng.rollout_step(st, step_io)


prof_step = profile(eager_steps, 10)
prof_rec = profile(lambda: [record_t(t) for t in range(10)], 10)


def device_kernels(fn, steps):
    """Per-kernel device time of `fn` (CUPTI through torch.profiler, in a pass of its own): what each kernel costs inside the
    replayed graphs, without the host gaps that the eager event bracketing above also counts."""
    import re
    from torch.profiler import ProfilerActivity, profile as tprofile
    fn()
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA or "memcpy" in ev.name.lower() or "memset" in ev.name.lower():
            continue
        m = re.search(r"(\w+kernels?\w*)(<(true|false|\d)[^>]*>)?", ev.name)
        key = (m.group(1) + (m.group(2) or "")) if m else ev.name[:60]
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        o = out.setdefault(key, {"us_per_step": 0.0, "launches_per_step": 0.0})
        o["us_per_step"] += us / steps
        o["launches_per_step"] += 1.0 / steps
    return out


def replay_steps():
    eng.step_state_rewind(st)
    for t in range(T):
        g_step.replay()


eng.scratch_lock(True)
dev_step = device_kernels(replay_steps, T)
dev_rec = device_kernels(g_rec.replay, T)
eng.scratch_lock(False)

# a whole iteration: PpoUpdater.step (replayed) x T + end_iteration against iteration() (replayed), both from zero carries
rc = lambda: {"t_single": torch.zeros(ld, **f32), "airtime": torch.zeros((2, ld), **f32),
              "prev_contact": torch.ones((2, ld), device=dev, dtype=torch.uint8)}
io_on, rc_on = make_io(), rc()


def online_iteration(capture=False):
    up.begin_iteration(io_on, N)
    for t in range(T):
        refill(t)
        if capture and t == 1:
            up.capture_step(io_t)
        up.step(io_t)
    return up.end_iteration(rc_on, N)


io_it, rc_it = make_io(), rc()
up.iteration(io_it, rc_it, N)
up.capture_iteration(io_it, rc_it, N)       # first: the T-step rollout needs the larger scratch, locked from here on
online_iteration()
online_iteration(capture=True)
on_ms, it_ms = [], []
for _ in range(3):
    for fn, acc in ((online_iteration, on_ms), (lambda: up.iteration(io_it, rc_it, N), it_ms)):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        acc.append(e0.elapsed_time(e1))
assert eng.device_status() == 0

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                     text=True).stdout.strip()
ms, mr = statistics.median(step_us), statistics.median(rec_us)
res = {"config": f"online rollout step, {N} envs, H {H}, FP16-split, value + critic_obs recorded, CUDA-graph replay",
       "gpu": smi or torch.cuda.get_device_name(0),
       "us_per_step_rollout_step": step_us, "us_per_step_record_T1": rec_us,
       "median_us_rollout_step": ms, "median_us_record_T1": mr,
       "spread_us_rollout_step": max(step_us) - min(step_us), "spread_us_record_T1": max(rec_us) - min(rec_us),
       "step_beats_record_by_more_than_spread": mr - ms > max(max(step_us) - min(step_us), max(rec_us) - min(rec_us)),
       "kernels_rollout_step_eager": prof_step, "kernels_record_T1_eager": prof_rec,
       "kernels_rollout_step_replayed_device": dev_step, "kernels_record_T1_replayed_device": dev_rec,
       "iteration_ms_steps_plus_end_iteration": on_ms, "iteration_ms_iteration_replayed": it_ms,
       "timing": "CUDA events; step: per replay, inputs refilled outside the window; record: a graph of T offset calls / T; "
                 "alternated rounds, median of reps per round; kernel breakdown: *_eager = kbs_profile_enable events around "
                 "eager launches (include host launch gaps), *_replayed_device = CUPTI kernel durations of the replayed graphs",
       "T": T}
line = json.dumps(res)
print(line, flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(line + "\n")
eng.close()
