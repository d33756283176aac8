#!/usr/bin/env python
"""bench.py -- env control-steps/s of the kbot-joystick rollout control step on B200 (BASELINE.json metric).

One "step" = one pass of the hot path over one batch of synthetic recorded state: a rollout of T control steps
(observations -> LSTM actor -> sample -> PD torque -> terminations -> command update, critic value) over n_envs
environments, followed by the 12 reward terms and the GAE scan -- BASELINE.json configs[1] (4096 envs, H = 256) at
the reference's rollout length T = 100 (train.py:1766,1776).  Environments shard across ranks with no data-path
collective (weak scaling: every rank owns `--envs` environments).

  value   device-resident inputs (CUDA events, max over ranks)
  e2e     the same step through the C-ABI with HOST (pinned) inputs: H2D of every input + D2H of the results
          inside the timed region, copies pipelined against compute on a second stream
  --impl reference   the CPU oracle restatement of the reference's JAX path (JAX/ksim are not installable here;
          see DESIGN.md) on the host cores, bounded sample of the same workload
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "env-steps/sec (obs + LSTM actor/critic + torque + terminations + rewards + GAE)"
UNIT = "env-steps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=4096, help="environments per GPU")
    ap.add_argument("--T", type=int, default=100, help="control steps per rollout")
    ap.add_argument("--hidden", type=int, default=256)
    ap.add_argument("--gemm", default="f16", choices=["f16", "tf32", "simt"],
                    help="LSTM/MLP datapath: tcgen05 2xFP16-split (default), tcgen05 3xTF32, or fp32 FFMA")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--graph", action="store_true",
                    help="replay the step as one CUDA graph instead of launching eagerly (measured slower: 10.9 vs 10.0 ms)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ppo", action="store_true", help="skip the PPO minibatch-update leg (BASELINE configs[3])")
    ap.add_argument("--ppo-traj", type=int, default=512, help="stored trajectories per GPU and update (train.py:1764 batch_size)")
    ap.add_argument("--ppo-large", type=int, default=8192,
                    help="second PPO leg: 65 536 envs / 8 GPUs = 8 192 trajectories per GPU in one update (0 = skip)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy in "
                         "float32: a fixed, seeded sample of environments, the same for every array, all of them if they "
                         "fit in 64 MB")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return a


def config_dict(a, world):
    return {"workload": "BASELINE configs[1]: kbot-headless joystick control step, 4096 envs/GPU, LSTM(2x256) "
                        "actor+critic fwd, rewards, GAE; rollout of T recorded steps",
            "n_envs_per_gpu": a.envs, "T": a.T, "hidden": a.hidden, "depth": 2, "n_gpus": world,
            "sharding": "envs (independent), weights replicated, no data-path collective",
            "l2": "inputs exceed L2 (recorded state is %.2f GB per step per GPU)" % (input_bytes(a.envs, a.T) / 1e9)}


def input_bytes(n, T):
    ld = (n + 3) // 4 * 4
    rows = 27 + 26 + 49 + 72 + 96 + 240 + 144 + 20 + 1 + 1 + 46 + 20 + 1 + 1 + 6 + 10
    return rows * 4 * ld * T


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays, n):
    """Write arrays (name -> (tensor, axis of the environment index)) as out_dir/<name>.npy in float32.  Every array keeps
    the same environments: all n if they fit in DUMP_BYTES, else a sample drawn with a fixed seed, so that two builds run
    with the same arguments can be compared file by file."""
    import numpy as np
    import torch

    per_env = sum(4 * t.numel() // t.shape[ax] for t, ax in arrays.values())
    k = min(n, DUMP_BYTES // per_env)
    idx = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, (t, ax) in arrays.items():
        sel = torch.from_numpy(idx).to(t.device)
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(ax, sel).float().cpu().numpy())


# ------------------------------------------------------------------------------------------------------------------
# CPU reference arm (oracle restatement; see module docstring)
# ------------------------------------------------------------------------------------------------------------------

def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def oracle_step(n, T, hidden, seed=4321):
    """Build a closure running one bounded sample (n envs x T steps) of the whole path in the CPU oracle."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import numpy as np
    import kbot_oracle as O
    from kbot_joystick_b200 import synth

    p = O.OracleParams(hidden_size=hidden)
    b = synth.make_batch(seed, T, n)
    wa = synth.make_weights(77, 65, 40, hidden, 2)
    wc = synth.make_weights(78, 475, 1, hidden, 2)
    r0 = b["cmd0_rand"]
    cmd0 = O.initial_command(r0["mode"], r0["u6"], r0["u_arms"], p)
    st = b["state"]

    def run():
        carry = {"actor": np.zeros((n, 2, 2, hidden), np.float32), "critic": np.zeros((n, 2, 2, hidden), np.float32),
                 "lpf_params": np.zeros((n, 20), np.float32)}
        r = O.rollout_control_steps(wa, wc, st, b["noise"], b["episode"], b["cmd_rand"], cmd0, carry,
                                    np.zeros((n, 3), np.float32), p)
        tr = {"xquat": st["xquat"], "xpos": st["xpos"], "qpos": st["qpos"], "qvel": st["qvel"], "ctrl": r["ctrl"],
              "command": r["command"], "touch_l": st["sensordata"][..., O.SD_TOUCH_L],
              "touch_r": st["sensordata"][..., O.SD_TOUCH_R], "com_distance": st["com_distance"], "done": r["done"]}
        _, total, _ = O.rewards(tr, O.reward_initial_carry((n,)), p)
        adv, tgt = O.compute_ppo_inputs(r["value"], total, r["done"], r["success"], p)
        return float(adv.sum())

    return run


def blas_threads(n):
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core, so lift the BLAS pool limit."""
    try:
        from threadpoolctl import threadpool_info, threadpool_limits

        threadpool_limits(limits=n)
        used = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
        return used
    except Exception:  # noqa: BLE001
        return 1


def time_oracle(a, seconds, steps=None, warmup=1):
    n, T = 512, 10
    run = oracle_step(n, T, a.hidden)
    threads = blas_threads(cpu_cores())
    for _ in range(warmup):
        run()
    t0 = time.perf_counter()
    k = 0
    while True:
        run()
        k += 1
        el = time.perf_counter() - t0
        if (steps is not None and k >= steps) or (steps is None and el >= seconds):
            break
    return {"value": n * T * k / el, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{k} x ({n} envs x {T} control steps + rewards + GAE), NumPy oracle restatement of train.py "
                      f"(JAX/ksim not installable), BLAS threads = host cores", "seconds": el, "n": n, "T": T, "k": k}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t = time_oracle(a, None, steps=max(a.steps, 1), warmup=max(min(a.warmup, 2), 1))
    ms = 1e3 * t["seconds"] / t["k"]
    line = {"metric": METRIC, "value": t["value"], "unit": UNIT, "impl": "reference", "n_gpus": a.gpus,
            "steps": t["k"], "warmup": max(min(a.warmup, 2), 1), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(a, a.gpus),
            "cpu_baseline": {k: t[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": t["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi fields via NVML)
# ------------------------------------------------------------------------------------------------------------------

class Clocks:
    def __init__(self, index):
        self.samples, self.reasons, self.stop, self.max_mhz, self.th = [], set(), False, None, None
        try:
            import pynvml as nv

            nv.nvmlInit()
            self.nv = nv
            self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self.th = threading.Thread(target=self._loop, daemon=True)
            self.th.start()

    def finish(self):
        self.stop = True
        if self.th:
            self.th.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------------------------
# NUMA placement of a rank (the e2e leg is bound by host memory / PCIe: pinned staging must live next to the rank's GPU)
# ------------------------------------------------------------------------------------------------------------------

def bind_to_gpu_numa_node(local):
    """Pin this process (and, by first touch + a preferred-node policy, its pinned host buffers) to the NUMA node of GPU
    `local`.  r01: with 8 ranks the end-to-end leg stopped at ~175 GB/s aggregate H2D because every rank staged through
    whatever node the launcher started it on.  Best effort: returns what it did; never raises."""
    info = {"numa_node": None, "cpus": None}
    try:
        import ctypes

        import torch

        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text().strip())
        info["pci"] = bus
        cpus = set()
        if node >= 0:
            for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        else:
            # containers often hide the PCI device's numa_node (-1): ask NVML for the GPU's ideal CPUs / memory node instead
            import pynvml as nv

            nv.nvmlInit()
            hdl = nv.nvmlDeviceGetHandleByPciBusId(bus.encode())
            words = (os.cpu_count() + 63) // 64
            for w, bits in enumerate(nv.nvmlDeviceGetCpuAffinity(hdl, words)):
                cpus.update(64 * w + b for b in range(64) if (int(bits) >> b) & 1)
            try:
                nodes = nv.nvmlDeviceGetMemoryAffinity(hdl, 4, nv.NVML_AFFINITY_SCOPE_NODE)
                ids = [64 * w + b for w, bits in enumerate(nodes) for b in range(64) if (int(bits) >> b) & 1]
                node = ids[0] if ids else -1
            except Exception:  # noqa: BLE001
                node = -1
            info["source"] = "nvml"
            if not cpus:
                return info
        use = cpus & os.sched_getaffinity(0)
        if use:
            os.sched_setaffinity(0, use)
            info["cpus"] = len(use)
        info["numa_node"] = node if node >= 0 else None
        if node < 0:
            return info
        try:                                       # set_mempolicy(MPOL_PREFERRED, {node}): x86-64 syscall 238
            mask = ctypes.c_ulong(1 << node)
            rc = ctypes.CDLL(None, use_errno=True).syscall(238, 1, ctypes.byref(mask), ctypes.c_ulong(65))
            info["mempolicy"] = "preferred" if rc == 0 else "errno %d" % ctypes.get_errno()
        except Exception as ex:  # noqa: BLE001
            info["mempolicy"] = repr(ex)
    except Exception as ex:  # noqa: BLE001
        info["error"] = repr(ex)
    return info


# ------------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------------

def run_b200(a):
    import torch
    import torch.distributed as dist

    import kbot_joystick_b200  # noqa: F401
    from kbot_joystick_b200 import _lib as L
    from kbot_joystick_b200 import spec, synth
    from kbot_joystick_b200.engine import KbotStep

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    N, T, H = a.envs, a.T, a.hidden
    ld = (N + 3) // 4 * 4
    path = {"f16": L.GEMM_TC_2XF16, "tf32": L.GEMM_TC_3XTF32, "simt": L.GEMM_SIMT_FP32}[a.gemm]
    eng = KbotStep(hidden_size=H, depth=2, gemm_path=path)
    eng.pack_weights(L.NET_ACTOR, synth.weights_to_device(synth.make_weights(77, 65, 40, H, 2), dev))
    eng.pack_weights(L.NET_CRITIC, synth.weights_to_device(synth.make_weights(78, 475, 1, H, 2), dev))

    d = synth.make_batch_device(1234 + 2 + 100 * rank, T, N, dev)      # SURVEY 8d: seed = 1234 + config number
    f32 = dict(device=dev, dtype=torch.float32)
    command = torch.zeros((T + 1, 16, ld), **f32)
    cmd0 = torch.zeros((16, ld), **f32)
    eng.command_update(cmd0, d["cmd_mode"][0], d["cmd_u6"][0], d["cmd_u_arms"][0], None, N)
    command[0] = cmd0
    io = {"state": d["state"], "noise": d["noise"], "episode": d["episode"], "eps_action": d["eps_action"],
          "u_switch": d["u_switch"], "cmd_mode": d["cmd_mode"], "cmd_u6": d["cmd_u6"], "cmd_u_arms": d["cmd_u_arms"],
          "command": command, "pg_carry": torch.zeros((3, ld), **f32),
          "actor_carry": torch.zeros((2, 2, N, H), **f32), "critic_carry": torch.zeros((2, 2, N, H), **f32),
          "lpf": torch.zeros((20, ld), **f32), "actor_obs": None, "action": torch.zeros((T, 20, ld), **f32),
          "log_prob": torch.zeros((T, ld), **f32), "ctrl": torch.zeros((T, 20, ld), **f32), "term_codes": None,
          "done": torch.zeros((T, ld), device=dev, dtype=torch.uint8),
          "success": torch.zeros((T, ld), device=dev, dtype=torch.uint8), "value": torch.zeros((T, ld), **f32), "T": T}
    rcarry = {"t_single": torch.zeros(ld, **f32), "airtime": torch.zeros((2, ld), **f32),
              "prev_contact": torch.ones((2, ld), device=dev, dtype=torch.uint8)}
    total = torch.zeros((T, ld), **f32)
    adv = torch.zeros((T, ld), **f32)
    tgt = torch.zeros((T, ld), **f32)

    def step(io_=io):
        eng.rollout(io_, N)
        eng.rewards(io_["state"], io_["command"][:T], io_["ctrl"], io_["done"], rcarry, total=total, n_envs=N)
        eng.gae(io_["value"], total, io_["done"], io_["success"], adv=adv, targets=tgt, n_envs=N)
        io_["command"][0].copy_(io_["command"][T])       # next rollout continues from the last command

    # ---- device-resident timing ------------------------------------------------------------------------------------
    # The step is ~330 kernel launches on two streams (the library forks its side stream from / joins it into the
    # caller's stream with events; nothing allocates after warm-up), so it can be captured into a CUDA graph (--graph);
    # eager launches are the default because the GPU-side step is long enough to hide the CPU launch cost.
    l_before = eng.launches
    step()
    launches_per_step = eng.launches - l_before
    run_step, launch_mode = step, "eager"
    if a.graph:
        try:
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step()
            run_step, launch_mode = graph.replay, "cuda-graph replay"
        except Exception as ex:  # noqa: BLE001
            print(f"[bench] CUDA graph capture failed ({ex!r}); timing eager launches", file=sys.stderr)
            torch.cuda.synchronize()
    for _ in range(max(a.warmup, 3)):
        run_step()
    barrier()
    clocks = Clocks(local)
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_cpu0 = time.perf_counter()
    for _ in range(a.steps):
        run_step()
    cpu_enqueue_ms = 1e3 * (time.perf_counter() - t_cpu0) / a.steps      # host time to enqueue one step (no sync inside)
    e1.record()
    barrier()
    ck_dev = clocks.finish()
    ms_total = max_ranks(e0.elapsed_time(e1))
    launches = int(sum_ranks(launches_per_step * a.steps))
    ms_step = ms_total / a.steps
    value = world * N * T / (ms_step * 1e-3)
    assert torch.isfinite(adv).all() and torch.isfinite(total).all(), "non-finite outputs"
    if a.dump_outputs and rank == 0:
        # the passes below run the step again: take its outputs now.  command row 0 is the input of the next step.
        dump_outputs(a.dump_outputs, {
            "action": (io["action"], 2), "log_prob": (io["log_prob"], 1), "ctrl": (io["ctrl"], 2),
            "done": (io["done"], 1), "success": (io["success"], 1), "value": (io["value"], 1),
            "command": (io["command"][1:], 2), "pg_carry": (io["pg_carry"], 1), "lpf": (io["lpf"], 1),
            "actor_carry": (io["actor_carry"], 2), "critic_carry": (io["critic_carry"], 2),
            "reward_total": (total, 1), "reward_t_single": (rcarry["t_single"], 0),
            "reward_airtime": (rcarry["airtime"], 1), "reward_prev_contact": (rcarry["prev_contact"], 1),
            "advantages": (adv, 1), "value_targets": (tgt, 1)}, N)

    # ---- per-kernel pass (CUDA events around every launch, same step) -> roofline of the dominant kernel ----------
    eng.profile(True)
    # the same loop again, instrumented: averaged over as many steps as were timed (at most 20), so that the kernels are measured
    # in the sustained power state of the timed region (a single step right behind it has read 10-25 % slow on some boxes)
    n_prof = max(3, min(a.steps, 20))
    for _ in range(n_prof):
        step()
    torch.cuda.synchronize()
    prof = eng.profile_read()
    eng.profile(False)
    overflow = prof.pop("_overflow")
    prof = {k: (v[0] / n_prof, v[1] // n_prof) for k, v in prof.items()}
    tot_prof = sum(v[0] for v in prof.values())
    dom_name, (dom_ms, dom_n) = max(prof.items(), key=lambda kv: kv[1][0])
    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    bf16_sus = peaks.get("bf16_tflops_sustained", 1400.0)
    which = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    flops_actor, flops_critic = spec.net_flops(65, 40, H, 2), spec.net_flops(475, 1, H, 2)
    lstm_layer_flops = 2 * (2 * H) * (4 * H)                      # one layer-step per env: [x|h] (2H) x 4H gates
    roof = None
    if dom_name in ("lstm_layer_tc_kernel", "gemm_nt_kernel(simt)", "rollout_persist_kernel"):
        if dom_name in ("lstm_layer_tc_kernel", "rollout_persist_kernel"):
            if dom_name == "rollout_persist_kernel":
                # one launch = the whole recurrence: T steps x (2 nets x depth LSTM layers + actor/critic output heads)
                # (+ the actor's input projection 2 x 65 x H, folded into its layer 0 since r01 session 4).  ALGORITHMIC
                # FLOPs = the reference's arithmetic for this work (SURVEY 8d), not the MMAs the kernel happens to issue.
                flops_per_launch = N * T * (2 * 2 * lstm_layer_flops + 2 * H * (40 + 1) + 2 * 65 * H)
            else:
                flops_per_launch = lstm_layer_flops * N * 2      # one launch = one layer-step of BOTH nets
            if a.gemm == "tf32":
                peak = bf16_sus / 6.0                             # 3xTF32: TF32 = bf16 / 2, three MMAs per product
                note = "fp32-accurate 3xTF32: peak = sustained bf16 / 6"
            else:
                peak = bf16_sus / 3.0                             # 2xFP16 split: f16 rate = bf16 rate, three MMAs per product
                note = "fp32-accurate 2xFP16-split: peak = sustained bf16 / 3"
        else:
            flops_per_launch = (2 * (flops_actor + flops_critic) * N * T) / max(dom_n, 1) / 2   # avg per SIMT GEMM launch
            peak = 72.0                                           # fp32 FFMA: 148 SMs x 128 lanes x 2 x ~1.9 GHz
            note = "fp32 FFMA path: peak = nominal FFMA rate (interim SIMT datapath)"
        ach = flops_per_launch / (dom_ms / dom_n * 1e-3) / 1e12
        # dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ncu --set full capture of this exact
        # configuration (profiles/r02_ncu_traffic.json <- tools/ncu_r02.sh); None for a configuration that was not captured
        traffic = None
        try:
            art = json.loads((ROOT / "profiles" / "r02_ncu_traffic.json").read_text())
            rec = art.get(dom_name, {}).get(f"N{N}_T{T}_H{H}_{a.gemm}")
            if rec:
                traffic = rec["dram_bytes_read"] + rec["dram_bytes_write"]
        except Exception:  # noqa: BLE001
            traffic = None
        roof = {"kernel": dom_name, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                "frac": ach / peak, "traffic": traffic, "launches": dom_n, "avg_launch_us": 1e3 * dom_ms / dom_n,
                "share_of_step": dom_ms / tot_prof, "peak_source": which, "note": note}
    else:
        roof = {"kernel": dom_name, "bound": "hbm", "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None,
                "traffic": None, "launches": dom_n, "avg_launch_us": 1e3 * dom_ms / dom_n,
                "share_of_step": dom_ms / tot_prof, "peak_source": which}
    breakdown = {k: {"ms": round(v[0], 4), "launches": v[1]} for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    # HBM-bound stages: algorithmic bytes per env-step (DESIGN.md section 4 / SURVEY 8d) x N x T / event time / HBM peak
    # obs: unique rows read (~160 floats: joints, noise, IMU, command, feet, base) + 65 actor / 107 critic rows written
    # (the 368-row cinert / cvel dump goes straight from the state into pack); command + lagged-gravity scans: the switch
    # draw, done, IMU quaternion in, 16 command rows + 3 gravity rows out (the new-command uniforms are read only at a
    # switch).  All within 5 % of ncu's dram__bytes per launch (profiles/r01_s4_phase_a_and_persist.md).
    # pack: the actor's 65 observation rows -> its 128-wide split operand (the critic's rows go straight into the projection
    # kernel: 475 rows read, H split outputs written)
    hbm_bytes = {"obs_kernel": 1210, "pack_kernels": 65 * 4 + 128 * 4, "proj_tc_kernel": 475 * 4 + H * 4,
                 "reward_terms_kernel": 340, "command_kernel": 100, "terminate_kernel": 46, "gae_kernel": 18}
    for k, b in hbm_bytes.items():
        if k in breakdown and breakdown[k]["ms"] > 0:
            gbs = b * N * T / (breakdown[k]["ms"] * 1e-3) / 1e9
            breakdown[k]["hbm_gbs"] = round(gbs, 1)
            breakdown[k]["hbm_frac"] = round(gbs / hbm_peak, 3)

    # ---- end-to-end: host (pinned) inputs -> H2D -> step -> D2H of the results -------------------------------------
    e2e = None
    ck = ck_dev
    if not a.no_e2e:
        clocks2 = Clocks(local)                            # the e2e loop is a timed region too: keep sampling through it
        clocks2.start()
        # headline e2e: the rollout's randomness is drawn ON THE DEVICE (kbs_generate_rollout_noise -- what jax.random does
        # inside the reference's jitted rollout), so only the recorded physics state crosses PCIe; e2e_host_noise keeps r01's
        # form (every PRNG-derived array uploaded from the host: the parity-test configuration)
        e2e = run_e2e(a, eng, io, rcarry, total, adv, tgt, dev, barrier, max_ranks, world, device_noise=True)
        e2e["host_noise_variant"] = run_e2e(a, eng, io, rcarry, total, adv, tgt, dev, barrier, max_ranks, world, device_noise=False)
        e2e["numa"] = numa
        # the roofline of the end-to-end leg is the host link: one large pinned H2D copy per rank, all ranks at once
        try:
            hb = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
            db = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
            db.copy_(hb, non_blocking=True)
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(8):
                db.copy_(hb, non_blocking=True)
            c1.record()
            barrier()
            link = 8 * hb.numel() / (max_ranks(c0.elapsed_time(c1)) * 1e-3) / 1e9
            e2e["host_link"] = {"h2d_gbs_per_gpu_all_ranks_copying": link,
                                "e2e_h2d_gbs_per_gpu": e2e["h2d_bytes_per_step"] / (e2e["ms_per_step"] * 1e-3) / 1e9,
                                "note": "plain 256 MB pinned cudaMemcpyAsync H2D on every rank simultaneously: what the platform's "
                                        "PCIe / host-memory path gives each GPU at this rank count"}
            e2e["host_link"]["frac"] = e2e["host_link"]["e2e_h2d_gbs_per_gpu"] / link
            del hb, db
        except Exception as ex:  # noqa: BLE001
            e2e["host_link"] = {"error": repr(ex)}
        ck2 = clocks2.finish()
        allv = sorted(clocks.samples + clocks2.samples)
        ck = {"sm_mhz": allv[len(allv) // 2] if allv else None, "sm_max_mhz": ck_dev["sm_max_mhz"],
              "reasons": sorted(set(ck_dev["reasons"]) | set(ck2["reasons"])), "samples": len(allv),
              "samples_device_loop": ck_dev["samples"], "note": "NVML samples over the device-timed loop and the e2e loop; the "
              "rollout kernel itself runs at ~1.47 GHz under the 1 000 W cap (clock64 / globaltimer, profiles/r01_persist_kernel.md)"}

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        t = time_oracle(a, a.cpu_seconds)
        cpu = {k: t[k] for k in ("value", "unit", "cores", "kind", "sample")}

    # ---- BASELINE configs[3]: the PPO minibatch update (the only collective of the path) ------------------------------
    ppo = None
    if not a.no_ppo and a.gemm == "f16":
        eng.close()
        del d, io
        torch.cuda.empty_cache()
        try:
            ppo = run_ppo_update(a, dev, world, barrier, max_ranks, peaks, a.ppo_traj)
            free, _tot = torch.cuda.mem_get_info()
            free = -max_ranks(-float(free))                  # the same decision on every rank (the leg has collectives)
            if a.ppo_large and free > 130e9:
                big = run_ppo_update(a, dev, world, barrier, max_ranks, peaks, a.ppo_large, steps=3)
                ppo["large"] = big
            elif a.ppo_large:
                ppo["large"] = {"skipped": "needs ~100 GB of free device memory, %.0f GB free" % (free / 1e9)}
        except Exception as ex:  # noqa: BLE001  the rollout numbers above must survive a failure here
            print(f"[bench] PPO update leg failed: {ex!r}", file=sys.stderr)
            ppo = {"error": repr(ex)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": max(a.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": {"f16": "f32 (tcgen05 2xFP16-split GEMMs, fp32 accumulate)",
                          "tf32": "f32 (tcgen05 3xTF32 GEMMs, fp32 accumulate)", "simt": "f32"}[a.gemm],
                "data": "synthetic", "config": config_dict(a, world), "clocks": ck, "gpu_launches": launches,
                "e2e": e2e, "roofline": roof, "cpu_baseline": cpu, "kernel_breakdown_ms": breakdown, "ppo_update": ppo,
                "profile_overflow": overflow, "gemm_path": a.gemm, "launch_mode": launch_mode,
                "cpu_enqueue_ms_per_step": cpu_enqueue_ms}
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def run_ppo_update(a, dev, world, barrier, max_ranks, peaks, n_traj, steps=8, breakdown=True):
    """BASELINE configs[3]: one PPO minibatch update per GPU on `n_traj` stored trajectories of T steps -- gradients of the
    PPO loss by BPTT through both LSTM stacks (kbs_ppo_grad: persistent tcgen05 forward + backward kernels, split-K
    weight-gradient GEMMs), the gradient all-reduce over NCCL (the path's only collective), global-norm clip + AdamW
    (train.py:1059-1065) and the weight re-pack; the whole update replayed as ONE CUDA graph.  Timed with CUDA events, max
    over ranks; the all-reduce is also timed alone against the measured 725 GB/s bus bandwidth (B200_PROFILING.md)."""
    import torch
    import torch.distributed as dist

    from kbot_joystick_b200 import _lib as L
    from kbot_joystick_b200 import synth
    from kbot_joystick_b200.engine import KbotStep
    from kbot_joystick_b200.ppo import PpoUpdater

    H, T, N = a.hidden, a.T, n_traj
    ld = (N + 3) // 4 * 4
    rank = int(os.environ.get("RANK", "0"))
    eng = KbotStep(hidden_size=H, depth=2, gemm_path=L.GEMM_TC_2XF16)
    up = PpoUpdater(eng, synth.make_weights(77, 65, 40, H, 2), synth.make_weights(78, 475, 1, H, 2))      # same weights on every rank
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    f32 = dict(device=dev, dtype=torch.float32)
    rn = lambda *s, sc=1.0: torch.randn(s, generator=g, **f32) * sc      # noqa: E731
    batch = {"actor_obs": rn(T, 65, ld, sc=0.7), "critic_obs": rn(T, 475, ld, sc=0.7), "action": rn(T, 20, ld, sc=0.3),
             "done": (torch.rand((T, ld), generator=g, device=dev) < 0.01).to(torch.uint8),
             "old_log_probs": rn(T, ld) - 20.0, "advantages": rn(T, ld), "value_targets": rn(T, ld, sc=0.5),
             "old_values": rn(T, ld, sc=0.5)}
    # old log-probs / values near the current policy, as in a real update (forward-only pass: kbs_ppo_variables)
    z = lambda: torch.zeros((2, 2, N, H), **f32)      # noqa: E731
    fwd = eng.ppo_variables(batch["actor_obs"], batch["action"], batch["done"], z(), torch.zeros((20, ld), **f32),
                            batch["critic_obs"], z(), want_std=False, n_envs=N)
    batch["old_log_probs"], batch["old_values"] = fwd["log_probs"] + rn(T, ld, sc=0.1), fwd["values"] + rn(T, ld, sc=0.2)
    del fwd
    for _ in range(2):
        up.update(batch, N)
    launches0 = eng.launches
    up.update(batch, N)
    launches_per_update = eng.launches - launches0
    mode = "cuda-graph replay (gradients + all-reduce + clip + AdamW + re-pack)"
    try:
        up.capture(batch, N)
        up.update(batch, N)
    except Exception as ex:  # noqa: BLE001
        print(f"[bench] PPO update: CUDA graph capture failed ({ex!r}); timing eager launches", file=sys.stderr)
        up._graph = None
        mode = "eager"
        torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = up.update(batch, N)
    e1.record()
    barrier()
    ms = max_ranks(e0.elapsed_time(e1) / steps)
    assert eng.device_status() == 0, "device health word set during the PPO update"
    assert torch.isfinite(up.param).all() and torch.isfinite(out["stats"]).all()
    res = {"trajectories_per_gpu": N, "T": T, "ms_per_update": ms, "env_steps_per_s": world * N * T / (ms * 1e-3),
           "updates_timed": steps, "launch_mode": mode, "kernel_launches_per_update": launches_per_update,
           "grad_floats": int(up.grad.numel()), "optimizer": "adamw lr 5e-4 wd 1e-5 + global-norm clip (train.py:1059-1065)",
           "loss": float(out["stats"][0])}
    if world > 1:                                  # the collective alone: 9 MB fp32 sum over NVLink / NVSwitch
        buf = up.grad.clone()
        for _ in range(3):
            dist.all_reduce(buf)
        barrier()
        e0.record()
        for _ in range(20):
            dist.all_reduce(buf)
        e1.record()
        barrier()
        us = max_ranks(e0.elapsed_time(e1) / 20) * 1e3
        nbytes = buf.numel() * 4
        res["allreduce"] = {"bytes": nbytes, "us": us, "bus_gbs": 2 * (world - 1) / world * nbytes / (us * 1e-6) / 1e9,
                            "bus_gbs_reference": 725.0, "note": "9 MB: latency-bound, overlapped: the critic's slice is reduced on a "
                            "second stream while the actor's weight-gradient GEMMs run (ppo.PpoUpdater._step)"}
        chk = up.param.double().sum().reshape(1).clone()          # replicas must stay bitwise identical
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        res["replicas_identical"] = bool(float(hi - lo) == 0.0)
    if breakdown:
        # per-kernel CUDA-event pass (eager, same minibatch) -> roofline of the two recurrence kernels.  ALGORITHMIC FLOPs:
        # forward 2 nets x 2 layers x 2 (2H)(4H) per row; backward [dx | dh] = dG [W_ih | W_hh]: the same count; weight
        # gradients dG^T [x | h]: the same again (+ input / output projections); fp32-accurate tensor peak = sustained bf16 / 3.
        eng.scratch_lock(False)
        os.environ["KBS_PPO_SIDE_PACK"] = "0"      # one stream for this pass: the events around a launch then time that launch alone
        eng.profile(True)
        up.grads(batch, N)
        torch.cuda.synchronize()
        prof = eng.profile_read()
        eng.profile(False)
        os.environ.pop("KBS_PPO_SIDE_PACK", None)
        prof.pop("_overflow", None)
        peak = peaks.get("bf16_tflops_sustained", 1400.0) / 3.0
        rows = N * T
        lstm = 2 * 2 * 2 * (2 * H) * (4 * H) * rows
        flops = {"rollout_persist_kernel": lstm, "bptt_persist_kernel": lstm,
                 "gemm_tn_tc_kernel": lstm + 2 * rows * H * (65 + 475) + 2 * rows * H * 41}
        kb = {}
        for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0]):
            kb[k] = {"ms": round(v[0], 4), "launches": v[1]}
            if k in flops and v[0] > 0:
                ach = flops[k] / (v[0] * 1e-3) / 1e12
                kb[k].update({"tflops": round(ach, 1), "frac_of_fp32_accurate_tensor_peak": round(ach / peak, 3)})
        res["kernel_breakdown_ms"] = kb
        res["roofline_note"] = ("rollout_persist_kernel here = lstm_fwd_save_kernel (forward with saved activations); at 512 "
                                "trajectories a slot of the wavefront holds 128 work items = one per SM: both recurrence kernels "
                                "are bound by the dependency chain of a slot (tcgen05 issue + operand fill + epilogue + publish / "
                                "poll hop), not by the tensor pipe; peak = sustained bf16 / 3 = %.0f TFLOP/s" % peak)
    eng.close()
    del up, batch
    torch.cuda.empty_cache()
    return res


def run_e2e(a, eng, io, rcarry, total, adv, tgt, dev, barrier, max_ranks, world, device_noise=True):
    """Same step with every input in pinned host memory.  The recorded state is uploaded in chunks of time steps on
    a copy stream while the compute stream runs kbs_rollout on the chunks already resident (the C-ABI takes plain
    device pointers + T, so a chunk is just an offset view); results come back with a D2H copy."""
    import torch

    N, T = a.envs, a.T
    # upload granularity: 25 steps (4 chunks per 100-step rollout) measured best: 0.94 of the link against 0.915 with 10-step
    # chunks (100 strided copies per step) and 0.905 with one chunk; KBS_E2E_CHUNK overrides
    chunk = int(os.environ.get("KBS_E2E_CHUNK", "0")) or (25 if T % 25 == 0 else 10 if T % 10 == 0 else T)
    if T % chunk:
        chunk = T
    host, h2d = {}, 0

    def pin(t):
        nonlocal h2d
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t)
        h2d += t.numel() * t.element_size()
        return h

    for grp in ("state",) if device_noise else ("state", "noise"):
        host[grp] = {k: pin(v) for k, v in io[grp].items()}
    # what kbs_upload_state moves instead of the whole state: measured by a dry call on the copy stream
    h2d -= sum(v.numel() * v.element_size() for v in io["state"].values())
    h2d += eng.upload_state(host["state"], io["state"])
    torch.cuda.synchronize()
    if not device_noise:
        for k in ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms"):
            host[k] = pin(io[k])
    host["episode"] = {k: pin(v) for k, v in io["episode"].items()}
    outs = {"adv": adv, "tgt": tgt, "total": total, "done": io["done"], "action": io["action"], "log_prob": io["log_prob"],
            "value": io["value"]}
    host_out = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in outs.items()}
    d2h = sum(v.numel() * v.element_size() for v in outs.values())
    copy_s = torch.cuda.Stream(device=dev)
    comp_s = torch.cuda.current_stream()
    # Two sets of device input buffers: the upload of step k + 1 runs while step k's last chunks, rewards, GAE and the
    # result read-back are still in flight (it only waits for step k - 1, the previous user of its buffer set).
    INPUTS = ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms")
    io_b = dict(io)
    for grp in ("state", "noise", "episode"):
        io_b[grp] = {k: torch.empty_like(v) for k, v in io[grp].items()}
    for k in INPUTS:
        io_b[k] = torch.empty_like(io[k])
    sets = [io, io_b]
    done_ev = [None, None]                                  # compute of the last step that used buffer set i
    count = [0]

    def sub_io(cur, t0, t1):
        s = dict(cur)
        s["state"] = {k: v[t0:t1] for k, v in cur["state"].items()}
        s["noise"] = {k: v[t0:t1] for k, v in cur["noise"].items()}
        for k in INPUTS + ("action", "log_prob", "ctrl", "done", "success", "value"):
            s[k] = cur[k][t0:t1]
        s["command"] = cur["command"][t0:t1 + 1]
        s["T"] = t1 - t0
        return s

    def step():
        which = count[0] & 1
        count[0] += 1
        cur = sets[which]
        evs = []
        with torch.cuda.stream(copy_s):
            if done_ev[which] is not None:
                copy_s.wait_event(done_ev[which])           # the readers of this buffer set (two steps ago) are done
            for k, v in host["episode"].items():
                cur["episode"][k].copy_(v, non_blocking=True)
            for t0 in range(0, T, chunk):
                t1 = t0 + chunk
                # recorded state: only the 473 of 676 MuJoCo rows the path reads cross PCIe (kbs_upload_state)
                eng.upload_state({k: v[t0:t1] for k, v in host["state"].items()},
                                 {k: v[t0:t1] for k, v in cur["state"].items()}, stream=copy_s.cuda_stream)
                if not device_noise:
                    for k, v in host["noise"].items():
                        cur["noise"][k][t0:t1].copy_(v[t0:t1], non_blocking=True)
                    for k in INPUTS:
                        cur[k][t0:t1].copy_(host[k][t0:t1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_s)
                evs.append(ev)
        for i, t0 in enumerate(range(0, T, chunk)):
            comp_s.wait_event(evs[i])
            sub = sub_io(cur, t0, t0 + chunk)
            if device_noise:
                eng.generate_rollout_noise(sub, N, seed=1234, step0=(count[0] - 1) * T + t0)
            eng.rollout(sub, N)
        eng.rewards(cur["state"], io["command"][:T], io["ctrl"], io["done"], rcarry, total=total, n_envs=N)
        eng.gae(io["value"], total, io["done"], io["success"], adv=adv, targets=tgt, n_envs=N)
        io["command"][0].copy_(io["command"][T])
        ev = torch.cuda.Event()
        ev.record(comp_s)
        done_ev[which] = ev
        for k, v in outs.items():
            host_out[k].copy_(v, non_blocking=True)

    for _ in range(2):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    k = max(2, min(a.steps, 5))
    for _ in range(k):
        step()
    e1.record()
    barrier()
    ms = max_ranks(e0.elapsed_time(e1)) / k
    assert torch.isfinite(host_out["adv"]).all()
    return {"value": world * N * T / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "ms_per_step": ms, "steps": k,
            "noise": "drawn on the device (kbs_generate_rollout_noise, Philox4x32-10)" if device_noise else "uploaded from the host",
            "pipeline": f"H2D in {chunk}-step chunks on a copy stream (state: only the 473 of 676 rows the path reads) into "
                        f"double-buffered device inputs, overlapped with kbs_rollout on the chunks already resident"}


if __name__ == "__main__":
    args = parse()
    # stdout carries exactly ONE line, the JSON: everything libraries write to file descriptor 1 on the way (NCCL prints
    # "NCCL version ..." there when its communicator comes up) goes to stderr instead
    sys.stdout.flush()
    _json_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(_json_fd, "w")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
    sys.stdout.flush()
