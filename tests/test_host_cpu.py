"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol include/kbotstep.h declares, the
ctypes structs match the C structs, constants agree between spec.py / the oracle / kbs_default_params, the Task mirror
exposes the reference's plugin surface, and the env sharding covers N > 1 (world_size-2 gloo)."""

import ctypes as C
import inspect
import os
import re
import socket
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import kbot_oracle as O

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol(lib_built):
    from kbot_joystick_b200 import _lib as L

    hdr = (ROOT / "include" / "kbotstep.h").read_text()
    declared = set(re.findall(r"^(?:int|int64_t|const char\*)\s+(kbs_\w+)\s*\(", hdr, flags=re.M))
    assert len(declared) >= 20
    lib = L.load()
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, f"declared in kbotstep.h but not exported: {missing}"
    assert declared == set(L.EXPORTS), declared ^ set(L.EXPORTS)
    assert lib.kbs_version() == 101
    assert b"aligned" in lib.kbs_error_string(-3)
    nm = subprocess.run(["nm", "-D", "--defined-only", os.fspath(L.LIB_PATH)], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (kbs_\w+)", nm))
    assert declared <= exported


def test_default_params_match_spec_and_oracle(lib_built):
    from kbot_joystick_b200 import _lib as L
    from kbot_joystick_b200 import spec

    p = L.default_params()               # pure host function: no GPU needed
    op = O.OracleParams()
    assert (p.hidden_size, p.depth) == (256, 2)
    np.testing.assert_array_equal(np.array(p.joint_bias[:], np.float32), O.joint_biases())
    np.testing.assert_array_equal(np.array(p.joint_range[:], np.float32), O.max_joint_range())
    np.testing.assert_array_equal(np.array(p.joint_bias[:], np.float32), np.array(spec.JOINT_BIASES, np.float32))
    np.testing.assert_array_equal(np.array(p.kp[:]), np.array(spec.KP, np.float32))
    np.testing.assert_array_equal(np.array(p.kd[:], np.float32), np.array(spec.KD, np.float32))
    np.testing.assert_array_equal(np.array(p.ctrl_limit[:]), np.array(spec.CTRL_LIMIT, np.float32))
    np.testing.assert_array_equal(np.array(p.reward_scale[:], np.float32), np.array(O.REWARD_SCALES, np.float32))
    np.testing.assert_array_equal(np.array(p.arm_lo[:], np.float32), O.JOINT_LIMITS64[10:, 0].astype(np.float32))
    np.testing.assert_array_equal(np.array(p.arm_hi[:], np.float32), O.JOINT_LIMITS64[10:, 1].astype(np.float32))
    for k in ("ctrl_dt", "min_std", "max_std", "var_scale", "gamma", "lam", "gravity", "eps_quat", "unhealthy_z",
              "max_tilt", "max_length_sec", "switch_prob", "lpf_alpha", "jpos_noise_mag", "jvel_noise_mag",
              "gyro_noise_std", "pg_noise_std", "linvel_es", "angvel_es", "rp_es", "rp_es_zero", "bh_es", "bh_standard",
              "bh_foot_origin", "arm_es", "grace_period", "touchdown_penalty", "feet_es", "com_es", "acc_es", "torque_es"):
        assert np.float32(getattr(p, k)) == np.float32(getattr(op, k)), k
    assert (p.body_base, p.body_lfoot, p.body_rfoot) == (spec.BODY_BASE, spec.BODY_LFOOT, spec.BODY_RFOOT)
    assert (p.sd_gyro, p.sd_imu_quat, p.sd_touch_l, p.sd_touch_r) == (19, 28, 47, 48)
    assert spec.net_flops(65, 40) == 2150912 and spec.net_flops(475, 1) == 2340864      # SURVEY 8d


def test_ctypes_structs_match_header(lib_built):
    """Field order of the ctypes mirrors == field order of the C structs (same names, same count)."""
    from kbot_joystick_b200 import _lib as L

    hdr = (ROOT / "include" / "kbotstep.h").read_text()

    def c_fields(name):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), hdr, flags=re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        out = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            names = re.sub(r"^(const\s+)?(kbs_\w+|float|double|int32_t|int64_t|uint8_t)\s*\*?\s*", "", decl)
            for nm in names.split(","):
                out.append(re.sub(r"[\*\s]|\[.*?\]", "", nm))
        return out

    for cname, cls in (("kbs_params", L.KbsParams), ("kbs_state_view", L.KbsStateView), ("kbs_noise_view", L.KbsNoiseView),
                       ("kbs_episode_view", L.KbsEpisodeView), ("kbs_net_weights", L.KbsNetWeights),
                       ("kbs_actor_out", L.KbsActorOut), ("kbs_traj_view", L.KbsTrajView),
                       ("kbs_reward_carry", L.KbsRewardCarry), ("kbs_rollout_io", L.KbsRolloutIO),
                       ("kbs_ppo_io", L.KbsPpoIO), ("kbs_ppo_loss_params", L.KbsPpoLossParams),
                       ("kbs_ppo_loss_io", L.KbsPpoLossIO), ("kbs_ppo_batch", L.KbsPpoBatch),
                       ("kbs_net_grads", L.KbsNetGrads), ("kbs_adamw_params", L.KbsAdamwParams),
                       ("kbs_actuator_rand_params", L.KbsActuatorRandParams)):
        assert c_fields(cname) == [f[0] for f in cls._fields_], cname
    assert C.sizeof(L.KbsStateView) == 11 * 8 and C.sizeof(L.KbsPpoIO) == 22 * 8    # 14 + 7 pointers + two floats


def test_product_fails_loudly_without_gpu_or_library(lib_built, monkeypatch):
    import torch

    from kbot_joystick_b200 import _lib as L
    from kbot_joystick_b200.engine import KbotStep

    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            KbotStep()
    monkeypatch.setattr(L, "_lib", None)
    monkeypatch.setattr(L, "LIB_PATH", ROOT / "kbot-joystick_b200" / "does_not_exist.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        L.load()


def test_product_never_imports_the_oracle():
    for f in (ROOT / "kbot-joystick_b200").rglob("*.py"):
        src = f.read_text()
        assert "kbot_oracle" not in src and "import oracle" not in src, f


def test_task_mirror_exposes_reference_plugin_surface():
    from kbot_joystick_b200.task import HumanoidWalkingTask, HumanoidWalkingTaskConfig

    for name in ("get_model", "get_initial_model_carry", "get_observations", "get_commands", "get_rewards",
                 "get_terminations", "get_actuators", "run_actor", "run_critic", "sample_action", "get_ppo_variables",
                 "mirror_joints", "mirror_obs"):                                    # train.py:1091-1582
        assert callable(getattr(HumanoidWalkingTask, name)), name
    assert "argmax" in inspect.signature(HumanoidWalkingTask.sample_action).parameters      # train.py:1555
    c = HumanoidWalkingTaskConfig()
    assert (c.hidden_size, c.num_envs, c.rollout_steps, c.gamma, c.lam) == (256, 4096, 100, 0.94, 0.94)   # train.py:1761-1776
    from kbot_joystick_b200 import spec

    j = np.arange(20, dtype=np.float32)
    np.testing.assert_array_equal(-j[list(spec.MIRROR_JOINT_SRC)], O.mirror_joints(j))   # the kernel's index table


def test_env_shard_partition():
    from kbot_joystick_b200.sharding import env_shard

    for n, w in ((4096, 8), (16384, 3), (7, 8), (65536, 8), (1, 1)):
        spans = [env_shard(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and sum(c for _, c in spans) == n
        for (s0, c0), (s1, _) in zip(spans, spans[1:]):
            assert s0 + c0 == s1
        assert max(c for _, c in spans) - min(c for _, c in spans) <= 1
    with pytest.raises(ValueError):
        env_shard(8, 8, 8)


_WORKER = r"""
import os, sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
import kbot_oracle as O
from kbot_joystick_b200 import synth
from kbot_joystick_b200.sharding import env_shard, max_over_ranks, sum_over_ranks
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
N, T = 37, 6
b = synth.make_batch(3, T, N)                       # every rank draws the same global batch ...
start, cnt = env_shard(N, rank, world)               # ... and owns a contiguous block of envs
rng = np.random.default_rng(0)
v = rng.standard_normal((T, N)).astype(np.float32); r = rng.random((T, N)).astype(np.float32)
done = rng.random((T, N)) < 0.1; succ = done & (rng.random((T, N)) < 0.5)
p = O.OracleParams()
adv_full, _ = O.compute_ppo_inputs(v, r, done, succ, p)
sl = slice(start, start + cnt)
adv_loc, _ = O.compute_ppo_inputs(v[:, sl], r[:, sl], done[:, sl], succ[:, sl], p)
assert np.array_equal(adv_loc, adv_full[:, sl])      # envs are independent: sharding needs no data-path collective
tot = sum_over_ranks(float(cnt))
assert tot == N, tot
t = max_over_ranks(1.0 + rank)
assert t == float(world), t
chk = sum_over_ranks(float(adv_loc.astype(np.float64).sum()))
assert abs(chk - float(adv_full.astype(np.float64).sum())) < 1e-6
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_env_sharding_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % (str(ROOT), str(ROOT / "oracle")))
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="2", OMP_NUM_THREADS="1")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o}"
        assert f"rank {r} ok" in o


_PPO_WORKER = r"""
import os, sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
import kbot_oracle as O
import ppo_grad_torch as G
from kbot_joystick_b200 import synth
from kbot_joystick_b200.ppo import NetParams, allreduce_sum_
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
T, N, H = 3, 8, 128
p = O.OracleParams(hidden_size=H)
wa, wc = synth.make_weights(1, 65, 40, H, 2), synth.make_weights(2, 475, 1, H, 2)
rng = np.random.default_rng(0)
f = np.float32
b = {"actor_obs": rng.normal(0, .7, (T, N, 65)).astype(f), "critic_obs": rng.normal(0, .7, (T, N, 475)).astype(f),
     "action": (.3 * rng.normal(size=(T, N, 20))).astype(f), "done": rng.random((T, N)) < .2,
     "advantages": rng.normal(size=(T, N)).astype(f), "value_targets": rng.normal(size=(T, N)).astype(f),
     "old_log_probs": rng.normal(-18, 1, (T, N)).astype(f), "old_values": rng.normal(size=(T, N)).astype(f)}
full = G.ppo_minibatch_grads(wa, wc, b, p)
sl = slice(rank * N // world, (rank + 1) * N // world)               # environments shard across ranks, weights replicated
loc = G.ppo_minibatch_grads(wa, wc, {k: v[:, sl] for k, v in b.items()}, p)
flat = torch.cat([NetParams(loc[2]).flat.double(), NetParams(loc[3]).flat.double()])
assert allreduce_sum_(flat) == world                                 # the PPO gradient all-reduce
flat /= world
ref = torch.cat([NetParams(full[2]).flat.double(), NetParams(full[3]).flat.double()])
assert flat.numel() == ref.numel() == sum(int(np.prod(s)) for s in NetParams(wa).shapes + NetParams(wc).shapes)
assert torch.allclose(flat, ref, rtol=1e-5, atol=2e-6 * float(ref.abs().max())), float((flat - ref).abs().max())   # NetParams is fp32
v = NetParams(wa).as_dict()                                           # flat <-> eqx-layout views round trip
assert np.array_equal(v["layers"][1]["w_hh"].numpy(), wa["layers"][1]["w_hh"]) and np.array_equal(v["b_out"].numpy(), wa["b_out"])
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_ppo_gradient_allreduce_world_size_2_gloo(tmp_path):
    """Data-parallel PPO update: per-rank gradients on an env shard, summed over ranks and divided by the world size,
    equal the gradients of the whole minibatch (equal shards); NetParams' flat layout round-trips."""
    script = tmp_path / "worker.py"
    script.write_text(_PPO_WORKER % (str(ROOT), str(ROOT / "oracle")))
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="2", OMP_NUM_THREADS="1")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o}"
        assert f"rank {r} ok" in o


def test_checkpoint_leaf_stream_round_trip(tmp_path):
    """8f-4: the eqx `tree_serialise_leaves` stream of Model(actor, critic) <-> the weight dicts kbs_weights_pack takes."""
    from kbot_joystick_b200 import checkpoint as ck
    from kbot_joystick_b200 import synth

    wa, wc = synth.make_weights(5, 65, 40, 128, 2), synth.make_weights(6, 475, 1, 128, 2)
    static = (65, 20, 0.01, 1.0, 0.5, 10.0, 0.02)          # Actor's scalar fields (train.py:853-860) ride along as 0-d leaves
    path = tmp_path / "model.eqx"
    ck.write_leaves(ck.weights_to_leaves(wa, wc, static_actor=static, static_critic=(475,)), path)
    a, c = ck.load_policy(path, hidden=128, depth=2)
    for got, ref in ((a, wa), (c, wc)):
        for k in ("w_in", "b_in", "w_out", "b_out"):
            np.testing.assert_array_equal(got[k], ref[k])
        for l in range(2):
            for k in ("w_ih", "w_hh", "b"):
                np.testing.assert_array_equal(got["layers"][l][k], ref["layers"][l][k])
    with pytest.raises(AssertionError):
        ck.load_policy(path, hidden=256, depth=2)            # wrong architecture is refused, not silently reshaped


def test_xla_ffi_shim_sources_agree():
    """The (uncompiled here: no jaxlib) XLA-FFI shim: jax_ffi.py imports without jax and registers exactly the handler
    symbols csrc/kbs_xla_ffi.cc defines; every handler forwards to an entry point include/kbotstep.h declares."""
    import re
    from pathlib import Path

    import kbot_joystick_b200.jax_ffi as kf

    root = Path(__file__).resolve().parent.parent
    cc = (root / "kbot-joystick_b200" / "csrc" / "kbs_xla_ffi.cc").read_text()
    header = (root / "include" / "kbotstep.h").read_text()
    defined = set(re.findall(r"XLA_FFI_DEFINE_HANDLER_SYMBOL\((\w+),", cc))
    assert defined == set(kf._TARGETS.values()), (defined, kf._TARGETS)
    for target in kf._TARGETS:
        assert re.search(rf"\bint {target}\(", header), target
        assert f"{target}(H(handle)" in cc, target


def test_xla_ffi_shim_compiles_against_stub_headers():
    """jaxlib's headers are not installable here, so csrc/kbs_xla_ffi.cc is type-checked with g++ against a stub of the FFI
    surface (tests/ffi_stub) whose Bind().To() static_asserts every handler against the context / attribute / argument /
    result types of its binding.  Catches typos and signature drift; the real build is `make ffi JAX_INCLUDE=...`."""
    import shutil

    if not shutil.which("g++"):
        pytest.skip("no g++")
    cuda_inc = "/usr/local/cuda/include"
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I" + str(ROOT / "tests" / "ffi_stub"), "-I" + str(ROOT / "include"),
           "-I" + cuda_inc, "-x", "c++", str(ROOT / "kbot-joystick_b200" / "csrc" / "kbs_xla_ffi.cc")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    # ... and the stub really checks: a handler bound with a wrong argument type must not compile
    src = (ROOT / "kbot-joystick_b200" / "csrc" / "kbs_xla_ffi.cc").read_text()
    bad = src.replace("XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsMirrorJoints, MirrorJointsImpl, KBS_BIND_N().Arg<F32>().Ret<F32>());",
                      "XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsMirrorJoints, MirrorJointsImpl, KBS_BIND_N().Arg<U8>().Ret<F32>());")
    assert bad != src
    r2 = subprocess.run(cmd[:-1] + ["-"], input=bad, capture_output=True, text=True)
    assert r2.returncode != 0 and "does not match its binding" in r2.stderr


def test_ffi_covers_every_hot_path_entry_point():
    """north_star: "a thin C-ABI exposed as JAX FFI custom calls".  Every compute entry point of include/kbotstep.h on the
    path has an XLA-FFI handler + a jax_ffi.py wrapper (debug / profiling / lifecycle symbols are host-side only)."""
    import kbot_joystick_b200.jax_ffi as kf

    need = {"kbs_observations", "kbs_command_update", "kbs_actor_step", "kbs_critic_step", "kbs_torque", "kbs_terminate",
            "kbs_rewards", "kbs_gae", "kbs_policy_step", "kbs_rollout", "kbs_ppo_variables", "kbs_mirror_observations",
            "kbs_mirror_joints", "kbs_com_distance", "kbs_ppo_grad", "kbs_adamw_step", "kbs_grad_norm",
            "kbs_sample_actuator_randomization"}
    assert need <= set(kf._TARGETS), need - set(kf._TARGETS)
    for t in need:
        assert callable(getattr(kf, t[len("kbs_"):])), t


def test_ksim_adapter_matches_reference_hook_signatures():
    """kbot_joystick_b200.ksim_adapter overrides the reference Task's model hooks with EXACTLY the reference's parameter
    lists (tests/golden/ref_signatures.json, extracted from the reference's train.py by tools/make_ref_signatures.py:
    regenerate it there when the reference changes), and lowers each to FFI targets jax_ffi registers.  Importing it
    needs neither jax nor ksim."""
    import json

    import kbot_joystick_b200.jax_ffi as kf
    import kbot_joystick_b200.ksim_adapter as ka

    fix = json.loads((ROOT / "tests" / "golden" / "ref_signatures.json").read_text())["hooks"]
    for name in ("run_actor", "run_critic", "sample_action", "get_ppo_variables", "get_initial_model_carry"):
        got = list(inspect.signature(getattr(ka.KbotFfiTaskMixin, name)).parameters)
        assert got == fix[name]["args"], (name, got, fix[name]["args"])
        for tgt in ka.HOOK_TARGETS[name]:
            assert tgt in kf._TARGETS, (name, tgt)
    # the batched torch mirror (task.py) keeps the same hook NAMES for the whole plugin surface
    from kbot_joystick_b200 import task as T

    for name in ("get_observations", "get_commands", "get_rewards", "get_terminations", "get_actuators", "get_model",
                 "get_initial_model_carry", "sample_action", "get_ppo_variables", "run_actor", "run_critic"):
        assert name in fix and hasattr(T.HumanoidWalkingTask, name), name
