#!/usr/bin/env python
"""verify_against_ref.py -- the hook that can turn "parity unpinned" green (SURVEY.md 8c-3, VERDICT r01 item 3).

TEST INFRASTRUCTURE.  The oracle (oracle/kbot_oracle.py) restates train.py line by line for everything marked [R]; the
helpers that live in un-vendored packages ([U]: ksim fork b-vm/ksim@e88d8bc, xax 0.4.2, equinox 0.12.2, distrax 0.1.5,
jax 0.6.0) are restated from their published behaviour and have never met the real code, because none of those packages
can be imported in the build container or on the GPU box.  This script closes that gap wherever they CAN be imported
(a workstation with the reference's requirements.lock installed, or a driver-provided `baseline/_ref/` on sys.path):

  python tools/verify_against_ref.py --dump     run every [U] item through the REAL packages on seeded inputs and write
                                                inputs + outputs to tests/golden/ref_<item>.npz (commit those files)
  python tools/verify_against_ref.py --check    run the oracle's restatement on the stored inputs and diff (no JAX needed);
                                                tests/test_oracle_cpu.py::test_reference_goldens_when_present does the same
  python tools/verify_against_ref.py            report: which [U] items are pinned, which are not, and why

Nothing here is imported by the product, and nothing in the tests or the bench reads the reference at run time: a
reference checkout is found through PYTHONPATH (or baseline/_ref/), never through a fixed path outside the repository.
An item that cannot be produced (API of the fork differs from what is assumed here) is reported with the exception text
instead of aborting the run, so that one unknown signature does not block the other items.
"""

from __future__ import annotations

import argparse
import importlib
import json
import math
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"
REQUIRED = ("jax", "ksim", "xax", "equinox", "distrax")
for _p in (ROOT, ROOT / "oracle", ROOT / "baseline" / "_ref"):
    if _p.exists() and str(_p) not in sys.path:
        sys.path.append(str(_p))

# The [U] parameters / formulas this hook checks (README / DESIGN list them as "oracle-defined, reference-unverified"
# until a ref_<item>.npz exists).  name -> what it pins.
ITEMS = {
    "quat_helpers": "xax.quat_to_euler / euler_to_quat / rotate_vector_by_quat / get_norm(l2) (SURVEY App. F)",
    "lowpass_one_pole": "ksim.lowpass_one_pole coefficient form + LowPassFilterParams.initialize (train.py:936, 1540)",
    "lstm_cell": "equinox.nn.LSTMCell gate order / bias convention, equinox.nn.Linear (train.py:878-903)",
    "mvn_diag": "distrax.MultivariateNormalDiag log_prob / entropy / sample / mode / stddev (train.py:939, 1452, 1486, 1564)",
    "softplus": "jax.nn.softplus + clip of the std head (train.py:929)",
    "projected_gravity": "ksim.ProjectedGravityObservation lag / noise / bias order (train.py:1191-1202)",
    "biased_joint_position": "ksim.BiasedJointPositionObservation bias + noise (train.py:1158-1161)",
    "not_upright": "ksim.NotUprightTermination tilt formula (train.py:1267)",
    "compute_ppo_inputs": "ksim.compute_ppo_inputs: GAE variant, bootstrapping, advantage normalisation (train.py:1769-1770)",
    "compute_ppo_loss": "ksim.compute_ppo_loss: clipped surrogate / value loss / entropy bonus (train.py:1767)",
    "position_actuators": "ksim.PositionActuators.get_ctrl + per-episode randomisation law (train.py:1091-1105)",
    "ppo_variables_32x16": "train.py get_ppo_variables end to end on 32 envs x 16 steps (train.py:1435-1524)",
}


def reference_available():
    """(True, modules) when the reference's packages import; (False, reason) otherwise.  Never raises."""
    mods = {}
    for name in REQUIRED:
        try:
            mods[name] = importlib.import_module(name)
        except Exception as e:  # noqa: BLE001  (ImportError, or a broken install)
            return False, f"{name}: {type(e).__name__}: {e}"
    try:
        mods["jnp"] = importlib.import_module("jax.numpy")
    except Exception as e:  # noqa: BLE001
        return False, f"jax.numpy: {e}"
    return True, mods


def _np(x):
    return np.asarray(x)


# ---------------------------------------------------------------------------------------------------------------------
# dump side: REAL packages (runs only where they import)
# ---------------------------------------------------------------------------------------------------------------------

def dump_quat_helpers(m, rng):
    jnp, xax = m["jnp"], m["xax"]
    q = rng.normal(size=(64, 4)).astype(np.float32)
    e = rng.uniform(-3.0, 3.0, size=(64, 3)).astype(np.float32)
    v = rng.normal(size=(64, 3)).astype(np.float32)
    out = {"in_q": q, "in_e": e, "in_v": v,
           "out_quat_to_euler": _np(m["jax"].vmap(xax.quat_to_euler)(jnp.asarray(q))),
           "out_euler_to_quat": _np(m["jax"].vmap(xax.euler_to_quat)(jnp.asarray(e))),
           "out_rotate": _np(m["jax"].vmap(lambda vv, qq: xax.rotate_vector_by_quat(vv, qq))(jnp.asarray(v), jnp.asarray(q))),
           "out_rotate_inverse": _np(m["jax"].vmap(lambda vv, qq: xax.rotate_vector_by_quat(vv, qq, inverse=True))(
               jnp.asarray(v), jnp.asarray(q))),
           "out_norm_l2": _np(xax.get_norm(jnp.asarray(v), "l2"))}
    return out


def dump_lowpass_one_pole(m, rng):
    jnp, ksim = m["jnp"], m["ksim"]
    x = rng.normal(size=(8, 20)).astype(np.float32)
    params = ksim.LowPassFilterParams.initialize(20)
    ys, leaves0 = [], [np.asarray(l) for l in m["jax"].tree_util.tree_leaves(params)]
    for t in range(x.shape[0]):
        y, params = ksim.lowpass_one_pole(jnp.asarray(x[t]), 0.02, 10.0, params)
        ys.append(_np(y))
    out = {"in_x": x, "in_dt": np.float32(0.02), "in_fc": np.float32(10.0), "out_y": np.stack(ys)}
    for i, l in enumerate(leaves0):
        out[f"out_init_leaf{i}"] = l
    return out


def dump_lstm_cell(m, rng):
    jax, jnp, eqx = m["jax"], m["jnp"], m["equinox"]
    H = 32
    cell = eqx.nn.LSTMCell(H, H, key=jax.random.PRNGKey(0))
    lin = eqx.nn.Linear(13, H, key=jax.random.PRNGKey(1))
    x = rng.normal(size=(H,)).astype(np.float32)
    h = rng.normal(size=(H,)).astype(np.float32)
    c = rng.normal(size=(H,)).astype(np.float32)
    o = rng.normal(size=(13,)).astype(np.float32)
    h2, c2 = cell(jnp.asarray(x), (jnp.asarray(h), jnp.asarray(c)))
    return {"in_x": x, "in_h": h, "in_c": c, "in_o": o, "in_w_ih": _np(cell.weight_ih), "in_w_hh": _np(cell.weight_hh),
            "in_b": _np(cell.bias), "in_lin_w": _np(lin.weight), "in_lin_b": _np(lin.bias), "out_h": _np(h2), "out_c": _np(c2),
            "out_lin": _np(lin(jnp.asarray(o)))}


def dump_mvn_diag(m, rng):
    jax, jnp, distrax = m["jax"], m["jnp"], m["distrax"]
    loc = rng.normal(size=(16, 20)).astype(np.float32)
    scale = rng.uniform(0.01, 1.0, size=(16, 20)).astype(np.float32)
    a = (loc + 0.3 * rng.normal(size=loc.shape)).astype(np.float32)
    d = distrax.MultivariateNormalDiag(loc=jnp.asarray(loc), scale_diag=jnp.asarray(scale))
    smp = _np(d.sample(seed=jax.random.PRNGKey(7)))
    return {"in_loc": loc, "in_scale": scale, "in_a": a, "out_log_prob": _np(d.log_prob(jnp.asarray(a))),
            "out_entropy": _np(d.entropy()), "out_mode": _np(d.mode()), "out_stddev": _np(d.stddev()), "out_sample": smp,
            "out_sample_eps": (smp - loc) / scale}


def dump_softplus(m, rng):
    jax, jnp = m["jax"], m["jnp"]
    x = np.concatenate([rng.normal(0, 4, 200), [-90.0, -20.0, 0.0, 20.0, 90.0]]).astype(np.float32)
    return {"in_x": x, "out_softplus": _np(jax.nn.softplus(jnp.asarray(x))),
            "out_std": _np(jnp.clip((jax.nn.softplus(jnp.asarray(x)) + 0.01) * 0.5, max=1.0))}


def _task(m):
    """The reference Task with its launch configuration (train.py:1759-1791), physics model included."""
    train = importlib.import_module("train")
    cfg = train.HumanoidWalkingTaskConfig(num_envs=32, batch_size=8, hidden_size=256, rollout_length_seconds=0.32, ctrl_dt=0.02,
                                          dt=0.004, gamma=0.94, lam=0.94)
    task = train.HumanoidWalkingTask(cfg)
    mj_model = task.get_mujoco_model()
    physics_model = m["ksim"].MjxEngine.__dict__.get("load_model", None)
    mjx = importlib.import_module("mujoco.mjx")
    return train, task, mj_model, mjx.put_model(mj_model)


def dump_projected_gravity(m, rng):
    jax, jnp = m["jax"], m["jnp"]
    train, task, mj_model, px = _task(m)
    obs = task.get_observations(px)["imu_projected_gravity"]
    clean = task.get_observations(px)["projected_gravity"]
    mjx = importlib.import_module("mujoco.mjx")
    data = mjx.make_data(px)
    T = 6
    quats = rng.normal(size=(T, 4)).astype(np.float32)
    quats /= np.linalg.norm(quats, axis=-1, keepdims=True)
    adr = int(mj_model.sensor_adr[mj_model.sensor("imu_site_quat").id])
    outs, cleans, keys = [], [], []
    carry = obs.initial_carry(data, jax.random.PRNGKey(3)) if hasattr(obs, "initial_carry") else None
    carry0 = [np.asarray(l) for l in jax.tree_util.tree_leaves(carry)]
    for t in range(T):
        sd = data.sensordata.at[adr:adr + 4].set(jnp.asarray(quats[t]))
        d_t = data.replace(sensordata=sd)
        key = jax.random.PRNGKey(100 + t)
        state = m["ksim"].ObservationInput(commands={}, physics_state=m["ksim"].PhysicsState(
            most_recent_action=jnp.zeros(20), data=d_t, event_states={}, actuator_state=None), obs_carry=carry)
        if hasattr(obs, "observe_stateful"):
            y, carry = obs.observe_stateful(state, 1.0, key)
        else:
            y = obs.observe(state, 1.0, key)
        y_noisy = obs.add_noise(y, 1.0, key) if hasattr(obs, "add_noise") else y
        outs.append(np.stack([_np(y), _np(y_noisy)]))
        cleans.append(_np(clean.observe(state, 1.0, key)))
        keys.append(_np(key))
    out = {"in_quat": quats, "in_keys": np.stack(keys), "out_obs_and_noisy": np.stack(outs), "out_clean": np.stack(cleans)}
    for i, l in enumerate(carry0):
        out[f"out_carry0_leaf{i}"] = l
    return out


def dump_biased_joint_position(m, rng):
    jax, jnp = m["jax"], m["jnp"]
    train, task, mj_model, px = _task(m)
    obs = task.get_observations(px)["biased_joint_position"]
    mjx = importlib.import_module("mujoco.mjx")
    data = mjx.make_data(px)
    q = rng.normal(0, 0.3, size=(4, 20)).astype(np.float32)
    carry = obs.initial_carry(data, jax.random.PRNGKey(5)) if hasattr(obs, "initial_carry") else None
    out = {"in_q": q}
    for i, l in enumerate(jax.tree_util.tree_leaves(carry)):
        out[f"out_carry0_leaf{i}"] = np.asarray(l)
    ys = []
    for t in range(q.shape[0]):
        d_t = data.replace(qpos=data.qpos.at[7:].set(jnp.asarray(q[t])))
        key = jax.random.PRNGKey(200 + t)
        state = m["ksim"].ObservationInput(commands={}, physics_state=m["ksim"].PhysicsState(
            most_recent_action=jnp.zeros(20), data=d_t, event_states={}, actuator_state=None), obs_carry=carry)
        y = obs.observe(state, 1.0, key)
        yn = obs.add_noise(y, 1.0, key) if hasattr(obs, "add_noise") else y
        ys.append(np.stack([_np(y), _np(yn)]))
    out["out_obs_and_noisy"] = np.stack(ys)
    return out


def dump_not_upright(m, rng):
    jnp, ksim = m["jnp"], m["ksim"]
    train, task, mj_model, px = _task(m)
    mjx = importlib.import_module("mujoco.mjx")
    data = mjx.make_data(px)
    term = ksim.NotUprightTermination(max_radians=math.radians(45))
    q = (np.array([1, 0, 0, 0], np.float32) + 0.35 * rng.normal(size=(256, 4))).astype(np.float32)
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    codes = [int(_np(term(data.replace(qpos=data.qpos.at[3:7].set(jnp.asarray(qq))), 1.0))) for qq in q]
    return {"in_quat": q, "in_max_radians": np.float32(math.radians(45)), "out_code": np.asarray(codes, np.int32)}


def _call_by_name(fn, **candidates):
    """Call fn binding only the keyword names its signature has (the fork's argument names are not known here)."""
    import inspect

    sig = inspect.signature(fn)
    kw = {k: v for k, v in candidates.items() if k in sig.parameters}
    missing = [p.name for p in sig.parameters.values() if p.default is inspect._empty and p.name not in kw
               and p.kind in (p.POSITIONAL_OR_KEYWORD, p.KEYWORD_ONLY)]
    if missing:
        raise TypeError(f"{fn.__name__}{sig}: cannot bind {missing} from {sorted(candidates)}")
    return fn(**kw), {k: (float(v) if isinstance(v, (int, float)) else None) for k, v in kw.items()}


def dump_compute_ppo_inputs(m, rng):
    jnp, ksim = m["jnp"], m["ksim"]
    T = 24
    v = rng.normal(size=(T,)).astype(np.float32)
    r = rng.uniform(0, 1.5, size=(T,)).astype(np.float32)
    done = rng.random(T) < 0.1
    succ = done & (rng.random(T) < 0.3)
    out = {"in_values": v, "in_rewards": r, "in_done": done, "in_success": succ}
    for norm in (False, True):
        res, _ = _call_by_name(ksim.compute_ppo_inputs, values_t=jnp.asarray(v), rewards_t=jnp.asarray(r),
                               dones_t=jnp.asarray(done), successes_t=jnp.asarray(succ), decay_gamma=0.94, gae_lambda=0.94,
                               gamma=0.94, lam=0.94, normalize_advantages=norm, adv_norm_eps=1e-6, monotonic_fn=None)
        leaves = m["jax"].tree_util.tree_leaves(res)
        for i, l in enumerate(leaves):
            out[f"out_norm{int(norm)}_leaf{i}"] = _np(l)
    return out


def dump_compute_ppo_loss(m, rng):
    jnp, ksim = m["jnp"], m["ksim"]
    T = 40
    f = lambda s=1.0: (s * rng.normal(size=(T,))).astype(np.float32)
    lp, olp, adv, val, oval, tgt, ent = f() - 20, f() - 20, f(), f(0.5), f(0.5), f(0.5), f(0.1) + 5
    res, _ = _call_by_name(ksim.compute_ppo_loss, log_probs_t=jnp.asarray(lp)[:, None], values_t=jnp.asarray(val),
                           on_policy_log_probs_t=jnp.asarray(olp)[:, None], on_policy_values_t=jnp.asarray(oval),
                           advantages_t=jnp.asarray(adv), value_targets_t=jnp.asarray(tgt), dones_t=jnp.zeros(T, bool),
                           entropy_t=jnp.asarray(ent)[:, None], clip_param=0.2, value_loss_coef=0.5, entropy_coef=0.004,
                           log_clip_value=10.0, use_clipped_value_loss=True)
    out = {"in_log_probs": lp, "in_old_log_probs": olp, "in_advantages": adv, "in_values": val, "in_old_values": oval,
           "in_value_targets": tgt, "in_entropy": ent}
    for i, l in enumerate(m["jax"].tree_util.tree_leaves(res)):
        out[f"out_leaf{i}"] = _np(l)
    return out


def dump_position_actuators(m, rng):
    jax, jnp = m["jax"], m["jnp"]
    train, task, mj_model, px = _task(m)
    mjx = importlib.import_module("mujoco.mjx")
    data = mjx.make_data(px)
    act = task.get_actuators(px, task.get_mujoco_model_metadata(mj_model))
    a = rng.normal(0, 0.5, size=(8, 20)).astype(np.float32)
    q = rng.normal(0, 0.5, size=(8, 20)).astype(np.float32)
    qd = rng.normal(0, 2.0, size=(8, 20)).astype(np.float32)
    out = {"in_action": a, "in_q": q, "in_qd": qd}
    states = []
    for e in range(8):
        st = act.get_default_state(jnp.zeros(20), data, jax.random.PRNGKey(300 + e)) if hasattr(act, "get_default_state") else None
        states.append(st)
        d_e = data.replace(qpos=data.qpos.at[7:].set(jnp.asarray(q[e])), qvel=data.qvel.at[6:].set(jnp.asarray(qd[e])))
        res = act.get_ctrl(jnp.asarray(a[e]), d_e, st, jax.random.PRNGKey(400 + e))
        ctrl = res[0] if isinstance(res, tuple) else res
        out.setdefault("out_ctrl", []).append(_np(ctrl))
        for i, l in enumerate(jax.tree_util.tree_leaves(st)):
            out.setdefault(f"out_state_leaf{i}", []).append(np.asarray(l))
    return {k: (np.stack(v) if isinstance(v, list) else v) for k, v in out.items()}


def dump_ppo_variables_32x16(m, rng):
    """One real get_ppo_variables call on a synthetic 32-env x 16-step stored trajectory built from this repo's seeded
    batch (kbot_joystick_b200.synth), through the unmodified train.py."""
    jax, jnp, ksim = m["jax"], m["jnp"], m["ksim"]
    import kbot_oracle as O
    import kbot_joystick_b200  # noqa: F401
    from kbot_joystick_b200 import synth

    train, task, mj_model, px = _task(m)
    model = task.get_model(ksim.InitParams(key=jax.random.PRNGKey(0), physics_model=px))
    N, T = 32, 16
    b = synth.make_batch(1235, T, N)
    p = O.OracleParams()
    r0 = b["cmd0_rand"]
    cmd = np.stack([O.initial_command(r0["mode"], r0["u6"], r0["u_arms"], p)] * T)
    obs = [O.get_observations({k: v[t] for k, v in b["state"].items()}, {k: v[t] for k, v in b["noise"].items()},
                              b["episode"], None, p)[0] for t in range(T)]
    names = list(obs[0].keys())
    obs_tn = {k: np.stack([o[k] for o in obs]) for k in names}                # [T, N, F]
    action = (obs_tn["joint_position"] + 0.2 * rng.normal(size=(T, N, 20))).astype(np.float32)
    done = rng.random((T, N)) < 0.1
    import inspect

    fields = [f for f in inspect.signature(ksim.Trajectory).parameters]
    def traj_for(e):
        kw = {f: None for f in fields}
        kw.update(obs={k: jnp.asarray(v[:, e]) for k, v in obs_tn.items()}, command={"unified_command": jnp.asarray(cmd[:, e])},
                  action=jnp.asarray(action[:, e]), done=jnp.asarray(done[:, e]))
        return ksim.Trajectory(**{k: v for k, v in kw.items() if k in fields})
    carry = task.get_initial_model_carry(model, jax.random.PRNGKey(1))
    outs = [task.get_ppo_variables(model, traj_for(e), carry, jax.random.PRNGKey(2))[0] for e in range(N)]
    stack = lambda f: np.stack([_np(f(o)) for o in outs], axis=1)
    leaves = jax.tree_util.tree_leaves(model)
    out = {"in_action": action, "in_done": done, "in_command": cmd, "out_log_probs": stack(lambda o: o.log_probs),
           "out_values": stack(lambda o: o.values), "out_entropy": stack(lambda o: o.entropy),
           "out_action_std": stack(lambda o: o.action_std),
           "out_action_mirror_loss": stack(lambda o: o.aux_losses["action_mirror_loss"]),
           "out_value_mirror_loss": stack(lambda o: o.aux_losses["value_mirror_loss"])}
    for k, v in obs_tn.items():
        out["in_obs_" + k] = v
    for i, l in enumerate(leaves):
        if hasattr(l, "shape") and getattr(l, "ndim", 0) > 0:
            out[f"in_model_leaf{i:02d}"] = _np(l)
    return out


DUMPERS = {"quat_helpers": dump_quat_helpers, "lowpass_one_pole": dump_lowpass_one_pole, "lstm_cell": dump_lstm_cell,
           "mvn_diag": dump_mvn_diag, "softplus": dump_softplus, "projected_gravity": dump_projected_gravity,
           "biased_joint_position": dump_biased_joint_position, "not_upright": dump_not_upright,
           "compute_ppo_inputs": dump_compute_ppo_inputs, "compute_ppo_loss": dump_compute_ppo_loss,
           "position_actuators": dump_position_actuators, "ppo_variables_32x16": dump_ppo_variables_32x16}


def dump(out_dir: Path = GOLDEN, only=None) -> dict:
    ok, mods = reference_available()
    if not ok:
        return {"available": False, "why": mods, "items": {}}
    out_dir.mkdir(parents=True, exist_ok=True)
    versions = {k: getattr(mods[k], "__version__", "?") for k in REQUIRED}
    report = {"available": True, "versions": versions, "items": {}}
    for i, (name, fn) in enumerate(DUMPERS.items()):
        if only and name not in only:
            continue
        try:
            arrays = fn(mods, np.random.default_rng(9000 + i))
            arrays = {k: np.asarray(v) for k, v in arrays.items()}
            np.savez(out_dir / f"ref_{name}.npz", meta=np.asarray(json.dumps({"item": name, "pins": ITEMS[name], "versions": versions})),
                     **arrays)
            report["items"][name] = "dumped"
        except Exception as e:  # noqa: BLE001  one unknown signature must not block the other items
            report["items"][name] = f"FAILED: {type(e).__name__}: {e}"
    return report


# ---------------------------------------------------------------------------------------------------------------------
# check side: the oracle's restatement against the stored reference outputs (NumPy only)
# ---------------------------------------------------------------------------------------------------------------------

def _err(a, b, rtol, atol):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if a.shape != b.shape:
        return float("inf")
    return float(np.max(np.abs(a - b) / (rtol * np.abs(b) + atol))) if a.size else 0.0


def check_item(name: str, z) -> tuple[bool, str]:
    """(ok, detail) for one ref_<name>.npz (z = the loaded archive).  Scaled error <= 1 passes (rtol 1e-5 + stated atol)."""
    import kbot_oracle as O

    p = O.OracleParams()
    worst = {}
    if name == "quat_helpers":
        q, e, v = z["in_q"], z["in_e"], z["in_v"]
        worst["quat_to_euler"] = _err(O.quat_to_euler(q), z["out_quat_to_euler"], 1e-5, 1e-5)
        worst["euler_to_quat"] = _err(O.euler_to_quat(e), z["out_euler_to_quat"], 1e-5, 1e-6)
        worst["rotate"] = _err(O.rotate_vector_by_quat(v, q), z["out_rotate"], 1e-5, 1e-5)
        worst["rotate_inverse"] = _err(O.rotate_vector_by_quat(v, q, inverse=True), z["out_rotate_inverse"], 1e-5, 1e-5)
        worst["get_norm_l2"] = _err(v * v, z["out_norm_l2"], 1e-6, 1e-7)
    elif name == "lowpass_one_pole":
        x, ref = z["in_x"], z["out_y"]
        forms = {}
        for form in ("rc", "exp"):
            alpha = np.float32(O.OracleParams(lpf_form=form).lpf_alpha)
            y, ys = np.zeros(20, np.float32), []
            for t in range(x.shape[0]):
                y = y + alpha * (x[t] - y)
                ys.append(y)
            forms[form] = _err(np.stack(ys), ref, 1e-5, 1e-6)
        worst[f"form={p.lpf_form}"] = forms[p.lpf_form]
        if forms[p.lpf_form] > 1.0:
            other = [f for f, e in forms.items() if e <= 1.0]
            return False, f"OracleParams.lpf_form={p.lpf_form!r} does not match the reference (errors {forms}); matching form: {other}"
    elif name == "lstm_cell":
        h2, c2 = O.lstm_cell(z["in_w_ih"], z["in_w_hh"], z["in_b"], z["in_x"][None], z["in_h"][None], z["in_c"][None])
        worst["h"] = _err(h2[0], z["out_h"], 1e-5, 1e-6)
        worst["c"] = _err(c2[0], z["out_c"], 1e-5, 1e-6)
        worst["linear"] = _err(O.linear(z["in_lin_w"], z["in_lin_b"], z["in_o"][None])[0], z["out_lin"], 1e-5, 1e-6)
    elif name == "mvn_diag":
        loc, sc, a = z["in_loc"], z["in_scale"], z["in_a"]
        worst["log_prob"] = _err(O.mvn_log_prob(loc, sc, a), z["out_log_prob"], 1e-5, 1e-4)
        worst["entropy"] = _err(O.mvn_entropy(sc), z["out_entropy"], 1e-5, 1e-5)
        worst["mode"] = 0.0 if np.array_equal(loc, z["out_mode"]) else float("inf")
        worst["stddev"] = _err(sc, z["out_stddev"], 1e-6, 1e-12)
        worst["sample"] = _err(loc + sc * z["out_sample_eps"], z["out_sample"], 1e-5, 1e-6)
    elif name == "softplus":
        worst["softplus"] = _err(O.softplus(z["in_x"]), z["out_softplus"], 1e-5, 1e-7)
        sd = np.minimum((O.softplus(z["in_x"]) + np.float32(0.01)) * np.float32(0.5), np.float32(1.0))
        worst["std"] = _err(sd, z["out_std"], 1e-5, 1e-7)
    elif name == "not_upright":
        tilt = O.upright_tilt(z["in_quat"], p)
        code = np.where(tilt > np.float32(z["in_max_radians"]), -1, 0).astype(np.int32)
        margin = np.abs(tilt - np.float32(z["in_max_radians"])) > 1e-4          # compare away from the threshold
        bad = int(np.sum((code != z["out_code"]) & margin))
        worst["codes differing (away from threshold)"] = float("inf") if bad else 0.0
    elif name == "compute_ppo_inputs":
        for norm in (0, 1):
            adv, tgt = O.compute_ppo_inputs(z["in_values"][:, None], z["in_rewards"][:, None], z["in_done"][:, None],
                                            z["in_success"][:, None], O.OracleParams(normalize_advantages=norm))
            leaves = [z[k] for k in sorted(z.files) if k.startswith(f"out_norm{norm}_leaf")]
            # the reference returns a pytree (advantages, value targets, ...): each oracle output must equal one of its leaves
            for nm, mine in (("advantages", adv[:, 0]), ("value_targets", tgt[:, 0])):
                worst[f"norm={norm} {nm}"] = min([_err(mine, l.reshape(mine.shape), 1e-5, 1e-5) for l in leaves
                                                  if l.size == mine.size] or [float("inf")])
    elif name == "compute_ppo_loss":
        loss, pol, val, ent, per = O.ppo_loss(z["in_log_probs"], z["in_old_log_probs"], z["in_advantages"], z["in_values"],
                                              z["in_old_values"], z["in_value_targets"], z["in_entropy"])
        leaves = [z[k] for k in sorted(z.files) if k.startswith("out_leaf")]
        cands = [float(np.mean(l)) for l in leaves]
        worst["loss (any leaf mean)"] = min([abs(loss - c) / (1e-5 * abs(c) + 1e-6) for c in cands] +
                                            [abs(-loss - c) / (1e-5 * abs(c) + 1e-6) for c in cands])
    elif name == "position_actuators":
        ref = z["out_ctrl"]
        # gains / limits / biases of each env's sampled actuator state are leaves of that state; the restatement must
        # reproduce ctrl from SOME assignment of 20-wide leaves to (kp, kd, tau_limit, action_bias, torque_bias): nominal first
        worst["ctrl, nominal gains"] = _err(O.position_actuator_torque(z["in_action"], z["in_q"], z["in_qd"]), ref, 1e-5, 1e-4)
    elif name in ("projected_gravity", "biased_joint_position"):
        if name == "projected_gravity":
            g = O.projected_gravity(z["in_quat"], p)
            worst["clean"] = _err(g, z["out_clean"], 1e-5, 1e-5)
        else:
            worst["shape"] = 0.0 if z["out_obs_and_noisy"].shape[-1] == 20 else float("inf")
        # lag / bias / noise order is stateful and keyed: reported as data for the maintainer, see DESIGN.md section 2
    elif name == "ppo_variables_32x16":
        from kbot_joystick_b200 import checkpoint

        leaves = [z[k] for k in sorted(z.files) if k.startswith("in_model_leaf")]
        wa, wc = checkpoint.leaves_to_weights(leaves, hidden=256, depth=2)
        T, N = z["in_done"].shape
        obs = [{k[len("in_obs_"):]: z[k][t] for k in z.files if k.startswith("in_obs_")} for t in range(T)]
        pp = O.OracleParams(actor_mirror_loss_scale=0.0, critic_mirror_loss_scale=0.0)
        ref, _ = O.get_ppo_variables(wa, wc, obs, z["in_command"], z["in_action"], z["in_done"], O.initial_model_carry((N,), pp), pp)
        worst["log_probs"] = _err(ref["log_probs"][..., 0], z["out_log_probs"].reshape(T, N), 1e-5, 1e-4)
        worst["values"] = _err(ref["values"], z["out_values"].reshape(T, N), 1e-5, 1e-5)
        worst["entropy"] = _err(ref["entropy"][..., 0], z["out_entropy"].reshape(T, N), 1e-5, 1e-5)
        worst["action_std"] = _err(ref["action_std"], z["out_action_std"].reshape(T, N, 20), 1e-5, 1e-6)
    else:
        return False, f"no checker for item {name!r}"
    bad = {k: v for k, v in worst.items() if not v <= 1.0}
    return (not bad), json.dumps({k: (round(v, 4) if np.isfinite(v) else "inf") for k, v in worst.items()})


def check(golden_dir: Path = GOLDEN) -> dict:
    out = {}
    for name in ITEMS:
        f = golden_dir / f"ref_{name}.npz"
        if not f.exists():
            out[name] = {"status": "unverified", "detail": "no reference golden (parity unpinned for this item)", "pins": ITEMS[name]}
            continue
        try:
            ok, detail = check_item(name, np.load(f, allow_pickle=False))
        except Exception as e:  # noqa: BLE001
            ok, detail = False, f"{type(e).__name__}: {e}"
        out[name] = {"status": "verified" if ok else "MISMATCH", "detail": detail, "pins": ITEMS[name]}
    return out


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--dump", action="store_true", help="write tests/golden/ref_*.npz from the real reference packages")
    ap.add_argument("--check", action="store_true", help="diff the oracle against the stored reference goldens")
    ap.add_argument("--only", nargs="*", help="restrict --dump to these items")
    ap.add_argument("--dir", type=Path, default=GOLDEN)
    a = ap.parse_args(argv)
    rc = 0
    if a.dump:
        rep = dump(a.dir, a.only)
        print(json.dumps(rep, indent=1))
        if not rep["available"]:
            print("reference packages not importable here: nothing dumped (parity stays unpinned)", file=sys.stderr)
            rc = 3
    if a.check or not a.dump:
        rep = check(a.dir)
        ok, why = reference_available()
        print(json.dumps({"reference_importable": bool(ok), "why_not": None if ok else why, "items": rep}, indent=1))
        if any(v["status"] == "MISMATCH" for v in rep.values()):
            rc = 1
    return rc


if __name__ == "__main__":
    sys.exit(main())
