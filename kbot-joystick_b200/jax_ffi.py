"""jax.ffi registration of the XLA-FFI handlers in libkbs_xla_ffi.so (csrc/kbs_xla_ffi.cc): the binding a JAX program
such as the reference (train.py on ksim) uses to call the C-ABI from inside jit on the CUDA platform.

Not importable in this image (no jax / jaxlib: SURVEY F5) and not used by the tests or the bench, which bind the same
C-ABI through ctypes + torch (`_lib.py`, `engine.py`).  Build the shim with `make ffi JAX_INCLUDE=...` first.  Every
wrapper below is one `jax.ffi.ffi_call` = one custom call in the jitted program; in-out arguments of the C-ABI (carries,
filter / reward / optimiser state) are aliased onto their results (`input_output_aliases`), so XLA updates them in place.

    import kbot_joystick_b200.jax_ffi as kf
    kf.register()                                   # once per process
    h = engine.handle_address                       # kbs_create / kbs_weights_pack done through ctypes as usual
    adv, targets = kf.gae(h, values_tn, rewards_tn, done_tn, success_tn, n_envs=N)

Layout at this boundary: env-major SoA `[F, ld]` (`ld` = n_envs rounded up to a multiple of 4), trajectories `[T, F, ld]`;
`ksim_adapter.py` converts from / to the single-env arrays the ksim Task hooks see (one custom call per vmapped hook).
"""
from __future__ import annotations

import ctypes
from pathlib import Path

# jax.ffi target name -> (handler symbol in libkbs_xla_ffi.so, the entry point of include/kbotstep.h it forwards to)
_TARGETS = {
    "kbs_gae": "KbsGae", "kbs_terminate": "KbsTerminate", "kbs_torque": "KbsTorque",
    "kbs_sample_actuator_randomization": "KbsSampleActuatorRandomization", "kbs_policy_step": "KbsPolicyStep",
    "kbs_observations": "KbsObservations", "kbs_command_update": "KbsCommandUpdate", "kbs_actor_step": "KbsActorStep",
    "kbs_critic_step": "KbsCriticStep", "kbs_rollout": "KbsRollout",
    "kbs_rollout_record": "KbsRolloutRecord", "kbs_ppo_variables": "KbsPpoVariables",
    "kbs_mirror_observations": "KbsMirrorObservations", "kbs_mirror_joints": "KbsMirrorJoints",
    "kbs_com_distance": "KbsComDistance", "kbs_rewards": "KbsRewards", "kbs_ppo_grad": "KbsPpoGrad",
    "kbs_grad_norm": "KbsGradNorm", "kbs_adamw_step": "KbsAdamwStep", "kbs_ppo_variables_vjp": "KbsPpoVariablesVjp",
}
STATE_ROWS = (("qpos", 27), ("qvel", 26), ("sensordata", 49), ("xpos", 72), ("xquat", 96), ("cinert", 240), ("cvel", 144),
              ("actuator_force", 20))


def register(path: str | None = None) -> None:
    import jax  # noqa: PLC0415 -- deliberately lazy: this module must import without jax

    lib = ctypes.cdll.LoadLibrary(path or str(Path(__file__).resolve().parent / "libkbs_xla_ffi.so"))
    for target, symbol in _TARGETS.items():
        jax.ffi.register_ffi_target(target, jax.ffi.pycapsule(getattr(lib, symbol)), platform="CUDA")


def _j():
    import jax
    import jax.numpy as jnp
    import numpy as np

    return jax, jnp, np


def _sds(jax, shape, dtype):
    return jax.ShapeDtypeStruct(tuple(shape), dtype)


def _h(np, handle, **attrs):
    out = {"handle": np.int64(handle)}
    for k, v in attrs.items():
        out[k] = np.float32(v) if isinstance(v, float) else np.int64(v)
    return out


def gae(handle: int, values, rewards, done, success, n_envs: int):
    """ksim.compute_ppo_inputs: values / rewards [T, ld] f32, done / success [T, ld] -> (advantages, value_targets)."""
    jax, jnp, np = _j()
    out = (_sds(jax, values.shape, jnp.float32),) * 2
    return jax.ffi.ffi_call("kbs_gae", out)(values, rewards, done.astype(jnp.uint8), success.astype(jnp.uint8),
                                            **_h(np, handle, n_envs=n_envs))


def terminate(handle: int, qpos, xpos, time, n_envs: int):
    """get_terminations: qpos [27, ld], xpos [72, ld], time [ld] -> (codes s32 [3, ld], done u8 [ld], success u8 [ld])."""
    jax, jnp, np = _j()
    ld = qpos.shape[-1]
    out = (_sds(jax, (3, ld), jnp.int32), _sds(jax, (ld,), jnp.uint8), _sds(jax, (ld,), jnp.uint8))
    return jax.ffi.ffi_call("kbs_terminate", out)(qpos, xpos, time, **_h(np, handle, n_envs=n_envs))


def torque(handle: int, action, qpos, qvel, kp, kd, tau_limit, action_bias, torque_bias, n_envs: int):
    """PositionActuators.get_ctrl: action [20, ld] + joint state + the per-episode actuator arrays [20, ld] -> ctrl [20, ld]."""
    jax, jnp, np = _j()
    return jax.ffi.ffi_call("kbs_torque", _sds(jax, action.shape, jnp.float32))(
        action, qpos, qvel, kp, kd, tau_limit, action_bias, torque_bias, **_h(np, handle, n_envs=n_envs))


def sample_actuator_randomization(handle: int, u, reset, kp, kd, tau_limit, action_bias, torque_bias, n_envs: int):
    """Per-episode PositionActuators randomisation: u [5, 20, ld] uniforms, reset u8 [ld]; the five arrays are updated in place."""
    jax, jnp, np = _j()
    out = tuple(_sds(jax, a.shape, jnp.float32) for a in (kp, kd, tau_limit, action_bias, torque_bias))
    call = jax.ffi.ffi_call("kbs_sample_actuator_randomization", out, input_output_aliases={2: 0, 3: 1, 4: 2, 5: 3, 6: 4})
    return call(u, reset.astype(jnp.uint8), kp, kd, tau_limit, action_bias, torque_bias, **_h(np, handle, n_envs=n_envs))


def policy_step(handle: int, joint_angles, joint_vel, projected_gravity, gyro, command, carry):
    """convert.py step_fn batched over envs: AoS [n, .] inputs + flat carry [n, depth*2*H + 20] -> (action [n, 20], carry)."""
    jax, jnp, np = _j()
    n = joint_angles.shape[0]
    out = (_sds(jax, (n, 20), jnp.float32), _sds(jax, carry.shape, jnp.float32))
    return jax.ffi.ffi_call("kbs_policy_step", out)(joint_angles, joint_vel, projected_gravity, gyro, command, carry,
                                                    **_h(np, handle))


def observations(handle: int, state: dict, noise, jpos_bias, pg_lag, pg_bias, command, pg_carry, pg_reset, n_envs: int):
    """get_observations + the run_actor / run_critic concatenations: state = {qpos [27, ld], ...} (STATE_ROWS), noise [46, ld]
    -> (pg_carry [3, ld], computed [78, ld], actor_obs [65, ld], critic_obs [475, ld])."""
    jax, jnp, np = _j()
    ld = state["qpos"].shape[-1]
    f32 = jnp.float32
    out = (_sds(jax, (3, ld), f32), _sds(jax, (78, ld), f32), _sds(jax, (65, ld), f32), _sds(jax, (475, ld), f32))
    call = jax.ffi.ffi_call("kbs_observations", out, input_output_aliases={13: 0})
    return call(*(state[k] for k, _ in STATE_ROWS), noise, jpos_bias, pg_lag, pg_bias, command, pg_carry,
                pg_reset.astype(jnp.uint8), **_h(np, handle, n_envs=n_envs))


def command_update(handle: int, command, u_switch, mode, u6, u_arms, n_envs: int, initial: bool = False):
    """UnifiedCommand.__call__ (initial=True: initial_command): command [16, ld] updated in place."""
    jax, jnp, np = _j()
    call = jax.ffi.ffi_call("kbs_command_update", _sds(jax, command.shape, jnp.float32), input_output_aliases={0: 0})
    return call(command, u_switch, mode.astype(jnp.int32), u6, u_arms, **_h(np, handle, n_envs=n_envs, always_resample=int(initial)))


def actor_step(handle: int, obs, carry, lpf, eps, done, n_envs: int, argmax: bool = False):
    """sample_action: obs [65, ld], carry [depth, 2, n, H], lpf [20, ld], eps [20, ld] N(0,1), done u8 [ld]
    -> (carry, lpf, action, mean, std [20, ld], log_prob, entropy [ld])."""
    jax, jnp, np = _j()
    ld = obs.shape[-1]
    f32 = jnp.float32
    out = (_sds(jax, carry.shape, f32), _sds(jax, lpf.shape, f32)) + (_sds(jax, (20, ld), f32),) * 3 + (_sds(jax, (ld,), f32),) * 2
    call = jax.ffi.ffi_call("kbs_actor_step", out, input_output_aliases={1: 0, 2: 1})
    return call(obs, carry, lpf, eps, done.astype(jnp.uint8), **_h(np, handle, n_envs=n_envs, argmax=int(argmax)))


def critic_step(handle: int, obs, carry, done, n_envs: int):
    """run_critic: obs [475, ld], carry [depth, 2, n, H], done u8 [ld] -> (carry, value [ld])."""
    jax, jnp, np = _j()
    out = (_sds(jax, carry.shape, jnp.float32), _sds(jax, (obs.shape[-1],), jnp.float32))
    call = jax.ffi.ffi_call("kbs_critic_step", out, input_output_aliases={1: 0})
    return call(obs, carry, done.astype(jnp.uint8), **_h(np, handle, n_envs=n_envs))


def rollout(handle: int, state: dict, noise: dict, episode, torque_bias, rand: dict, command0, pg_carry, actor_carry,
            critic_carry, lpf, n_envs: int):
    """The fused control step over T recorded steps (kbs_rollout).  state: {name: [T, rows, ld]} incl. com_distance / time
    [T, ld]; noise: eps_jpos, eps_jvel [T, 20, ld], eps_gyro, eps_pg [T, 3, ld]; episode [84 + 20, ld] packed as the handler
    documents; rand: eps_action [T, 20, ld], u_switch [T, ld], cmd_mode s32 [T, ld], cmd_u6 [T, 6, ld], cmd_u_arms [T, 10, ld].
    -> dict(command [T + 1, 16, ld], pg_carry, actor_carry, critic_carry, lpf, actor_obs, action, log_prob, ctrl, term_codes,
    done, success, value)."""
    jax, jnp, np = _j()
    T, _, ld = state["qpos"].shape
    f32 = jnp.float32
    names = ("command", "pg_carry", "actor_carry", "critic_carry", "lpf", "actor_obs", "action", "log_prob", "ctrl", "term_codes",
             "done", "success", "value")
    out = (_sds(jax, (T + 1, 16, ld), f32), _sds(jax, pg_carry.shape, f32), _sds(jax, actor_carry.shape, f32),
           _sds(jax, critic_carry.shape, f32), _sds(jax, lpf.shape, f32), _sds(jax, (T, 65, ld), f32), _sds(jax, (T, 20, ld), f32),
           _sds(jax, (T, ld), f32), _sds(jax, (T, 20, ld), f32), _sds(jax, (T, 3, ld), jnp.int32), _sds(jax, (T, ld), jnp.uint8),
           _sds(jax, (T, ld), jnp.uint8), _sds(jax, (T, ld), f32))
    call = jax.ffi.ffi_call("kbs_rollout", out, input_output_aliases={22: 1, 23: 2, 24: 3, 25: 4})
    res = call(*(state[k] for k, _ in STATE_ROWS), state["com_distance"], state["time"], noise["eps_jpos"], noise["eps_jvel"],
               noise["eps_gyro"], noise["eps_pg"], episode, torque_bias, rand["eps_action"], rand["u_switch"],
               rand["cmd_mode"].astype(jnp.int32), rand["cmd_u6"], rand["cmd_u_arms"], command0, pg_carry, actor_carry, critic_carry,
               lpf, **_h(np, handle, n_envs=n_envs))
    return dict(zip(names, res))


def rollout_record(handle: int, state: dict, noise: dict, episode, torque_bias, rand: dict, command0, pg_carry, actor_carry,
                   critic_carry, lpf, done_prev, n_envs: int):
    """rollout() continued across calls (kbs_rollout_record): done_prev [ld] is the previous call's done[T-1] (zeros on the
    first call), so the lag state restarts where an episode ended on the previous call's last step -- with one step per call,
    as ksim's engine loop makes it, that is every episode end.  -> rollout()'s dict plus critic_obs [T, 475, ld], the
    critic's concatenation of every step."""
    jax, jnp, np = _j()
    T, _, ld = state["qpos"].shape
    f32 = jnp.float32
    names = ("command", "pg_carry", "actor_carry", "critic_carry", "lpf", "actor_obs", "action", "log_prob", "ctrl", "term_codes",
             "done", "success", "value", "critic_obs")
    out = (_sds(jax, (T + 1, 16, ld), f32), _sds(jax, pg_carry.shape, f32), _sds(jax, actor_carry.shape, f32),
           _sds(jax, critic_carry.shape, f32), _sds(jax, lpf.shape, f32), _sds(jax, (T, 65, ld), f32), _sds(jax, (T, 20, ld), f32),
           _sds(jax, (T, ld), f32), _sds(jax, (T, 20, ld), f32), _sds(jax, (T, 3, ld), jnp.int32), _sds(jax, (T, ld), jnp.uint8),
           _sds(jax, (T, ld), jnp.uint8), _sds(jax, (T, ld), f32), _sds(jax, (T, 475, ld), f32))
    call = jax.ffi.ffi_call("kbs_rollout_record", out, input_output_aliases={22: 1, 23: 2, 24: 3, 25: 4})
    res = call(*(state[k] for k, _ in STATE_ROWS), state["com_distance"], state["time"], noise["eps_jpos"], noise["eps_jvel"],
               noise["eps_gyro"], noise["eps_pg"], episode, torque_bias, rand["eps_action"], rand["u_switch"],
               rand["cmd_mode"].astype(jnp.int32), rand["cmd_u6"], rand["cmd_u_arms"], command0, pg_carry, actor_carry, critic_carry,
               lpf, done_prev.astype(jnp.uint8), **_h(np, handle, n_envs=n_envs))
    return dict(zip(names, res))


def ppo_variables(handle: int, actor_obs, critic_obs, actor_obs_mirror, critic_obs_mirror, action, done, actor_carry, critic_carry,
                  lpf, actor_mirror_carry, critic_mirror_carry, lpf_mirror, n_envs: int, actor_mirror_loss_scale: float = 1.0,
                  critic_mirror_loss_scale: float = 0.01):
    """get_ppo_variables on a stored trajectory ([T, F, ld] SoA), aux_losses included: -> (actor_carry, critic_carry, lpf,
    actor_mirror_carry, critic_mirror_carry, lpf_mirror, log_probs, values, entropy [T, ld], action_std [T, 20, ld],
    action_mirror_loss, value_mirror_loss [T, ld]); the six carries alias their inputs."""
    jax, jnp, np = _j()
    T, _, ld = actor_obs.shape
    f32 = jnp.float32
    carries = (actor_carry, critic_carry, lpf, actor_mirror_carry, critic_mirror_carry, lpf_mirror)
    out = tuple(_sds(jax, c.shape, f32) for c in carries) + (_sds(jax, (T, ld), f32),) * 3 + (_sds(jax, (T, 20, ld), f32),) + \
        (_sds(jax, (T, ld), f32),) * 2
    call = jax.ffi.ffi_call("kbs_ppo_variables", out, input_output_aliases={6: 0, 7: 1, 8: 2, 9: 3, 10: 4, 11: 5})
    return call(actor_obs, critic_obs, actor_obs_mirror, critic_obs_mirror, action, done.astype(jnp.uint8), *carries,
                **_h(np, handle, n_envs=n_envs, actor_mirror_loss_scale=float(actor_mirror_loss_scale),
                     critic_mirror_loss_scale=float(critic_mirror_loss_scale)))


def mirror_observations(handle: int, state: dict, computed, command, n_envs: int):
    """mirror_obs + mirror_cmd + concatenations for T stored steps -> (actor_obs [T, 65, ld], critic_obs [T, 475, ld], command)."""
    jax, jnp, np = _j()
    T, _, ld = computed.shape
    out = (_sds(jax, (T, 65, ld), jnp.float32), _sds(jax, (T, 475, ld), jnp.float32), _sds(jax, command.shape, jnp.float32))
    return jax.ffi.ffi_call("kbs_mirror_observations", out)(*(state[k] for k, _ in STATE_ROWS), computed, command,
                                                            **_h(np, handle, n_envs=n_envs))


def mirror_joints(handle: int, x, n_envs: int):
    jax, jnp, np = _j()
    return jax.ffi.ffi_call("kbs_mirror_joints", _sds(jax, x.shape, jnp.float32))(x, **_h(np, handle, n_envs=n_envs))


def com_distance(handle: int, geom1, geom2, pos, subtree_com_base, n_envs: int):
    """COMDistanceObservation for T steps: geom1 / geom2 s32 [T, ncon, ld], pos [T, 3 ncon, ld], subtree_com [T, 3, ld] -> [T, ld]."""
    jax, jnp, np = _j()
    T, _, ld = geom1.shape
    return jax.ffi.ffi_call("kbs_com_distance", _sds(jax, (T, ld), jnp.float32))(
        geom1.astype(jnp.int32), geom2.astype(jnp.int32), pos, subtree_com_base, **_h(np, handle, n_envs=n_envs))


def rewards(handle: int, state: dict, command, ctrl, done, t_single, airtime, prev_contact, n_envs: int):
    """get_rewards on a trajectory -> (t_single, airtime, prev_contact, total [T, ld], components [T, 12, ld])."""
    jax, jnp, np = _j()
    T, _, ld = command.shape
    f32 = jnp.float32
    out = (_sds(jax, t_single.shape, f32), _sds(jax, airtime.shape, f32), _sds(jax, prev_contact.shape, jnp.uint8),
           _sds(jax, (T, ld), f32), _sds(jax, (T, 12, ld), f32))
    call = jax.ffi.ffi_call("kbs_rewards", out, input_output_aliases={9: 0, 10: 1, 11: 2})
    return call(state["qpos"], state["qvel"], state["sensordata"], state["xpos"], state["xquat"], state["com_distance"], command, ctrl,
                done.astype(jnp.uint8), t_single, airtime, prev_contact.astype(jnp.uint8), **_h(np, handle, n_envs=n_envs))


def net_param_count(num_in: int, num_out: int, hidden: int, depth: int) -> int:
    return hidden * num_in + hidden + depth * (8 * hidden * hidden + 4 * hidden) + num_out * hidden + num_out


def ppo_grad(handle: int, batch: dict, actor_carry0, critic_carry0, lpf0, n_envs: int, hidden: int = 256, depth: int = 2):
    """Gradients of the PPO minibatch loss (kbs_ppo_grad): batch = {actor_obs [T, 65, ld], critic_obs [T, 475, ld], action,
    done, old_log_probs, advantages, value_targets, old_values} -> (grad_actor flat, grad_critic flat, log_probs, values,
    entropy [T, ld], stats [4]); flat layout = w_in, b_in, (w_ih, w_hh, b) per layer, w_out, b_out."""
    jax, jnp, np = _j()
    T, _, ld = batch["actor_obs"].shape
    f32 = jnp.float32
    out = (_sds(jax, (net_param_count(65, 40, hidden, depth),), f32), _sds(jax, (net_param_count(475, 1, hidden, depth),), f32)) + \
        (_sds(jax, (T, ld), f32),) * 3 + (_sds(jax, (4,), f32),)
    return jax.ffi.ffi_call("kbs_ppo_grad", out)(
        batch["actor_obs"], batch["critic_obs"], batch["action"], batch["done"].astype(jnp.uint8), batch["old_log_probs"],
        batch["advantages"], batch["value_targets"], batch["old_values"], actor_carry0, critic_carry0, lpf0,
        **_h(np, handle, n_envs=n_envs, hidden=hidden, depth=depth))


def ppo_variables_vjp(handle: int, batch: dict, actor_carry0, critic_carry0, lpf0, cotangents: dict, n_envs: int, hidden: int = 256,
                      depth: int = 2):
    """VJP of the PPO variables (kbs_ppo_variables_vjp), the backward rule of a jax.custom_vjp around get_ppo_variables:
    batch = {actor_obs [T, 65, ld], critic_obs [T, 475, ld], action, done}, cotangents = {log_probs, values, entropy [T, ld],
    action_std [T, 20, ld]} -> (grad_actor flat, grad_critic flat, log_probs, values, entropy [T, ld]); flat layout as ppo_grad.
    The parameter cotangent is summed over the minibatch's envs: under vmap it must not be reduced again."""
    jax, jnp, np = _j()
    T, _, ld = batch["actor_obs"].shape
    f32 = jnp.float32
    out = (_sds(jax, (net_param_count(65, 40, hidden, depth),), f32), _sds(jax, (net_param_count(475, 1, hidden, depth),), f32)) + \
        (_sds(jax, (T, ld), f32),) * 3
    return jax.ffi.ffi_call("kbs_ppo_variables_vjp", out)(
        batch["actor_obs"], batch["critic_obs"], batch["action"], batch["done"].astype(jnp.uint8), actor_carry0, critic_carry0, lpf0,
        cotangents["log_probs"], cotangents["values"], cotangents["entropy"], cotangents["action_std"],
        **_h(np, handle, n_envs=n_envs, hidden=hidden, depth=depth))


def grad_norm(handle: int, grad):
    jax, jnp, np = _j()
    return jax.ffi.ffi_call("kbs_grad_norm", _sds(jax, (1,), jnp.float32))(grad, **_h(np, handle))


def adamw_step(handle: int, param, grad, m, v, grad_norm_, step, lr: float = 5e-4, weight_decay: float = 1e-5, grad_scale: float = 1.0,
               max_grad_norm: float = 10.0):
    """optax.adamw + ksim's clip on one flat parameter vector; step = int64 [1] count of applied updates -> (param, m, v, step)."""
    jax, jnp, np = _j()
    out = (_sds(jax, param.shape, jnp.float32),) * 3 + (_sds(jax, (1,), jnp.int64),)
    call = jax.ffi.ffi_call("kbs_adamw_step", out, input_output_aliases={0: 0, 2: 1, 3: 2, 5: 3})
    return call(param, grad, m, v, grad_norm_, step, **_h(np, handle, lr=float(lr), weight_decay=float(weight_decay),
                                                          grad_scale=float(grad_scale), max_grad_norm=float(max_grad_norm)))
