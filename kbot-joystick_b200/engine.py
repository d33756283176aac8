"""Host-side driver of libkbotstep.so: torch tensors in, C-ABI calls out.

Layouts (see include/kbotstep.h): per-env fields are SoA `[F, ld]` (env contiguous, `ld` = n_envs rounded
up to a multiple of 4); trajectories are `[T, F, ld]`; recurrent carries are AoS `[depth, 2, n, H]`.
torch is plumbing only (allocation + current stream); all arithmetic happens inside the CUDA library.
"""

from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import torch

from . import _lib as L

STATE_ROWS = {"qpos": 27, "qvel": 26, "sensordata": 49, "xpos": 72, "xquat": 96, "cinert": 240, "cvel": 144,
              "actuator_force": 20, "com_distance": 1, "time": 1}
NOISE_ROWS = {"eps_jpos": 20, "eps_jvel": 20, "eps_gyro": 3, "eps_pg": 3}
EPISODE_ROWS = {"jpos_bias": 20, "pg_lag": 1, "pg_bias": 3, "kp": 20, "kd": 20, "tau_limit": 20,
                "action_bias": 20, "torque_bias": 20}
COMPUTED_OBS_ROWS = {  # rows of the `computed` block written by kbs_observations
    "biased_joint_position": (0, 20), "noisy_biased_joint_position": (20, 40), "noisy_joint_velocity": (40, 60),
    "noisy_imu_gyro": (60, 63), "feet_position": (63, 69), "projected_gravity": (69, 72),
    "imu_projected_gravity": (72, 75), "noisy_imu_projected_gravity": (75, 78)}


def round_up4(n: int) -> int:
    return (n + 3) // 4 * 4


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _view(cls, rows: dict, tensors: dict | None, ld: int | None = None, host: bool = False):
    v = cls()
    if tensors:
        for k in rows:
            t = tensors.get(k)
            if t is not None:
                setattr(v, k, L.host_ptr(t) if host else L.ptr(t))
    if ld is not None:
        v.ld = ld
    return v


def _ppo_batch(batch: dict):
    """kbs_ppo_batch over a minibatch dict ([T, F, ld] arrays; missing keys are NULL)."""
    T, _, ld = batch["actor_obs"].shape
    b = L.KbsPpoBatch()
    for k in ("actor_obs", "critic_obs", "action", "done", "old_log_probs", "advantages", "value_targets", "old_values",
              "actor_carry0", "critic_carry0", "lpf0"):
        setattr(b, k, L.ptr(batch.get(k)))
    b.T, b.ld = T, ld
    return b


def _net_grads(g: dict):
    """kbs_net_grads over an eqx-layout dict of gradient tensors."""
    s = L.KbsNetGrads()
    s.w_in, s.b_in, s.w_out, s.b_out = (L.ptr(g[k]) for k in ("w_in", "b_in", "w_out", "b_out"))
    for i, lw in enumerate(g["layers"]):
        s.w_ih[i], s.w_hh[i], s.b[i] = L.ptr(lw["w_ih"]), L.ptr(lw["w_hh"]), L.ptr(lw["b"])
    return s


@dataclass
class KbotStep:
    """One handle of the B200 control-step library bound to the current CUDA device."""

    hidden_size: int = 256
    depth: int = 2
    gemm_path: int = L.GEMM_SIMT_FP32
    overrides: dict = field(default_factory=dict)

    def __post_init__(self) -> None:
        if not torch.cuda.is_available():
            raise RuntimeError("kbot-joystick_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = L.load()
        p = L.default_params()
        p.hidden_size, p.depth, p.gemm_path = self.hidden_size, self.depth, self.gemm_path
        for k, v in self.overrides.items():
            setattr(p, k, v)
        self.params = p
        h = C.c_void_p()
        L.check(self.lib.kbs_create(C.byref(p), C.byref(h)), "kbs_create")
        self._h = h
        self._keep: list = []

    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.kbs_destroy(self._h)
            self._h = None

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self) -> int:
        return int(self.lib.kbs_launch_count(self._h))

    @property
    def handle_address(self) -> int:
        """The kbs_handle* as an integer: the `handle` attribute of the XLA-FFI calls (jax_ffi.py, csrc/kbs_xla_ffi.cc)."""
        return int(self._h.value)

    def device_status(self) -> int:
        """0 = healthy; != 0 = a dependency wait of the persistent rollout kernel timed out (synchronises)."""
        v = C.c_int(0)
        L.check(self.lib.kbs_device_status(self._h, C.byref(v)), "kbs_device_status")
        return int(v.value)

    def device_status_reset(self) -> None:
        L.check(self.lib.kbs_device_status_reset(self._h), "kbs_device_status_reset")

    def scratch_lock(self, on: bool) -> None:
        """While locked, a call that would have to reallocate the library's scratch fails instead (CUDA-graph safety)."""
        L.check(self.lib.kbs_scratch_lock(self._h, 1 if on else 0), "kbs_scratch_lock")

    def profile(self, on: bool) -> None:
        L.check(self.lib.kbs_profile_enable(self._h, 1 if on else 0), "kbs_profile_enable")

    def profile_read(self) -> dict:
        """{kernel name: (total ms, launches)} for the launches made while profiling was enabled."""
        ms = (C.c_double * L.NUM_KERNEL_IDS)()
        cnt = (C.c_int64 * L.NUM_KERNEL_IDS)()
        rc = self.lib.kbs_profile_read(self._h, L.NUM_KERNEL_IDS, ms, cnt)
        if rc not in (0, 1):
            L.check(rc, "kbs_profile_read")
        out = {self.lib.kbs_kernel_name(i).decode(): (ms[i], int(cnt[i])) for i in range(L.NUM_KERNEL_IDS) if cnt[i]}
        out["_overflow"] = bool(rc)
        return out

    # ---- weights -------------------------------------------------------------------------------------
    def pack_weights(self, net: int, w: dict, sync: bool = True) -> None:
        """w: eqx-layout CUDA tensors {w_in,b_in,w_out,b_out, layers:[{w_ih,w_hh,b}]} (train.py:847-1004).  sync=False: only
        enqueue (stream-ordered; required inside CUDA-graph capture)."""
        s = L.KbsNetWeights()
        s.w_in, s.b_in, s.w_out, s.b_out = (L.ptr(w[k]) for k in ("w_in", "b_in", "w_out", "b_out"))
        for i, lw in enumerate(w["layers"]):
            s.w_ih[i], s.w_hh[i], s.b[i] = L.ptr(lw["w_ih"]), L.ptr(lw["w_hh"]), L.ptr(lw["b"])
        L.check(self.lib.kbs_weights_pack(self._h, net, C.byref(s), _stream()), "kbs_weights_pack")
        if sync:
            torch.cuda.current_stream().synchronize()

    # ---- stages --------------------------------------------------------------------------------------
    def observations(self, state: dict, command, noise: dict | None = None, episode: dict | None = None,
                     pg_carry=None, computed=None, actor_obs=None, critic_obs=None, n_envs: int | None = None,
                     pg_reset=None):
        ld = state["qpos"].shape[-1]
        n = n_envs or ld
        sv = _view(L.KbsStateView, STATE_ROWS, state, ld)
        nv = _view(L.KbsNoiseView, NOISE_ROWS, noise)
        ev = _view(L.KbsEpisodeView, EPISODE_ROWS, episode)
        L.check(self.lib.kbs_observations(self._h, C.byref(sv), C.byref(nv), C.byref(ev), L.ptr(command),
                                          L.ptr(pg_carry), L.ptr(pg_reset), L.ptr(computed), L.ptr(actor_obs),
                                          L.ptr(critic_obs), n,
                                          _stream()), "kbs_observations")

    def ppo_loss(self, log_probs, old_log_probs, advantages, values, old_values, value_targets, entropy,
                 per_step=None, n_envs: int | None = None, **hyper) -> torch.Tensor:
        """ksim.compute_ppo_loss on [T, ld] arrays -> device tensor [loss, mean policy, mean value, mean entropy].
        hyper: clip_param, value_loss_coef, entropy_coef, log_clip_value, use_clipped_value_loss (kbs_ppo_loss_params)."""
        T, ld = log_probs.shape
        lp = L.KbsPpoLossParams()
        L.check(self.lib.kbs_ppo_loss_default_params(C.byref(lp)), "kbs_ppo_loss_default_params")
        for k, v in hyper.items():
            setattr(lp, k, v)
        out = torch.empty((4,), device=log_probs.device)
        io = L.KbsPpoLossIO()
        io.log_probs, io.old_log_probs, io.advantages = L.ptr(log_probs), L.ptr(old_log_probs), L.ptr(advantages)
        io.values, io.old_values, io.value_targets = L.ptr(values), L.ptr(old_values), L.ptr(value_targets)
        io.entropy, io.per_step, io.out = L.ptr(entropy), L.ptr(per_step), L.ptr(out)
        io.T, io.ld = T, ld
        L.check(self.lib.kbs_ppo_loss(self._h, C.byref(lp), C.byref(io), n_envs or ld, _stream()), "kbs_ppo_loss")
        return out

    def ppo_grad(self, batch: dict, grads_actor: dict, grads_critic: dict, n_envs: int | None = None, critic_ready=None,
                 **hyper) -> dict:
        """Gradients of the PPO minibatch loss (kbs_ppo_grad).  batch: actor_obs [T,65,ld], critic_obs [T,475,ld],
        action [T,20,ld], done u8 [T,ld], old_log_probs / advantages / value_targets / old_values [T,ld], optional
        actor_carry0 / critic_carry0 [depth,2,n,H], lpf0 [20,ld].  grads_*: eqx-layout dicts of CUDA tensors (written).
        Returns {"stats": [loss, policy, value, entropy] (device), "log_probs", "values", "entropy": [T, ld]}."""
        T, _, ld = batch["actor_obs"].shape
        dev = batch["actor_obs"].device
        lp = L.KbsPpoLossParams()
        L.check(self.lib.kbs_ppo_loss_default_params(C.byref(lp)), "kbs_ppo_loss_default_params")
        for k, v in hyper.items():
            setattr(lp, k, v)
        b = _ppo_batch(batch)
        ga, gc = _net_grads(grads_actor), _net_grads(grads_critic)
        # critic_ready: a torch.cuda.Event the library records on the stream once the critic's gradients are final (its
        # all-reduce can then overlap the actor's weight-gradient GEMMs)
        L.check(self.lib.kbs_ppo_grad_set_events(self._h, critic_ready.cuda_event if critic_ready is not None else None),
                "kbs_ppo_grad_set_events")
        out = {"stats": torch.empty((4,), device=dev), "log_probs": torch.empty((T, ld), device=dev),
               "values": torch.empty((T, ld), device=dev), "entropy": torch.empty((T, ld), device=dev)}
        L.check(self.lib.kbs_ppo_grad(self._h, C.byref(lp), C.byref(b), C.byref(ga), C.byref(gc), L.ptr(out["log_probs"]),
                                      L.ptr(out["values"]), L.ptr(out["entropy"]), L.ptr(out["stats"]), n_envs or ld, _stream()),
                "kbs_ppo_grad")
        return out

    def ppo_variables_vjp(self, batch: dict, cotangents: dict, grads_actor: dict, grads_critic: dict, n_envs: int | None = None,
                          critic_ready=None) -> dict:
        """Vector-Jacobian product of the PPO variables (kbs_ppo_variables_vjp): grads_* (written, eqx layout) = the gradient
        of sum(ct * var) over the minibatch for cotangents {"log_probs", "values", "entropy": [T, ld], "action_std":
        [T, 20, ld]} (a missing key is a zero cotangent), through the same forward and BPTT as ppo_grad.  batch as for
        ppo_grad; old_log_probs / advantages / value_targets / old_values are not read.  critic_ready as for ppo_grad.
        Returns the forward's {"log_probs", "values", "entropy": [T, ld]}."""
        T, _, ld = batch["actor_obs"].shape
        dev = batch["actor_obs"].device
        b = _ppo_batch(batch)
        ct = L.KbsPpoCotangents()
        for k in ("log_probs", "values", "entropy", "action_std"):
            setattr(ct, k, L.ptr(cotangents.get(k)))
        ga, gc = _net_grads(grads_actor), _net_grads(grads_critic)
        L.check(self.lib.kbs_ppo_grad_set_events(self._h, critic_ready.cuda_event if critic_ready is not None else None),
                "kbs_ppo_grad_set_events")
        out = {k: torch.empty((T, ld), device=dev) for k in ("log_probs", "values", "entropy")}
        L.check(self.lib.kbs_ppo_variables_vjp(self._h, C.byref(b), C.byref(ct), C.byref(ga), C.byref(gc),
                                               L.ptr(out["log_probs"]), L.ptr(out["values"]), L.ptr(out["entropy"]),
                                               n_envs or ld, _stream()), "kbs_ppo_variables_vjp")
        return out

    def adam_step(self, param, grad, m, v, step: int, lr=5e-4, b1=0.9, b2=0.999, eps=1e-8, grad_scale=1.0) -> None:
        """optax.adam on one flat parameter tensor (train.py:1057-1063)."""
        L.check(self.lib.kbs_adam_step(self._h, L.ptr(param), L.ptr(grad), L.ptr(m), L.ptr(v), param.numel(), lr, b1, b2, eps,
                                       grad_scale, step, _stream()), "kbs_adam_step")

    def grad_norm(self, grad, out=None):
        """optax.global_norm of one flat gradient tensor -> device tensor [1] (deterministic, double accumulation)."""
        if out is None:
            out = torch.empty((1,), device=grad.device)
        L.check(self.lib.kbs_grad_norm(self._h, L.ptr(grad), grad.numel(), L.ptr(out), _stream()), "kbs_grad_norm")
        return out

    def adamw_step(self, param, grad, m, v, step: int = 0, grad_norm=None, step_dev=None, **opt) -> None:
        """optax.adamw (train.py:1064-1065) + ksim's global-norm clip / non-finite skip [U] on one flat parameter tensor.
        opt: lr, b1, b2, eps, weight_decay, grad_scale, max_grad_norm (kbs_adamw_params; defaults = the launch config).
        step_dev: device int64 [1] counter of applied updates (advanced here) or None -> `step` (>= 1) is used."""
        o = L.KbsAdamwParams()
        L.check(self.lib.kbs_adamw_default_params(C.byref(o)), "kbs_adamw_default_params")
        for k, val in opt.items():
            setattr(o, k, val)
        L.check(self.lib.kbs_adamw_step(self._h, L.ptr(param), L.ptr(grad), L.ptr(m), L.ptr(v), param.numel(), C.byref(o),
                                        L.ptr(grad_norm), L.ptr(step_dev), step, _stream()), "kbs_adamw_step")

    def minibatch_permutation(self, pass_dev, n_envs: int, seed: int = 0, env0: int = 0, out=None):
        """A uniform random permutation of the env axis (kbs_minibatch_permutation) -> int32 [n_envs] on the device.
        pass_dev: device int64 [1] pass counter (read, then advanced by one); env0: the rank's global env offset."""
        if out is None:
            out = torch.empty((n_envs,), dtype=torch.int32, device=pass_dev.device)
        L.check(self.lib.kbs_minibatch_permutation(self._h, seed, L.ptr(pass_dev), env0, L.ptr(out), n_envs, _stream()),
                "kbs_minibatch_permutation")
        return out

    MINIBATCH_FIELDS = ("actor_obs", "critic_obs", "action", "done", "old_log_probs", "advantages", "value_targets",
                        "old_values", "actor_carry0", "critic_carry0", "lpf0")

    def minibatch_buffers(self, T: int, num_batches: int, batch_size: int, device) -> dict:
        """Uninitialised destination of shuffle_minibatches, start carries included."""
        e = lambda *s, dt=torch.float32: torch.empty((num_batches,) + s, dtype=dt, device=device)
        dst = {"actor_obs": e(T, L.ACTOR_OBS, batch_size), "critic_obs": e(T, L.CRITIC_OBS, batch_size),
               "action": e(T, L.NUM_JOINTS, batch_size), "done": e(T, batch_size, dt=torch.uint8)}
        for k in ("old_log_probs", "advantages", "value_targets", "old_values"):
            dst[k] = e(T, batch_size)
        for k in ("actor_carry0", "critic_carry0"):
            dst[k] = e(self.depth, 2, batch_size, self.hidden_size)
        dst["lpf0"] = e(L.NUM_JOINTS, batch_size)
        return dst

    def shuffle_minibatches(self, perm, src: dict, n_envs: int, batch_size: int, dst: dict | None = None) -> dict:
        """The rollout `src` (a ppo_grad batch over all n_envs trajectories at its ld) cut into n_envs / batch_size dense
        minibatches (kbs_shuffle_minibatches): column j of minibatch b is env perm[b * batch_size + j].  dst (allocated when
        None): every array [B, T, F, batch_size] ([B, T, batch_size] for the [T, ld] fields), carries [B, depth, 2,
        batch_size, H], lpf0 [B, 20, batch_size]; the carries are present where src has them."""
        T, _, ld = src["actor_obs"].shape
        if dst is None:
            dst = self.minibatch_buffers(T, n_envs // batch_size, batch_size, src["actor_obs"].device)
            dst = {k: t for k, t in dst.items() if not k.endswith("0") or src.get(k) is not None}
        s, d = L.KbsPpoBatch(), L.KbsPpoMinibatches()
        for k in self.MINIBATCH_FIELDS:
            setattr(s, k, L.ptr(src.get(k)))
            setattr(d, k, L.ptr(dst.get(k)))
        s.T, s.ld = T, ld
        d.batch_size, d.num_batches = batch_size, dst["actor_obs"].shape[0]
        L.check(self.lib.kbs_shuffle_minibatches(self._h, L.ptr(perm), C.byref(s), C.byref(d), n_envs, _stream()),
                "kbs_shuffle_minibatches")
        return dst

    def sample_actuator_randomization(self, u, episode: dict, reset=None, n_envs: int | None = None, **scales) -> None:
        """Per-episode PositionActuators randomisation (train.py:1097-1105): u [5, 20, ld] uniforms -> episode["kp"], ["kd"],
        ["tau_limit"], ["action_bias"], ["torque_bias"] ([20, ld] each, written where reset != 0 / everywhere)."""
        ld = u.shape[-1]
        rp = L.KbsActuatorRandParams()
        L.check(self.lib.kbs_actuator_rand_default_params(C.byref(rp)), "kbs_actuator_rand_default_params")
        for k, val in scales.items():
            setattr(rp, k, val)
        ev = _view(L.KbsEpisodeView, EPISODE_ROWS, episode)
        L.check(self.lib.kbs_sample_actuator_randomization(self._h, C.byref(rp), L.ptr(u), L.ptr(reset), C.byref(ev), ld,
                                                           n_envs or ld, _stream()), "kbs_sample_actuator_randomization")

    def com_distance(self, geom1, geom2, pos, subtree_com_base, out=None, n_envs: int | None = None):
        """COMDistanceObservation (train.py:509-659) for T steps: geom1/geom2 int32 [T, ncon, ld], pos [T, 3 ncon, ld],
        subtree_com_base [T, 3, ld] -> [T, ld]."""
        T, ncon, ld = geom1.shape
        if out is None:
            out = torch.empty((T, ld), device=pos.device)
        L.check(self.lib.kbs_com_distance(self._h, L.ptr(geom1), L.ptr(geom2), L.ptr(pos), L.ptr(subtree_com_base), L.ptr(out),
                                          ncon, T, ld, n_envs or ld, _stream()), "kbs_com_distance")
        return out

    def upload_state(self, host_state: dict, dev_state: dict, stream: int | None = None) -> int:
        """Enqueue the H2D copy of T recorded steps ([T][rows][ld] per array; host tensors pinned): only the rows the path
        reads (kbs_upload_state).  Returns the bytes enqueued."""
        T, ld = dev_state["qpos"].shape[0], dev_state["qpos"].shape[-1]
        hv = _view(L.KbsStateView, STATE_ROWS, host_state, ld, host=True)
        dv = _view(L.KbsStateView, STATE_ROWS, dev_state, ld)
        n = C.c_int64(0)
        L.check(self.lib.kbs_upload_state(self._h, C.byref(hv), C.byref(dv), T, C.byref(n),
                                          _stream() if stream is None else stream), "kbs_upload_state")
        return int(n.value)

    def mirror_observations(self, state: dict, computed, command, actor_obs=None, critic_obs=None, command_out=None,
                            n_envs: int | None = None) -> None:
        """mirror_obs / mirror_cmd + the actor / critic concatenations (train.py:1463-1481, 1584-1756) for T stored steps:
        every array is time-major [T][rows][ld]."""
        T, ld = computed.shape[0], computed.shape[-1]
        sv = _view(L.KbsStateView, STATE_ROWS, state, ld)
        L.check(self.lib.kbs_mirror_observations(self._h, C.byref(sv), L.ptr(computed), L.ptr(command), L.ptr(actor_obs),
                                                 L.ptr(critic_obs), L.ptr(command_out), T, n_envs or ld, _stream()),
                "kbs_mirror_observations")

    def mirror_joints(self, x, out=None, n_envs: int | None = None):
        """mirror_joints (train.py:1574-1582) on [T][20][ld] (or [20][ld])."""
        ld = x.shape[-1]
        T = x.shape[0] if x.dim() == 3 else 1
        if out is None:
            out = torch.empty_like(x)
        L.check(self.lib.kbs_mirror_joints(self._h, L.ptr(x), L.ptr(out), T, ld, n_envs or ld, _stream()), "kbs_mirror_joints")
        return out

    def command_update(self, command, mode, u6, u_arms, u_switch=None, n_envs: int | None = None) -> None:
        ld = command.shape[-1]
        L.check(self.lib.kbs_command_update(self._h, L.ptr(command), L.ptr(u_switch), L.ptr(mode), L.ptr(u6),
                                            L.ptr(u_arms), ld, n_envs or ld, _stream()), "kbs_command_update")

    def actor_step(self, obs, carry, lpf, eps=None, action_in=None, done=None, out: dict | None = None,
                   n_envs: int | None = None) -> dict:
        ld = obs.shape[-1]
        n = n_envs or ld
        if out is None:
            out = {k: torch.empty((20, ld), device=obs.device) for k in ("action", "mean", "std")}
            out["log_prob"] = torch.empty((ld,), device=obs.device)
            out["entropy"] = torch.empty((ld,), device=obs.device)
        o = L.KbsActorOut()
        for k in ("action", "mean", "std", "log_prob", "entropy"):
            setattr(o, k, L.ptr(out.get(k)))
        L.check(self.lib.kbs_actor_step(self._h, L.ptr(obs), ld, L.ptr(carry), L.ptr(lpf), L.ptr(eps),
                                        L.ptr(action_in), L.ptr(done), C.byref(o), n, _stream()), "kbs_actor_step")
        return out

    def critic_step(self, obs, carry, done=None, value=None, n_envs: int | None = None):
        ld = obs.shape[-1]
        if value is None:
            value = torch.empty((ld,), device=obs.device)
        L.check(self.lib.kbs_critic_step(self._h, L.ptr(obs), ld, L.ptr(carry), L.ptr(done), L.ptr(value),
                                         n_envs or ld, _stream()), "kbs_critic_step")
        return value

    def torque(self, action, state: dict, episode: dict | None = None, ctrl=None, n_envs: int | None = None):
        ld = action.shape[-1]
        if ctrl is None:
            ctrl = torch.empty_like(action)
        sv = _view(L.KbsStateView, STATE_ROWS, state, ld)
        ev = _view(L.KbsEpisodeView, EPISODE_ROWS, episode)
        L.check(self.lib.kbs_torque(self._h, L.ptr(action), C.byref(sv), C.byref(ev), L.ptr(ctrl), n_envs or ld,
                                    _stream()), "kbs_torque")
        return ctrl

    def torque_substeps(self, action, prev_action, u_drop, latency, q_sub, qd_sub, episode: dict | None = None, ctrl=None,
                        sub_dt: float = 0.004, drop_prob: float = 0.05, n_envs: int | None = None):
        """Per-physics-sub-step actuator path (latency / dropped commands, train.py:1775-1781): q_sub / qd_sub [S, 20, ld]
        -> ctrl [S, 20, ld]; prev_action [20, ld] is updated in place to the action that was applied."""
        S, _, ld = q_sub.shape
        if ctrl is None:
            ctrl = torch.empty_like(q_sub)
        ev = _view(L.KbsEpisodeView, EPISODE_ROWS, episode)
        L.check(self.lib.kbs_torque_substeps(self._h, L.ptr(action), L.ptr(prev_action), L.ptr(u_drop), L.ptr(latency),
                                             L.ptr(q_sub), L.ptr(qd_sub), C.byref(ev), L.ptr(ctrl), S, sub_dt, drop_prob, ld,
                                             n_envs or ld, _stream()), "kbs_torque_substeps")
        return ctrl

    def terminate(self, state: dict, n_envs: int | None = None, want_pre: bool = False) -> dict:
        ld = state["qpos"].shape[-1]
        dev = state["qpos"].device
        out = {"codes": torch.empty((3, ld), dtype=torch.int32, device=dev),
               "done": torch.empty((ld,), dtype=torch.uint8, device=dev),
               "success": torch.empty((ld,), dtype=torch.uint8, device=dev),
               "pre": torch.empty((2, ld), device=dev) if want_pre else None}
        sv = _view(L.KbsStateView, STATE_ROWS, state, ld)
        L.check(self.lib.kbs_terminate(self._h, C.byref(sv), L.ptr(out["codes"]), L.ptr(out["done"]),
                                       L.ptr(out["success"]), L.ptr(out["pre"]), n_envs or ld, _stream()),
                "kbs_terminate")
        return out

    def rewards(self, traj_state: dict, command, ctrl, done, carry: dict, total=None, components=None,
                n_envs: int | None = None):
        T, _, ld = command.shape
        tv = L.KbsTrajView()
        tv.state = _view(L.KbsStateView, STATE_ROWS, traj_state, ld)
        tv.command, tv.ctrl, tv.done, tv.T = L.ptr(command), L.ptr(ctrl), L.ptr(done), T
        cv = L.KbsRewardCarry()
        cv.t_single, cv.airtime, cv.prev_contact = (L.ptr(carry[k]) for k in ("t_single", "airtime", "prev_contact"))
        if total is None:
            total = torch.empty((T, ld), device=command.device)
        L.check(self.lib.kbs_rewards(self._h, C.byref(tv), C.byref(cv), L.ptr(total), L.ptr(components),
                                     n_envs or ld, _stream()), "kbs_rewards")
        return total

    def gae(self, values, rewards, done, success, adv=None, targets=None, n_envs: int | None = None):
        T, ld = values.shape
        adv = torch.empty_like(values) if adv is None else adv
        targets = torch.empty_like(values) if targets is None else targets
        L.check(self.lib.kbs_gae(self._h, L.ptr(values), L.ptr(rewards), L.ptr(done), L.ptr(success), L.ptr(adv),
                                 L.ptr(targets), T, ld, n_envs or ld, _stream()), "kbs_gae")
        return adv, targets

    def policy_step(self, joint_angles, joint_vel, projected_gravity, gyro, command, carry):
        n = joint_angles.shape[0]
        carry_out = torch.empty_like(carry)
        action = torch.empty((n, 20), device=carry.device)
        L.check(self.lib.kbs_policy_step(self._h, L.ptr(joint_angles), L.ptr(joint_vel), L.ptr(projected_gravity),
                                         L.ptr(gyro), L.ptr(command), L.ptr(carry), L.ptr(carry_out), L.ptr(action),
                                         n, _stream()), "kbs_policy_step")
        return action, carry_out

    def ppo_variables(self, actor_obs, action, done, actor_carry, lpf, critic_obs=None, critic_carry=None,
                      want_std: bool = True, want_mean: bool = False, n_envs: int | None = None, mirror: dict | None = None) -> dict:
        """get_ppo_variables on a stored trajectory (train.py:1510-1524): returns log_probs/values/entropy/action_std.
        mirror (aux_losses, train.py:1462-1481): {"actor_obs", "critic_obs" (mirrored concatenations from
        mirror_observations), "actor_carry", "critic_carry", "lpf" (the *_mirror carries, in/out), "actor_scale",
        "critic_scale"} -> out["action_mirror_loss"], out["value_mirror_loss"] [T, ld]."""
        T, _, ld = actor_obs.shape
        dev = actor_obs.device
        out = {"log_probs": torch.empty((T, ld), device=dev), "entropy": torch.empty((T, ld), device=dev),
               "values": torch.empty((T, ld), device=dev) if critic_obs is not None else None,
               "action_std": torch.empty((T, 20, ld), device=dev) if want_std else None,
               "mean": torch.empty((T, 20, ld), device=dev) if want_mean else None}
        io = L.KbsPpoIO()
        if mirror is not None:
            out["action_mirror_loss"] = torch.empty((T, ld), device=dev)
            out["value_mirror_loss"] = torch.empty((T, ld), device=dev) if mirror.get("critic_obs") is not None else None
            io.actor_obs_mirror, io.critic_obs_mirror = L.ptr(mirror["actor_obs"]), L.ptr(mirror.get("critic_obs"))
            io.actor_mirror_carry, io.critic_mirror_carry = L.ptr(mirror["actor_carry"]), L.ptr(mirror.get("critic_carry"))
            io.lpf_mirror = L.ptr(mirror["lpf"])
            io.action_mirror_loss, io.value_mirror_loss = L.ptr(out["action_mirror_loss"]), L.ptr(out["value_mirror_loss"])
            io.actor_mirror_loss_scale = mirror.get("actor_scale", 1.0)       # train.py:115-122 defaults (launch: 0.0)
            io.critic_mirror_loss_scale = mirror.get("critic_scale", 0.01)
        io.actor_obs, io.critic_obs, io.action, io.done = L.ptr(actor_obs), L.ptr(critic_obs), L.ptr(action), L.ptr(done)
        io.actor_carry, io.critic_carry, io.lpf = L.ptr(actor_carry), L.ptr(critic_carry), L.ptr(lpf)
        io.log_probs, io.values, io.entropy = L.ptr(out["log_probs"]), L.ptr(out["values"]), L.ptr(out["entropy"])
        io.action_std, io.mean = L.ptr(out["action_std"]), L.ptr(out["mean"])
        io.T, io.ld = T, ld
        L.check(self.lib.kbs_ppo_variables(self._h, C.byref(io), n_envs or ld, _stream()), "kbs_ppo_variables")
        return out

    def generate_rollout_noise(self, io: dict, n_envs: int, seed: int, step0: int = 0) -> None:
        """Fill the randomness of a kbs_rollout_io (io["noise"], eps_action, u_switch, cmd_mode, cmd_u6, cmd_u_arms) on the device
        with counter-based Philox draws (kbs_generate_rollout_noise): what jax.random does inside the reference's jitted rollout.
        Parity tests pass these arrays explicitly instead."""
        ld = io["u_switch"].shape[-1]
        T = io["u_switch"].shape[0]
        nv = _view(L.KbsNoiseView, NOISE_ROWS, io.get("noise"))
        L.check(self.lib.kbs_generate_rollout_noise(self._h, seed, step0, C.byref(nv), L.ptr(io.get("eps_action")), L.ptr(io.get("u_switch")),
                                                    L.ptr(io.get("cmd_mode")), L.ptr(io.get("cmd_u6")), L.ptr(io.get("cmd_u_arms")), T, ld,
                                                    n_envs, _stream()), "kbs_generate_rollout_noise")

    def rollout(self, io: dict, n_envs: int) -> None:
        """io: tensors named as the fields of kbs_rollout_io (state/noise/episode are nested dicts).  With io["done_prev"]
        (u8 [ld], the previous call's done[T-1]) or io["critic_obs"] ([T, 475, ld], written) present and not None, the call
        is kbs_rollout_record: the lag state restarts on step 0 where done_prev != 0, and every step's critic concatenation
        is recorded."""
        r = L.KbsRolloutIO()
        ld = io["state"]["qpos"].shape[-1]
        r.state = _view(L.KbsStateView, STATE_ROWS, io["state"], ld)
        r.noise = _view(L.KbsNoiseView, NOISE_ROWS, io.get("noise"))
        r.episode = _view(L.KbsEpisodeView, EPISODE_ROWS, io.get("episode"))
        for k, _ in L.KbsRolloutIO._fields_:
            if k in ("state", "noise", "episode", "T"):
                continue
            setattr(r, k, L.ptr(io.get(k)))
        r.T = io["T"]
        if io.get("done_prev") is None and io.get("critic_obs") is None:
            L.check(self.lib.kbs_rollout(self._h, C.byref(r), n_envs, _stream()), "kbs_rollout")
            return
        rec = L.KbsRolloutRecord(L.ptr(io.get("done_prev")), L.ptr(io.get("critic_obs")))
        L.check(self.lib.kbs_rollout_record(self._h, C.byref(r), C.byref(rec), n_envs, _stream()), "kbs_rollout_record")

    # ---- the online rollout: one control step per call ----------------------------------------------------------------------
    def step_state(self, n_envs: int, with_critic: bool = True, carry: dict | None = None) -> "StepState":
        """A device step state for n_envs (kbs_step_state): the carries in the kernels' own layouts, lpf, pg_carry, the command,
        done_prev and the step index, loaded from `carry` (see step_state_load; None = zeros)."""
        nb = C.c_uint64(0)
        L.check(self.lib.kbs_step_state_bytes(self._h, n_envs, 1 if with_critic else 0, C.byref(nb)), "kbs_step_state_bytes")
        buf = torch.empty((int(nb.value),), dtype=torch.uint8, device=torch.device("cuda", torch.cuda.current_device()))
        st = StepState(buf, L.KbsStepState(buf.data_ptr(), int(nb.value), n_envs, 1 if with_critic else 0))
        self.step_state_load(st, carry or {})
        return st

    def step_state_load(self, st: "StepState", carry: dict) -> None:
        """carry: any of actor_carry / critic_carry [depth,2,n,H], lpf [20,ld], pg_carry [3,ld], command [16,ld], done_prev u8
        [ld] (missing = zeros).  The step index becomes 0."""
        c = L.KbsStepCarry(*(L.ptr(carry.get(k)) for k, _ in L.KbsStepCarry._fields_))
        L.check(self.lib.kbs_step_state_load(self._h, C.byref(st.desc), C.byref(c), _stream()), "kbs_step_state_load")

    def step_state_store(self, st: "StepState", out: dict) -> dict:
        """Write the state's carries into the tensors of `out` (same keys as step_state_load; missing = not written)."""
        c = L.KbsStepCarry(*(L.ptr(out.get(k)) for k, _ in L.KbsStepCarry._fields_))
        L.check(self.lib.kbs_step_state_store(self._h, C.byref(st.desc), C.byref(c), _stream()), "kbs_step_state_store")
        return out

    def step_state_rewind(self, st: "StepState") -> None:
        """Step index back to 0; nothing else changes."""
        L.check(self.lib.kbs_step_state_rewind(self._h, C.byref(st.desc), _stream()), "kbs_step_state_rewind")

    def rollout_step(self, st: "StepState", io: dict) -> None:
        """One control step (kbs_rollout_step).  io: state / noise / episode (dicts of this step's [F, ld] tensors), eps_action,
        u_switch, cmd_mode, cmd_u6, cmd_u_arms of this step; trajectories command [T+1,16,ld], actor_obs, critic_obs, action,
        log_prob, ctrl, term_codes, done, success, value ([T, ..., ld]; optional ones may be missing or None) and traj_state
        (dict of [T, F, ld] tensors recording this step's state fields).  Slot t = the state's device step index."""
        r = L.KbsStepIO()
        ld = io["state"]["qpos"].shape[-1]
        r.state = _view(L.KbsStateView, STATE_ROWS, io["state"], ld)
        r.noise = _view(L.KbsNoiseView, NOISE_ROWS, io.get("noise"))
        r.episode = _view(L.KbsEpisodeView, EPISODE_ROWS, io.get("episode"))
        r.traj_state = _view(L.KbsStateView, STATE_ROWS, io.get("traj_state"), ld)
        for k, _ in L.KbsStepIO._fields_:
            if k not in ("state", "noise", "episode", "traj_state", "T"):
                setattr(r, k, L.ptr(io.get(k)))
        r.T = io["command"].shape[0] - 1 if io.get("command") is not None else 0
        L.check(self.lib.kbs_rollout_step(self._h, C.byref(st.desc), C.byref(r), _stream()), "kbs_rollout_step")

    # ---- the physics sub-steps between two online control steps ---------------------------------------------------------------
    def actuator_state(self, n_envs: int, n_substeps: int, prev_action=None) -> "ActuatorState":
        """A device actuator state for n_envs and n_substeps sub-steps per control step (kbs_actuator_state): the sub-step index,
        the last applied action and this control step's latched one, loaded from prev_action [20, ld] (None = zeros)."""
        nb = C.c_uint64(0)
        L.check(self.lib.kbs_actuator_state_bytes(self._h, n_envs, C.byref(nb)), "kbs_actuator_state_bytes")
        buf = torch.empty((int(nb.value),), dtype=torch.uint8, device=torch.device("cuda", torch.cuda.current_device()))
        ast = ActuatorState(buf, L.KbsActuatorState(buf.data_ptr(), int(nb.value), n_envs, n_substeps))
        self.actuator_state_load(ast, prev_action)
        return ast

    def actuator_state_load(self, ast: "ActuatorState", prev_action=None) -> None:
        """prev_action [20, ld] (None = zeros); the sub-step index becomes 0."""
        L.check(self.lib.kbs_actuator_state_load(self._h, C.byref(ast.desc), L.ptr(prev_action), _stream()),
                "kbs_actuator_state_load")

    def actuator_state_store(self, ast: "ActuatorState", prev_action=None):
        """The state's last applied action, written into prev_action [20, ld] (allocated when None) and returned."""
        if prev_action is None:
            prev_action = torch.empty((L.NUM_JOINTS, round_up4(ast.desc.n_envs)), device=ast.buf.device)
        L.check(self.lib.kbs_actuator_state_store(self._h, C.byref(ast.desc), L.ptr(prev_action), _stream()),
                "kbs_actuator_state_store")
        return prev_action

    def actuator_substep(self, st: "StepState", ast: "ActuatorState", io_k: dict) -> None:
        """One physics sub-step after the control step st just ran (kbs_actuator_substep).  io_k: action [T, 20, ld] (the
        trajectory the steps record), u_drop / latency [ld] of this control step, qpos [27, ld] / qvel [26, ld] of this sub-step,
        episode (dict of [F, ld] tensors, optional), ctrl [20, ld] (written); sub_dt / drop_prob (default 0.004 / 0.05).  The
        sub-step index and the step index are read on the device."""
        r = L.KbsSubstepIO()
        for k in ("action", "u_drop", "latency", "qpos", "qvel", "ctrl"):
            setattr(r, k, L.ptr(io_k.get(k)))
        r.T = io_k["action"].shape[0] if io_k.get("action") is not None else 0
        r.episode = _view(L.KbsEpisodeView, EPISODE_ROWS, io_k.get("episode"))
        r.sub_dt, r.drop_prob = io_k.get("sub_dt", 0.004), io_k.get("drop_prob", 0.05)
        L.check(self.lib.kbs_actuator_substep(self._h, C.byref(st.desc), C.byref(ast.desc), C.byref(r), _stream()),
                "kbs_actuator_substep")


@dataclass
class StepState:
    """A step state's device buffer and its kbs_step_state descriptor (keeps the buffer alive)."""

    buf: torch.Tensor
    desc: L.KbsStepState


@dataclass
class ActuatorState:
    """An actuator state's device buffer and its kbs_actuator_state descriptor (keeps the buffer alive)."""

    buf: torch.Tensor
    desc: L.KbsActuatorState
