"""ctypes binding of libkbotstep.so (include/kbotstep.h).

PyTorch is used only for device memory and streams; every compute call goes through the C-ABI.  There is no
CPU fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""

from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["KBS_LIB_PATH"]) if os.environ.get("KBS_LIB_PATH") else _PKG_DIR / "libkbotstep.so"   # override: A/B builds

NUM_JOINTS = 20
NUM_COMMANDS = 16
ACTOR_OBS = 65
CRITIC_OBS = 475
MAX_DEPTH = 4
NUM_REWARDS = 12
NET_ACTOR, NET_CRITIC = 0, 1
GEMM_TC_3XTF32, GEMM_SIMT_FP32, GEMM_TC_2XF16 = 0, 1, 2

_f, _i32, _i64, _vp = C.c_float, C.c_int32, C.c_int64, C.c_void_p


class KbsParams(C.Structure):
    _fields_ = [
        ("hidden_size", _i32), ("depth", _i32), ("gemm_path", _i32), ("normalize_advantages", _i32),
        ("ctrl_dt", _f), ("min_std", _f), ("max_std", _f), ("var_scale", _f), ("lpf_alpha", _f),
        ("gamma", _f), ("lam", _f), ("adv_eps", _f),
        ("jpos_noise_mag", _f), ("jvel_noise_mag", _f), ("gyro_noise_std", _f), ("pg_noise_std", _f),
        ("gravity", _f), ("eps_quat", _f),
        ("unhealthy_z", _f), ("max_tilt", _f), ("max_length_sec", _f), ("switch_prob", _f),
        ("cmd_lo", _f * 6), ("cmd_hi", _f * 6),
        ("joint_bias", _f * 20), ("joint_range", _f * 20), ("arm_lo", _f * 10), ("arm_hi", _f * 10),
        ("kp", _f * 20), ("kd", _f * 20), ("ctrl_limit", _f * 20), ("reward_scale", _f * 12),
        ("linvel_es", _f), ("angvel_es", _f), ("rp_es", _f), ("rp_es_zero", _f), ("bh_es", _f),
        ("bh_standard", _f), ("bh_foot_origin", _f), ("arm_es", _f), ("grace_period", _f),
        ("touchdown_penalty", _f), ("feet_es", _f), ("com_es", _f), ("acc_es", _f), ("torque_es", _f),
        ("body_base", _i32), ("body_lfoot", _i32), ("body_rfoot", _i32),
        ("sd_gyro", _i32), ("sd_imu_quat", _i32), ("sd_touch_l", _i32), ("sd_touch_r", _i32),
    ]


class KbsStateView(C.Structure):
    _fields_ = [(k, _vp) for k in ("qpos", "qvel", "sensordata", "xpos", "xquat", "cinert", "cvel",
                                   "actuator_force", "com_distance", "time")] + [("ld", _i64)]


class KbsNoiseView(C.Structure):
    _fields_ = [(k, _vp) for k in ("eps_jpos", "eps_jvel", "eps_gyro", "eps_pg")]


class KbsEpisodeView(C.Structure):
    _fields_ = [(k, _vp) for k in ("jpos_bias", "pg_lag", "pg_bias", "kp", "kd", "tau_limit", "action_bias",
                                   "torque_bias")]


class KbsNetWeights(C.Structure):
    _fields_ = [("w_in", _vp), ("b_in", _vp), ("w_ih", _vp * MAX_DEPTH), ("w_hh", _vp * MAX_DEPTH),
                ("b", _vp * MAX_DEPTH), ("w_out", _vp), ("b_out", _vp)]


class KbsActorOut(C.Structure):
    _fields_ = [(k, _vp) for k in ("action", "mean", "std", "log_prob", "entropy")]


class KbsTrajView(C.Structure):
    _fields_ = [("state", KbsStateView), ("command", _vp), ("ctrl", _vp), ("done", _vp), ("T", _i64)]


class KbsRewardCarry(C.Structure):
    _fields_ = [("t_single", _vp), ("airtime", _vp), ("prev_contact", _vp)]


class KbsRolloutIO(C.Structure):
    _fields_ = [("state", KbsStateView), ("noise", KbsNoiseView), ("episode", KbsEpisodeView)] + [
        (k, _vp) for k in ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms", "command", "pg_carry",
                           "actor_carry", "critic_carry", "lpf", "actor_obs", "action", "log_prob", "ctrl",
                           "term_codes", "done", "success", "value")] + [("T", _i64)]


class KbsRolloutRecord(C.Structure):
    """struct kbs_rollout_record (kbs_rollout_record's optional outputs / boundary input)."""
    _fields_ = [("done_prev", _vp), ("critic_obs", _vp)]


class KbsStepState(C.Structure):
    """kbs_step_state: the caller-owned device buffer of the online rollout and what it was sized for."""
    _fields_ = [("buf", _vp), ("bytes", C.c_uint64), ("n_envs", _i64), ("with_critic", C.c_int32)]


class KbsStepCarry(C.Structure):
    """kbs_step_carry: the ABI form of what a step state carries (load / store)."""
    _fields_ = [(k, _vp) for k in ("actor_carry", "critic_carry", "lpf", "pg_carry", "command", "done_prev")]


class KbsStepIO(C.Structure):
    """kbs_step_io: one step's inputs, and the trajectories whose slot t it writes."""
    _fields_ = [("state", KbsStateView), ("noise", KbsNoiseView), ("episode", KbsEpisodeView)] + [
        (k, _vp) for k in ("eps_action", "u_switch", "cmd_mode", "cmd_u6", "cmd_u_arms", "command", "actor_obs", "critic_obs",
                           "action", "log_prob", "ctrl", "term_codes", "done", "success", "value")] + [
        ("traj_state", KbsStateView), ("T", _i64)]


class KbsActuatorState(C.Structure):
    """kbs_actuator_state: the caller-owned device buffer of the physics sub-steps (k, prev_action, applied)."""
    _fields_ = [("buf", _vp), ("bytes", C.c_uint64), ("n_envs", _i64), ("n_substeps", C.c_int32)]


class KbsSubstepIO(C.Structure):
    """kbs_substep_io: one physics sub-step's inputs and its ctrl."""
    _fields_ = [("action", _vp), ("T", _i64), ("u_drop", _vp), ("latency", _vp), ("qpos", _vp), ("qvel", _vp),
                ("episode", KbsEpisodeView), ("ctrl", _vp), ("sub_dt", _f), ("drop_prob", _f)]


class KbsPpoIO(C.Structure):
    _fields_ = [(k, _vp) for k in ("actor_obs", "critic_obs", "action", "done", "actor_carry", "critic_carry", "lpf",
                                   "log_probs", "values", "entropy", "action_std", "mean")] + [("T", _i64), ("ld", _i64)] + [
        (k, _vp) for k in ("actor_obs_mirror", "critic_obs_mirror", "actor_mirror_carry", "critic_mirror_carry", "lpf_mirror",
                           "action_mirror_loss", "value_mirror_loss")] + [("actor_mirror_loss_scale", _f),
                                                                          ("critic_mirror_loss_scale", _f)]


class KbsAdamwParams(C.Structure):
    _fields_ = [("b1", C.c_double), ("b2", C.c_double)] + [(k, _f) for k in ("lr", "eps", "weight_decay", "grad_scale",
                                                                            "max_grad_norm")]


class KbsActuatorRandParams(C.Structure):
    _fields_ = [(k, _f) for k in ("kp_scale", "kd_scale", "torque_limit_scale_low", "action_bias_scale", "torque_bias_scale")]


class KbsPpoLossParams(C.Structure):
    _fields_ = [("clip_param", C.c_float), ("value_loss_coef", C.c_float), ("entropy_coef", C.c_float),
                ("log_clip_value", C.c_float), ("use_clipped_value_loss", C.c_int32)]


class KbsPpoLossIO(C.Structure):
    _fields_ = [(k, _vp) for k in ("log_probs", "old_log_probs", "advantages", "values", "old_values", "value_targets",
                                   "entropy", "per_step", "out")] + [("T", _i64), ("ld", _i64)]


class KbsPpoBatch(C.Structure):
    _fields_ = [(k, _vp) for k in ("actor_obs", "critic_obs", "action", "done", "old_log_probs", "advantages", "value_targets",
                                   "old_values", "actor_carry0", "critic_carry0", "lpf0")] + [("T", _i64), ("ld", _i64)]


class KbsPpoMinibatches(C.Structure):
    _fields_ = [(k, _vp) for k in ("actor_obs", "critic_obs", "action", "done", "old_log_probs", "advantages", "value_targets",
                                   "old_values", "actor_carry0", "critic_carry0", "lpf0")] + [("batch_size", _i64),
                                                                                             ("num_batches", _i64)]


class KbsNetGrads(C.Structure):
    _fields_ = [("w_in", _vp), ("b_in", _vp), ("w_ih", _vp * MAX_DEPTH), ("w_hh", _vp * MAX_DEPTH), ("b", _vp * MAX_DEPTH),
                ("w_out", _vp), ("b_out", _vp)]


class KbsPpoCotangents(C.Structure):
    _fields_ = [(k, _vp) for k in ("log_probs", "values", "entropy", "action_std")]


# every symbol include/kbotstep.h declares (tests check the .so exports all of them)
EXPORTS = (
    "kbs_version", "kbs_error_string", "kbs_default_params", "kbs_create", "kbs_destroy", "kbs_get_params",
    "kbs_weights_pack", "kbs_observations", "kbs_command_update", "kbs_actor_step", "kbs_critic_step",
    "kbs_torque", "kbs_terminate", "kbs_rewards", "kbs_gae", "kbs_policy_step", "kbs_rollout", "kbs_ppo_variables",
    "kbs_launch_count", "kbs_device_status", "kbs_mirror_observations", "kbs_mirror_joints", "kbs_upload_state", "kbs_com_distance", "kbs_ppo_loss_default_params", "kbs_ppo_loss", "kbs_ppo_grad", "kbs_adam_step", "kbs_torque_substeps", "kbs_profile_enable", "kbs_profile_read", "kbs_kernel_name", "kbs_debug_tc_gates", "kbs_debug_tc_trace", "kbs_debug_tc_trace_attach",
    "kbs_adamw_default_params", "kbs_adamw_step", "kbs_grad_norm", "kbs_scratch_lock", "kbs_actuator_rand_default_params",
    "kbs_sample_actuator_randomization", "kbs_device_status_reset", "kbs_ppo_grad_set_events", "kbs_generate_rollout_noise",
    "kbs_minibatch_permutation", "kbs_shuffle_minibatches", "kbs_rollout_record", "kbs_step_state_bytes", "kbs_step_state_load",
    "kbs_step_state_store", "kbs_step_state_rewind", "kbs_rollout_step", "kbs_actuator_state_bytes", "kbs_actuator_state_load",
    "kbs_actuator_state_store", "kbs_actuator_substep", "kbs_ppo_variables_vjp",
)
VERSION = 101
STATUS_TIMEOUT_LSTM, STATUS_TIMEOUT_HEAD, STATUS_F16_RANGE, STATUS_STEP_RANGE = 1, 2, 0x100, 0x200
STATUS_SUBSTEP_RANGE = 0x400
NUM_KERNEL_IDS = 26
MAX_PERMUTATION_ENVS = 16384

_lib = None


def load() -> C.CDLL:
    """Load libkbotstep.so.  Raises (never falls back) when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make`). kbot-joystick_b200 has no CPU fallback.")
    lib = C.CDLL(os.fspath(LIB_PATH))
    P = C.POINTER
    lib.kbs_version.restype = C.c_int
    lib.kbs_error_string.restype = C.c_char_p
    lib.kbs_error_string.argtypes = [C.c_int]
    lib.kbs_default_params.argtypes = [P(KbsParams)]
    lib.kbs_create.argtypes = [P(KbsParams), P(_vp)]
    lib.kbs_destroy.argtypes = [_vp]
    lib.kbs_get_params.argtypes = [_vp, P(KbsParams)]
    lib.kbs_weights_pack.argtypes = [_vp, C.c_int, P(KbsNetWeights), _vp]
    lib.kbs_observations.argtypes = [_vp, P(KbsStateView), P(KbsNoiseView), P(KbsEpisodeView), _vp, _vp, _vp, _vp,
                                     _vp, _vp, _i64, _vp]
    lib.kbs_mirror_observations.argtypes = [_vp, P(KbsStateView), _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]
    lib.kbs_ppo_loss_default_params.argtypes = [P(KbsPpoLossParams)]
    lib.kbs_ppo_loss.argtypes = [_vp, P(KbsPpoLossParams), P(KbsPpoLossIO), _i64, _vp]
    lib.kbs_ppo_grad.argtypes = [_vp, P(KbsPpoLossParams), P(KbsPpoBatch), P(KbsNetGrads), P(KbsNetGrads), _vp, _vp, _vp, _vp,
                                 _i64, _vp]
    lib.kbs_adam_step.argtypes = [_vp, _vp, _vp, _vp, _vp, _i64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _i64, _vp]
    lib.kbs_adamw_default_params.argtypes = [P(KbsAdamwParams)]
    lib.kbs_adamw_step.argtypes = [_vp, _vp, _vp, _vp, _vp, _i64, P(KbsAdamwParams), _vp, _vp, _i64, _vp]
    lib.kbs_ppo_grad_set_events.argtypes = [_vp, _vp]
    lib.kbs_ppo_variables_vjp.argtypes = [_vp, P(KbsPpoBatch), P(KbsPpoCotangents), P(KbsNetGrads), P(KbsNetGrads), _vp, _vp,
                                          _vp, _i64, _vp]
    lib.kbs_generate_rollout_noise.argtypes = [_vp, C.c_uint64, _i64, P(KbsNoiseView), _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp]
    lib.kbs_grad_norm.argtypes = [_vp, _vp, _i64, _vp, _vp]
    lib.kbs_minibatch_permutation.argtypes = [_vp, C.c_uint64, _vp, _i64, _vp, _i64, _vp]
    lib.kbs_shuffle_minibatches.argtypes = [_vp, _vp, P(KbsPpoBatch), P(KbsPpoMinibatches), _i64, _vp]
    lib.kbs_scratch_lock.argtypes = [_vp, C.c_int]
    lib.kbs_device_status_reset.argtypes = [_vp]
    lib.kbs_actuator_rand_default_params.argtypes = [P(KbsActuatorRandParams)]
    lib.kbs_sample_actuator_randomization.argtypes = [_vp, P(KbsActuatorRandParams), _vp, _vp, P(KbsEpisodeView), _i64, _i64, _vp]
    lib.kbs_torque_substeps.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, P(KbsEpisodeView), _vp, C.c_int32, C.c_float, C.c_float,
                                        _i64, _i64, _vp]
    lib.kbs_com_distance.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, _i64, _i64, _i64, _vp]
    lib.kbs_upload_state.argtypes = [_vp, P(KbsStateView), P(KbsStateView), _i64, P(_i64), _vp]
    lib.kbs_mirror_joints.argtypes = [_vp, _vp, _vp, _i64, _i64, _i64, _vp]
    lib.kbs_command_update.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]
    lib.kbs_actor_step.argtypes = [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, P(KbsActorOut), _i64, _vp]
    lib.kbs_critic_step.argtypes = [_vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp]
    lib.kbs_torque.argtypes = [_vp, _vp, P(KbsStateView), P(KbsEpisodeView), _vp, _i64, _vp]
    lib.kbs_terminate.argtypes = [_vp, P(KbsStateView), _vp, _vp, _vp, _vp, _i64, _vp]
    lib.kbs_rewards.argtypes = [_vp, P(KbsTrajView), P(KbsRewardCarry), _vp, _vp, _i64, _vp]
    lib.kbs_gae.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp]
    lib.kbs_policy_step.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
    lib.kbs_rollout.argtypes = [_vp, P(KbsRolloutIO), _i64, _vp]
    lib.kbs_rollout_record.argtypes = [_vp, P(KbsRolloutIO), P(KbsRolloutRecord), _i64, _vp]
    lib.kbs_ppo_variables.argtypes = [_vp, P(KbsPpoIO), _i64, _vp]
    lib.kbs_step_state_bytes.argtypes = [_vp, _i64, C.c_int, P(C.c_uint64)]
    lib.kbs_step_state_load.argtypes = [_vp, P(KbsStepState), P(KbsStepCarry), _vp]
    lib.kbs_step_state_store.argtypes = [_vp, P(KbsStepState), P(KbsStepCarry), _vp]
    lib.kbs_step_state_rewind.argtypes = [_vp, P(KbsStepState), _vp]
    lib.kbs_rollout_step.argtypes = [_vp, P(KbsStepState), P(KbsStepIO), _vp]
    lib.kbs_actuator_state_bytes.argtypes = [_vp, _i64, P(C.c_uint64)]
    lib.kbs_actuator_state_load.argtypes = [_vp, P(KbsActuatorState), _vp, _vp]
    lib.kbs_actuator_state_store.argtypes = [_vp, P(KbsActuatorState), _vp, _vp]
    lib.kbs_actuator_substep.argtypes = [_vp, P(KbsStepState), P(KbsActuatorState), P(KbsSubstepIO), _vp]
    lib.kbs_launch_count.argtypes = [_vp]
    lib.kbs_launch_count.restype = _i64
    lib.kbs_device_status.argtypes = [_vp, P(C.c_int)]
    lib.kbs_profile_enable.argtypes = [_vp, C.c_int]
    lib.kbs_profile_read.argtypes = [_vp, C.c_int, P(C.c_double), P(_i64)]
    lib.kbs_debug_tc_gates.argtypes = [_vp, C.c_int, C.c_int, _vp, _vp, _vp, _i64, _vp]
    lib.kbs_debug_tc_trace.argtypes = [_vp, _vp, _i64, _vp]
    lib.kbs_debug_tc_trace_attach.argtypes = [_vp, _vp, _i64, C.c_int]
    lib.kbs_kernel_name.argtypes = [C.c_int]
    lib.kbs_kernel_name.restype = C.c_char_p
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("kbs_error_string", "kbs_launch_count", "kbs_kernel_name"):
            fn.restype = C.c_int
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().kbs_error_string(rc).decode()
        raise RuntimeError(f"{what} failed: [{rc}] {msg}")


def default_params() -> KbsParams:
    p = KbsParams()
    check(load().kbs_default_params(C.byref(p)), "kbs_default_params")
    return p


def host_ptr(t) -> int | None:
    """Pointer of a pinned host tensor (None -> NULL): source of the asynchronous uploads."""
    if t is None:
        return None
    assert (not t.is_cuda) and t.is_contiguous() and t.is_pinned(), "uploads take contiguous pinned host tensors"
    return t.data_ptr()


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "kbotstep takes contiguous CUDA tensors"
    return t.data_ptr()
