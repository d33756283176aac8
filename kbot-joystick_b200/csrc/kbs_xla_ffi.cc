// kbs_xla_ffi.cc -- XLA FFI (jax.ffi) handlers over the C-ABI of libkbotstep.so: the binding a maintainer of the reference
// (a JAX program) adds so that the jitted ksim Task hooks lower to these kernels on the CUDA platform (INTEGRATION.md 2).
//
// NOT BUILT IN THIS IMAGE: jaxlib and its headers (xla/ffi/api/ffi.h) are not installable here (SURVEY F5), so the shared
// object is produced only where they exist:
//     make ffi JAX_INCLUDE=$(python -c "import jax.ffi; print(jax.ffi.include_dir())")
// What IS checked here: `make ffi-check` (and tests/test_host_cpu.py) type-check this file with g++ against a stub of the
// FFI surface (tests/ffi_stub/xla/ffi/api/ffi.h) whose Bind().To() static_asserts every handler against its binding.
// The file adds nothing to the product path: every handler unpacks buffers and forwards to ONE entry point of
// include/kbotstep.h on XLA's stream; errors come back as ffi::Error (no throw across the ABI, no CPU fallback).
//
// Handle: the Python side creates the kbs_handle once (kbs_create / kbs_weights_pack through ctypes, jax_ffi.py) and
// passes the pointer as the int64 attribute "handle" of every call.  Layout at the boundary: env-major SoA [F][ld]
// (ld = n_envs rounded up to 4), trajectories [T][F][ld] -- see INTEGRATION.md "Layout contract".  In-out arguments of
// the C-ABI (carries, filter state, reward carries, optimiser state) are input + result pairs that jax_ffi.py aliases
// (input_output_aliases); a handler copies input -> result first when XLA did not alias them.
#if __has_include("xla/ffi/api/ffi.h")
#include <cstdint>

#include <cuda_runtime_api.h>

#include "kbotstep.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

namespace {

using F32 = ffi::Buffer<ffi::F32>;
using U8 = ffi::Buffer<ffi::U8>;
using S32 = ffi::Buffer<ffi::S32>;
using S64 = ffi::Buffer<ffi::S64>;
using RF32 = ffi::ResultBuffer<ffi::F32>;
using RU8 = ffi::ResultBuffer<ffi::U8>;
using RS32 = ffi::ResultBuffer<ffi::S32>;
using RS64 = ffi::ResultBuffer<ffi::S64>;

inline kbs_handle* H(int64_t handle) { return reinterpret_cast<kbs_handle*>(static_cast<intptr_t>(handle)); }
inline ffi::Error Rc(int rc) { return rc == 0 ? ffi::Error::Success() : ffi::Error::Internal(kbs_error_string(rc)); }
template <typename B>
inline int64_t Dim(const B& b, int i) { return static_cast<int64_t>(b.dimensions()[i]); }
// in-out pair: aliased -> nothing to do; otherwise the result starts as a copy of the input
template <typename In, typename Out>
inline bool Carry(cudaStream_t stream, const In& in, Out& out) {
  return in.typed_data() == out->typed_data() ||
         cudaMemcpyAsync(out->typed_data(), in.typed_data(), in.size_bytes(), cudaMemcpyDeviceToDevice, stream) == cudaSuccess;
}

// ---- ksim.compute_ppo_inputs (GAE), gamma / lam live in the handle's kbs_params (train.py:1769-1770) --------------------
ffi::Error GaeImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, F32 values, F32 rewards, U8 done, U8 success, RF32 adv,
                   RF32 targets) {
  const int64_t T = Dim(values, 0), ld = Dim(values, 1);
  return Rc(kbs_gae(H(handle), values.typed_data(), rewards.typed_data(), done.typed_data(), success.typed_data(),
                    adv->typed_data(), targets->typed_data(), T, ld, n_envs, stream));
}

// ---- get_terminations (train.py:1258-1269, 817-823): qpos [27][ld], xpos [72][ld], time [ld] -> codes / done / success ----
ffi::Error TerminateImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, F32 qpos, F32 xpos, F32 time, RS32 codes, RU8 done,
                         RU8 success) {
  kbs_state_view s{};
  s.qpos = qpos.typed_data(); s.xpos = xpos.typed_data(); s.time = time.typed_data(); s.ld = Dim(qpos, 1);
  return Rc(kbs_terminate(H(handle), &s, codes->typed_data(), done->typed_data(), success->typed_data(), nullptr, n_envs,
                          stream));
}

// ---- get_actuators().get_ctrl (train.py:1091-1105): action [20][ld], qpos [27][ld], qvel [26][ld], the five per-episode
//      actuator arrays [20][ld] (kbs_sample_actuator_randomization) -> ctrl [20][ld] ----------------------------------------
ffi::Error TorqueImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, F32 action, F32 qpos, F32 qvel, F32 kp, F32 kd,
                      F32 tau_limit, F32 action_bias, F32 torque_bias, RF32 ctrl) {
  kbs_state_view s{};
  s.qpos = qpos.typed_data(); s.qvel = qvel.typed_data(); s.ld = Dim(qpos, 1);
  kbs_episode_view ep{};
  ep.kp = kp.typed_data(); ep.kd = kd.typed_data(); ep.tau_limit = tau_limit.typed_data();
  ep.action_bias = action_bias.typed_data(); ep.torque_bias = torque_bias.typed_data();
  return Rc(kbs_torque(H(handle), action.typed_data(), &s, &ep, ctrl->typed_data(), n_envs, stream));
}

// ---- per-episode actuator randomisation (train.py:1097-1105): u [5][20][ld], reset u8 [ld], the five arrays in-out ---------
ffi::Error ActuatorRandImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, F32 u, U8 reset, F32 kp, F32 kd, F32 tau_limit,
                            F32 action_bias, F32 torque_bias, RF32 kp_o, RF32 kd_o, RF32 tau_o, RF32 ab_o, RF32 tb_o) {
  if (!Carry(stream, kp, kp_o) || !Carry(stream, kd, kd_o) || !Carry(stream, tau_limit, tau_o) || !Carry(stream, action_bias, ab_o) ||
      !Carry(stream, torque_bias, tb_o))
    return ffi::Error::Internal("kbs_sample_actuator_randomization: carry copy failed");
  kbs_actuator_rand_params rp;
  kbs_actuator_rand_default_params(&rp);
  kbs_episode_view ep{};
  ep.kp = kp_o->typed_data(); ep.kd = kd_o->typed_data(); ep.tau_limit = tau_o->typed_data();
  ep.action_bias = ab_o->typed_data(); ep.torque_bias = tb_o->typed_data();
  return Rc(kbs_sample_actuator_randomization(H(handle), &rp, u.typed_data(), reset.typed_data(), &ep, Dim(u, 2), n_envs, stream));
}

// ---- convert.py:84-119 step_fn, batched over envs (AoS rows as the exported function takes them) -------------------------
ffi::Error PolicyStepImpl(cudaStream_t stream, int64_t handle, F32 joint_angles, F32 joint_vel, F32 projected_gravity, F32 gyro,
                          F32 command, F32 carry, RF32 action, RF32 carry_out) {
  return Rc(kbs_policy_step(H(handle), joint_angles.typed_data(), joint_vel.typed_data(), projected_gravity.typed_data(),
                            gyro.typed_data(), command.typed_data(), carry.typed_data(), carry_out->typed_data(),
                            action->typed_data(), Dim(joint_angles, 0), stream));
}

// ---- get_observations (train.py:1155-1204) + the run_actor / run_critic concatenations (train.py:1351-1431) -----------------
// state rows as kbs_state_view; noise [46][ld] = eps_jpos 20 | eps_jvel 20 | eps_gyro 3 | eps_pg 3; episode: jpos_bias [20][ld],
// pg_lag [ld], pg_bias [3][ld]; command [16][ld]; pg_carry [3][ld] in-out; pg_reset u8 [ld]
ffi::Error ObservationsImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, F32 qpos, F32 qvel, F32 sensordata, F32 xpos,
                            F32 xquat, F32 cinert, F32 cvel, F32 actuator_force, F32 noise, F32 jpos_bias, F32 pg_lag, F32 pg_bias,
                            F32 command, F32 pg_carry, U8 pg_reset, RF32 pg_carry_out, RF32 computed, RF32 actor_obs,
                            RF32 critic_obs) {
  if (!Carry(stream, pg_carry, pg_carry_out)) return ffi::Error::Internal("kbs_observations: carry copy failed");
  const int64_t ld = Dim(qpos, 1);
  kbs_state_view s{};
  s.qpos = qpos.typed_data(); s.qvel = qvel.typed_data(); s.sensordata = sensordata.typed_data(); s.xpos = xpos.typed_data();
  s.xquat = xquat.typed_data(); s.cinert = cinert.typed_data(); s.cvel = cvel.typed_data();
  s.actuator_force = actuator_force.typed_data(); s.ld = ld;
  kbs_noise_view nz{};
  nz.eps_jpos = noise.typed_data(); nz.eps_jvel = nz.eps_jpos + 20 * ld; nz.eps_gyro = nz.eps_jvel + 20 * ld; nz.eps_pg = nz.eps_gyro + 3 * ld;
  kbs_episode_view ep{};
  ep.jpos_bias = jpos_bias.typed_data(); ep.pg_lag = pg_lag.typed_data(); ep.pg_bias = pg_bias.typed_data();
  return Rc(kbs_observations(H(handle), &s, &nz, &ep, command.typed_data(), pg_carry_out->typed_data(), pg_reset.typed_data(),
                             computed->typed_data(), actor_obs->typed_data(), critic_obs->typed_data(), n_envs, stream));
}

// ---- get_commands: UnifiedCommand.__call__ (train.py:768-785); always_resample != 0 = initial_command (train.py:724-766) -----
ffi::Error CommandUpdateImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, int64_t always_resample, F32 command,
                             F32 u_switch, S32 mode, F32 u6, F32 u_arms, RF32 command_out) {
  if (!Carry(stream, command, command_out)) return ffi::Error::Internal("kbs_command_update: carry copy failed");
  return Rc(kbs_command_update(H(handle), command_out->typed_data(), always_resample ? nullptr : u_switch.typed_data(),
                               mode.typed_data(), u6.typed_data(), u_arms.typed_data(), Dim(command, 1), n_envs, stream));
}

// ---- sample_action -> run_actor -> Actor.forward (train.py:1545-1572, 913-941); argmax != 0: dist.mode() ---------------------
ffi::Error ActorStepImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, int64_t argmax, F32 obs, F32 carry, F32 lpf, F32 eps,
                         U8 done, RF32 carry_out, RF32 lpf_out, RF32 action, RF32 mean, RF32 std, RF32 log_prob, RF32 entropy) {
  if (!Carry(stream, carry, carry_out) || !Carry(stream, lpf, lpf_out)) return ffi::Error::Internal("kbs_actor_step: carry copy failed");
  kbs_actor_out o{};
  o.action = action->typed_data(); o.mean = mean->typed_data(); o.std = std->typed_data();
  o.log_prob = log_prob->typed_data(); o.entropy = entropy->typed_data();
  return Rc(kbs_actor_step(H(handle), obs.typed_data(), Dim(obs, 1), carry_out->typed_data(), lpf_out->typed_data(),
                           argmax ? nullptr : eps.typed_data(), nullptr, done.typed_data(), &o, n_envs, stream));
}

// ---- run_critic -> Critic.forward (train.py:1381-1433, 993-1004) --------------------------------------------------------------
ffi::Error CriticStepImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, F32 obs, F32 carry, U8 done, RF32 carry_out,
                          RF32 value) {
  if (!Carry(stream, carry, carry_out)) return ffi::Error::Internal("kbs_critic_step: carry copy failed");
  return Rc(kbs_critic_step(H(handle), obs.typed_data(), Dim(obs, 1), carry_out->typed_data(), done.typed_data(),
                            value->typed_data(), n_envs, stream));
}

// ---- the fused control step over T recorded steps (ksim step_engine around mjx.step, SURVEY 3.2) -------------------------------
// state [T][rows][ld] x 10; noise [T][46][ld]; episode [88][ld] = jpos_bias 20 | pg_lag 1 | pg_bias 3 | kp 20 | kd 20 | tau_limit
// 20 | action_bias 20 ... (torque_bias: a separate [20][ld]); randomness eps_action [T][20][ld], u_switch [T][ld], cmd_mode s32
// [T][ld], cmd_u6 [T][6][ld], cmd_u_arms [T][10][ld]; command0 [16][ld]; carries in-out.
// RolloutIo: the in-out copies and the kbs_rollout_io both rollout handlers pass; false = a copy failed.
bool RolloutIo(cudaStream_t stream, F32& qpos, F32& qvel, F32& sensordata, F32& xpos, F32& xquat, F32& cinert, F32& cvel,
               F32& actuator_force, F32& com_distance, F32& time, F32& eps_jpos, F32& eps_jvel, F32& eps_gyro, F32& eps_pg,
               F32& episode, F32& torque_bias, F32& eps_action, F32& u_switch, S32& cmd_mode, F32& cmd_u6, F32& cmd_u_arms,
               F32& command0, F32& pg_carry, F32& actor_carry, F32& critic_carry, F32& lpf, RF32& command, RF32& pg_carry_out,
               RF32& actor_carry_out, RF32& critic_carry_out, RF32& lpf_out, RF32& actor_obs, RF32& action, RF32& log_prob,
               RF32& ctrl, RS32& term_codes, RU8& done, RU8& success, RF32& value, kbs_rollout_io& io) {
  if (!Carry(stream, pg_carry, pg_carry_out) || !Carry(stream, actor_carry, actor_carry_out) ||
      !Carry(stream, critic_carry, critic_carry_out) || !Carry(stream, lpf, lpf_out))
    return false;
  const int64_t T = Dim(qpos, 0), ld = Dim(qpos, 2);
  // row 0 of the [T + 1][16][ld] command trajectory is the command at step 0 (input)
  if (cudaMemcpyAsync(command->typed_data(), command0.typed_data(), command0.size_bytes(), cudaMemcpyDeviceToDevice, stream) != cudaSuccess)
    return false;
  io = kbs_rollout_io{};
  io.state.qpos = qpos.typed_data(); io.state.qvel = qvel.typed_data(); io.state.sensordata = sensordata.typed_data();
  io.state.xpos = xpos.typed_data(); io.state.xquat = xquat.typed_data(); io.state.cinert = cinert.typed_data();
  io.state.cvel = cvel.typed_data(); io.state.actuator_force = actuator_force.typed_data();
  io.state.com_distance = com_distance.typed_data(); io.state.time = time.typed_data(); io.state.ld = ld;
  io.noise.eps_jpos = eps_jpos.typed_data(); io.noise.eps_jvel = eps_jvel.typed_data(); io.noise.eps_gyro = eps_gyro.typed_data();
  io.noise.eps_pg = eps_pg.typed_data();
  const float* e = episode.typed_data();
  io.episode.jpos_bias = e; io.episode.pg_lag = e + 20 * ld; io.episode.pg_bias = e + 21 * ld; io.episode.kp = e + 24 * ld;
  io.episode.kd = e + 44 * ld; io.episode.tau_limit = e + 64 * ld; io.episode.action_bias = e + 84 * ld;
  io.episode.torque_bias = torque_bias.typed_data();
  io.eps_action = eps_action.typed_data(); io.u_switch = u_switch.typed_data(); io.cmd_mode = cmd_mode.typed_data();
  io.cmd_u6 = cmd_u6.typed_data(); io.cmd_u_arms = cmd_u_arms.typed_data();
  io.command = command->typed_data(); io.pg_carry = pg_carry_out->typed_data(); io.actor_carry = actor_carry_out->typed_data();
  io.critic_carry = critic_carry_out->typed_data(); io.lpf = lpf_out->typed_data(); io.actor_obs = actor_obs->typed_data();
  io.action = action->typed_data(); io.log_prob = log_prob->typed_data(); io.ctrl = ctrl->typed_data();
  io.term_codes = term_codes->typed_data(); io.done = done->typed_data(); io.success = success->typed_data();
  io.value = value->typed_data(); io.T = T;
  return true;
}
#define KBS_ROLLOUT_PARAMS                                                                                                      \
  F32 qpos, F32 qvel, F32 sensordata, F32 xpos, F32 xquat, F32 cinert, F32 cvel, F32 actuator_force, F32 com_distance, F32 time, \
      F32 eps_jpos, F32 eps_jvel, F32 eps_gyro, F32 eps_pg, F32 episode, F32 torque_bias, F32 eps_action, F32 u_switch,          \
      S32 cmd_mode, F32 cmd_u6, F32 cmd_u_arms, F32 command0, F32 pg_carry, F32 actor_carry, F32 critic_carry, F32 lpf
#define KBS_ROLLOUT_RESULTS                                                                                                    \
  RF32 command, RF32 pg_carry_out, RF32 actor_carry_out, RF32 critic_carry_out, RF32 lpf_out, RF32 actor_obs, RF32 action,      \
      RF32 log_prob, RF32 ctrl, RS32 term_codes, RU8 done, RU8 success, RF32 value
#define KBS_ROLLOUT_IO_ARGS                                                                                                    \
  qpos, qvel, sensordata, xpos, xquat, cinert, cvel, actuator_force, com_distance, time, eps_jpos, eps_jvel, eps_gyro, eps_pg, \
      episode, torque_bias, eps_action, u_switch, cmd_mode, cmd_u6, cmd_u_arms, command0, pg_carry, actor_carry, critic_carry,  \
      lpf, command, pg_carry_out, actor_carry_out, critic_carry_out, lpf_out, actor_obs, action, log_prob, ctrl, term_codes,   \
      done, success, value
ffi::Error RolloutImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, KBS_ROLLOUT_PARAMS, KBS_ROLLOUT_RESULTS) {
  kbs_rollout_io io;
  if (!RolloutIo(stream, KBS_ROLLOUT_IO_ARGS, io)) return ffi::Error::Internal("kbs_rollout: carry copy failed");
  return Rc(kbs_rollout(H(handle), &io, n_envs, stream));
}

// ---- the same step, continued across calls (ksim's engine loop: one step per call) and recording what the update trains on:
//      done_prev u8 [ld] = the previous call's done[T-1] (zeros on the first call); critic_obs [T][475][ld] out ----------------
ffi::Error RolloutRecordImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, KBS_ROLLOUT_PARAMS, U8 done_prev,
                             KBS_ROLLOUT_RESULTS, RF32 critic_obs) {
  kbs_rollout_io io;
  if (!RolloutIo(stream, KBS_ROLLOUT_IO_ARGS, io)) return ffi::Error::Internal("kbs_rollout_record: carry copy failed");
  struct kbs_rollout_record rec{done_prev.typed_data(), critic_obs->typed_data()};
  return Rc(kbs_rollout_record(H(handle), &io, &rec, n_envs, stream));
}

// ---- get_ppo_variables -> xax.scan(_ppo_scan_fn) (train.py:1435-1524) on a stored trajectory, aux_losses included ------------
ffi::Error PpoVariablesImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, float actor_mirror_loss_scale,
                            float critic_mirror_loss_scale, F32 actor_obs, F32 critic_obs, F32 actor_obs_mirror,
                            F32 critic_obs_mirror, F32 action, U8 done, F32 actor_carry, F32 critic_carry, F32 lpf,
                            F32 actor_mirror_carry, F32 critic_mirror_carry, F32 lpf_mirror, RF32 actor_carry_out,
                            RF32 critic_carry_out, RF32 lpf_out, RF32 actor_mirror_carry_out, RF32 critic_mirror_carry_out,
                            RF32 lpf_mirror_out, RF32 log_probs, RF32 values, RF32 entropy, RF32 action_std,
                            RF32 action_mirror_loss, RF32 value_mirror_loss) {
  if (!Carry(stream, actor_carry, actor_carry_out) || !Carry(stream, critic_carry, critic_carry_out) || !Carry(stream, lpf, lpf_out) ||
      !Carry(stream, actor_mirror_carry, actor_mirror_carry_out) || !Carry(stream, critic_mirror_carry, critic_mirror_carry_out) ||
      !Carry(stream, lpf_mirror, lpf_mirror_out))
    return ffi::Error::Internal("kbs_ppo_variables: carry copy failed");
  kbs_ppo_io io{};
  io.actor_obs = actor_obs.typed_data(); io.critic_obs = critic_obs.typed_data(); io.action = action.typed_data();
  io.done = done.typed_data();
  io.actor_carry = actor_carry_out->typed_data(); io.critic_carry = critic_carry_out->typed_data(); io.lpf = lpf_out->typed_data();
  io.log_probs = log_probs->typed_data(); io.values = values->typed_data(); io.entropy = entropy->typed_data();
  io.action_std = action_std->typed_data(); io.mean = nullptr;
  io.T = Dim(actor_obs, 0); io.ld = Dim(actor_obs, 2);
  io.actor_obs_mirror = actor_obs_mirror.typed_data(); io.critic_obs_mirror = critic_obs_mirror.typed_data();
  io.actor_mirror_carry = actor_mirror_carry_out->typed_data(); io.critic_mirror_carry = critic_mirror_carry_out->typed_data();
  io.lpf_mirror = lpf_mirror_out->typed_data();
  io.action_mirror_loss = action_mirror_loss->typed_data(); io.value_mirror_loss = value_mirror_loss->typed_data();
  io.actor_mirror_loss_scale = actor_mirror_loss_scale; io.critic_mirror_loss_scale = critic_mirror_loss_scale;
  return Rc(kbs_ppo_variables(H(handle), &io, n_envs, stream));
}

// ---- mirror_obs / mirror_cmd + concatenations (train.py:1463-1481, 1584-1756); mirror_joints (train.py:1574-1582) -------------
ffi::Error MirrorObservationsImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, F32 qpos, F32 qvel, F32 sensordata, F32 xpos,
                                  F32 xquat, F32 cinert, F32 cvel, F32 actuator_force, F32 computed, F32 command, RF32 actor_obs,
                                  RF32 critic_obs, RF32 command_out) {
  kbs_state_view s{};
  s.qpos = qpos.typed_data(); s.qvel = qvel.typed_data(); s.sensordata = sensordata.typed_data(); s.xpos = xpos.typed_data();
  s.xquat = xquat.typed_data(); s.cinert = cinert.typed_data(); s.cvel = cvel.typed_data();
  s.actuator_force = actuator_force.typed_data(); s.ld = Dim(qpos, 2);
  return Rc(kbs_mirror_observations(H(handle), &s, computed.typed_data(), command.typed_data(), actor_obs->typed_data(),
                                    critic_obs->typed_data(), command_out->typed_data(), Dim(qpos, 0), n_envs, stream));
}
ffi::Error MirrorJointsImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, F32 in, RF32 out) {
  return Rc(kbs_mirror_joints(H(handle), in.typed_data(), out->typed_data(), Dim(in, 0), Dim(in, 2), n_envs, stream));
}

// ---- COMDistanceObservation.observe (train.py:509-659) --------------------------------------------------------------------------
ffi::Error ComDistanceImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, S32 geom1, S32 geom2, F32 pos, F32 subtree_com,
                           RF32 com_distance) {
  return Rc(kbs_com_distance(H(handle), geom1.typed_data(), geom2.typed_data(), pos.typed_data(), subtree_com.typed_data(),
                             com_distance->typed_data(), int(Dim(geom1, 1)), Dim(geom1, 0), Dim(geom1, 2), n_envs, stream));
}

// ---- get_rewards table + scale-and-sum (train.py:125-506, 1224-1256) on a trajectory ------------------------------------------
ffi::Error RewardsImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, F32 qpos, F32 qvel, F32 sensordata, F32 xpos, F32 xquat,
                       F32 com_distance, F32 command, F32 ctrl, U8 done, F32 t_single, F32 airtime, U8 prev_contact,
                       RF32 t_single_out, RF32 airtime_out, RU8 prev_contact_out, RF32 total, RF32 components) {
  if (!Carry(stream, t_single, t_single_out) || !Carry(stream, airtime, airtime_out) || !Carry(stream, prev_contact, prev_contact_out))
    return ffi::Error::Internal("kbs_rewards: carry copy failed");
  kbs_traj_view tr{};
  tr.state.qpos = qpos.typed_data(); tr.state.qvel = qvel.typed_data(); tr.state.sensordata = sensordata.typed_data();
  tr.state.xpos = xpos.typed_data(); tr.state.xquat = xquat.typed_data(); tr.state.com_distance = com_distance.typed_data();
  tr.state.ld = Dim(qpos, 2);
  tr.command = command.typed_data(); tr.ctrl = ctrl.typed_data(); tr.done = done.typed_data(); tr.T = Dim(qpos, 0);
  kbs_reward_carry rc{t_single_out->typed_data(), airtime_out->typed_data(), prev_contact_out->typed_data()};
  return Rc(kbs_rewards(H(handle), &tr, &rc, total->typed_data(), components->typed_data(), n_envs, stream));
}

// ---- jax.grad of the PPO minibatch loss (train.py:1435-1524 under jax.grad; ksim.compute_ppo_loss) ----------------------------
// grads: ONE flat f32 buffer per network in the order w_in, b_in, (w_ih, w_hh, b) per layer, w_out, b_out (ppo.NetParams)
void GradViews(float* p, int64_t hidden, int64_t depth, int64_t num_in, int64_t num_out, kbs_net_grads* g) {
  const int64_t Hh = hidden;
  g->w_in = p; p += Hh * num_in; g->b_in = p; p += Hh;
  for (int64_t l = 0; l < depth && l < KBS_MAX_DEPTH; ++l) {
    g->w_ih[l] = p; p += 4 * Hh * Hh; g->w_hh[l] = p; p += 4 * Hh * Hh; g->b[l] = p; p += 4 * Hh;
  }
  g->w_out = p; p += num_out * Hh; g->b_out = p;
}
ffi::Error PpoGradImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, int64_t hidden, int64_t depth, F32 actor_obs,
                       F32 critic_obs, F32 action, U8 done, F32 old_log_probs, F32 advantages, F32 value_targets, F32 old_values,
                       F32 actor_carry0, F32 critic_carry0, F32 lpf0, RF32 grad_actor, RF32 grad_critic, RF32 log_probs, RF32 values,
                       RF32 entropy, RF32 stats) {
  kbs_ppo_loss_params lp;
  kbs_ppo_loss_default_params(&lp);
  kbs_ppo_batch b{};
  b.actor_obs = actor_obs.typed_data(); b.critic_obs = critic_obs.typed_data(); b.action = action.typed_data();
  b.done = done.typed_data(); b.old_log_probs = old_log_probs.typed_data(); b.advantages = advantages.typed_data();
  b.value_targets = value_targets.typed_data(); b.old_values = old_values.typed_data();
  b.actor_carry0 = actor_carry0.typed_data(); b.critic_carry0 = critic_carry0.typed_data(); b.lpf0 = lpf0.typed_data();
  b.T = Dim(actor_obs, 0); b.ld = Dim(actor_obs, 2);
  kbs_net_grads ga{}, gc{};
  GradViews(grad_actor->typed_data(), hidden, depth, KBS_ACTOR_OBS, KBS_ACTOR_OUT, &ga);
  GradViews(grad_critic->typed_data(), hidden, depth, KBS_CRITIC_OBS, 1, &gc);
  return Rc(kbs_ppo_grad(H(handle), &lp, &b, &ga, &gc, log_probs->typed_data(), values->typed_data(), entropy->typed_data(),
                         stats->typed_data(), n_envs, stream));
}

// ---- VJP of get_ppo_variables (train.py:1484-1487): the backward rule of a jax.custom_vjp around it (INTEGRATION.md) ----------
// ct_*: the cotangents of log_probs / values / entropy [T][ld] and action_std [T][20][ld]; grads flat as for KbsPpoGrad
ffi::Error PpoVariablesVjpImpl(cudaStream_t stream, int64_t handle, int64_t n_envs, int64_t hidden, int64_t depth, F32 actor_obs,
                               F32 critic_obs, F32 action, U8 done, F32 actor_carry0, F32 critic_carry0, F32 lpf0, F32 ct_log_probs,
                               F32 ct_values, F32 ct_entropy, F32 ct_action_std, RF32 grad_actor, RF32 grad_critic, RF32 log_probs,
                               RF32 values, RF32 entropy) {
  kbs_ppo_batch b{};
  b.actor_obs = actor_obs.typed_data(); b.critic_obs = critic_obs.typed_data(); b.action = action.typed_data();
  b.done = done.typed_data();
  b.actor_carry0 = actor_carry0.typed_data(); b.critic_carry0 = critic_carry0.typed_data(); b.lpf0 = lpf0.typed_data();
  b.T = Dim(actor_obs, 0); b.ld = Dim(actor_obs, 2);
  kbs_ppo_cotangents ct{ct_log_probs.typed_data(), ct_values.typed_data(), ct_entropy.typed_data(), ct_action_std.typed_data()};
  kbs_net_grads ga{}, gc{};
  GradViews(grad_actor->typed_data(), hidden, depth, KBS_ACTOR_OBS, KBS_ACTOR_OUT, &ga);
  GradViews(grad_critic->typed_data(), hidden, depth, KBS_CRITIC_OBS, 1, &gc);
  return Rc(kbs_ppo_variables_vjp(H(handle), &b, &ct, &ga, &gc, log_probs->typed_data(), values->typed_data(),
                                  entropy->typed_data(), n_envs, stream));
}

// ---- optax.global_norm + optax.adamw with ksim's clip (train.py:1059-1065) on one flat parameter vector ------------------------
ffi::Error GradNormImpl(cudaStream_t stream, int64_t handle, F32 grad, RF32 norm) {
  return Rc(kbs_grad_norm(H(handle), grad.typed_data(), Dim(grad, 0), norm->typed_data(), stream));
}
ffi::Error AdamwStepImpl(cudaStream_t stream, int64_t handle, float lr, float weight_decay, float grad_scale, float max_grad_norm,
                         F32 param, F32 grad, F32 m, F32 v, F32 grad_norm, S64 step, RF32 param_out, RF32 m_out, RF32 v_out,
                         RS64 step_out) {
  if (!Carry(stream, param, param_out) || !Carry(stream, m, m_out) || !Carry(stream, v, v_out) || !Carry(stream, step, step_out))
    return ffi::Error::Internal("kbs_adamw_step: carry copy failed");
  kbs_adamw_params o;
  kbs_adamw_default_params(&o);
  o.lr = lr; o.weight_decay = weight_decay; o.grad_scale = grad_scale; o.max_grad_norm = max_grad_norm;
  return Rc(kbs_adamw_step(H(handle), param_out->typed_data(), grad.typed_data(), m_out->typed_data(), v_out->typed_data(),
                           Dim(param, 0), &o, grad_norm.typed_data(), step_out->typed_data(), 0, stream));
}

}  // namespace

#define KBS_BIND() ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Attr<int64_t>("handle")
#define KBS_BIND_N() KBS_BIND().Attr<int64_t>("n_envs")
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsGae, GaeImpl, KBS_BIND_N().Arg<F32>().Arg<F32>().Arg<U8>().Arg<U8>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsTerminate, TerminateImpl,
                              KBS_BIND_N().Arg<F32>().Arg<F32>().Arg<F32>().Ret<S32>().Ret<U8>().Ret<U8>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsTorque, TorqueImpl,
                              KBS_BIND_N().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsSampleActuatorRandomization, ActuatorRandImpl,
                              KBS_BIND_N().Arg<F32>().Arg<U8>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsPolicyStep, PolicyStepImpl,
                              KBS_BIND().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsObservations, ObservationsImpl,
                              KBS_BIND_N().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<U8>()
                                  .Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsCommandUpdate, CommandUpdateImpl,
                              KBS_BIND_N().Attr<int64_t>("always_resample").Arg<F32>().Arg<F32>().Arg<S32>().Arg<F32>().Arg<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsActorStep, ActorStepImpl,
                              KBS_BIND_N().Attr<int64_t>("argmax").Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<U8>()
                                  .Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsCriticStep, CriticStepImpl, KBS_BIND_N().Arg<F32>().Arg<F32>().Arg<U8>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsRollout, RolloutImpl,
                              KBS_BIND_N().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<S32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>()
                                  .Ret<S32>().Ret<U8>().Ret<U8>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsRolloutRecord, RolloutRecordImpl,
                              KBS_BIND_N().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<S32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<U8>()
                                  .Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>()
                                  .Ret<S32>().Ret<U8>().Ret<U8>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsPpoVariables, PpoVariablesImpl,
                              KBS_BIND_N().Attr<float>("actor_mirror_loss_scale").Attr<float>("critic_mirror_loss_scale")
                                  .Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<U8>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>()
                                  .Ret<F32>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsMirrorObservations, MirrorObservationsImpl,
                              KBS_BIND_N().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<F32>().Arg<F32>().Ret<F32>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsMirrorJoints, MirrorJointsImpl, KBS_BIND_N().Arg<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsComDistance, ComDistanceImpl, KBS_BIND_N().Arg<S32>().Arg<S32>().Arg<F32>().Arg<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsRewards, RewardsImpl,
                              KBS_BIND_N().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<F32>().Arg<U8>().Arg<F32>().Arg<F32>().Arg<U8>()
                                  .Ret<F32>().Ret<F32>().Ret<U8>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsPpoGrad, PpoGradImpl,
                              KBS_BIND_N().Attr<int64_t>("hidden").Attr<int64_t>("depth")
                                  .Arg<F32>().Arg<F32>().Arg<F32>().Arg<U8>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<F32>().Arg<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsPpoVariablesVjp, PpoVariablesVjpImpl,
                              KBS_BIND_N().Attr<int64_t>("hidden").Attr<int64_t>("depth")
                                  .Arg<F32>().Arg<F32>().Arg<F32>().Arg<U8>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>()
                                  .Arg<F32>().Arg<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsGradNorm, GradNormImpl, KBS_BIND().Arg<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(KbsAdamwStep, AdamwStepImpl,
                              KBS_BIND().Attr<float>("lr").Attr<float>("weight_decay").Attr<float>("grad_scale").Attr<float>("max_grad_norm")
                                  .Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Arg<S64>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<S64>());
#else
#error "kbs_xla_ffi.cc needs jaxlib's XLA FFI headers: make ffi JAX_INCLUDE=$(python -c 'import jax.ffi; print(jax.ffi.include_dir())')"
#endif
