/*
 * kbotstep.h -- C-ABI of libkbotstep.so: the B200-native (sm_100a) rollout control step of the
 * kbot-joystick task.  Plain pointers and sizes; no torch / JAX types.  Every entry point cites the
 * reference interface (file:line under kscalelabs/kbot-joystick) it replaces.
 *
 * Conventions
 *  - All pointers are DEVICE pointers owned by the caller unless stated otherwise.  The library owns
 *    only the packed weights and scratch held by the opaque handle.
 *  - Work is enqueued on the caller's stream (a cudaStream_t passed as void*); calls are asynchronous.
 *  - Return value: 0 ok; <0 invalid argument (KBS_E_*); >0 a cudaError_t.  Nothing throws; there is no
 *    CPU fallback.
 *  - Layout "SoA[F][ld]": feature-major, env index contiguous, row f at base + f*ld.  ld >= n_envs,
 *    ld % 4 == 0, base 16-byte aligned (float4 access).  Trajectories are [T][F][ld]: step t at
 *    base + t*F*ld.
 *  - Layout "AoS[n][W]": row-major per env (used for recurrent carries, K-major GEMM operands).
 *  - fp32 everywhere; termination codes int32; done/success uint8 (0/1).
 */
#ifndef KBOTSTEP_H_
#define KBOTSTEP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KBS_VERSION 101
#define KBS_NUM_JOINTS 20
#define KBS_NUM_COMMANDS 16
#define KBS_ACTOR_OBS 65    /* train.py:1290-1295 */
#define KBS_CRITIC_OBS 475  /* train.py:1297-1312 */
#define KBS_ACTOR_OUT 40
#define KBS_MAX_DEPTH 4
#define KBS_NUM_REWARDS 12
#define KBS_NQ 27
#define KBS_NV 26
#define KBS_NBODY 24
#define KBS_NSENSORDATA 49
#define KBS_NUM_COMPUTED_OBS 78

/* error codes */
#define KBS_OK 0
#define KBS_E_NULL (-1)       /* required pointer is NULL */
#define KBS_E_SHAPE (-2)      /* n_envs / ld / T / hidden size not supported */
#define KBS_E_ALIGN (-3)      /* pointer not 16-byte aligned or ld % 4 != 0 */
#define KBS_E_STATE (-4)      /* weights not packed / handle not ready */
#define KBS_E_PARAM (-5)      /* bad scalar parameter */
#define KBS_E_DEVICE (-6)     /* the device health word is non-zero (kbs_device_status): a persistent kernel's dependency
                                 wait timed out, or an FP16-split operand left its range; sticky until kbs_device_status_reset */

enum { KBS_NET_ACTOR = 0, KBS_NET_CRITIC = 1 };
/* GEMM datapath for the LSTM/MLP contractions.  All are sm_100a CUDA in this library (no vendor library, no
 * fallback).  TC_* = tcgen05.mma with fp32 TMEM accumulators on operands split into two tensor-core-exact planes
 * (fp32-accurate: hi.hi + hi.lo + lo.hi): 3XTF32 = TF32 planes, 2XF16 = FP16 planes (lo scaled by 2^11; operands must
 * stay below 65504 in magnitude; half the bytes and twice the MMA rate).  The FP16 split represents an operand element x
 * to within 2^-22 |x| + 2^-36: below fp16's normal range (|x| < 2^-14) the floor 2^-36 is absolute, so an operand whose
 * elements all sit near it keeps only its leading bits.  SIMT = plain fp32 FFMA. */
enum { KBS_GEMM_TC_3XTF32 = 0, KBS_GEMM_SIMT_FP32 = 1, KBS_GEMM_TC_2XF16 = 2 };

/* Scalars of the path.  Defaults = the reference launch config (train.py:1761-1791) and tables
 * train.py:22-70, 1206-1269; robot/kbot/metadata.json; robot/kbot/robot.mjcf. */
typedef struct kbs_params {
  int32_t hidden_size;          /* train.py:1773 (256); 128 also supported */
  int32_t depth;                /* train.py:82 (2).  1 .. KBS_MAX_DEPTH; kbs_create refuses others with KBS_E_SHAPE.
                                 * The persistent tensor-core kernels hold at most 2 layers.  Above 2, on the tensor-core
                                 * datapaths (3xTF32, FP16-split), these refuse with KBS_E_SHAPE before launching anything:
                                 *   kbs_ppo_variables with mean or the mirror pass;
                                 *   kbs_step_state_bytes / _load and so kbs_rollout_step (no online step state).
                                 * Everything else runs the per-step launches instead of the persistent kernels. */
  int32_t gemm_path;            /* KBS_GEMM_* */
  int32_t normalize_advantages; /* ksim compute_ppo_inputs flag [unverified]: 0 none, 1 per-trajectory a/(std+eps) */
  float ctrl_dt;                /* train.py:1776 */
  float min_std, max_std, var_scale; /* train.py:1320-1322 */
  float lpf_alpha;              /* ksim.lowpass_one_pole coefficient, y' = y + alpha (x - y) */
  float gamma, lam, adv_eps;    /* train.py:1769-1770 */
  float jpos_noise_mag, jvel_noise_mag, gyro_noise_std, pg_noise_std; /* train.py:1160,1162,1176,1194 */
  float gravity, eps_quat;
  float unhealthy_z, max_tilt, max_length_sec; /* train.py:1265-1268 */
  float switch_prob;            /* train.py:1220 */
  float cmd_lo[6], cmd_hi[6];   /* vx vy wz bh rx ry, train.py:1212-1217 */
  float joint_bias[KBS_NUM_JOINTS];   /* train.py:24-45 */
  float joint_range[KBS_NUM_JOINTS];  /* max(bias-min, max-bias), train.py:1332 */
  float arm_lo[10], arm_hi[10];       /* JOINT_LIMITS[10:20], train.py:1207-1209 */
  float kp[KBS_NUM_JOINTS], kd[KBS_NUM_JOINTS], ctrl_limit[KBS_NUM_JOINTS];
  float reward_scale[KBS_NUM_REWARDS]; /* train.py:1224-1256 table order */
  float linvel_es, angvel_es, rp_es, rp_es_zero, bh_es, bh_standard, bh_foot_origin, arm_es;
  float grace_period, touchdown_penalty, feet_es, com_es, acc_es, torque_es;
  int32_t body_base, body_lfoot, body_rfoot;           /* 1, 7, 12 */
  int32_t sd_gyro, sd_imu_quat, sd_touch_l, sd_touch_r; /* 19, 28, 47, 48 */
} kbs_params;

/* One control step of physics state, SoA[F][ld] per field (ksim PhysicsData fields the Task reads). */
typedef struct kbs_state_view {
  const float* qpos;           /* [27][ld] */
  const float* qvel;           /* [26][ld] */
  const float* sensordata;     /* [49][ld] */
  const float* xpos;           /* [72][ld]  row 3*body+k */
  const float* xquat;          /* [96][ld]  row 4*body+k, (w,x,y,z) */
  const float* cinert;         /* [240][ld] row 10*body+k */
  const float* cvel;           /* [144][ld] row 6*body+k */
  const float* actuator_force; /* [20][ld] */
  const float* com_distance;   /* [ld]  COMDistanceObservation consumed as a recorded scalar */
  const float* time;           /* [ld]  episode time, seconds */
  int64_t ld;
} kbs_state_view;

/* PRNG-derived noise, supplied explicitly (parity mode: "identical inputs and PRNG-derived noise"). */
typedef struct kbs_noise_view {
  const float* eps_jpos;   /* [20][ld] U(-1,1)  AdditiveUniformNoise train.py:1160 */
  const float* eps_jvel;   /* [20][ld] U(-1,1)  train.py:1162 */
  const float* eps_gyro;   /* [3][ld]  N(0,1)   train.py:1176 */
  const float* eps_pg;     /* [3][ld]  N(0,1)   train.py:1194 */
} kbs_noise_view;

/* Per-episode randomisation (SURVEY F8): any pointer may be NULL = nominal / zero. */
typedef struct kbs_episode_view {
  const float* jpos_bias;  /* [20][ld] BiasedJointPositionObservation train.py:1158 */
  const float* pg_lag;     /* [ld]     ProjectedGravityObservation lag, train.py:1195-1196 */
  const float* pg_bias;    /* [3][ld]  train.py:1197 */
  const float* kp;         /* [20][ld] PositionActuators kp_scale etc., train.py:1097-1105 */
  const float* kd;         /* [20][ld] */
  const float* tau_limit;  /* [20][ld] */
  const float* action_bias;/* [20][ld] */
  const float* torque_bias;/* [20][ld] */
} kbs_episode_view;

/* eqx-layout weights of one network (device pointers). Linear.weight [out][in], LSTMCell.weight_ih
 * [4H][H], weight_hh [4H][H], bias [4H], gate order i,f,g,o (train.py:878-903, 964-989). */
typedef struct kbs_net_weights {
  const float* w_in;  const float* b_in;
  const float* w_ih[KBS_MAX_DEPTH]; const float* w_hh[KBS_MAX_DEPTH]; const float* b[KBS_MAX_DEPTH];
  const float* w_out; const float* b_out;
} kbs_net_weights;

/* Outputs of the actor head (any pointer may be NULL = not written). */
typedef struct kbs_actor_out {
  float* action;    /* [20][ld]  mode() or mean + std*eps      train.py:1564 */
  float* mean;      /* [20][ld]  low-pass-filtered mean        train.py:933-936 */
  float* std;       /* [20][ld]  train.py:929, PPOVariables.action_std 1487 */
  float* log_prob;  /* [ld]      of `action` (or of action_in) train.py:1452 */
  float* entropy;   /* [ld]      train.py:1486 */
} kbs_actor_out;

typedef struct kbs_handle kbs_handle;

int kbs_version(void);
const char* kbs_error_string(int code);
/* Fill *p with the reference launch configuration. */
int kbs_default_params(kbs_params* p);
int kbs_create(const kbs_params* p, kbs_handle** out);
int kbs_destroy(kbs_handle* h);
int kbs_get_params(const kbs_handle* h, kbs_params* out);

/* Replaces: equinox parameter pytrees of Actor/Critic (train.py:847-1004), loaded by
 * task.load_ckpt (convert.py:36-39).  Repacks into the kernel layouts (gate-interleaved, hi/lo split). */
int kbs_weights_pack(kbs_handle* h, int net, const kbs_net_weights* w, void* stream);

/* Replaces: HumanoidWalkingTask.get_observations + every Observation.observe (train.py:1155-1204, 682-707)
 * and the obs concatenations of run_actor / run_critic (train.py:1351-1431).
 *   computed   [78][ld] or NULL: rows 0-19 biased_joint_position, 20-39 noisy_biased_joint_position,
 *              40-59 noisy_joint_velocity, 60-62 noisy_imu_gyro, 63-68 feet_position, 69-71 projected_gravity,
 *              72-74 imu_projected_gravity, 75-77 noisy_imu_projected_gravity  (all other table entries are
 *              row slices of kbs_state_view and are not copied)
 *   actor_obs  [65][ld] or NULL;  critic_obs [475][ld] or NULL
 *   pg_carry   [3][ld] in/out lagged projected gravity state (may be NULL when episode->pg_lag is NULL)
 *   pg_reset   u8 [ld] or NULL: 1 = first step of a new episode, the lag state restarts at the current value
 *   noise may be NULL (then noisy twins = clean values). */
int kbs_observations(kbs_handle* h, const kbs_state_view* s, const kbs_noise_view* noise,
                     const kbs_episode_view* ep, const float* command, float* pg_carry,
                     const uint8_t* pg_reset, float* computed, float* actor_obs, float* critic_obs,
                     int64_t n_envs, void* stream);

/* Replaces: the per-physics-sub-step actuator path of ksim's engine (SURVEY 8f-2; train.py:1775-1781: dt 0.004,
 * ctrl_dt 0.02 => 5 sub-steps, action_latency_range (0.003, 0.01) s, drop_action_prob 0.05; engine semantics unverified):
 * a dropped command (u_drop < drop_prob) repeats the last applied action; sub-step k sees the new action once
 * k * sub_dt >= latency, the previous one before; ctrl_k = PositionActuators.get_ctrl on the sub-step's joint state.
 *   action [20][ld]; prev_action [20][ld] in/out (last applied action); u_drop, latency [ld];
 *   q_sub, qd_sub [S][20][ld] joint positions / velocities at each sub-step; ctrl_out [S][20][ld]. */
int kbs_torque_substeps(kbs_handle* h, const float* action, float* prev_action, const float* u_drop, const float* latency,
                        const float* q_sub, const float* qd_sub, const kbs_episode_view* ep, float* ctrl_out, int32_t n_substeps,
                        float sub_dt, float drop_prob, int64_t ld, int64_t n_envs, void* stream);

/* Replaces: ksim.compute_ppo_loss inside PPOTask (hyper-parameters: entropy_coef train.py:1767; the rest are ksim defaults,
 * unverified): clipped surrogate + (clipped) value loss + entropy bonus over a stored trajectory, reduced to means.
 *   ratio = exp(clip(log_probs - old_log_probs, +-log_clip_value)); policy = min(ratio A, clip(ratio, 1 +- eps) A)
 *   value = 0.5 max((tgt - v)^2, (tgt - (v_old + clip(v - v_old, +-eps)))^2)  (0.5 (tgt - v)^2 when not clipped)
 *   objective = policy - value_loss_coef value + entropy_coef entropy
 * All inputs [T][ld] (log-probs / entropy summed over the action dimensions, as kbs_ppo_variables returns them).
 * out (device, 4 floats): loss = -mean(objective), mean policy, mean value, mean entropy; the reduction order is fixed
 * (bitwise reproducible).  per_step [T][ld] optional: the objective per transition. */
typedef struct kbs_ppo_loss_params {
  float clip_param, value_loss_coef, entropy_coef, log_clip_value;
  int32_t use_clipped_value_loss;
} kbs_ppo_loss_params;
typedef struct kbs_ppo_loss_io {
  const float* log_probs; const float* old_log_probs; const float* advantages;
  const float* values; const float* old_values; const float* value_targets; const float* entropy;
  float* per_step;
  float* out;
  int64_t T, ld;
} kbs_ppo_loss_io;
int kbs_ppo_loss_default_params(kbs_ppo_loss_params* p);
int kbs_ppo_loss(kbs_handle* h, const kbs_ppo_loss_params* params, const kbs_ppo_loss_io* io, int64_t n_envs, void* stream);

/* Replaces: jax.grad of the PPO minibatch loss through get_ppo_variables (train.py:1435-1524) -- back-propagation through
 * time through both LSTM stacks, the projections, the actor head (softplus std, clamp, one-pole low-pass of the mean) and
 * ksim.compute_ppo_loss [U] (kbs_ppo_loss_params) -- for one minibatch of n stored trajectories of T steps (BASELINE
 * configs[3]; the per-rank gradients are then all-reduced over NCCL by the caller, see INTEGRATION.md).
 *   batch: env-major SoA arrays as kbs_ppo_variables takes them; *_carry0 [depth][2][n][H] / lpf0 [20][ld] = the carries
 *          at the first step (NULL = zeros, get_initial_model_carry)
 *   actor / critic: gradient buffers in the eqx layout of kbs_net_weights (written): w_in [H][num_in], b_in [H],
 *          w_ih / w_hh [4H][H], b [4H] per layer, w_out [num_out][H], b_out [num_out]
 *   log_probs / values / entropy [T][ld]: the forward outputs (written); stats_out: device, 4 floats as kbs_ppo_loss.
 * First version: fp32 FFMA GEMMs, deterministic (no atomics). */
typedef struct kbs_ppo_batch {
  const float* actor_obs;      /* [T][65][ld] */
  const float* critic_obs;     /* [T][475][ld] */
  const float* action;         /* [T][20][ld] */
  const uint8_t* done;         /* [T][ld] */
  const float* old_log_probs;  /* [T][ld] */
  const float* advantages;     /* [T][ld] */
  const float* value_targets;  /* [T][ld] */
  const float* old_values;     /* [T][ld] */
  const float* actor_carry0;   /* [depth][2][n][H] or NULL */
  const float* critic_carry0;  /* [depth][2][n][H] or NULL */
  const float* lpf0;           /* [20][ld] or NULL */
  int64_t T, ld;
} kbs_ppo_batch;
typedef struct kbs_net_grads {
  float* w_in;  float* b_in;
  float* w_ih[KBS_MAX_DEPTH]; float* w_hh[KBS_MAX_DEPTH]; float* b[KBS_MAX_DEPTH];
  float* w_out; float* b_out;
} kbs_net_grads;
int kbs_ppo_grad(kbs_handle* h, const kbs_ppo_loss_params* params, const kbs_ppo_batch* batch, const kbs_net_grads* actor,
                 const kbs_net_grads* critic, float* log_probs, float* values, float* entropy, float* stats_out,
                 int64_t n_envs, void* stream);
/* Overlap hook for the gradient all-reduce (the only collective of the path): kbs_ppo_grad finishes the critic's gradients
 * before the actor's; when `critic_ready` (a cudaEvent_t) is set, the next kbs_ppo_grad calls record it on their stream at
 * that point, so the caller can start reducing the critic's gradients on another stream while the actor's weight-gradient
 * GEMMs still run.  NULL clears it.  (The torch datapaths without the persistent kernels record it at the end.) */
int kbs_ppo_grad_set_events(kbs_handle* h, void* critic_ready);
/* Vector-Jacobian product of get_ppo_variables (train.py:1484-1487) on one minibatch: the gradient of a caller's loss, given
 * its cotangents d loss / d (log_probs, values, entropy, action_std), back-propagated through the same forward and BPTT as
 * kbs_ppo_grad.  Writes into actor / critic (layout of kbs_ppo_grad) sum_{t,e} ct . d var / d theta at the weights packed in
 * the handle, and the forward's log_probs / values / entropy [T][ld] (bitwise those of kbs_ppo_grad on the same batch).
 *   batch: as kbs_ppo_grad; old_log_probs, advantages, value_targets and old_values are not read (may be NULL).  The start
 *          carries, observations, actions and done are constants.  No mirror pass.
 *   ct: any member may be NULL (= zero cotangent).
 * Same datapaths as kbs_ppo_grad, selected the same way; honours kbs_ppo_grad_set_events; no host synchronisation (capturable).
 * Each network's cotangents are scaled on the device by a power of two chosen from their largest magnitude, and its gradients
 * by the inverse (exact), so any loss scale suits the FP16-split datapath: VJP(2^k ct) == 2^k VJP(ct) bitwise while nothing
 * leaves the normal range.  All-zero cotangents give zero gradients; a non-finite one propagates into its network's gradient. */
typedef struct kbs_ppo_cotangents {
  const float* log_probs;   /* [T][ld] */
  const float* values;      /* [T][ld] */
  const float* entropy;     /* [T][ld] */
  const float* action_std;  /* [T][20][ld] */
} kbs_ppo_cotangents;
int kbs_ppo_variables_vjp(kbs_handle* h, const kbs_ppo_batch* batch, const kbs_ppo_cotangents* ct, const kbs_net_grads* actor,
                          const kbs_net_grads* critic, float* log_probs, float* values, float* entropy, int64_t n_envs,
                          void* stream);
/* Replaces: optax.adam -- the adam_weight_decay == 0.0 branch of get_optimizer (train.py:1062-1063; NOT the branch the launch
 * config takes: see kbs_adamw_step): scale_by_adam, eps_root = 0, then -learning_rate, on one flat parameter array: g = grad * grad_scale (1 / world_size after a sum all-reduce, or a global-norm clip factor);
 * m = b1 m + (1 - b1) g; v = b2 v + (1 - b2) g^2; p -= lr (m / (1 - b1^step)) / (sqrt(v / (1 - b2^step)) + eps).  step >= 1. */
int kbs_adam_step(kbs_handle* h, float* param, const float* grad, float* m, float* v, int64_t count, float lr, float b1,
                  float b2, float eps, float grad_scale, int64_t step, void* stream);

/* Replaces: optax.adamw (train.py:1062-1065: the launch config keeps adam_weight_decay = 1e-5, train.py:99-102, so
 * get_optimizer returns optax.adamw(lr, weight_decay): scale_by_adam(b1, b2, eps, eps_root = 0) -> add_decayed_weights(wd)
 * -> scale by -lr) and ksim's gradient clipping around optimizer.update [U: global-norm clip to `max_grad_norm`, update
 * skipped when the norm is not finite].  One flat parameter array:
 *   g = grad * grad_scale * clip,  clip = min(1, max_grad_norm / max(norm * grad_scale, 1e-6))  (1 when grad_norm is NULL
 *       or max_grad_norm <= 0);  m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;
 *   p -= lr ((m / (1 - b1^step)) / (sqrt(v / (1 - b2^step)) + eps) + weight_decay p)
 * grad_norm: device, 1 float = the global L2 norm of `grad` (kbs_grad_norm), or NULL.  A non-finite norm leaves p, m, v
 * and the step counter untouched.  step_dev: device int64 = number of updates applied so far (read, then advanced by one
 * when the update is applied), so that the whole update can be replayed as one CUDA graph; NULL = use `step` (>= 1). */
typedef struct kbs_adamw_params {
  double b1, b2;   /* doubles: (1 - b) is formed in double (1.0f - 0.999f != 0.001f); m and v are updated in double and rounded once */
  float lr, eps, weight_decay, grad_scale, max_grad_norm;
} kbs_adamw_params;
int kbs_adamw_default_params(kbs_adamw_params* p);   /* lr 5e-4, b1 0.9, b2 0.999, eps 1e-8, wd 1e-5 [R]; clip 10.0 [U] */
int kbs_adamw_step(kbs_handle* h, float* param, const float* grad, float* m, float* v, int64_t count,
                   const kbs_adamw_params* o, const float* grad_norm, int64_t* step_dev, int64_t step, void* stream);
/* Replaces: optax.global_norm over the gradient pytree: norm_out (device, 1 float) = sqrt(sum grad^2), accumulated in
 * double in a fixed order (bitwise reproducible; identical on every rank after the all-reduce). */
int kbs_grad_norm(kbs_handle* h, const float* grad, int64_t count, float* norm_out, void* stream);

/* The update phase of a PPO epoch (train.py:1763-1766: num_passes 3, batch_size 512 trajectories): num_passes passes over the
 * stored rollout, each over a fresh random permutation of the env axis cut into n_envs / batch_size minibatches of whole
 * trajectories [U: ksim's update loop is not vendored; this is the library's reading of it].  ppo.PpoUpdater.epoch chains
 * kbs_ppo_variables -> kbs_gae -> per pass (kbs_minibatch_permutation -> kbs_shuffle_minibatches -> one update per
 * minibatch), all on the device.
 *
 * Replaces: jax.random.permutation over the env axis [U].  perm_out int32 [n_envs] = a uniform random permutation of
 * 0..n_envs-1, drawn on the device:
 *   key(e)   = word 0 of Philox4x32-10(counter = (pass lo, pass hi, env0 + e, 0xFFFFFFFF), key = seed)   (the function of
 *              kbs_generate_rollout_noise; no rollout-noise counter has 0xFFFFFFFF as its fourth word)
 *   perm_out = the low 32 bits of the 64-bit values (key(e) << 32) | e sorted ascending (ties broken by e: always a permutation)
 * pass_dev: device int64, read and then advanced by one (as step_dev of kbs_adamw_step), so a replayed CUDA graph draws a
 * new permutation on every pass.  env0: the rank's global env offset (rank * n_envs): with one seed, ranks draw different
 * permutations.  One CTA sorts in shared memory: n_envs <= KBS_MAX_PERMUTATION_ENVS, else KBS_E_SHAPE. */
#define KBS_MAX_PERMUTATION_ENVS 16384
int kbs_minibatch_permutation(kbs_handle* h, uint64_t seed, int64_t* pass_dev, int64_t env0, int32_t* perm_out, int64_t n_envs,
                              void* stream);
/* The rollout buffer cut into dense minibatches: column j of minibatch b is env perm[b * batch_size + j] of `src`.
 *   src: the whole rollout as kbs_ppo_grad takes a minibatch (SoA at src->ld, carries [depth][2][n_envs][H]).
 *   dst: every array [num_batches][T][F][batch_size] (done u8, the [T] fields with F = 1); carries
 *        [num_batches][depth][2][batch_size][H], lpf0 [num_batches][20][batch_size].  Minibatch b is then an ordinary
 *        kbs_ppo_batch with ld = batch_size at offset b of every array (whole 128-row panels keep kbs_ppo_grad's fast path).
 *   A NULL src carry / lpf0 (zeros at the first step) requires a NULL dst one.
 * batch_size % 4 == 0, num_batches * batch_size == n_envs <= KBS_MAX_PERMUTATION_ENVS, src->ld >= n_envs, src->ld % 4 == 0;
 * float arrays and perm 16-byte aligned, done 4-byte aligned.  An index of perm outside [0, n_envs) is never read through:
 * its float columns are written as NaN (done 0), so the update's non-finite skip refuses that minibatch.  One pass over
 * the buffer: a CTA stages one [T][F] row of n_envs values in shared memory and writes its num_batches segments. */
typedef struct kbs_ppo_minibatches {
  float* actor_obs; float* critic_obs; float* action; uint8_t* done;
  float* old_log_probs; float* advantages; float* value_targets; float* old_values;
  float* actor_carry0; float* critic_carry0; float* lpf0;
  int64_t batch_size, num_batches;
} kbs_ppo_minibatches;
int kbs_shuffle_minibatches(kbs_handle* h, const int32_t* perm, const kbs_ppo_batch* src, const kbs_ppo_minibatches* dst,
                            int64_t n_envs, void* stream);

/* Pins the handle's scratch allocation: while locked, a call that would have to grow (free + reallocate) the scratch
 * returns KBS_E_STATE instead -- a captured CUDA graph holds pointers into it (ppo.PpoUpdater.capture). */
int kbs_scratch_lock(kbs_handle* h, int on);

/* Replaces: the per-episode randomisation of ksim.PositionActuators (train.py:1097-1105: kp_scale = kd_scale = 1.4,
 * torque_limit_scale_low = 0.5, action_bias_scale = 0.02 rad, torque_bias_scale = 0.0 N m; fork b-vm/ksim [U]: the sampling
 * law below is this library's reading, every scale is a parameter).  Randomness explicit: u [5][20][ld] U[0,1) rows for
 * (kp, kd, tau_limit, action_bias, torque_bias).
 *   kp  = kp_nominal  * (1/kp_scale + u (kp_scale - 1/kp_scale));   kd likewise with kd_scale
 *   tau_limit = ctrl_limit * (low + u (1 - low));   action_bias = (2u - 1) action_bias_scale;  torque_bias likewise
 * reset u8 [ld] or NULL: only envs with reset != 0 are resampled (episode boundaries), the others keep their values.
 * Writes the kp / kd / tau_limit / action_bias / torque_bias arrays of *ep ([20][ld] each; NULL = skipped). */
typedef struct kbs_actuator_rand_params {
  float kp_scale, kd_scale, torque_limit_scale_low, action_bias_scale, torque_bias_scale;
} kbs_actuator_rand_params;
int kbs_actuator_rand_default_params(kbs_actuator_rand_params* p);
int kbs_sample_actuator_randomization(kbs_handle* h, const kbs_actuator_rand_params* rp, const float* u, const uint8_t* reset,
                                      const kbs_episode_view* ep, int64_t ld, int64_t n_envs, void* stream);

/* Replaces: COMDistanceObservation.observe (train.py:509-659): distance between subtree_com[2].xy and the centroid of the
 * convex hull (Andrew's monotone chain) of the floor-contact points, -1 when fewer than 3 distinct contact.geom2 values.
 *   contact_geom1 / contact_geom2  int32 [T][ncon][ld]   (MJX contact.geom1 / geom2, padding included)
 *   contact_pos                    [T][3 ncon][ld]       row 3 c + k = contact.pos[c][k]
 *   subtree_com_base               [T][3][ld]            data.subtree_com[2]
 *   com_distance                   [T][ld] out           (what kbs_state_view.com_distance / the COM reward consume)
 * 3 <= ncon <= 32. */
int kbs_com_distance(kbs_handle* h, const int32_t* contact_geom1, const int32_t* contact_geom2, const float* contact_pos,
                     const float* subtree_com_base, float* com_distance, int ncon, int64_t T, int64_t ld, int64_t n_envs,
                     void* stream);

/* Host -> device upload of T recorded steps of MuJoCo-shaped state ([T][rows][ld] per array, pinned host memory for
 * asynchronous copies): only the rows the path reads cross PCIe -- qpos, qvel, actuator_force, com_distance, time in
 * full; sensordata rows imu_gyro / imu_site_quat / foot touch; xpos / xquat of base and both feet; cinert[1:], cvel[1:]
 * (473 of the 676 rows, row indices from kbs_params).  One cudaMemcpy2DAsync per row range on `stream`; arrays whose
 * pointer is NULL in either view are skipped.  *bytes_out (optional) = bytes enqueued. */
int kbs_upload_state(kbs_handle* h, const kbs_state_view* host, const kbs_state_view* dev, int64_t T, int64_t* bytes_out,
                     void* stream);

/* Replaces: mirror_obs + mirror_cmd (train.py:1584-1756) followed by the run_actor / run_critic concatenations on the
 * mirrored observations (train.py:1463-1481), for T stored steps.  The mirror acts on the RAW named observations, so it
 * is built from what the rollout stored: `computed` [T][78][ld] (kbs_observations), the recorded state (time-major
 * [T][rows][ld] arrays in *s) and `command` [T][16][ld].
 *   actor_obs [T][65][ld] / critic_obs [T][475][ld] / command_out [T][16][ld]: any may be NULL (not all). */
int kbs_mirror_observations(kbs_handle* h, const kbs_state_view* s, const float* computed, const float* command,
                            float* actor_obs, float* critic_obs, float* command_out, int64_t T, int64_t n_envs,
                            void* stream);
/* Replaces: mirror_joints (train.py:1574-1582): out = -[in[5:10], in[0:5], in[10:15], in[15:20]] on [T][20][ld]
 * (legs swapped, arm halves NOT exchanged -- as the reference writes it).  in != out. */
int kbs_mirror_joints(kbs_handle* h, const float* in, float* out, int64_t T, int64_t ld, int64_t n_envs, void* stream);

/* Replaces: UnifiedCommand.__call__/initial_command (train.py:724-785).  Randomness explicit:
 *   u_switch [ld] U[0,1); mode int32 [ld] in 0..5; u6 [6][ld]; u_arms [10][ld].  u_switch NULL = always
 *   resample (initial_command).  command [16][ld] in/out. */
int kbs_command_update(kbs_handle* h, float* command, const float* u_switch, const int32_t* mode,
                       const float* u6, const float* u_arms, int64_t ld, int64_t n_envs, void* stream);

/* Replaces: sample_action -> run_actor -> Actor.forward (train.py:1545-1572, 1351-1379, 913-941) and the
 * actor half of _ppo_scan_fn (train.py:1443-1452, 1486-1487).
 *   obs [65][ld]; carry AoS [depth][2][n][H] in/out; lpf [20][ld] in/out; eps [20][ld] or NULL (argmax);
 *   action_in [20][ld] or NULL: if given, log_prob is evaluated at action_in (stored transition);
 *   done [ld] or NULL: carries and lpf reset to initial (zeros) where done (train.py:1502-1506). */
int kbs_actor_step(kbs_handle* h, const float* obs, int64_t ld, float* carry, float* lpf, const float* eps,
                   const float* action_in, const uint8_t* done, const kbs_actor_out* out, int64_t n_envs,
                   void* stream);

/* Replaces: run_critic -> Critic.forward (train.py:1381-1433, 993-1004). obs [475][ld]; value [ld]. */
int kbs_critic_step(kbs_handle* h, const float* obs, int64_t ld, float* carry, const uint8_t* done,
                    float* value, int64_t n_envs, void* stream);

/* Replaces: get_actuators -> ksim.PositionActuators.get_ctrl (train.py:1091-1105).
 *   action, ctrl_out [20][ld]; q = qpos rows 7.., qd = qvel rows 6.. of the state view. */
int kbs_torque(kbs_handle* h, const float* action, const kbs_state_view* s, const kbs_episode_view* ep,
               float* ctrl_out, int64_t n_envs, void* stream);

/* Replaces: get_terminations + TerrainBadZTermination.__call__ (train.py:1258-1269, 817-823) and ksim's
 * done/success reduction.  codes int32 [3][ld] (bad_z, not_upright, episode_length); done/success u8 [ld];
 * pre [2][ld] or NULL: pre-threshold values (height, tilt) for tolerance-based checking. */
int kbs_terminate(kbs_handle* h, const kbs_state_view* s, int32_t* codes, uint8_t* done, uint8_t* success,
                  float* pre, int64_t n_envs, void* stream);

/* Trajectory-wise inputs of get_rewards: T steps of state plus the recorded command / ctrl / done. */
typedef struct kbs_traj_view {
  kbs_state_view state;   /* each field [T][F][ld] */
  const float* command;   /* [T][16][ld] */
  const float* ctrl;      /* [T][20][ld]  Trajectory.ctrl (train.py:504) */
  const uint8_t* done;    /* [T][ld] */
  int64_t T;
} kbs_traj_view;

/* Reward carries (train.py:135-136, 175-178), in/out: t_single [ld], airtime [2][ld], prev_contact u8 [2][ld]. */
typedef struct kbs_reward_carry {
  float* t_single; float* airtime; uint8_t* prev_contact;
} kbs_reward_carry;

/* Replaces: get_rewards table + the 12 Reward.get_reward[_stateful] (train.py:125-506, 1224-1256) and
 * ksim's scale-and-sum.  total [T][ld]; components [T][12][ld] or NULL. */
int kbs_rewards(kbs_handle* h, const kbs_traj_view* traj, const kbs_reward_carry* carry, float* total,
                float* components, int64_t n_envs, void* stream);

/* Replaces: ksim.compute_ppo_inputs (GAE; PPOConfig gamma/lam train.py:1769-1770).
 * values, rewards [T][ld]; done, success u8 [T][ld]; advantages, value_targets [T][ld]. */
int kbs_gae(kbs_handle* h, const float* values, const float* rewards, const uint8_t* done,
            const uint8_t* success, float* advantages, float* value_targets, int64_t T, int64_t ld,
            int64_t n_envs, void* stream);

/* Replaces: convert.py:84-119 step_fn (kinfer policy step).  AoS inputs as the exported function takes them:
 * joint_angles [n][20], joint_vel [n][20], projected_gravity [n][3], gyro [n][3], command [n][16],
 * carry [n][depth*2*H+20] in -> carry_out; action_out [n][20] = dist.mode(). */
int kbs_policy_step(kbs_handle* h, const float* joint_angles, const float* joint_vel,
                    const float* projected_gravity, const float* gyro, const float* command,
                    const float* carry_in, float* carry_out, float* action_out, int64_t n_envs, void* stream);

/* Fused rollout control step over T recorded steps (T=1: the per-step call ksim's engine loop makes):
 * observations -> actor -> sample -> torque -> terminations -> command update -> carry reset on done,
 * and (if critic_value != NULL) critic obs -> critic -> value.  Replaces the body of ksim's step_engine
 * around mjx.step (SURVEY 3.2) for recorded/synthetic state.
 * All per-step arrays are trajectories [T][...][ld]. */
typedef struct kbs_rollout_io {
  kbs_state_view state;           /* [T][F][ld] */
  kbs_noise_view noise;           /* [T][..][ld] */
  kbs_episode_view episode;       /* per-env, no time axis */
  const float* eps_action;        /* [T][20][ld] N(0,1) or NULL (argmax) */
  const float* u_switch;          /* [T][ld] */
  const int32_t* cmd_mode;        /* [T][ld] */
  const float* cmd_u6;            /* [T][6][ld] */
  const float* cmd_u_arms;        /* [T][10][ld] */
  float* command;                 /* [T+1][16][ld]: row 0 = command at step 0 (input); row t+1 written */
  float* pg_carry;                /* [3][ld] in/out */
  float* actor_carry;             /* AoS [depth][2][n][H] in/out */
  float* critic_carry;            /* AoS [depth][2][n][H] in/out (used if value != NULL) */
  float* lpf;                     /* [20][ld] in/out */
  float* actor_obs;               /* [T][65][ld] or NULL (stored for the PPO pass) */
  float* action;                  /* [T][20][ld] */
  float* log_prob;                /* [T][ld] or NULL */
  float* ctrl;                    /* [T][20][ld] */
  int32_t* term_codes;            /* [T][3][ld] or NULL */
  uint8_t* done;                  /* [T][ld] */
  uint8_t* success;               /* [T][ld] */
  float* value;                   /* [T][ld] or NULL */
  int64_t T;
} kbs_rollout_io;

int kbs_rollout(kbs_handle* h, const kbs_rollout_io* io, int64_t n_envs, void* stream);

/* kbs_rollout plus what crosses a call boundary and what the PPO update trains on.  kbs_rollout(h, io, n, s) is
 * kbs_rollout_record(h, io, NULL, n, s); either pointer of `rec` may be NULL.
 *
 * done_prev [ld] u8 (4-byte aligned): done of the step before this call's step 0, i.e. the previous call's done[T-1].  On
 * step 0, where done_prev[e] != 0, the lagged projected-gravity state (pg_carry) restarts at the current value, exactly as it
 * does inside a call on the step after done[t-1].  That is the only stage that reads the previous step's done: the actor /
 * critic carries and the action filter (lpf) are reset after step t from done[t] within the step, command[t+1] is drawn
 * from done[t], and kbs_rewards pads t = 0 of a trajectory as the reference does (no previous step).  So a rollout split
 * into calls, each passing the previous call's done[T-1] here, is the same rollout as one call over all steps; without it,
 * an episode that ends on a call's last step keeps its lag state into the next episode.  T = 1 calls (one per control step
 * around the simulator) need it at every episode end.
 *
 * critic_obs [T][475][ld] (16-byte aligned): the run_critic concatenation of every step, all 475 rows, as
 * kbs_observations(critic_obs) writes it -- what kbs_ppo_variables / kbs_ppo_grad train the critic on.  It may be requested
 * with io->value == NULL (the rows are written, the critic is not run); it needs the state rows the concatenation reads
 * (cinert, cvel, actuator_force; else KBS_E_NULL).  Requesting it changes no other output of the call.
 *
 * Declared as a plain struct tag (like POSIX `struct stat` / stat()): the function owns the ordinary name. */
struct kbs_rollout_record {
  const uint8_t* done_prev;   /* [ld] or NULL */
  float* critic_obs;          /* [T][475][ld] or NULL */
};
int kbs_rollout_record(kbs_handle* h, const kbs_rollout_io* io, const struct kbs_rollout_record* rec, int64_t n_envs,
                       void* stream);

/* The online rollout: one control step per call, the form a simulator loop around mjx.step drives (state t+1 depends on
 * the ctrl of step t).  What crosses a step boundary stays on the device in a caller-owned STEP STATE: one device buffer of
 * kbs_step_state_bytes bytes, 256-byte aligned (any cudaMalloc'd or torch-allocated buffer is).  The library keeps none of
 * it in its scratch, which every other entry point reuses between steps.  It holds:
 *   - the actor and critic carries in the operand layouts the rollout kernels read and write: on the tensor-core datapaths
 *     the split-blocked h operand in two slots with a device word naming the slot the next step reads, and the fp32 c and h;
 *     on SIMT the ABI carries;
 *   - lpf, pg_carry, the current command row and done_prev (the previous step's done);
 *   - the step index t (device int64): every kbs_rollout_step reads it and then advances it by one, like step_dev of
 *     kbs_adamw_step, so one captured CUDA graph of the step serves every step of an iteration.
 * Its per-env rows are at ld = n_envs rounded up to a multiple of 4; the arrays kbs_rollout_step takes use that ld too. */
typedef struct kbs_step_state {
  void* buf;                  /* device, 256-byte aligned */
  uint64_t bytes;             /* size of buf: >= kbs_step_state_bytes(h, n_envs, with_critic) */
  int64_t n_envs;
  int32_t with_critic;        /* room for the critic's carries (kbs_rollout_step with value != NULL needs it) */
} kbs_step_state;
int kbs_step_state_bytes(kbs_handle* h, int64_t n_envs, int with_critic, uint64_t* bytes);

/* ABI form of what a step state carries.  On load any pointer may be NULL (= zeros: get_initial_model_carry, no previous
 * done); on store NULL = not written. */
typedef struct kbs_step_carry {
  float* actor_carry;         /* AoS [depth][2][n][H] */
  float* critic_carry;        /* AoS [depth][2][n][H] (with_critic states only) */
  float* lpf;                 /* [20][ld] */
  float* pg_carry;            /* [3][ld] */
  float* command;             /* [16][ld]: the command of the next step (row 0 of a rollout's command) */
  uint8_t* done_prev;         /* [ld], 4-byte aligned: the done of the step before the next one */
} kbs_step_carry;
/* Fills the state from `in` and sets t = 0 and the h slot to 0. */
int kbs_step_state_load(kbs_handle* h, const kbs_step_state* st, const kbs_step_carry* in, void* stream);
/* The reverse, leaving the state as it is.  After the same steps, the carries, lpf, pg_carry and command are bitwise what
 * kbs_rollout_record leaves in io (command: row T), and done_prev is its done[T-1]. */
int kbs_step_state_store(kbs_handle* h, const kbs_step_state* st, const kbs_step_carry* out, void* stream);
/* Sets the step index back to 0 and changes nothing else: the next iteration of an online rollout records into slot 0 again.
 * It does not repair a state that a step past T left behind (see kbs_rollout_step): load that one again. */
int kbs_step_state_rewind(kbs_handle* h, const kbs_step_state* st, void* stream);

/* One control step of the online rollout.  Inputs are this step's [F][ld] arrays.  Outputs are trajectories; slot t is
 * written, t being the state's step index read on the device.  The stages are those of kbs_rollout_record, and T calls from a
 * loaded state give bitwise the outputs of one T-step kbs_rollout_record call (with done_prev, and critic_obs where asked)
 * from the same carries. */
typedef struct kbs_step_io {
  kbs_state_view state;       /* this step: [F][ld] */
  kbs_noise_view noise;       /* this step: [..][ld] */
  kbs_episode_view episode;   /* per env */
  const float* eps_action;    /* [20][ld] N(0,1) or NULL (argmax) */
  const float* u_switch;      /* [ld] */
  const int32_t* cmd_mode;    /* [ld] */
  const float* cmd_u6;        /* [6][ld] */
  const float* cmd_u_arms;    /* [10][ld] */
  /* trajectories [T][..][ld], slot t written */
  float* command;             /* [T+1][16][ld]: rows t (the state's command) and t+1 (the next one) */
  float* actor_obs;           /* [T][65][ld] or NULL */
  float* critic_obs;          /* [T][475][ld] or NULL (needs cinert, cvel, actuator_force in state) */
  float* action;              /* [T][20][ld] */
  float* log_prob;            /* [T][ld] or NULL */
  float* ctrl;                /* [T][20][ld] */
  int32_t* term_codes;        /* [T][3][ld] or NULL */
  uint8_t* done;              /* [T][ld] */
  uint8_t* success;           /* [T][ld] */
  float* value;               /* [T][ld] or NULL (the critic is not run); needs a with_critic state and cinert, cvel,
                                 actuator_force */
  kbs_state_view traj_state;  /* [T][F][ld]: copies of this step's state fields (what kbs_rewards reads afterwards); a NULL
                                 field is not recorded, and needs a non-NULL state field otherwise; ld ignored */
  int64_t T;                  /* trajectory length */
} kbs_step_io;
/* The step's index is only known on the device.  A step that finds t >= T records nothing and leaves t as it is; it sets
 * KBS_STATUS_STEP_RANGE in the health word, so the next fused call returns KBS_E_DEVICE.  The carries in the state did
 * advance: load it again.  On the tensor-core datapaths the recurrence is the persistent kernel with T = 1 (KBS_E_SHAPE for an
 * n_envs it cannot take). */
int kbs_rollout_step(kbs_handle* h, const kbs_step_state* st, const kbs_step_io* io, void* stream);

/* The physics sub-steps between two online control steps (ksim's engine loop: S = ctrl_dt / dt calls of mjx.step per control
 * step, train.py:1775-1781: dt 0.004, ctrl_dt 0.02 => 5, action_latency_range (0.003, 0.01) s, drop_action_prob 0.05).
 * Before each mjx.step the engine calls PositionActuators.get_ctrl on that sub-step's joint state.  The rule [U], the same as
 * kbs_torque_substeps and oracle.position_actuator_substeps:
 *   applied = u_drop < drop_prob ? prev_action : action         (a dropped command repeats the last applied action)
 *   ctrl_k  = PD(k * sub_dt >= latency ? applied : prev_action, q_k, qd_k)          k = 0 .. S-1
 *   after sub-step S-1: prev_action = applied
 * With a simulator in the loop the joint state of sub-step k+1 depends on ctrl_k, so the sub-steps are one call each.  What
 * crosses a sub-step stays on the device in a caller-owned ACTUATOR STATE, beside the step state: one device buffer of
 * kbs_actuator_state_bytes bytes, 256-byte aligned, holding the sub-step index k (device int32), prev_action [20][ld] (the last
 * applied action) and applied [20][ld] (this control step's latched action), rows at ld = n_envs rounded up to a multiple of 4. */
typedef struct kbs_actuator_state {
  void* buf;                  /* device, 256-byte aligned */
  uint64_t bytes;             /* size of buf: >= kbs_actuator_state_bytes(h, n_envs) */
  int64_t n_envs;
  int32_t n_substeps;         /* S: sub-steps per control step (> 0) */
} kbs_actuator_state;
int kbs_actuator_state_bytes(kbs_handle* h, int64_t n_envs, uint64_t* bytes);
/* prev_action [20][ld] or NULL (= zeros); sets k = 0. */
int kbs_actuator_state_load(kbs_handle* h, const kbs_actuator_state* ast, const float* prev_action, void* stream);
/* prev_action [20][ld] <- the state's last applied action; the state is left as it is. */
int kbs_actuator_state_store(kbs_handle* h, const kbs_actuator_state* ast, float* prev_action, void* stream);

/* One sub-step's inputs and output.  Arrays are [F][ld] at the states' ld unless stated otherwise. */
typedef struct kbs_substep_io {
  const float* action;        /* [T][20][ld]: the action trajectory the control steps record (kbs_step_io.action) */
  int64_t T;
  const float* u_drop;        /* [ld] U[0,1) of this control step */
  const float* latency;       /* [ld] seconds, of this control step */
  const float* qpos;          /* [27][ld] this sub-step's joint state: rows 7.. are q (as kbs_torque reads them) */
  const float* qvel;          /* [26][ld] rows 6.. are qd */
  kbs_episode_view episode;   /* gains, limits and biases; NULL fields = nominal / zero */
  float* ctrl;                /* [20][ld] out */
  float sub_dt;               /* > 0 (dt of the physics step) */
  float drop_prob;            /* in [0, 1] */
} kbs_substep_io;
/* Sub-step k of the control step that kbs_rollout_step just ran, t being the step state's device index (already advanced, so
 * the step's action is action[t-1]).  At k = 0 it latches `applied`; it writes ctrl; it then advances k, and after sub-step S-1
 * it sets prev_action = applied and k = 0.  So S calls after a step give bitwise the S rows of ctrl, and the same prev_action,
 * that kbs_torque_substeps gives for action[t-1] and the S joint states stacked.  t and k are read on the device: one captured
 * sub-step replays for every sub-step of every control step.  Run the sub-steps of step T-1 before the step state is rewound.
 * A sub-step that finds t = 0 (no step since load or rewind), t > T or k >= S writes nothing and leaves k as it is; it sets
 * KBS_STATUS_SUBSTEP_RANGE, so the next fused call returns KBS_E_DEVICE.
 * KBS_E_SHAPE: the two states' n_envs differ, n_substeps <= 0, T <= 0.  KBS_E_PARAM: sub_dt <= 0, drop_prob outside [0, 1]. */
int kbs_actuator_substep(kbs_handle* h, const kbs_step_state* st, const kbs_actuator_state* ast, const kbs_substep_io* io,
                         void* stream);

/* Replaces: the jax.random draws the reference makes ON THE DEVICE during a rollout -- observation noise (train.py:1160, 1162,
 * 1176, 1194), the action sample (train.py:1564), the command resampling (train.py:725-737, 752-753, 782-783) -- for callers
 * that do not need bit parity with JAX's threefry streams (parity mode hands these arrays to kbs_rollout explicitly).
 * Counter-based Philox4x32-10: value (row r, step step0 + t, env e) depends only on (seed, r, step0 + t, e), so any split of a
 * rollout into calls gives the same numbers.  Fills, for T steps (any pointer may be NULL = skipped):
 *   noise->eps_jpos, eps_jvel [T][20][ld] U(-1,1); eps_gyro, eps_pg [T][3][ld] N(0,1); eps_action [T][20][ld] N(0,1);
 *   u_switch [T][ld] U[0,1); cmd_mode int32 [T][ld] in 0..5; cmd_u6 [T][6][ld], cmd_u_arms [T][10][ld] U[0,1). */
int kbs_generate_rollout_noise(kbs_handle* h, uint64_t seed, int64_t step0, const kbs_noise_view* noise, float* eps_action,
                               float* u_switch, int32_t* cmd_mode, float* cmd_u6, float* cmd_u_arms, int64_t T, int64_t ld,
                               int64_t n_envs, void* stream);

/* Replaces: get_ppo_variables -> xax.scan(_ppo_scan_fn) (train.py:1435-1524): on a STORED trajectory, re-run actor and
 * critic step by step from `*_carry`, carries reset to initial where done[t] (train.py:1502-1506), and return what
 * ksim.PPOVariables holds.  The observations are the stored ones (Trajectory.obs): actor_obs [T][65][ld] is the
 * run_actor concat of the noisy observations, critic_obs [T][475][ld] the run_critic concat (both are outputs of
 * kbs_observations / kbs_rollout).  The mirror passes (aux_losses, scaled by 0.0 in the launch config
 * train.py:1771-1772) are evaluated by calling this function again on mirrored observations (see INTEGRATION.md). */
typedef struct kbs_ppo_io {
  const float* actor_obs;   /* [T][65][ld] */
  const float* critic_obs;  /* [T][475][ld] or NULL (then values is not written) */
  const float* action;      /* [T][20][ld]  Trajectory.action */
  const uint8_t* done;      /* [T][ld] */
  float* actor_carry;       /* AoS [depth][2][n][H] in/out */
  float* critic_carry;      /* AoS [depth][2][n][H] in/out (if critic_obs) */
  float* lpf;               /* [20][ld] in/out */
  float* log_probs;         /* [T][ld]      PPOVariables.log_probs  train.py:1484 */
  float* values;            /* [T][ld]      PPOVariables.values     train.py:1485 */
  float* entropy;           /* [T][ld]      PPOVariables.entropy    train.py:1486 */
  float* action_std;        /* [T][20][ld]  PPOVariables.action_std train.py:1487, or NULL */
  float* mean;              /* [T][20][ld]  dist.mean() (for the mirror loss), or NULL */
  int64_t T, ld;
  /* aux_losses of PPOVariables (train.py:1462-1481, 1488-1491): the actor and the critic run a second time on the MIRRORED
   * observations (kbs_mirror_observations: mirror_obs + mirror_cmd followed by the run_actor / run_critic concatenations)
   * with their own carries, and
   *   action_mirror_loss = mean_j (mean - mirror_joints(mean_mirrored))^2 * actor_mirror_loss_scale
   *   value_mirror_loss  = (value - value_mirrored)^2 * critic_mirror_loss_scale
   * All NULL = not evaluated.  The launch config scales both by 0.0 (train.py:1771-1772); the defaults are 1.0 / 0.01. */
  const float* actor_obs_mirror;   /* [T][65][ld] */
  const float* critic_obs_mirror;  /* [T][475][ld] or NULL (then value_mirror_loss is not written) */
  float* actor_mirror_carry;       /* AoS [depth][2][n][H] in/out  (carry["actor_mirror"]) */
  float* critic_mirror_carry;      /* AoS [depth][2][n][H] in/out  (carry["critic_mirror"]) */
  float* lpf_mirror;               /* [20][ld] in/out              (carry["lpf_params_mirror"]) */
  float* action_mirror_loss;       /* [T][ld] */
  float* value_mirror_loss;        /* [T][ld] */
  float actor_mirror_loss_scale, critic_mirror_loss_scale;
} kbs_ppo_io;
int kbs_ppo_variables(kbs_handle* h, const kbs_ppo_io* io, int64_t n_envs, void* stream);

/* Number of kernel launches this library has enqueued since the handle was created (bench bookkeeping). */
int64_t kbs_launch_count(const kbs_handle* h);

/* Device-side health word of the fused rollout (kbs_rollout / kbs_ppo_variables on the tensor-core paths run all T
 * steps as one persistent kernel whose CTAs wait on each other's progress counters; a wait that times out is recorded
 * here instead of hanging).  Synchronises with the device.  *status_out == 0: healthy. */
int kbs_device_status(kbs_handle* h, int* status_out);
/* Status bits: 1 / 2 = a dependency wait of an LSTM / head item timed out (the kernel then drains without waiting: its
 * outputs are garbage); 0x100 = a value handed to the FP16-split tensor-core datapath was non-finite or >= 65504 in
 * magnitude (it would silently become inf: use KBS_GEMM_TC_3XTF32 / KBS_GEMM_SIMT_FP32 for such inputs).  The word is
 * sticky; the fused entry points (kbs_rollout, kbs_ppo_variables, kbs_policy_step, kbs_ppo_grad) copy it to the host after
 * their kernels and return KBS_E_DEVICE at the next call that finds it set.  Reset: synchronises and clears it. */
#define KBS_STATUS_TIMEOUT_LSTM 1
#define KBS_STATUS_TIMEOUT_HEAD 2
#define KBS_STATUS_F16_RANGE 0x100
#define KBS_STATUS_STEP_RANGE 0x200   /* kbs_rollout_step found its step index t >= T */
#define KBS_STATUS_SUBSTEP_RANGE 0x400 /* kbs_actuator_substep found t = 0, t > T or k >= S */
int kbs_device_status_reset(kbs_handle* h);

/* Per-kernel device timing for bench.py's roofline line: while enabled, every kernel launch of this handle is
 * bracketed by CUDA events on its launch stream (up to 8192 launches; do not enable during stream capture).
 * kbs_profile_read sums elapsed ms and launch counts per kernel id (ids 0..KBS_NUM_KERNEL_IDS-1, names from
 * kbs_kernel_name); returns 1 if the event pool overflowed (totals partial), 0 ok. */
/* Test hook of the tcgen05 datapath: pre-activation gates [n][4H] (eqx order i,f,g,o, bias added) of LSTM layer
 * `layer` of `net` for row-major x [n][H], h [n][H].  Needs a tensor-core gemm_path (KBS_GEMM_TC_3XTF32 or
 * KBS_GEMM_TC_2XF16) and packed weights: x and h are split as that datapath splits its operands. */
int kbs_debug_tc_gates(kbs_handle* h, int net, int layer, const float* x_rm, const float* h_rm, float* gates_out,
                       int64_t n_envs, void* stream);

/* Profiling hook: one LSTM layer launch (both nets) with per-CTA clock64 stamps, trace_out device int64 [ctas][8]
 * (start, setup done, first stage landed, MMAs issued, accumulators ready, epilogue done, smid, -). */
int kbs_debug_tc_trace(kbs_handle* h, long long* trace_out, int64_t n_envs, void* stream);
/* Same stamps for LSTM layer `layer` at step `step` of subsequent kbs_rollout calls (trace_out NULL detaches). */
int kbs_debug_tc_trace_attach(kbs_handle* h, long long* trace_out, int64_t step, int layer);

#define KBS_NUM_KERNEL_IDS 26
int kbs_profile_enable(kbs_handle* h, int on);
int kbs_profile_read(kbs_handle* h, int max_ids, double* total_ms, int64_t* launches);
const char* kbs_kernel_name(int id);

#ifdef __cplusplus
}
#endif
#endif /* KBOTSTEP_H_ */
