// kbs_api.cu -- the extern "C" boundary of libkbotstep.so (include/kbotstep.h): argument validation, scratch
// management and stage orchestration.  No CPU fallback: every entry point enqueues sm_100a kernels or fails.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "kbs_common.cuh"

namespace {

inline int64_t round_up4(int64_t n) { return (n + 3) / 4 * 4; }

int check_ld(int64_t ld, int64_t n) {
  if (n <= 0) return KBS_E_SHAPE;
  if (ld < round_up4(n)) return KBS_E_SHAPE;
  if (ld % 4) return KBS_E_ALIGN;
  return KBS_OK;
}

#define REQ(p)            \
  do {                    \
    if (!(p)) return KBS_E_NULL; \
  } while (0)
#define AL(p)                                     \
  do {                                            \
    if ((p) && !kbs_aligned16(p)) return KBS_E_ALIGN; \
  } while (0)

int check_state(const kbs_state_view* s, int64_t n, bool need_priv) {
  REQ(s);
  REQ(s->qpos); REQ(s->qvel);
  int rc = check_ld(s->ld, n);
  if (rc) return rc;
  AL(s->qpos); AL(s->qvel); AL(s->sensordata); AL(s->xpos); AL(s->xquat); AL(s->cinert); AL(s->cvel);
  AL(s->actuator_force); AL(s->com_distance); AL(s->time);
  if (need_priv) { REQ(s->sensordata); REQ(s->xpos); REQ(s->xquat); }
  return KBS_OK;
}

kbs_state_view state_at(const kbs_state_view& s, int64_t t) {
  kbs_state_view o = s;
  const int64_t ld = s.ld;
  if (s.qpos) o.qpos = s.qpos + t * KBS_NQ * ld;
  if (s.qvel) o.qvel = s.qvel + t * KBS_NV * ld;
  if (s.sensordata) o.sensordata = s.sensordata + t * KBS_NSENSORDATA * ld;
  if (s.xpos) o.xpos = s.xpos + t * 3 * KBS_NBODY * ld;
  if (s.xquat) o.xquat = s.xquat + t * 4 * KBS_NBODY * ld;
  if (s.cinert) o.cinert = s.cinert + t * 10 * KBS_NBODY * ld;
  if (s.cvel) o.cvel = s.cvel + t * 6 * KBS_NBODY * ld;
  if (s.actuator_force) o.actuator_force = s.actuator_force + t * KBS_NUM_JOINTS * ld;
  if (s.com_distance) o.com_distance = s.com_distance + t * ld;
  if (s.time) o.time = s.time + t * ld;
  return o;
}

kbs_noise_view noise_at(const kbs_noise_view& z, int64_t t, int64_t ld) {
  kbs_noise_view o = z;
  if (z.eps_jpos) o.eps_jpos = z.eps_jpos + t * 20 * ld;
  if (z.eps_jvel) o.eps_jvel = z.eps_jvel + t * 20 * ld;
  if (z.eps_gyro) o.eps_gyro = z.eps_gyro + t * 3 * ld;
  if (z.eps_pg) o.eps_pg = z.eps_pg + t * 3 * ld;
  return o;
}

constexpr int kOutLd = 64;  // row stride of the trunk output buffer

// Workspace of one trunk evaluation: the exact-fp32 trunk's, or the tensor-core LSTM stack's plus its row-major input and
// top-layer output [n][H]; then the trunk's output out_rm [n][kOutLd].
struct TrunkWs { KbsSimtTrunkWs simt; KbsTcStackWs tc; float* x_rm; float* hbuf; float* out_rm; };
TrunkWs trunk_ws(KbsScratch& s, const kbs_handle* h, int64_t n) {
  TrunkWs w{};
  if (h->p.gemm_path == KBS_GEMM_SIMT_FP32) {
    w.simt = kbs_simt_trunk_ws(s, h, n);
  } else {
    w.tc = kbs_tc_stack_ws(s, h, n);
    w.x_rm = s.take<float>(size_t(n) * h->p.hidden_size);
    w.hbuf = s.take<float>(size_t(n) * h->p.hidden_size);
  }
  w.out_rm = s.take<float>(size_t(n) * kOutLd);
  return w;
}

int trunk(kbs_handle* h, int net, const float* obs, int64_t ld, float* carry, const uint8_t* done, const TrunkWs& ws, int64_t n,
          cudaStream_t st) {
  if (h->p.gemm_path == KBS_GEMM_SIMT_FP32) return kbs_simt_trunk(h, net, obs, ld, carry, done, ws.out_rm, ws.simt, n, st);
  // tensor-core path: input_proj (FFMA, K = 65 / 475) -> LSTM stack on tcgen05 -> output_proj (FFMA, N = 40 / 1)
  int rc;
  if ((rc = kbs_simt_in_proj(h, net, obs, ld, ws.x_rm, n, st))) return rc;
  if ((rc = kbs_tc_lstm_stack(h, net, ws.x_rm, carry, done, ws.hbuf, ws.tc, n, false, st))) return rc;
  return kbs_simt_out_proj(h, net, ws.hbuf, ws.out_rm, n, st);
}

// Fused rollout on the tensor-core path.  The state is recorded, so everything that does not depend on the networks
// is evaluated for all T steps first (terminations, command law, lagged gravity, observations, input projections:
// big HBM-bound launches), then the whole recurrence runs as ONE persistent kernel (kbs_tc_rollout_recurrent; the per-step
// form -- 2 LSTM layer launches for both nets + a head launch per step -- stays behind KBS_TC_PER_STEP=1).
// done_prev restarts the lag scan at step 0; critic_obs (when given) replaces the per-chunk scratch of the critic's
// observations and gets all 475 rows, the input projection still reads cinert / cvel straight from the state.
// Observation assembly + input projections can run in chunks of CT steps on the handle's aux stream while the
// recurrence of the previous chunk runs on the caller's stream (KBS_ROLLOUT_CHUNKS = 2..8).  MEASURED: slower
// (9.97 vs 8.89 ms per 100-step rollout): the persistent recurrence kernel wants every SM to itself, so the
// concurrent kernels delay its CTAs more than they hide.  Default = 1 chunk: phase A first, then the recurrence.
int rollout_chunks() {
  const char* e = getenv("KBS_ROLLOUT_CHUNKS");
  const int c = e ? atoi(e) : 1;
  return (c < 1 || c > kKbsMaxChunks) ? 1 : c;
}

// Workspace of rollout_fused_tc: the recurrence's, the lag states of all T steps (when pg_carry is carried), the actor's
// observations when the caller keeps none, the critic's when it records none, and the operands of the input projections.
struct FusedTcWs { KbsTcRolloutWs r; float *lagged, *aobs, *cobs, *xsb_a, *xsb_c, *osb_a, *osb_c; };
FusedTcWs fused_tc_ws(KbsScratch& s, const kbs_handle* h, int64_t n, int64_t ld, int64_t T, int chunks, bool critic, bool pg,
                      bool own_aobs, bool own_cobs) {
  const int64_t CT = (T + chunks - 1) / chunks;
  const size_t sbf = size_t(kbs_tc_sb_floats(h, n));
  FusedTcWs w{};
  w.r = kbs_tc_rollout_ws(s, h, n, critic ? 2 : 1);
  w.lagged = pg ? s.take<float>(size_t(T) * 3 * ld) : nullptr;
  w.aobs = own_aobs ? nullptr : s.take<float>(size_t(T) * KBS_ACTOR_OBS * ld);
  w.cobs = (critic && !own_cobs) ? s.take<float>(size_t(CT) * KBS_CRITIC_OBS * ld) : nullptr;
  w.xsb_a = s.take<float>(size_t(T) * sbf);
  w.xsb_c = critic ? s.take<float>(size_t(T) * sbf) : nullptr;
  w.osb_a = s.take<float>(kbs_tc_obs_sb_floats(h, KBS_NET_ACTOR, n, CT));
  w.osb_c = critic ? s.take<float>(kbs_tc_obs_sb_floats(h, KBS_NET_CRITIC, n, CT)) : nullptr;
  return w;
}

// res (kbs_rollout_step): the carries are resident in a step state (KbsTcRolloutArgs::res_*), io->*_carry are not read.
int rollout_fused_tc(kbs_handle* h, const kbs_rollout_io* io, const uint8_t* done_prev, float* critic_obs, const FusedTcWs& w,
                     int chunks_cfg, const KbsTcRolloutArgs* res, int64_t n, cudaStream_t st) {
  const int64_t ld = io->state.ld, T = io->T;
  const bool critic = io->value != nullptr;
  const int64_t CT = (T + chunks_cfg - 1) / chunks_cfg;
  const size_t sbf = size_t(kbs_tc_sb_floats(h, n));
  KbsTcRolloutArgs r{};
  if (res) { for (int k = 0; k < 2; ++k) { r.res_hsb[k] = res->res_hsb[k]; r.res_fb[k] = res->res_fb[k]; } r.res_hsb_slot = res->res_hsb_slot; }
  r.ws = w.r;
  float* lagged = w.lagged;
  float* aobs = io->actor_obs ? io->actor_obs : w.aobs;
  float* cobs = critic_obs ? critic_obs : w.cobs;
  float *xsb_a = w.xsb_a, *xsb_c = w.xsb_c, *osb_a = w.osb_a, *osb_c = w.osb_c;
  int rc;

  if ((rc = kbs_launch_terminate(h, io->state, io->term_codes, io->done, io->success, nullptr, n, st, T))) return rc;
  if (lagged) {
    if ((rc = kbs_launch_phase_a_scans(h, io->command, io->u_switch, io->cmd_mode, io->cmd_u6, io->cmd_u_arms, io->done,
                                       done_prev, io->state.sensordata, io->episode.pg_lag, io->pg_carry, lagged, T, ld, n,
                                       st)))
      return rc;
  } else if ((rc = kbs_launch_command_scan(h, io->command, io->u_switch, io->cmd_mode, io->cmd_u6, io->cmd_u_arms, io->done,
                                           T, ld, n, st))) {
    return rc;
  }
  if ((rc = kbs_side_stream_init(h))) return rc;
  const bool overlap = chunks_cfg > 1;
  cudaStream_t aux = overlap ? h->aux_stream : st;
  if (overlap) {
    KBS_CUDA_TRY(cudaEventRecord(h->ev_pre, st));           // scans done; previous call's readers of the staging buffers too
    KBS_CUDA_TRY(cudaStreamWaitEvent(aux, h->ev_pre, 0));
  }
  r.x_sb_all[0] = xsb_a; r.x_sb_all[1] = xsb_c;
  int n_chunks = 0;
  for (int64_t t0 = 0; t0 < T; t0 += CT, ++n_chunks) {
    const int64_t tc = (T - t0 < CT) ? T - t0 : CT;
    const kbs_state_view s = state_at(io->state, t0);
    const kbs_noise_view nz = noise_at(io->noise, t0, ld);
    float* aobs_c = aobs + t0 * KBS_ACTOR_OBS * ld;
    float* cobs_c = critic_obs ? critic_obs + t0 * KBS_CRITIC_OBS * ld : cobs;
    if ((rc = kbs_launch_observations(h, s, &nz, &io->episode, io->command + t0 * KBS_NUM_COMMANDS * ld, nullptr, nullptr,
                                      nullptr, aobs_c, cobs_c, n, aux, tc, lagged ? lagged + t0 * 3 * ld : nullptr,
                                      /*skip_dump=*/critic_obs == nullptr, /*one_step=*/res != nullptr)))
      return rc;
    const float* obs_soa[2] = {aobs_c, cobs_c};
    float* obs_sb[2] = {osb_a, osb_c};
    float* xsb[2] = {xsb_a + size_t(t0) * sbf, critic ? xsb_c + size_t(t0) * sbf : nullptr};
    // one chunk (default): the actor's input projection is folded into layer 0 of the persistent kernel (r.x_is_obs)
    if ((rc = kbs_tc_input_proj_all(h, critic ? 2 : 1, obs_soa, obs_sb, xsb, ld, n, tc, aux,
                                    critic ? s.cinert : nullptr, critic ? s.cvel : nullptr, chunks_cfg == 1 ? &r : nullptr)))
      return rc;
    if (overlap) KBS_CUDA_TRY(cudaEventRecord(h->ev_chunk[n_chunks], aux));
  }

  r.chunk_len = overlap ? CT : 0; r.chunk_events = h->ev_chunk;
  r.n = n; r.ld = ld; r.T = T; r.with_critic = critic;
  r.carry[0] = io->actor_carry; r.carry[1] = io->critic_carry;
  r.done = io->done; r.actor_obs = aobs; r.lpf = io->lpf; r.eps_action = io->eps_action;
  r.qpos = io->state.qpos; r.qvel = io->state.qvel; r.ep = io->episode;
  r.action = io->action; r.log_prob = io->log_prob; r.ctrl = io->ctrl; r.value = io->value;
  return kbs_tc_rollout_recurrent(h, r, st);
}

// Workspace of rollout_simt: the trunk's, and one step of observations the caller does not keep.
struct SimtRolloutWs { TrunkWs trunk; float* aobs; float* cobs; };
SimtRolloutWs simt_rollout_ws(KbsScratch& s, const kbs_handle* h, int64_t n, int64_t ld) {
  SimtRolloutWs w{};
  w.trunk = trunk_ws(s, h, n);
  w.aobs = s.take<float>(size_t(KBS_ACTOR_OBS) * ld);
  w.cobs = s.take<float>(size_t(KBS_CRITIC_OBS) * ld);
  return w;
}
int rollout_simt(kbs_handle* h, const kbs_rollout_io* io, const uint8_t* done_prev, float* critic_obs, const SimtRolloutWs& w,
                 int64_t n, cudaStream_t st, bool one_step = false);

}  // namespace

int kbs_side_stream_init(kbs_handle* h) {
  if (h->side_stream) return 0;
  KBS_CUDA_TRY(cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking));
  KBS_CUDA_TRY(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
  KBS_CUDA_TRY(cudaEventCreateWithFlags(&h->ev_pre, cudaEventDisableTiming));
  for (int i = 0; i < kKbsMaxChunks; ++i) KBS_CUDA_TRY(cudaEventCreateWithFlags(&h->ev_chunk[i], cudaEventDisableTiming));
  for (int i = 0; i < 2; ++i) {
    KBS_CUDA_TRY(cudaEventCreateWithFlags(&h->ev_lstm[i], cudaEventDisableTiming));
    KBS_CUDA_TRY(cudaEventCreateWithFlags(&h->ev_head[i], cudaEventDisableTiming));
  }
  return 0;
}

int kbs_status_init(kbs_handle* h) {
  if (h->persist_status) return KBS_OK;
  KBS_CUDA_TRY(cudaMalloc(&h->persist_status, 256));
  KBS_CUDA_TRY(cudaMemset(h->persist_status, 0, 256));
  KBS_CUDA_TRY(cudaHostAlloc(&h->status_host, 64, cudaHostAllocDefault));
  *h->status_host = 0u;
  return KBS_OK;
}

// refresh the pinned host copy of the (sticky) device health word once the work enqueued so far on `st` has run
int kbs_status_publish(kbs_handle* h, cudaStream_t st) {
  if (!h->persist_status) return KBS_OK;
  KBS_CUDA_TRY(cudaMemcpyAsync(h->status_host, h->persist_status, 4, cudaMemcpyDeviceToHost, st));
  return KBS_OK;
}

// entry check of the fused entry points: the handle belongs to one device (its kernels' shared-memory opt-in, its
// weights and scratch live there), and a health word left non-zero by an earlier call is an error, not a silent result
int kbs_enter(kbs_handle* h) {
  int dev = -1;
  KBS_CUDA_TRY(cudaGetDevice(&dev));
  if (dev != h->device) return KBS_E_STATE;
  if (h->status_host && *reinterpret_cast<volatile unsigned int*>(h->status_host) != 0u) return KBS_E_DEVICE;
  return KBS_OK;
}

int kbs_scratch_reserve(kbs_handle* h, size_t floats) {
  if (floats <= h->scratch_floats) return KBS_OK;
  if (h->scratch_locked) return KBS_E_STATE;       // a captured graph holds pointers into the current allocation
  if (h->scratch) { KBS_CUDA_TRY(cudaFree(h->scratch)); h->scratch = nullptr; h->scratch_floats = 0; }
  const size_t want = floats + floats / 8 + 1024;
  KBS_CUDA_TRY(cudaMalloc(&h->scratch, want * sizeof(float)));
  h->scratch_floats = want;
  return KBS_OK;
}

extern "C" {

int kbs_version(void) { return KBS_VERSION; }

const char* kbs_error_string(int code) {
  switch (code) {
    case KBS_OK: return "ok";
    case KBS_E_NULL: return "required pointer is NULL";
    case KBS_E_SHAPE: return "unsupported shape (n_envs / ld / T / hidden_size)";
    case KBS_E_ALIGN: return "pointer not 16-byte aligned or ld % 4 != 0";
    case KBS_E_STATE: return "handle not ready (weights not packed, or datapath unavailable)";
    case KBS_E_PARAM: return "bad scalar parameter";
    case KBS_E_DEVICE: return "device health word set (dependency-wait timeout or FP16-split operand out of range): kbs_device_status";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown kbs error";
  }
}

int kbs_default_params(kbs_params* p) {
  REQ(p);
  memset(p, 0, sizeof(*p));
  p->hidden_size = 256; p->depth = 2; p->gemm_path = KBS_GEMM_SIMT_FP32; p->normalize_advantages = 0;
  p->ctrl_dt = 0.02f; p->min_std = 0.01f; p->max_std = 1.0f; p->var_scale = 0.5f;
  {
    const double w = 2.0 * M_PI * 10.0, dt = 0.02;   // cutoff_frequency = 10 Hz, train.py:90-93
    p->lpf_alpha = (float)(w * dt / (1.0 + w * dt));
  }
  p->gamma = 0.94f; p->lam = 0.94f; p->adv_eps = 1e-6f;
  p->jpos_noise_mag = (float)(3.0 * M_PI / 180.0); p->jvel_noise_mag = (float)(15.0 * M_PI / 180.0);
  p->gyro_noise_std = (float)(10.0 * M_PI / 180.0); p->pg_noise_std = (float)(3.0 * M_PI / 180.0);
  p->gravity = 9.81f; p->eps_quat = 1e-6f;
  p->unhealthy_z = 0.4f; p->max_tilt = (float)(45.0 * M_PI / 180.0); p->max_length_sec = 12.0f;
  p->switch_prob = (float)(0.02 / 5);
  const float lo[6] = {-0.5f, -0.5f, -1.0f, -0.25f, -0.25f, -0.25f};
  const float hi[6] = {1.2f, 0.5f, 1.0f, 0.05f, 0.25f, 0.25f};
  memcpy(p->cmd_lo, lo, sizeof(lo)); memcpy(p->cmd_hi, hi, sizeof(hi));
  const double deg[20] = {20, 0, 0, 50, -30, -20, -0.0, 0, -50, 30, 0, -10, 0, 90, 0, 0, 10, 0, -90, 0};
  const double lim[20][2] = {{-1.047198, 2.216568}, {-0.20944, 2.268928}, {-1.570796, 1.570796}, {0.0, 2.70526},
                             {-1.134464, 0.261799}, {-2.216568, 1.047198}, {-2.268928, 0.20944}, {-1.570796, 1.570796},
                             {-2.70526, 0.0}, {-0.261799, 1.134464}, {-3.490658, 1.047198}, {-1.658063, 0.436332},
                             {-1.671886, 1.671886}, {0.0, 2.478368}, {-1.37881, 1.37881}, {-1.047198, 3.490658},
                             {-0.436332, 1.658063}, {-1.671886, 1.671886}, {-2.478368, 0.0}, {-1.37881, 1.37881}};
  for (int j = 0; j < 20; ++j) {
    const float b = (float)(deg[j] * M_PI / 180.0), mn = (float)lim[j][0], mx = (float)lim[j][1];
    p->joint_bias[j] = b;
    p->joint_range[j] = fmaxf(b - mn, mx - b);   // evaluated in fp32 like jnp (train.py:1332)
    if (j >= 10) { p->arm_lo[j - 10] = mn; p->arm_hi[j - 10] = mx; }
  }
  const float kp[20] = {150, 200, 100, 150, 40, 150, 200, 100, 150, 40, 100, 100, 40, 40, 20, 100, 100, 40, 40, 20};
  const float kd[20] = {24.722f, 26.387f, 3.419f, 8.654f, 0.990f, 24.722f, 26.387f, 3.419f, 8.654f, 0.990f,
                        8.284f, 8.257f, 0.945f, 1.266f, 0.295f, 8.284f, 8.257f, 0.945f, 1.266f, 0.295f};
  const float cl[20] = {120, 60, 60, 120, 17, 120, 60, 60, 120, 17, 60, 60, 17, 17, 14, 60, 60, 17, 17, 14};
  memcpy(p->kp, kp, sizeof(kp)); memcpy(p->kd, kd, sizeof(kd)); memcpy(p->ctrl_limit, cl, sizeof(cl));
  const float rs[12] = {0.2f, 0.1f, 0.2f, 0.2f, 0.2f, 0.1f, 0.1f, 1.5f, 0.1f, 0.05f, 0.1f, 0.1f};
  memcpy(p->reward_scale, rs, sizeof(rs));
  p->linvel_es = 0.2f; p->angvel_es = 0.2f; p->rp_es = 0.03f; p->rp_es_zero = 0.01f; p->bh_es = 0.02f;
  p->bh_standard = 0.80f; p->bh_foot_origin = 0.06f; p->arm_es = 0.1f; p->grace_period = 2.0f;
  p->touchdown_penalty = 0.4f; p->feet_es = 0.02f; p->com_es = 0.04f; p->acc_es = 5.0f; p->torque_es = 5.0f;
  p->body_base = 1; p->body_lfoot = 7; p->body_rfoot = 12;
  p->sd_gyro = 19; p->sd_imu_quat = 28; p->sd_touch_l = 47; p->sd_touch_r = 48;
  return KBS_OK;
}

int kbs_create(const kbs_params* p, kbs_handle** out) {
  REQ(p); REQ(out);
  if (p->hidden_size != 128 && p->hidden_size != 256) return KBS_E_SHAPE;
  if (p->depth < 1 || p->depth > KBS_MAX_DEPTH) return KBS_E_SHAPE;
  if (p->gemm_path != KBS_GEMM_TC_3XTF32 && p->gemm_path != KBS_GEMM_SIMT_FP32 && p->gemm_path != KBS_GEMM_TC_2XF16)
    return KBS_E_PARAM;
  int dev = 0;
  KBS_CUDA_TRY(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  KBS_CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) {
    fprintf(stderr, "libkbotstep: device %d is sm_%d%d; this library is built for sm_100a only\n", dev, prop.major,
            prop.minor);
    return (int)cudaErrorNoKernelImageForDevice;
  }
  kbs_handle* h = new (std::nothrow) kbs_handle();
  if (!h) return (int)cudaErrorMemoryAllocation;
  h->p = *p;
  h->device = dev;
  h->num_sms = prop.multiProcessorCount;
  *out = h;
  return KBS_OK;
}

int kbs_destroy(kbs_handle* h) {
  if (!h) return KBS_OK;
  for (int k = 0; k < 2; ++k) {
    KbsNet& N = h->net[k];
    cudaFree(N.w_in); cudaFree(N.b_in); cudaFree(N.w_out); cudaFree(N.b_out); cudaFree(N.tc_image); cudaFree(N.tc_bwd_image); cudaFree(N.tc_bwd_image64); cudaFree(N.tc_fwd8_image);
    for (int l = 0; l < KBS_MAX_DEPTH; ++l) { cudaFree(N.w_ih[l]); cudaFree(N.w_hh[l]); cudaFree(N.b[l]); }
  }
  cudaFree(h->scratch);
  cudaFree(h->persist_status);
  if (h->status_host) cudaFreeHost(h->status_host);
  cudaFree(h->loss_ticket);
  cudaFree(h->norm_partial);
  if (h->side_stream) {
    cudaStreamDestroy(h->side_stream);
    cudaStreamDestroy(h->aux_stream);
    cudaEventDestroy(h->ev_pre);
    for (int i = 0; i < kKbsMaxChunks; ++i) cudaEventDestroy(h->ev_chunk[i]);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(h->ev_lstm[i]); cudaEventDestroy(h->ev_head[i]); }
  }
  if (h->prof_ev) {
    for (int i = 0; i < 2 * kKbsProfMaxPairs; ++i) cudaEventDestroy(h->prof_ev[i]);
    delete[] h->prof_ev; delete[] h->prof_id;
  }
  delete h;
  return KBS_OK;
}

int kbs_get_params(const kbs_handle* h, kbs_params* out) {
  REQ(h); REQ(out);
  *out = h->p;
  return KBS_OK;
}

int64_t kbs_launch_count(const kbs_handle* h) { return h ? h->launches : -1; }

int kbs_device_status(kbs_handle* h, int* status_out) {
  REQ(h); REQ(status_out);
  *status_out = 0;
  if (!h->persist_status) return KBS_OK;
  unsigned int v = 0;
  KBS_CUDA_TRY(cudaDeviceSynchronize());
  KBS_CUDA_TRY(cudaMemcpy(&v, h->persist_status, 4, cudaMemcpyDeviceToHost));
  *h->status_host = v;
  *status_out = int(v);
  return KBS_OK;
}

int kbs_device_status_reset(kbs_handle* h) {
  REQ(h);
  if (!h->persist_status) return KBS_OK;
  KBS_CUDA_TRY(cudaDeviceSynchronize());
  KBS_CUDA_TRY(cudaMemset(h->persist_status, 0, 4));
  *h->status_host = 0u;
  return KBS_OK;
}

int kbs_scratch_lock(kbs_handle* h, int on) {
  REQ(h);
  h->scratch_locked = on != 0;
  return KBS_OK;
}

int kbs_debug_tc_trace_attach(kbs_handle* h, long long* trace_out, int64_t step, int layer) {
  REQ(h);
  h->trace_buf = trace_out; h->trace_step = step; h->trace_layer = layer;
  return KBS_OK;
}

int kbs_debug_tc_trace(kbs_handle* h, long long* trace_out, int64_t n, void* stream) {
  REQ(h); REQ(trace_out);
  if (n <= 0) return KBS_E_SHAPE;
  KbsTcRolloutWs ws;
  int rc = kbs_scratch(h, [&](KbsScratch& s) { ws = kbs_tc_rollout_ws(s, h, n, 1); });
  if (rc) return rc;
  return kbs_tc_debug_trace(h, trace_out, ws, n, (cudaStream_t)stream);
}

int kbs_debug_tc_gates(kbs_handle* h, int net, int layer, const float* x_rm, const float* h_rm, float* gates_out,
                       int64_t n, void* stream) {
  REQ(h); REQ(x_rm); REQ(h_rm); REQ(gates_out);
  if (n <= 0 || layer < 0 || layer >= h->p.depth) return KBS_E_SHAPE;
  float* ws;   // x and h as SB operands
  int rc = kbs_scratch(h, [&](KbsScratch& s) { ws = s.take<float>(2 * size_t(kbs_tc_sb_floats(h, n))); });
  if (rc) return rc;
  return kbs_tc_debug_gates(h, net, layer, x_rm, h_rm, gates_out, ws, n, (cudaStream_t)stream);
}

int kbs_profile_enable(kbs_handle* h, int on) {
  REQ(h);
  if (on && !h->prof_ev) {
    h->prof_ev = new (std::nothrow) cudaEvent_t[2 * kKbsProfMaxPairs];
    h->prof_id = new (std::nothrow) int8_t[kKbsProfMaxPairs];
    if (!h->prof_ev || !h->prof_id) return (int)cudaErrorMemoryAllocation;
    for (int i = 0; i < 2 * kKbsProfMaxPairs; ++i) KBS_CUDA_TRY(cudaEventCreate(&h->prof_ev[i]));
  }
  h->prof_on = on != 0;
  if (on) h->prof_n = 0;
  return KBS_OK;
}

int kbs_profile_read(kbs_handle* h, int max_ids, double* total_ms, int64_t* launches) {
  REQ(h); REQ(total_ms); REQ(launches);
  for (int i = 0; i < max_ids; ++i) { total_ms[i] = 0.0; launches[i] = 0; }
  for (int i = 0; i < h->prof_n; ++i) {
    float ms = 0.f;
    KBS_CUDA_TRY(cudaEventSynchronize(h->prof_ev[2 * i + 1]));
    KBS_CUDA_TRY(cudaEventElapsedTime(&ms, h->prof_ev[2 * i], h->prof_ev[2 * i + 1]));
    const int id = h->prof_id[i];
    if (id >= 0 && id < max_ids) { total_ms[id] += ms; launches[id]++; }
  }
  return h->prof_n >= kKbsProfMaxPairs ? 1 : 0;   // 1 = event pool exhausted, totals are partial
}

const char* kbs_kernel_name(int id) {
  static const char* names[KBS_K_COUNT] = {
      "obs_kernel", "command_kernel", "torque_kernel", "terminate_kernel", "reward_rot_kernel", "reward_terms_kernel",
      "reward_scan_kernel", "gae_kernel", "adv_norm_kernel", "policy_io_kernels", "gemm_nt_kernel(simt)",
      "lstm_cell_kernel", "actor_head_kernel", "critic_head_kernel", "pack_kernels", "lstm_layer_tc_kernel",
      "proj_tc_kernel", "rollout_persist_kernel", "bptt_persist_kernel", "gemm_tn_tc_kernel", "sb_to_tn_kernel", "tn_reduce_kernel",
      "step_record_kernel", "actuator_substep_kernel", "minibatch_permutation_kernel", "shuffle_minibatches_kernels"};
  return (id >= 0 && id < KBS_K_COUNT) ? names[id] : "?";
}

int kbs_weights_pack(kbs_handle* h, int net, const kbs_net_weights* w, void* stream) {
  REQ(h); REQ(w);
  if (net != KBS_NET_ACTOR && net != KBS_NET_CRITIC) return KBS_E_PARAM;
  { int dev = -1; KBS_CUDA_TRY(cudaGetDevice(&dev)); if (dev != h->device) return KBS_E_STATE; }
  REQ(w->w_in); REQ(w->b_in); REQ(w->w_out); REQ(w->b_out);
  for (int l = 0; l < h->p.depth; ++l) { REQ(w->w_ih[l]); REQ(w->w_hh[l]); REQ(w->b[l]); }
  cudaStream_t st = (cudaStream_t)stream;
  int rc = kbs_simt_pack(h, net, w, st);
  if (rc) return rc;
  if (h->p.gemm_path != KBS_GEMM_SIMT_FP32) rc = kbs_tc_pack(h, net, st);
  return rc;
}

int kbs_observations(kbs_handle* h, const kbs_state_view* s, const kbs_noise_view* noise,
                     const kbs_episode_view* ep, const float* command, float* pg_carry,
                     const uint8_t* pg_reset, float* computed, float* actor_obs, float* critic_obs, int64_t n,
                     void* stream) {
  REQ(h); REQ(command);
  int rc = check_state(s, n, true);
  if (rc) return rc;
  if (critic_obs) { REQ(s->cinert); REQ(s->cvel); REQ(s->actuator_force); }
  if (noise && noise->eps_jpos) { REQ(noise->eps_jvel); REQ(noise->eps_gyro); REQ(noise->eps_pg); }
  AL(command); AL(pg_carry); AL(computed); AL(actor_obs); AL(critic_obs);
  if (!computed && !actor_obs && !critic_obs) return KBS_E_NULL;
  if (reinterpret_cast<uintptr_t>(pg_reset) & 3u) return KBS_E_ALIGN;
  return kbs_launch_observations(h, *s, noise, ep, command, pg_carry, pg_reset, computed, actor_obs, critic_obs, n,
                                 (cudaStream_t)stream);
}

int kbs_ppo_loss_default_params(kbs_ppo_loss_params* p) {
  REQ(p);
  p->clip_param = 0.2f; p->value_loss_coef = 0.5f; p->entropy_coef = 0.004f /* train.py:1767 */; p->log_clip_value = 10.0f;
  p->use_clipped_value_loss = 1;
  return KBS_OK;
}

int kbs_ppo_loss(kbs_handle* h, const kbs_ppo_loss_params* params, const kbs_ppo_loss_io* io, int64_t n, void* stream) {
  REQ(h); REQ(params); REQ(io);
  REQ(io->log_probs); REQ(io->old_log_probs); REQ(io->advantages); REQ(io->values); REQ(io->value_targets); REQ(io->entropy);
  REQ(io->out);
  if (params->use_clipped_value_loss) REQ(io->old_values);
  if (io->T <= 0) return KBS_E_SHAPE;
  if (n <= 0 || io->ld < n) return KBS_E_SHAPE;
  return kbs_launch_ppo_loss(h, *params, *io, n, (cudaStream_t)stream);
}

int kbs_com_distance(kbs_handle* h, const int32_t* contact_geom1, const int32_t* contact_geom2, const float* contact_pos,
                     const float* subtree_com_base, float* com_distance, int ncon, int64_t T, int64_t ld, int64_t n,
                     void* stream) {
  REQ(h); REQ(contact_geom1); REQ(contact_geom2); REQ(contact_pos); REQ(subtree_com_base); REQ(com_distance);
  if (T <= 0 || T > 65535) return KBS_E_SHAPE;
  int rc = check_ld(ld, n);
  if (rc) return rc;
  return kbs_launch_com_distance(h, contact_geom1, contact_geom2, contact_pos, subtree_com_base, com_distance, ncon, T, ld, n,
                                 (cudaStream_t)stream);
}

int kbs_upload_state(kbs_handle* h, const kbs_state_view* host, const kbs_state_view* dev, int64_t T, int64_t* bytes_out,
                     void* stream) {
  REQ(h); REQ(host); REQ(dev);
  if (T <= 0 || host->ld != dev->ld || host->ld <= 0) return KBS_E_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t ldb = size_t(host->ld) * sizeof(float);
  const int bb = h->p.body_base, bl = h->p.body_lfoot, br = h->p.body_rfoot;
  struct Range { const float* src; const float* dst; int rows, r0, r1; };
  const Range rs[] = {
      {host->qpos, dev->qpos, KBS_NQ, 0, KBS_NQ},
      {host->qvel, dev->qvel, KBS_NV, 0, KBS_NV},
      {host->sensordata, dev->sensordata, KBS_NSENSORDATA, h->p.sd_gyro, h->p.sd_gyro + 3},
      {host->sensordata, dev->sensordata, KBS_NSENSORDATA, h->p.sd_imu_quat, h->p.sd_imu_quat + 4},
      {host->sensordata, dev->sensordata, KBS_NSENSORDATA, h->p.sd_touch_l, h->p.sd_touch_l + 1},
      {host->sensordata, dev->sensordata, KBS_NSENSORDATA, h->p.sd_touch_r, h->p.sd_touch_r + 1},
      {host->xpos, dev->xpos, 3 * KBS_NBODY, 3 * bb, 3 * bb + 3},
      {host->xpos, dev->xpos, 3 * KBS_NBODY, 3 * bl, 3 * bl + 3},
      {host->xpos, dev->xpos, 3 * KBS_NBODY, 3 * br, 3 * br + 3},
      {host->xquat, dev->xquat, 4 * KBS_NBODY, 4 * bb, 4 * bb + 4},
      {host->xquat, dev->xquat, 4 * KBS_NBODY, 4 * bl, 4 * bl + 4},
      {host->xquat, dev->xquat, 4 * KBS_NBODY, 4 * br, 4 * br + 4},
      {host->cinert, dev->cinert, 10 * KBS_NBODY, 10, 10 * KBS_NBODY},       // cinert[1:]
      {host->cvel, dev->cvel, 6 * KBS_NBODY, 6, 6 * KBS_NBODY},              // cvel[1:]
      {host->actuator_force, dev->actuator_force, KBS_NUM_JOINTS, 0, KBS_NUM_JOINTS},
      {host->com_distance, dev->com_distance, 1, 0, 1},
      {host->time, dev->time, 1, 0, 1},
  };
  int64_t bytes = 0;
  for (const Range& r : rs) {
    if (!r.src || !r.dst) continue;
    const size_t pitch = size_t(r.rows) * ldb, width = size_t(r.r1 - r.r0) * ldb;
    KBS_CUDA_TRY(cudaMemcpy2DAsync(const_cast<float*>(r.dst) + size_t(r.r0) * host->ld, pitch, r.src + size_t(r.r0) * host->ld,
                                   pitch, width, size_t(T), cudaMemcpyHostToDevice, st));
    bytes += int64_t(width) * T;
  }
  if (bytes_out) *bytes_out = bytes;
  return KBS_OK;
}

int kbs_mirror_observations(kbs_handle* h, const kbs_state_view* s, const float* computed, const float* command,
                            float* actor_obs, float* critic_obs, float* command_out, int64_t T, int64_t n, void* stream) {
  REQ(h); REQ(computed); REQ(command);
  if (T <= 0 || T > 65535) return KBS_E_SHAPE;
  int rc = check_state(s, n, true);
  if (rc) return rc;
  if (critic_obs) { REQ(s->cinert); REQ(s->cvel); REQ(s->actuator_force); REQ(s->xpos); }
  if (!actor_obs && !critic_obs && !command_out) return KBS_E_NULL;
  AL(computed); AL(command); AL(actor_obs); AL(critic_obs); AL(command_out);
  return kbs_launch_mirror_obs(h, *s, computed, command, actor_obs, critic_obs, command_out, n, T, (cudaStream_t)stream);
}

int kbs_mirror_joints(kbs_handle* h, const float* in, float* out, int64_t T, int64_t ld, int64_t n, void* stream) {
  REQ(h); REQ(in); REQ(out);
  if (T <= 0 || T > 65535 || in == out) return KBS_E_SHAPE;
  int rc = check_ld(ld, n);
  if (rc) return rc;
  AL(in); AL(out);
  return kbs_launch_mirror_joints(h, in, out, ld, n, T, (cudaStream_t)stream);
}

int kbs_command_update(kbs_handle* h, float* command, const float* u_switch, const int32_t* mode, const float* u6,
                       const float* u_arms, int64_t ld, int64_t n, void* stream) {
  REQ(h); REQ(command); REQ(mode); REQ(u6); REQ(u_arms);
  int rc = check_ld(ld, n);
  if (rc) return rc;
  AL(command); AL(u_switch); AL(mode); AL(u6); AL(u_arms);
  return kbs_launch_command(h, command, command, u_switch, mode, u6, u_arms, nullptr, ld, n, (cudaStream_t)stream);
}

int kbs_actor_step(kbs_handle* h, const float* obs, int64_t ld, float* carry, float* lpf, const float* eps,
                   const float* action_in, const uint8_t* done, const kbs_actor_out* out, int64_t n, void* stream) {
  REQ(h); REQ(obs); REQ(carry); REQ(lpf); REQ(out);
  int rc = check_ld(ld, n);
  if (rc) return rc;
  AL(obs); AL(carry); AL(lpf); AL(eps); AL(action_in);
  cudaStream_t st = (cudaStream_t)stream;
  TrunkWs ws;
  if ((rc = kbs_scratch(h, [&](KbsScratch& s) { ws = trunk_ws(s, h, n); }))) return rc;
  if ((rc = trunk(h, KBS_NET_ACTOR, obs, ld, carry, done, ws, n, st))) return rc;
  return kbs_launch_actor_head(h, ws.out_rm, kOutLd, obs, ld, lpf, eps, action_in, done, *out, n, st);
}

int kbs_critic_step(kbs_handle* h, const float* obs, int64_t ld, float* carry, const uint8_t* done, float* value,
                    int64_t n, void* stream) {
  REQ(h); REQ(obs); REQ(carry); REQ(value);
  int rc = check_ld(ld, n);
  if (rc) return rc;
  AL(obs); AL(carry);
  cudaStream_t st = (cudaStream_t)stream;
  TrunkWs ws;
  if ((rc = kbs_scratch(h, [&](KbsScratch& s) { ws = trunk_ws(s, h, n); }))) return rc;
  if ((rc = trunk(h, KBS_NET_CRITIC, obs, ld, carry, done, ws, n, st))) return rc;
  return kbs_launch_critic_head(h, ws.out_rm, kOutLd, value, n, st);
}

int kbs_torque(kbs_handle* h, const float* action, const kbs_state_view* s, const kbs_episode_view* ep,
               float* ctrl_out, int64_t n, void* stream) {
  REQ(h); REQ(action); REQ(ctrl_out);
  int rc = check_state(s, n, false);
  if (rc) return rc;
  AL(action); AL(ctrl_out);
  return kbs_launch_torque(h, action, *s, ep, ctrl_out, n, (cudaStream_t)stream);
}

int kbs_torque_substeps(kbs_handle* h, const float* action, float* prev_action, const float* u_drop, const float* latency,
                        const float* q_sub, const float* qd_sub, const kbs_episode_view* ep, float* ctrl_out, int32_t n_substeps,
                        float sub_dt, float drop_prob, int64_t ld, int64_t n, void* stream) {
  REQ(h); REQ(action); REQ(prev_action); REQ(u_drop); REQ(latency); REQ(q_sub); REQ(qd_sub); REQ(ctrl_out);
  if (n_substeps <= 0 || n_substeps > 64) return KBS_E_SHAPE;
  int rc = check_ld(ld, n);
  if (rc) return rc;
  AL(action); AL(prev_action); AL(u_drop); AL(latency); AL(q_sub); AL(qd_sub); AL(ctrl_out);
  return kbs_launch_torque_substeps(h, action, prev_action, u_drop, latency, q_sub, qd_sub, ep, ctrl_out, n_substeps, sub_dt,
                                    drop_prob, ld, n, (cudaStream_t)stream);
}

int kbs_terminate(kbs_handle* h, const kbs_state_view* s, int32_t* codes, uint8_t* done, uint8_t* success, float* pre,
                  int64_t n, void* stream) {
  REQ(h);
  int rc = check_state(s, n, false);
  if (rc) return rc;
  REQ(s->xpos); REQ(s->time);
  AL(codes); AL(pre);
  if ((reinterpret_cast<uintptr_t>(done) & 3u) || (reinterpret_cast<uintptr_t>(success) & 3u)) return KBS_E_ALIGN;
  return kbs_launch_terminate(h, *s, codes, done, success, pre, n, (cudaStream_t)stream);
}

int kbs_rewards(kbs_handle* h, const kbs_traj_view* traj, const kbs_reward_carry* carry, float* total,
                float* components, int64_t n, void* stream) {
  REQ(h); REQ(traj); REQ(carry); REQ(total);
  if (traj->T <= 0 || traj->T > 65535) return KBS_E_SHAPE;
  int rc = check_state(&traj->state, n, true);
  if (rc) return rc;
  REQ(traj->state.com_distance); REQ(traj->command); REQ(traj->ctrl); REQ(traj->done);
  REQ(carry->t_single); REQ(carry->airtime); REQ(carry->prev_contact);
  AL(traj->command); AL(traj->ctrl); AL(total); AL(components);
  if (reinterpret_cast<uintptr_t>(traj->done) & 3u) return KBS_E_ALIGN;
  return kbs_launch_rewards(h, *traj, *carry, total, components, n, (cudaStream_t)stream);
}

int kbs_gae(kbs_handle* h, const float* values, const float* rewards, const uint8_t* done, const uint8_t* success,
            float* advantages, float* value_targets, int64_t T, int64_t ld, int64_t n, void* stream) {
  REQ(h); REQ(values); REQ(rewards); REQ(done); REQ(success); REQ(advantages); REQ(value_targets);
  if (T <= 0) return KBS_E_SHAPE;
  if (n <= 0 || ld < n) return KBS_E_SHAPE;
  return kbs_launch_gae(h, values, rewards, done, success, advantages, value_targets, T, ld, n, (cudaStream_t)stream);
}

int kbs_policy_step(kbs_handle* h, const float* joint_angles, const float* joint_vel, const float* projected_gravity,
                    const float* gyro, const float* command, const float* carry_in, float* carry_out,
                    float* action_out, int64_t n, void* stream) {
  REQ(h); REQ(joint_angles); REQ(joint_vel); REQ(projected_gravity); REQ(gyro); REQ(command); REQ(carry_in);
  REQ(carry_out); REQ(action_out);
  if (n <= 0) return KBS_E_SHAPE;
  { const int rc0 = kbs_enter(h); if (rc0) return rc0; }
  cudaStream_t st = (cudaStream_t)stream;
  const int H = h->p.hidden_size, d2 = 2 * h->p.depth;
  const int64_t ld = round_up4(n);
  {
    const char* legacy_env = getenv("KBS_TC_PER_STEP");
    if (h->p.gemm_path != KBS_GEMM_SIMT_FP32 && !(legacy_env && atoi(legacy_env)) && d2 <= 8 &&
        kbs_tc_persistent_available(h, n, 1, 1)) {
      // Tensor-core form: input projection on tcgen05, then the persistent recurrence kernel with T = 1 (128 x 256 tiles,
      // output head fused into its epilogue; action = dist.mode() because no sampling noise is passed).  The flat carry
      // records [n][d2 * H + 20] are converted straight to / from the kernel's operand layouts: one pass each way
      // instead of flat -> [d2][n][H] -> SB / FB (and back), which was 2/3 of the step's HBM traffic at large n.
      const int carry_w = d2 * H + 20;
      KbsTcRolloutArgs r{};
      float *xsb, *osb, *obs, *lpf, *act;
      int rc = kbs_scratch(h, [&](KbsScratch& s) {
        r.ws = kbs_tc_rollout_ws(s, h, n, 1);
        xsb = s.take<float>(kbs_tc_sb_floats(h, n));
        osb = s.take<float>(kbs_tc_obs_sb_floats(h, KBS_NET_ACTOR, n, 1));
        obs = s.take<float>(size_t(KBS_ACTOR_OBS) * ld);
        lpf = s.take<float>(size_t(20) * ld);
        act = s.take<float>(size_t(20) * ld);
      });
      if (rc) return rc;
      if ((rc = kbs_launch_policy_pack(h, joint_angles, joint_vel, projected_gravity, gyro, command, carry_in, obs, nullptr,
                                       lpf, ld, n, st)))
        return rc;
      const float* obs_soa[2] = {obs, nullptr};
      float* obs_sb[2] = {osb, nullptr};
      float* x_all[2] = {xsb, nullptr};
      if ((rc = kbs_tc_input_proj_all(h, 1, obs_soa, obs_sb, x_all, ld, n, 1, st, nullptr, nullptr, &r))) return rc;
      r.n = n; r.ld = ld; r.T = 1; r.with_critic = false;
      r.carry[0] = const_cast<float*>(carry_in); r.carry_out[0] = carry_out; r.carry_ld = carry_w;
      r.actor_obs = obs; r.lpf = lpf; r.action = act;
      if ((rc = kbs_tc_rollout_recurrent(h, r, st))) return rc;
      return kbs_launch_policy_unpack(h, nullptr, lpf, act, carry_out, action_out, ld, n, st);
    }
  }
  TrunkWs ws;
  float *obs, *lpf, *mean, *carry;
  int rc = kbs_scratch(h, [&](KbsScratch& s) {
    ws = trunk_ws(s, h, n);
    obs = s.take<float>(size_t(KBS_ACTOR_OBS) * ld);
    lpf = s.take<float>(size_t(20) * ld);
    mean = s.take<float>(size_t(20) * ld);
    carry = s.take<float>(size_t(d2) * n * H);
  });
  if (rc) return rc;
  if ((rc = kbs_launch_policy_pack(h, joint_angles, joint_vel, projected_gravity, gyro, command, carry_in, obs, carry,
                                   lpf, ld, n, st)))
    return rc;
  if ((rc = trunk(h, KBS_NET_ACTOR, obs, ld, carry, nullptr, ws, n, st))) return rc;
  kbs_actor_out o{};
  o.mean = mean;
  if ((rc = kbs_launch_actor_head(h, ws.out_rm, kOutLd, obs, ld, lpf, nullptr, nullptr, nullptr, o, n, st))) return rc;
  return kbs_launch_policy_unpack(h, carry, lpf, mean, carry_out, action_out, ld, n, st);
}

// Workspace of ppo_variables_pass: the exact-fp32 trunk's, or the tensor-core recurrence's and the input projections' of all T
// steps for actor [+ critic].
struct VarsWs { TrunkWs trunk; KbsTcRolloutWs rollout; float* xsb[2]; float* osb[2]; };
VarsWs vars_ws(KbsScratch& s, const kbs_handle* h, const kbs_ppo_io* io, int64_t n) {
  VarsWs w{};
  if (h->p.gemm_path == KBS_GEMM_SIMT_FP32) { w.trunk = trunk_ws(s, h, n); return w; }
  const int nets = io->critic_obs ? 2 : 1;
  w.rollout = kbs_tc_rollout_ws(s, h, n, nets);
  for (int k = 0; k < nets; ++k) w.xsb[k] = s.take<float>(size_t(io->T) * kbs_tc_sb_floats(h, n));
  for (int k = 0; k < nets; ++k) w.osb[k] = s.take<float>(kbs_tc_obs_sb_floats(h, k, n, io->T));
  return w;
}

// One pass of _ppo_scan_fn's networks over a stored trajectory (actor [+ critic]).
static int ppo_variables_pass(kbs_handle* h, const kbs_ppo_io* io, const VarsWs& ws, int64_t n, cudaStream_t st) {
  int rc;
  const bool critic = io->critic_obs != nullptr;
  const int64_t ld = io->ld, T = io->T;
  if (h->p.gemm_path == KBS_GEMM_SIMT_FP32) {
    // stage-by-stage form (exact-fp32 datapath): T x (actor step, critic step)
    for (int64_t t = 0; t < T; ++t) {
      const uint8_t* done_t = io->done + t * ld;
      if ((rc = trunk(h, KBS_NET_ACTOR, io->actor_obs + t * KBS_ACTOR_OBS * ld, ld, io->actor_carry, done_t, ws.trunk, n, st)))
        return rc;
      kbs_actor_out o{};
      o.log_prob = io->log_probs ? io->log_probs + t * ld : nullptr;
      o.entropy = io->entropy ? io->entropy + t * ld : nullptr;
      o.std = io->action_std ? io->action_std + t * KBS_NUM_JOINTS * ld : nullptr;
      o.mean = io->mean ? io->mean + t * KBS_NUM_JOINTS * ld : nullptr;
      if ((rc = kbs_launch_actor_head(h, ws.trunk.out_rm, kOutLd, io->actor_obs + t * KBS_ACTOR_OBS * ld, ld, io->lpf, nullptr,
                                      io->action + t * KBS_NUM_JOINTS * ld, done_t, o, n, st)))
        return rc;
      if (critic) {
        if ((rc = trunk(h, KBS_NET_CRITIC, io->critic_obs + t * KBS_CRITIC_OBS * ld, ld, io->critic_carry, done_t, ws.trunk,
                        n, st)))
          return rc;
        if ((rc = kbs_launch_critic_head(h, ws.trunk.out_rm, kOutLd, io->values + t * ld, n, st))) return rc;
      }
    }
    return KBS_OK;
  }
  // tensor-core form: input projections of all T steps (critic: one launch; actor: folded into layer 0), then the persistent
  // recurrence kernel with the stored actions (log-prob / entropy / std / mean of the stored action instead of sampling)
  KbsTcRolloutArgs r{};
  {
    const float* obs_soa[2] = {io->actor_obs, io->critic_obs};
    float* obs_sb[2] = {ws.osb[0], critic ? ws.osb[1] : nullptr};
    float* xsb[2] = {ws.xsb[0], critic ? ws.xsb[1] : nullptr};
    if ((rc = kbs_tc_input_proj_all(h, critic ? 2 : 1, obs_soa, obs_sb, xsb, ld, n, T, st, nullptr, nullptr, &r))) return rc;
  }
  r.n = n; r.ld = ld; r.T = T; r.with_critic = critic;
  r.carry[0] = io->actor_carry; r.carry[1] = io->critic_carry;
  r.done = io->done; r.actor_obs = io->actor_obs; r.lpf = io->lpf;
  r.action_in = io->action; r.log_prob = io->log_probs; r.entropy = io->entropy; r.action_std = io->action_std;
  r.mean = io->mean;
  r.value = io->values;
  r.ws = ws.rollout;
  return kbs_tc_rollout_recurrent(h, r, st);
}

int kbs_ppo_variables(kbs_handle* h, const kbs_ppo_io* io, int64_t n, void* stream) {
  REQ(h); REQ(io);
  REQ(io->actor_obs); REQ(io->action); REQ(io->done); REQ(io->actor_carry); REQ(io->lpf); REQ(io->log_probs);
  REQ(io->entropy);
  if (io->T <= 0) return KBS_E_SHAPE;
  int rc = check_ld(io->ld, n);
  if (rc) return rc;
  if ((rc = kbs_enter(h))) return rc;
  const bool critic = io->critic_obs != nullptr;
  if (critic) { REQ(io->critic_carry); REQ(io->values); }
  AL(io->actor_obs); AL(io->critic_obs); AL(io->action); AL(io->lpf); AL(io->log_probs); AL(io->values); AL(io->entropy);
  AL(io->action_std); AL(io->mean);
  const bool mirror = io->actor_obs_mirror != nullptr;
  if (mirror) {
    REQ(io->actor_mirror_carry); REQ(io->lpf_mirror); REQ(io->action_mirror_loss);
    if (io->critic_obs_mirror) { REQ(io->critic_mirror_carry); REQ(io->value_mirror_loss); if (!critic) return KBS_E_NULL; }
    AL(io->actor_obs_mirror); AL(io->critic_obs_mirror); AL(io->lpf_mirror); AL(io->action_mirror_loss); AL(io->value_mirror_loss);
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t ld = io->ld, T = io->T;
  const bool tc = h->p.gemm_path != KBS_GEMM_SIMT_FP32;
  // dist.mean() -- asked for, or taken internally by the mirror pass -- is an output of the persistent kernel only: refuse
  // before anything is launched, so the outputs and carries stay as they were
  if (tc && (io->mean || mirror) && !kbs_tc_persistent_available(h, n, T, critic ? 2 : 1)) return KBS_E_SHAPE;
  // the mirror pass's intermediates: mean, mean_m [T][20][ld], value_m, lp_m, ent_m [T][ld]; then both passes' workspace
  float *mean = nullptr, *mean_m = nullptr, *value_m = nullptr, *lp_m = nullptr, *ent_m = nullptr;
  VarsWs ws;
  rc = kbs_scratch(h, [&](KbsScratch& s) {
    if (mirror) {
      mean = s.take<float>(size_t(T) * KBS_NUM_JOINTS * ld);
      mean_m = s.take<float>(size_t(T) * KBS_NUM_JOINTS * ld);
      value_m = s.take<float>(size_t(T) * ld);
      lp_m = s.take<float>(size_t(T) * ld);
      ent_m = s.take<float>(size_t(T) * ld);
    }
    ws = vars_ws(s, h, io, n);
  });
  if (rc) return rc;
  kbs_ppo_io a = *io;
  if (mirror && !a.mean) a.mean = mean;
  if ((rc = ppo_variables_pass(h, &a, ws, n, st))) return rc;
  if (!mirror) return KBS_OK;
  // the mirrored passes (train.py:1462-1481): same networks, mirrored observations, their own carries
  kbs_ppo_io m = *io;
  m.actor_obs = io->actor_obs_mirror; m.critic_obs = io->critic_obs_mirror;
  m.actor_carry = io->actor_mirror_carry; m.critic_carry = io->critic_mirror_carry; m.lpf = io->lpf_mirror;
  m.log_probs = lp_m; m.entropy = ent_m; m.values = io->critic_obs_mirror ? value_m : nullptr; m.action_std = nullptr;
  m.mean = mean_m;
  if ((rc = ppo_variables_pass(h, &m, ws, n, st))) return rc;
  return kbs_launch_mirror_loss(h, a.mean, mean_m, io->values, value_m, io->action_mirror_loss,
                                io->critic_obs_mirror ? io->value_mirror_loss : nullptr, io->actor_mirror_loss_scale,
                                io->critic_mirror_loss_scale, T, ld, n, st);
}

int kbs_generate_rollout_noise(kbs_handle* h, uint64_t seed, int64_t step0, const kbs_noise_view* noise, float* eps_action,
                               float* u_switch, int32_t* cmd_mode, float* cmd_u6, float* cmd_u_arms, int64_t T, int64_t ld, int64_t n,
                               void* stream) {
  REQ(h);
  if (T <= 0 || T > 65535) return KBS_E_SHAPE;
  int rc = check_ld(ld, n);
  if (rc) return rc;
  if (noise) { AL(noise->eps_jpos); AL(noise->eps_jvel); AL(noise->eps_gyro); AL(noise->eps_pg); }
  AL(eps_action); AL(u_switch); AL(cmd_mode); AL(cmd_u6); AL(cmd_u_arms);
  return kbs_launch_rollout_noise(h, seed, step0, noise, eps_action, u_switch, cmd_mode, cmd_u6, cmd_u_arms, T, ld, n,
                                  (cudaStream_t)stream);
}

int kbs_minibatch_permutation(kbs_handle* h, uint64_t seed, int64_t* pass_dev, int64_t env0, int32_t* perm_out, int64_t n,
                              void* stream) {
  REQ(h); REQ(pass_dev); REQ(perm_out);
  if (n <= 0 || n > KBS_MAX_PERMUTATION_ENVS) return KBS_E_SHAPE;
  if (env0 < 0) return KBS_E_PARAM;
  if ((reinterpret_cast<uintptr_t>(pass_dev) & 7u) || (reinterpret_cast<uintptr_t>(perm_out) & 3u)) return KBS_E_ALIGN;
  return kbs_launch_minibatch_permutation(h, seed, pass_dev, env0, perm_out, n, (cudaStream_t)stream);
}

int kbs_shuffle_minibatches(kbs_handle* h, const int32_t* perm, const kbs_ppo_batch* src, const kbs_ppo_minibatches* dst, int64_t n,
                            void* stream) {
  REQ(h); REQ(perm); REQ(src); REQ(dst);
  REQ(src->actor_obs); REQ(src->critic_obs); REQ(src->action); REQ(src->done); REQ(src->old_log_probs); REQ(src->advantages);
  REQ(src->value_targets); REQ(src->old_values);
  REQ(dst->actor_obs); REQ(dst->critic_obs); REQ(dst->action); REQ(dst->done); REQ(dst->old_log_probs); REQ(dst->advantages);
  REQ(dst->value_targets); REQ(dst->old_values);
  // a start carry is copied when the rollout has one and left out (zeros at the first step) when it has none
  if (!src->actor_carry0 != !dst->actor_carry0 || !src->critic_carry0 != !dst->critic_carry0 || !src->lpf0 != !dst->lpf0)
    return KBS_E_NULL;
  const int64_t bs = dst->batch_size;
  if (src->T <= 0 || n <= 0 || n > KBS_MAX_PERMUTATION_ENVS || bs <= 0 || bs % 4 || n % bs || dst->num_batches != n / bs)
    return KBS_E_SHAPE;
  if (src->ld < n || (src->ld & 3)) return KBS_E_SHAPE;
  AL(perm);
  AL(src->actor_obs); AL(src->critic_obs); AL(src->action); AL(src->old_log_probs); AL(src->advantages); AL(src->value_targets);
  AL(src->old_values); AL(src->actor_carry0); AL(src->critic_carry0); AL(src->lpf0);
  AL(dst->actor_obs); AL(dst->critic_obs); AL(dst->action); AL(dst->old_log_probs); AL(dst->advantages); AL(dst->value_targets);
  AL(dst->old_values); AL(dst->actor_carry0); AL(dst->critic_carry0); AL(dst->lpf0);
  if ((reinterpret_cast<uintptr_t>(src->done) & 3u) || (reinterpret_cast<uintptr_t>(dst->done) & 3u)) return KBS_E_ALIGN;
  return kbs_launch_shuffle_minibatches(h, perm, *src, *dst, n, (cudaStream_t)stream);
}

int kbs_adamw_default_params(kbs_adamw_params* p) {
  REQ(p);
  p->lr = 5e-4f; p->b1 = 0.9; p->b2 = 0.999; p->eps = 1e-8f;   /* train.py:95-98, optax.adamw defaults */
  p->weight_decay = 1e-5f;                                       /* train.py:99-102 */
  p->grad_scale = 1.0f;
  p->max_grad_norm = 10.0f;                                      /* ksim RLConfig global gradient clip [U] */
  return KBS_OK;
}

int kbs_actuator_rand_default_params(kbs_actuator_rand_params* p) {
  REQ(p);
  p->kp_scale = 1.4f; p->kd_scale = 1.4f; p->torque_limit_scale_low = 0.5f; p->action_bias_scale = 0.02f;   /* train.py:1097-1105 */
  p->torque_bias_scale = 0.0f;
  return KBS_OK;
}

int kbs_sample_actuator_randomization(kbs_handle* h, const kbs_actuator_rand_params* rp, const float* u, const uint8_t* reset,
                                      const kbs_episode_view* ep, int64_t ld, int64_t n, void* stream) {
  REQ(h); REQ(rp); REQ(u); REQ(ep);
  int rc = check_ld(ld, n);
  if (rc) return rc;
  if (!(rp->kp_scale > 0.0f) || !(rp->kd_scale > 0.0f)) return KBS_E_PARAM;
  AL(u); AL(ep->kp); AL(ep->kd); AL(ep->tau_limit); AL(ep->action_bias); AL(ep->torque_bias);
  if (reinterpret_cast<uintptr_t>(reset) & 3u) return KBS_E_ALIGN;
  return kbs_launch_actuator_rand(h, *rp, u, reset, *ep, ld, n, (cudaStream_t)stream);
}

int kbs_rollout(kbs_handle* h, const kbs_rollout_io* io, int64_t n, void* stream) {
  return kbs_rollout_record(h, io, nullptr, n, stream);
}

int kbs_rollout_record(kbs_handle* h, const kbs_rollout_io* io, const struct kbs_rollout_record* rec, int64_t n,
                       void* stream) {
  REQ(h); REQ(io);
  if (io->T <= 0) return KBS_E_SHAPE;
  int rc = check_state(&io->state, n, true);
  if (rc) return rc;
  if ((rc = kbs_enter(h))) return rc;
  REQ(io->state.time); REQ(io->command); REQ(io->actor_carry); REQ(io->lpf); REQ(io->action); REQ(io->ctrl);
  REQ(io->done); REQ(io->success); REQ(io->cmd_mode); REQ(io->cmd_u6); REQ(io->cmd_u_arms); REQ(io->u_switch);
  if (io->value) { REQ(io->critic_carry); REQ(io->state.cinert); REQ(io->state.cvel); REQ(io->state.actuator_force); }
  const uint8_t* done_prev = rec ? rec->done_prev : nullptr;
  float* critic_obs = rec ? rec->critic_obs : nullptr;
  if (critic_obs) { REQ(io->state.cinert); REQ(io->state.cvel); REQ(io->state.actuator_force); }
  AL(critic_obs);
  if (reinterpret_cast<uintptr_t>(done_prev) & 3u) return KBS_E_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t ld = io->state.ld;
  if (h->p.gemm_path != KBS_GEMM_SIMT_FP32) {
    const int chunks = rollout_chunks();
    FusedTcWs w;
    if ((rc = kbs_scratch(h, [&](KbsScratch& s) {
           w = fused_tc_ws(s, h, n, ld, io->T, chunks, io->value != nullptr, io->pg_carry != nullptr, io->actor_obs != nullptr,
                           critic_obs != nullptr);
         })))
      return rc;
    return rollout_fused_tc(h, io, done_prev, critic_obs, w, chunks, nullptr, n, st);
  }
  SimtRolloutWs ws;
  if ((rc = kbs_scratch(h, [&](KbsScratch& s) { ws = simt_rollout_ws(s, h, n, ld); }))) return rc;
  return rollout_simt(h, io, done_prev, critic_obs, ws, n, st);
}

}  // extern "C"

namespace {

// The exact-fp32 rollout: T x (terminate, observations, actor trunk + head, torque, [critic trunk + head], command)
// one_step: kbs_rollout_step's T = 1 call (the observation kernel's one-step launch shape)
int rollout_simt(kbs_handle* h, const kbs_rollout_io* io, const uint8_t* done_prev, float* critic_obs, const SimtRolloutWs& w,
                 int64_t n, cudaStream_t st, bool one_step) {
  const int64_t ld = io->state.ld;
  const TrunkWs& ws = w.trunk;
  float* aobs_scratch = w.aobs;
  float* cobs = w.cobs;
  int rc;
  for (int64_t t = 0; t < io->T; ++t) {
    const kbs_state_view s = state_at(io->state, t);
    const kbs_noise_view nz = noise_at(io->noise, t, ld);
    const float* cmd_t = io->command + t * KBS_NUM_COMMANDS * ld;
    float* cmd_n = io->command + (t + 1) * KBS_NUM_COMMANDS * ld;
    float* aobs = io->actor_obs ? io->actor_obs + t * KBS_ACTOR_OBS * ld : aobs_scratch;
    float* cobs_t = critic_obs ? critic_obs + t * KBS_CRITIC_OBS * ld : io->value ? cobs : nullptr;
    uint8_t* done_t = io->done + t * ld;
    // terminations of the recorded state decide which carries reset after this step (train.py:1502-1506)
    if ((rc = kbs_launch_terminate(h, s, io->term_codes ? io->term_codes + t * 3 * ld : nullptr, done_t,
                                   io->success + t * ld, nullptr, n, st)))
      return rc;
    if ((rc = kbs_launch_observations(h, s, &nz, &io->episode, cmd_t, io->pg_carry, t > 0 ? done_t - ld : done_prev,
                                      nullptr, aobs, cobs_t, n, st, 1, nullptr, false, one_step)))
      return rc;
    if ((rc = trunk(h, KBS_NET_ACTOR, aobs, ld, io->actor_carry, done_t, ws, n, st))) return rc;
    kbs_actor_out o{};
    o.action = io->action + t * KBS_NUM_JOINTS * ld;
    o.log_prob = io->log_prob ? io->log_prob + t * ld : nullptr;
    if ((rc = kbs_launch_actor_head(h, ws.out_rm, kOutLd, aobs, ld, io->lpf,
                                    io->eps_action ? io->eps_action + t * KBS_NUM_JOINTS * ld : nullptr, nullptr, done_t,
                                    o, n, st)))
      return rc;
    if ((rc = kbs_launch_torque(h, o.action, s, &io->episode, io->ctrl + t * KBS_NUM_JOINTS * ld, n, st))) return rc;
    if (io->value) {
      if ((rc = trunk(h, KBS_NET_CRITIC, cobs_t, ld, io->critic_carry, done_t, ws, n, st))) return rc;
      if ((rc = kbs_launch_critic_head(h, ws.out_rm, kOutLd, io->value + t * ld, n, st))) return rc;
    }
    if ((rc = kbs_launch_command(h, cmd_t, cmd_n, io->u_switch + t * ld, io->cmd_mode + t * ld,
                                 io->cmd_u6 + t * 6 * ld, io->cmd_u_arms + t * 10 * ld, done_t, ld, n, st)))
      return rc;
  }
  return KBS_OK;
}

}  // namespace

// ---- the online rollout: one control step per call on a caller-owned step state ----------------------------------------------
namespace {

struct StepHeader { int64_t t; int32_t hsb_slot; uint32_t ticket; };
// Layout of a step state, carved from the caller's buffer like scratch (rows at ld = round_up4(n)).
struct StepState {
  StepHeader* hdr; uint8_t* done_prev; float* command /* [2][16][ld]: current, next */; float* lpf; float* pg_carry;
  KbsTcStepNet tc[2]; float* carry[2];
};
StepState step_state(KbsScratch& s, const kbs_handle* h, int64_t n, bool critic) {
  const int64_t ld = round_up4(n);
  StepState w{};
  w.hdr = s.take<StepHeader>(1);
  w.done_prev = s.take<uint8_t>(size_t(ld));
  w.command = s.take<float>(size_t(2) * KBS_NUM_COMMANDS * ld);
  w.lpf = s.take<float>(size_t(KBS_NUM_JOINTS) * ld);
  w.pg_carry = s.take<float>(size_t(3) * ld);
  for (int k = 0; k < (critic ? 2 : 1); ++k) {
    if (h->p.gemm_path == KBS_GEMM_SIMT_FP32) w.carry[k] = s.take<float>(size_t(h->p.depth) * 2 * n * h->p.hidden_size);
    else w.tc[k] = kbs_tc_step_net(s, h, n);
  }
  return w;
}

uint64_t step_state_bytes(const kbs_handle* h, int64_t n, bool critic) {
  KbsScratch s{nullptr};
  step_state(s, h, n, critic);
  return s.bytes;
}

// the descriptor's checks, then the layout on its buffer
int step_state_at(const kbs_handle* h, const kbs_step_state* st, StepState* w) {
  REQ(st); REQ(st->buf);
  if (st->n_envs <= 0) return KBS_E_SHAPE;
  if (reinterpret_cast<uintptr_t>(st->buf) & 255u) return KBS_E_ALIGN;
  if (st->bytes < step_state_bytes(h, st->n_envs, st->with_critic != 0)) return KBS_E_SHAPE;
  if (h->p.gemm_path != KBS_GEMM_SIMT_FP32 && !kbs_tc_persistent_available(h, st->n_envs, 1, st->with_critic ? 2 : 1))
    return KBS_E_SHAPE;
  KbsScratch s{static_cast<char*>(st->buf)};
  *w = step_state(s, h, st->n_envs, st->with_critic != 0);
  return KBS_OK;
}

int check_step_carry(const kbs_step_state* st, const kbs_step_carry* c) {
  REQ(c);
  if (c->critic_carry && !st->with_critic) return KBS_E_PARAM;
  AL(c->actor_carry); AL(c->critic_carry); AL(c->lpf); AL(c->pg_carry); AL(c->command);
  if (reinterpret_cast<uintptr_t>(c->done_prev) & 3u) return KBS_E_ALIGN;
  return KBS_OK;
}

// dst <- src (bytes), or zeros when src is NULL
int copy_or_zero(void* dst, const void* src, size_t bytes, cudaStream_t st) {
  if (src) KBS_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st));
  else KBS_CUDA_TRY(cudaMemsetAsync(dst, 0, bytes, st));
  return KBS_OK;
}

}  // namespace

extern "C" {

int kbs_step_state_bytes(kbs_handle* h, int64_t n, int with_critic, uint64_t* bytes) {
  REQ(h); REQ(bytes);
  if (n <= 0) return KBS_E_SHAPE;
  // the tensor-core datapaths keep the carries in the persistent kernel's layouts: a shape it cannot run has no state
  if (h->p.gemm_path != KBS_GEMM_SIMT_FP32 && !kbs_tc_persistent_available(h, n, 1, with_critic ? 2 : 1)) return KBS_E_SHAPE;
  *bytes = step_state_bytes(h, n, with_critic != 0);
  return KBS_OK;
}

int kbs_step_state_load(kbs_handle* h, const kbs_step_state* st, const kbs_step_carry* in, void* stream) {
  REQ(h);
  StepState w;
  int rc = step_state_at(h, st, &w);
  if (rc || (rc = check_step_carry(st, in)) || (rc = kbs_enter(h))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n = st->n_envs, ld = round_up4(n);
  KBS_CUDA_TRY(cudaMemsetAsync(w.hdr, 0, sizeof(StepHeader), s));
  if ((rc = copy_or_zero(w.done_prev, in->done_prev, size_t(ld), s))) return rc;
  if ((rc = copy_or_zero(w.command, in->command, size_t(KBS_NUM_COMMANDS) * ld * 4, s))) return rc;
  KBS_CUDA_TRY(cudaMemsetAsync(w.command + size_t(KBS_NUM_COMMANDS) * ld, 0, size_t(KBS_NUM_COMMANDS) * ld * 4, s));
  if ((rc = copy_or_zero(w.lpf, in->lpf, size_t(KBS_NUM_JOINTS) * ld * 4, s))) return rc;
  if ((rc = copy_or_zero(w.pg_carry, in->pg_carry, size_t(3) * ld * 4, s))) return rc;
  float* carry[2] = {in->actor_carry, in->critic_carry};
  for (int k = 0; k < (st->with_critic ? 2 : 1); ++k) {
    if (h->p.gemm_path == KBS_GEMM_SIMT_FP32)
      rc = copy_or_zero(w.carry[k], carry[k], size_t(h->p.depth) * 2 * n * h->p.hidden_size * 4, s);
    else
      rc = kbs_tc_step_carry(h, carry[k], w.tc[k], n, true, s);
    if (rc) return rc;
  }
  return KBS_OK;
}

int kbs_step_state_store(kbs_handle* h, const kbs_step_state* st, const kbs_step_carry* out, void* stream) {
  REQ(h);
  StepState w;
  int rc = step_state_at(h, st, &w);
  if (rc || (rc = check_step_carry(st, out)) || (rc = kbs_enter(h))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n = st->n_envs, ld = round_up4(n);
  auto copy = [&](void* dst, const void* src, size_t bytes) -> int {
    if (dst) KBS_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s));
    return KBS_OK;
  };
  if ((rc = copy(out->done_prev, w.done_prev, size_t(ld)))) return rc;
  if ((rc = copy(out->command, w.command, size_t(KBS_NUM_COMMANDS) * ld * 4))) return rc;
  if ((rc = copy(out->lpf, w.lpf, size_t(KBS_NUM_JOINTS) * ld * 4))) return rc;
  if ((rc = copy(out->pg_carry, w.pg_carry, size_t(3) * ld * 4))) return rc;
  float* carry[2] = {out->actor_carry, out->critic_carry};
  for (int k = 0; k < (st->with_critic ? 2 : 1); ++k) {
    if (!carry[k]) continue;
    if (h->p.gemm_path == KBS_GEMM_SIMT_FP32)
      rc = copy(carry[k], w.carry[k], size_t(h->p.depth) * 2 * n * h->p.hidden_size * 4);
    else
      rc = kbs_tc_step_carry(h, carry[k], w.tc[k], n, false, s);
    if (rc) return rc;
  }
  return KBS_OK;
}

int kbs_step_state_rewind(kbs_handle* h, const kbs_step_state* st, void* stream) {
  REQ(h);
  StepState w;
  if (const int rc = step_state_at(h, st, &w)) return rc;
  KBS_CUDA_TRY(cudaMemsetAsync(&w.hdr->t, 0, sizeof(int64_t), (cudaStream_t)stream));
  return KBS_OK;
}

int kbs_rollout_step(kbs_handle* h, const kbs_step_state* st, const kbs_step_io* io, void* stream) {
  REQ(h); REQ(io);
  StepState w;
  int rc = step_state_at(h, st, &w);
  if (rc) return rc;
  const int64_t n = st->n_envs, ld = round_up4(n);
  if (io->T <= 0) return KBS_E_SHAPE;
  if ((rc = check_state(&io->state, n, true))) return rc;
  if (io->state.ld != ld) return KBS_E_SHAPE;
  if ((rc = kbs_enter(h))) return rc;
  REQ(io->state.time); REQ(io->command); REQ(io->action); REQ(io->ctrl); REQ(io->done); REQ(io->success);
  REQ(io->cmd_mode); REQ(io->cmd_u6); REQ(io->cmd_u_arms); REQ(io->u_switch);
  if (io->value || io->critic_obs) { REQ(io->state.cinert); REQ(io->state.cvel); REQ(io->state.actuator_force); }
  if (io->value && !st->with_critic) return KBS_E_PARAM;
  if (!h->net[KBS_NET_ACTOR].packed || (io->value && !h->net[KBS_NET_CRITIC].packed)) return KBS_E_STATE;
  if (io->noise.eps_jpos) { REQ(io->noise.eps_jvel); REQ(io->noise.eps_gyro); REQ(io->noise.eps_pg); }
  AL(io->noise.eps_jpos); AL(io->noise.eps_jvel); AL(io->noise.eps_gyro); AL(io->noise.eps_pg);
  AL(io->eps_action); AL(io->u_switch); AL(io->cmd_mode); AL(io->cmd_u6); AL(io->cmd_u_arms);
  AL(io->command); AL(io->actor_obs); AL(io->critic_obs); AL(io->action); AL(io->log_prob); AL(io->ctrl); AL(io->term_codes);
  AL(io->value);
  if ((reinterpret_cast<uintptr_t>(io->done) & 3u) || (reinterpret_cast<uintptr_t>(io->success) & 3u)) return KBS_E_ALIGN;
  // the recorded state: (step field, trajectory field, rows)
  const kbs_state_view& a = io->state;
  const kbs_state_view& b = io->traj_state;
  const struct { const float* src; const float* dst; int rows; } rows[] = {
      {a.qpos, b.qpos, KBS_NQ}, {a.qvel, b.qvel, KBS_NV}, {a.sensordata, b.sensordata, KBS_NSENSORDATA},
      {a.xpos, b.xpos, 3 * KBS_NBODY}, {a.xquat, b.xquat, 4 * KBS_NBODY}, {a.cinert, b.cinert, 10 * KBS_NBODY},
      {a.cvel, b.cvel, 6 * KBS_NBODY}, {a.actuator_force, b.actuator_force, KBS_NUM_JOINTS}, {a.com_distance, b.com_distance, 1},
      {a.time, b.time, 1}};
  for (const auto& r : rows) {
    if (r.dst && !r.src) return KBS_E_NULL;
    AL(r.dst);
  }
  cudaStream_t s = (cudaStream_t)stream;
  const bool tc = h->p.gemm_path != KBS_GEMM_SIMT_FP32, critic = io->value != nullptr;

  // this step's outputs in scratch (the rollout kernels' addressing stays that of a T = 1 call), then one record pass
  float *aobs, *cobs, *action, *log_prob, *ctrl, *value;
  int32_t* codes;
  uint8_t *done, *success;
  FusedTcWs tw;
  SimtRolloutWs sw;
  rc = kbs_scratch(h, [&](KbsScratch& sc) {
    aobs = sc.take<float>(size_t(KBS_ACTOR_OBS) * ld);
    cobs = io->critic_obs ? sc.take<float>(size_t(KBS_CRITIC_OBS) * ld) : nullptr;
    action = sc.take<float>(size_t(KBS_NUM_JOINTS) * ld);
    log_prob = sc.take<float>(size_t(ld));
    ctrl = sc.take<float>(size_t(KBS_NUM_JOINTS) * ld);
    value = critic ? sc.take<float>(size_t(ld)) : nullptr;
    codes = io->term_codes ? sc.take<int32_t>(size_t(3) * ld) : nullptr;
    done = sc.take<uint8_t>(size_t(ld));
    success = sc.take<uint8_t>(size_t(ld));
    if (tc) tw = fused_tc_ws(sc, h, n, ld, 1, 1, critic, true, true, io->critic_obs != nullptr);
    else sw = simt_rollout_ws(sc, h, n, ld);
  });
  if (rc) return rc;
  kbs_rollout_io r1{};
  r1.state = io->state; r1.noise = io->noise; r1.episode = io->episode;
  r1.eps_action = io->eps_action; r1.u_switch = io->u_switch; r1.cmd_mode = io->cmd_mode; r1.cmd_u6 = io->cmd_u6;
  r1.cmd_u_arms = io->cmd_u_arms;
  r1.command = w.command; r1.pg_carry = w.pg_carry; r1.lpf = w.lpf;
  r1.actor_carry = w.carry[0]; r1.critic_carry = w.carry[1];          // SIMT; the tensor-core kernels read w.tc in place
  r1.actor_obs = aobs; r1.action = action; r1.log_prob = log_prob; r1.ctrl = ctrl; r1.term_codes = codes;
  r1.done = done; r1.success = success; r1.value = value; r1.T = 1;
  if (tc) {
    KbsTcRolloutArgs res{};
    for (int k = 0; k < 2; ++k) { res.res_hsb[k] = w.tc[k].hsb; res.res_fb[k] = w.tc[k].fb; }
    res.res_hsb_slot = &w.hdr->hsb_slot;
    rc = rollout_fused_tc(h, &r1, w.done_prev, cobs, tw, 1, &res, n, s);
  } else {
    rc = rollout_simt(h, &r1, w.done_prev, cobs, sw, n, s, /*one_step=*/true);
  }
  if (rc) return rc;

  KbsStepRecord R{};
  int j = 0;
  auto job = [&](const void* src, void* dst, int64_t words) {
    if (!dst) return;
    R.job[j].src = src; R.job[j].dst = dst; R.job[j].words = words; R.job[j].dst_step = words; ++j;
  };
  job(aobs, io->actor_obs, KBS_ACTOR_OBS * ld);
  job(cobs, io->critic_obs, KBS_CRITIC_OBS * ld);
  job(action, io->action, KBS_NUM_JOINTS * ld);
  job(log_prob, io->log_prob, ld);
  job(ctrl, io->ctrl, KBS_NUM_JOINTS * ld);
  job(value, io->value, ld);
  job(codes, io->term_codes, 3 * ld);
  job(done, io->done, ld / 4);
  job(success, io->success, ld / 4);
  for (const auto& rr : rows) job(rr.src, const_cast<float*>(rr.dst), rr.rows * ld);
  job(done, w.done_prev, ld / 4);
  R.job[j - 1].dst_step = 0;                                           // done_prev: no time axis
  R.job[j].src = w.command; R.job[j].dst = io->command; R.job[j].words = KBS_NUM_COMMANDS * ld;
  R.job[j].dst_step = KBS_NUM_COMMANDS * ld; R.job[j].shift = 1; ++j;
  R.jobs = j;
  R.T = io->T; R.t = &w.hdr->t; R.hsb_slot = tc ? &w.hdr->hsb_slot : nullptr; R.ticket = &w.hdr->ticket;
  if ((rc = kbs_status_init(h))) return rc;
  R.status = h->persist_status;
  if ((rc = kbs_launch_step_record(h, R, s))) return rc;
  return kbs_status_publish(h, s);
}

}  // extern "C"

// ---- the physics sub-steps between two online control steps, on a caller-owned actuator state ------------------------------
namespace {

struct ActuatorHeader { int32_t k; uint32_t ticket; };
// Layout of an actuator state, carved from the caller's buffer like scratch (rows at ld = round_up4(n)).
struct ActuatorState { ActuatorHeader* hdr; float* prev_action; float* applied; };
ActuatorState actuator_state(KbsScratch& s, int64_t n) {
  const int64_t ld = round_up4(n);
  ActuatorState w{};
  w.hdr = s.take<ActuatorHeader>(1);
  w.prev_action = s.take<float>(size_t(KBS_NUM_JOINTS) * ld);
  w.applied = s.take<float>(size_t(KBS_NUM_JOINTS) * ld);
  return w;
}

uint64_t actuator_state_bytes(int64_t n) {
  KbsScratch s{nullptr};
  actuator_state(s, n);
  return s.bytes;
}

// the descriptor's checks, then the layout on its buffer
int actuator_state_at(const kbs_actuator_state* ast, ActuatorState* w) {
  REQ(ast); REQ(ast->buf);
  if (ast->n_envs <= 0 || ast->n_substeps <= 0) return KBS_E_SHAPE;
  if (reinterpret_cast<uintptr_t>(ast->buf) & 255u) return KBS_E_ALIGN;
  if (ast->bytes < actuator_state_bytes(ast->n_envs)) return KBS_E_SHAPE;
  KbsScratch s{static_cast<char*>(ast->buf)};
  *w = actuator_state(s, ast->n_envs);
  return KBS_OK;
}

}  // namespace

extern "C" {

int kbs_actuator_state_bytes(kbs_handle* h, int64_t n, uint64_t* bytes) {
  REQ(h); REQ(bytes);
  if (n <= 0) return KBS_E_SHAPE;
  *bytes = actuator_state_bytes(n);
  return KBS_OK;
}

int kbs_actuator_state_load(kbs_handle* h, const kbs_actuator_state* ast, const float* prev_action, void* stream) {
  REQ(h);
  ActuatorState w;
  int rc = actuator_state_at(ast, &w);
  if (rc) return rc;
  AL(prev_action);
  if ((rc = kbs_enter(h))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t rows = size_t(KBS_NUM_JOINTS) * round_up4(ast->n_envs) * 4;
  KBS_CUDA_TRY(cudaMemsetAsync(w.hdr, 0, sizeof(ActuatorHeader), s));
  if ((rc = copy_or_zero(w.prev_action, prev_action, rows, s))) return rc;
  KBS_CUDA_TRY(cudaMemsetAsync(w.applied, 0, rows, s));
  return KBS_OK;
}

int kbs_actuator_state_store(kbs_handle* h, const kbs_actuator_state* ast, float* prev_action, void* stream) {
  REQ(h); REQ(prev_action);
  ActuatorState w;
  int rc = actuator_state_at(ast, &w);
  if (rc) return rc;
  AL(prev_action);
  if ((rc = kbs_enter(h))) return rc;
  KBS_CUDA_TRY(cudaMemcpyAsync(prev_action, w.prev_action, size_t(KBS_NUM_JOINTS) * round_up4(ast->n_envs) * 4,
                               cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return KBS_OK;
}

int kbs_actuator_substep(kbs_handle* h, const kbs_step_state* st, const kbs_actuator_state* ast, const kbs_substep_io* io,
                         void* stream) {
  REQ(h); REQ(io);
  StepState w;
  ActuatorState aw;
  int rc = step_state_at(h, st, &w);
  if (rc || (rc = actuator_state_at(ast, &aw))) return rc;
  REQ(io->action); REQ(io->u_drop); REQ(io->latency); REQ(io->qpos); REQ(io->qvel); REQ(io->ctrl);
  if (st->n_envs != ast->n_envs || io->T <= 0) return KBS_E_SHAPE;
  if (!(io->sub_dt > 0.f) || !(io->drop_prob >= 0.f && io->drop_prob <= 1.f)) return KBS_E_PARAM;
  AL(io->action); AL(io->u_drop); AL(io->latency); AL(io->qpos); AL(io->qvel); AL(io->ctrl);
  const kbs_episode_view& ep = io->episode;
  AL(ep.kp); AL(ep.kd); AL(ep.tau_limit); AL(ep.action_bias); AL(ep.torque_bias);
  if ((rc = kbs_enter(h))) return rc;
  if ((rc = kbs_status_init(h))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  KbsSubstepArgs a{};
  a.action = io->action; a.T = io->T; a.t = &w.hdr->t;
  a.k = &aw.hdr->k; a.ticket = &aw.hdr->ticket; a.prev_action = aw.prev_action; a.applied = aw.applied;
  a.u_drop = io->u_drop; a.latency = io->latency; a.qpos = io->qpos; a.qvel = io->qvel; a.ep = ep; a.ctrl = io->ctrl;
  a.S = ast->n_substeps; a.sub_dt = io->sub_dt; a.drop_prob = io->drop_prob;
  a.n = st->n_envs; a.ld = round_up4(st->n_envs); a.status = h->persist_status;
  if ((rc = kbs_launch_actuator_substep(h, a, s))) return rc;
  return kbs_status_publish(h, s);
}

}  // extern "C"
