// kbs_elementwise.cu -- HBM-bound stages of the control step: observations, command law, PD torque map,
// terminations, the 12 reward terms and the GAE scan.  Env-major SoA, float4 per thread (4 consecutive envs),
// streaming loads/stores.  Compiled with -fmad=false so the operation order is exactly the one written here
// (the reference's jnp expressions, train.py line ranges cited per kernel); HBM-bound, FMA rate is irrelevant.
#include <math.h>

#include "kbs_common.cuh"

namespace {

constexpr int kThreads = 128;
constexpr float kHalfPi = 1.57079632679489662f;
constexpr float kPi = 3.14159265358979324f;

// ---- xax quaternion helpers (SURVEY Appendix F), (w,x,y,z) -------------------------------------------
__device__ __forceinline__ void quat_norm_eps(float (&q)[4], float eps) {
  const float n = sqrtf(((q[0] * q[0] + q[1] * q[1]) + q[2] * q[2]) + q[3] * q[3]) + eps;
  q[0] /= n; q[1] /= n; q[2] /= n; q[3] /= n;
}

__device__ __forceinline__ void quat_to_euler(const float (&qin)[4], float eps, float (&e)[3]) {
  float q[4] = {qin[0], qin[1], qin[2], qin[3]};
  quat_norm_eps(q, eps);
  const float w = q[0], x = q[1], y = q[2], z = q[3];
  e[0] = atan2f(2.0f * (w * x + y * z), 1.0f - 2.0f * (x * x + y * y));
  const float sinp = 2.0f * (w * y - z * x);
  e[1] = (fabsf(sinp) >= 1.0f) ? copysignf(kHalfPi, sinp) : asinf(sinp);
  e[2] = atan2f(2.0f * (w * z + x * y), 1.0f - 2.0f * (y * y + z * z));
}

__device__ __forceinline__ void euler_to_quat(float roll, float pitch, float yaw, float (&q)[4]) {
  const float r = roll * 0.5f, p = pitch * 0.5f, y = yaw * 0.5f;
  const float cr = cosf(r), sr = sinf(r), cp = cosf(p), sp = sinf(p), cy = cosf(y), sy = sinf(y);
  q[0] = cr * cp * cy + sr * sp * sy;
  q[1] = sr * cp * cy - cr * sp * sy;
  q[2] = cr * sp * cy + sr * cp * sy;
  q[3] = cr * cp * sy - sr * sp * cy;
  const float n = sqrtf(((q[0] * q[0] + q[1] * q[1]) + q[2] * q[2]) + q[3] * q[3]);
  q[0] /= n; q[1] /= n; q[2] /= n; q[3] /= n;
}

__device__ __forceinline__ void rotate_vec(const float (&v)[3], const float (&qin)[4], bool inverse, float eps,
                                           float (&o)[3]) {
  float q[4] = {qin[0], qin[1], qin[2], qin[3]};
  quat_norm_eps(q, eps);
  const float w = q[0];
  const float x = inverse ? -q[1] : q[1], y = inverse ? -q[2] : q[2], z = inverse ? -q[3] : q[3];
  const float vx = v[0], vy = v[1], vz = v[2];
  const float t = 2.0f;
  o[0] = w * w * vx + t * y * w * vz - t * z * w * vy + x * x * vx + t * y * x * vy + t * z * x * vz - z * z * vx - y * y * vx;
  o[1] = t * x * y * vx + y * y * vy + t * z * y * vz + t * w * z * vx - z * z * vy + w * w * vy - t * w * x * vz - x * x * vy;
  o[2] = t * x * z * vx + t * y * z * vy + z * z * vz - t * w * y * vx + w * w * vz + t * w * x * vy - y * y * vz - x * x * vz;
}

__device__ __forceinline__ bool zero_cmd(float c0, float c1, float c2) {
  return sqrtf((c0 * c0 + c1 * c1) + c2 * c2) < 1e-3f;
}

// encode_projected_gravity, train.py:1338-1349
__device__ __forceinline__ void encode_pg(const float (&g)[3], float (&o)[5]) {
  o[0] = atan2f(g[1], -g[2]);
  o[1] = atan2f(-g[0], sqrtf(g[1] * g[1] + g[2] * g[2]));
  const float n = sqrtf((g[0] * g[0] + g[1] * g[1]) + g[2] * g[2]);
  o[2] = g[0] / n; o[3] = g[1] / n; o[4] = g[2] / n;
}

// =====================================================================================================
// observations: get_observations table + run_actor / run_critic concats.
// train.py:1155-1204, 682-707, 1329-1431.  grid = (env groups, 1 + copy sections).
// =====================================================================================================
// Sections of obs_kernel.  The trajectory form (T steps per launch): joints in 2 sections, IMU + command in one, feet + the
// critic's small copies in one, then the 368 pure-copy rows (cinert 230 + cvel 138) in 8 sections.  The one-step form
// (kbs_rollout_step: a few thousand envs, one step per launch) cuts the same rows 6x finer -- one joint per section, the command
// apart from the IMU, 8 copy rows per section -- so one step fills the SMs instead of running on a few blocks per SM.
template <bool ONE_STEP> struct ObsSections {
  static constexpr int kJoint = ONE_STEP ? 20 : 2;           // joint sections, KBS_NUM_JOINTS / kJoint joints each
  static constexpr int kImu = kJoint;
  static constexpr int kCmd = ONE_STEP ? kImu + 1 : kImu;     // the trajectory form does both in one section
  static constexpr int kFeet = kCmd + 1;
  static constexpr int kComputed = kFeet + 1;                 // sections before the copy sections
  static constexpr int kCopyRows = ONE_STEP ? 8 : 46;
  static constexpr int kCopy = 368 / kCopyRows;
};
constexpr int kCopyRowsPerSection = 46;  // mirror_obs_kernel's copy sections (the trajectory form's)
static_assert(368 % ObsSections<true>::kCopyRows == 0 && 368 % ObsSections<false>::kCopyRows == 0, "copy sections");

template <bool ONE_STEP>
__global__ void __launch_bounds__(kThreads)
obs_kernel(const __grid_constant__ kbs_params P, kbs_state_view s, kbs_noise_view nz,
           const kbs_episode_view ep, const float* __restrict__ command, float* __restrict__ pg_carry,
           const uint8_t* __restrict__ pg_reset, const float* __restrict__ pg_lagged, float* __restrict__ computed,
           float* __restrict__ actor_obs, float* __restrict__ critic_obs, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  const int64_t ld = s.ld;
  {  // time axis of a trajectory call: every [T][F][ld] array advances by t * F * ld
    const int64_t t = blockIdx.z;
    s.qpos += t * KBS_NQ * ld; s.qvel += t * KBS_NV * ld; s.sensordata += t * KBS_NSENSORDATA * ld;
    s.xpos += t * 3 * KBS_NBODY * ld; s.xquat += t * 4 * KBS_NBODY * ld;
    if (s.cinert) s.cinert += t * 10 * KBS_NBODY * ld;
    if (s.cvel) s.cvel += t * 6 * KBS_NBODY * ld;
    if (s.actuator_force) s.actuator_force += t * KBS_NUM_JOINTS * ld;
    if (nz.eps_jpos) { nz.eps_jpos += t * 20 * ld; nz.eps_jvel += t * 20 * ld; nz.eps_gyro += t * 3 * ld; nz.eps_pg += t * 3 * ld; }
    command += t * KBS_NUM_COMMANDS * ld;
    if (pg_lagged) pg_lagged += t * 3 * ld;
    if (computed) computed += t * KBS_NUM_COMPUTED_OBS * ld;
    if (actor_obs) actor_obs += t * KBS_ACTOR_OBS * ld;
    if (critic_obs) critic_obs += t * KBS_CRITIC_OBS * ld;
  }

  // blockIdx.y = section: the rows of one env-step are independent, so they are spread over the sections x as many
  // threads (one thread doing all ~250 rows of its 4 envs left 21 warps per SM and 2.4 TB/s).  Trajectory form:
  //   0 / 1: joints 0-9 / 10-19   2: IMU + command slots   3: feet positions + the critic's small copies   4..: dump
  using S = ObsSections<ONE_STEP>;
  const int sec = blockIdx.y;
  if (sec >= S::kComputed) {
    // critic privileged dump: center_of_mass_inertia = cinert[1:], center_of_mass_velocity = cvel[1:]
    const int i0 = (sec - S::kComputed) * S::kCopyRows;
#pragma unroll 8
    for (int i = i0; i < i0 + S::kCopyRows; ++i) {
      if (i < 230) kbs_copy4(s.cinert, 10 + i, critic_obs, 80 + i, ld, n0);
      else if (i < 368) kbs_copy4(s.cvel, 6 + (i - 230), critic_obs, 310 + (i - 230), ld, n0);
    }
    return;
  }

  const bool has_noise = nz.eps_jpos != nullptr;

  // joints: slots 0-19 / 20-39
  if (sec < S::kJoint) {
  constexpr int kPer = KBS_NUM_JOINTS / S::kJoint;
#pragma unroll 5
  for (int j = sec * kPer; j < sec * kPer + kPer; ++j) {
    float q[4], qd[4], jb[4] = {0, 0, 0, 0}, e1[4] = {0, 0, 0, 0}, e2[4] = {0, 0, 0, 0};
    kbs_ld4(s.qpos, 7 + j, ld, n0, q);
    kbs_ld4(s.qvel, 6 + j, ld, n0, qd);
    if (ep.jpos_bias) kbs_ld4(ep.jpos_bias, j, ld, n0, jb);
    if (has_noise) { kbs_ld4(nz.eps_jpos, j, ld, n0, e1); kbs_ld4(nz.eps_jvel, j, ld, n0, e2); }
    float bj[4], nbj[4], nv[4], a0[4], a1[4], c0[4], c1[4];
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      bj[l] = q[l] + jb[l];
      nbj[l] = bj[l] + P.jpos_noise_mag * e1[l];
      nv[l] = qd[l] + P.jvel_noise_mag * e2[l];
      a0[l] = (nbj[l] - P.joint_bias[j]) / P.joint_range[j];
      a1[l] = nv[l] / 10.0f;
      c0[l] = (q[l] - P.joint_bias[j]) / P.joint_range[j];
      c1[l] = qd[l] / 10.0f;
    }
    if (computed) { kbs_st4(computed, j, ld, n0, bj); kbs_st4(computed, 20 + j, ld, n0, nbj); kbs_st4(computed, 40 + j, ld, n0, nv); }
    if (actor_obs) { kbs_st4(actor_obs, j, ld, n0, a0); kbs_st4(actor_obs, 20 + j, ld, n0, a1); }
    if (critic_obs) { kbs_st4(critic_obs, j, ld, n0, c0); kbs_st4(critic_obs, 20 + j, ld, n0, c1); }
  }
  return;
  }

  // IMU: projected gravity (clean + lagged/biased/noisy twin) and gyro
  if (sec == S::kImu) {
    float iq[4][4], gy[3][4];
#pragma unroll
    for (int k = 0; k < 4; ++k) kbs_ld4(s.sensordata, P.sd_imu_quat + k, ld, n0, iq[k]);
#pragma unroll
    for (int k = 0; k < 3; ++k) kbs_ld4(s.sensordata, P.sd_gyro + k, ld, n0, gy[k]);
    float lag[4] = {0, 0, 0, 0}, pgb[3][4] = {}, epg[3][4] = {}, egy[3][4] = {}, prev[3][4];
    if (ep.pg_lag) kbs_ld4(ep.pg_lag, 0, ld, n0, lag);
    if (ep.pg_bias) { for (int k = 0; k < 3; ++k) kbs_ld4(ep.pg_bias, k, ld, n0, pgb[k]); }
    if (has_noise) {
      for (int k = 0; k < 3; ++k) { kbs_ld4(nz.eps_pg, k, ld, n0, epg[k]); kbs_ld4(nz.eps_gyro, k, ld, n0, egy[k]); }
    }
    if (pg_carry) { for (int k = 0; k < 3; ++k) kbs_ld4(pg_carry, k, ld, n0, prev[k]); }
    float lagged[3][4];
    if (pg_lagged) { for (int k = 0; k < 3; ++k) kbs_ld4(pg_lagged, k, ld, n0, lagged[k]); }
    bool rs[4] = {false, false, false, false};  // new episode: EMA state restarts at the current value
    if (pg_reset) {
      const uchar4 r4 = *reinterpret_cast<const uchar4*>(pg_reset + n0);
      rs[0] = r4.x != 0; rs[1] = r4.y != 0; rs[2] = r4.z != 0; rs[3] = r4.w != 0;
    }
    float o_pg[3][4], o_ipg[3][4], o_nipg[3][4], o_ngy[3][4], o_carry[3][4], enc_a[5][4], enc_c[5][4];
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const float q[4] = {iq[0][l], iq[1][l], iq[2][l], iq[3][l]};
      const float g[3] = {0.0f, 0.0f, -P.gravity};
      float gb[3];
      rotate_vec(g, q, true, P.eps_quat, gb);
      float na[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float pv = (pg_carry && !rs[l]) ? prev[k][l] : gb[k];
        const float nc = pg_lagged ? lagged[k][l] : lag[l] * pv + (1.0f - lag[l]) * gb[k];
        o_carry[k][l] = nc;
        o_pg[k][l] = gb[k];
        o_ipg[k][l] = nc + pgb[k][l];
        o_nipg[k][l] = o_ipg[k][l] + P.pg_noise_std * epg[k][l];
        o_ngy[k][l] = gy[k][l] + P.gyro_noise_std * egy[k][l];
        na[k] = o_nipg[k][l];
      }
      float ea[5], ec[5];
      encode_pg(na, ea);
      encode_pg(gb, ec);
#pragma unroll
      for (int k = 0; k < 5; ++k) { enc_a[k][l] = ea[k]; enc_c[k][l] = ec[k]; }
    }
    if (pg_carry) { for (int k = 0; k < 3; ++k) kbs_st4(pg_carry, k, ld, n0, o_carry[k]); }
    if (computed) {
      for (int k = 0; k < 3; ++k) {
        kbs_st4(computed, 60 + k, ld, n0, o_ngy[k]);
        kbs_st4(computed, 69 + k, ld, n0, o_pg[k]);
        kbs_st4(computed, 72 + k, ld, n0, o_ipg[k]);
        kbs_st4(computed, 75 + k, ld, n0, o_nipg[k]);
      }
    }
    if (actor_obs) {
      for (int k = 0; k < 5; ++k) kbs_st4(actor_obs, 40 + k, ld, n0, enc_a[k]);
      for (int k = 0; k < 3; ++k) kbs_st4(actor_obs, 45 + k, ld, n0, o_ngy[k]);
    }
    if (critic_obs) {
      for (int k = 0; k < 5; ++k) kbs_st4(critic_obs, 40 + k, ld, n0, enc_c[k]);
      for (int k = 0; k < 3; ++k) kbs_st4(critic_obs, 45 + k, ld, n0, gy[k]);
    }
    if (S::kCmd != S::kImu) return;
  }

  // zero_cmd flag + command: slots 48, 49-64
  if (sec == S::kCmd) {
  float c[16][4];
#pragma unroll
  for (int k = 0; k < 16; ++k) kbs_ld4(command, k, ld, n0, c[k]);
  float zc[4];
#pragma unroll
  for (int l = 0; l < 4; ++l) zc[l] = zero_cmd(c[0][l], c[1][l], c[2][l]) ? 1.0f : 0.0f;
  if (actor_obs) {
    kbs_st4(actor_obs, 48, ld, n0, zc);
#pragma unroll
    for (int k = 0; k < 16; ++k) kbs_st4(actor_obs, 49 + k, ld, n0, c[k]);
  }
  if (critic_obs) {
    kbs_st4(critic_obs, 48, ld, n0, zc);
#pragma unroll
    for (int k = 0; k < 16; ++k) kbs_st4(critic_obs, 49 + k, ld, n0, c[k]);
  }
  return;
  }

  if (computed || critic_obs) {
    // FeetPositionObservation train.py:682-699
    float bp[3][4], lp[3][4], rp[3][4], bq[4][4], fpos[6][4];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      kbs_ld4(s.xpos, 3 * P.body_base + k, ld, n0, bp[k]);
      kbs_ld4(s.xpos, 3 * P.body_lfoot + k, ld, n0, lp[k]);
      kbs_ld4(s.xpos, 3 * P.body_rfoot + k, ld, n0, rp[k]);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) kbs_ld4(s.xquat, 4 * P.body_base + k, ld, n0, bq[k]);
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const float q[4] = {bq[0][l], bq[1][l], bq[2][l], bq[3][l]};
      float e[3], qy[4], o[3];
      quat_to_euler(q, P.eps_quat, e);
      euler_to_quat(0.0f, 0.0f, e[2], qy);
      const float dl[3] = {lp[0][l] - bp[0][l], lp[1][l] - bp[1][l], lp[2][l] - bp[2][l]};
      rotate_vec(dl, qy, true, P.eps_quat, o);
      fpos[0][l] = o[0]; fpos[1][l] = o[1]; fpos[2][l] = o[2];
      const float dr[3] = {rp[0][l] - bp[0][l], rp[1][l] - bp[1][l], rp[2][l] - bp[2][l]};
      rotate_vec(dr, qy, true, P.eps_quat, o);
      fpos[3][l] = o[0]; fpos[4][l] = o[1]; fpos[5][l] = o[2];
    }
    if (computed) { for (int k = 0; k < 6; ++k) kbs_st4(computed, 63 + k, ld, n0, fpos[k]); }
    if (critic_obs) {
      for (int k = 0; k < 6; ++k) kbs_st4(critic_obs, 67 + k, ld, n0, fpos[k]);
      kbs_copy4(s.sensordata, P.sd_touch_l, critic_obs, 65, ld, n0);
      kbs_copy4(s.sensordata, P.sd_touch_r, critic_obs, 66, ld, n0);
      for (int k = 0; k < 7; ++k) kbs_copy4(s.qpos, k, critic_obs, 73 + k, ld, n0);   // base pos + quat
      for (int k = 0; k < 6; ++k) kbs_copy4(s.qvel, k, critic_obs, 448 + k, ld, n0);  // base lin + ang vel
#pragma unroll 4
      for (int j = 0; j < KBS_NUM_JOINTS; ++j) {
        float f[4];
        kbs_ld4(s.actuator_force, j, ld, n0, f);
#pragma unroll
        for (int l = 0; l < 4; ++l) f[l] = f[l] / 4.0f;
        kbs_st4(critic_obs, 454 + j, ld, n0, f);
      }
      kbs_st4(critic_obs, 474, ld, n0, bp[2]);  // base_height = xpos[1, 2]
    }
  }
}

// =====================================================================================================
// X1: mirror_obs / mirror_cmd / mirror_joints (train.py:1574-1756) followed by the run_actor / run_critic
// concatenations on the MIRRORED observations -- what _ppo_scan_fn feeds the *_mirror carries (train.py:1463-1481).
// The mirror acts on the raw named observations (before normalisation), so it is built from the stored raw
// observations (`computed`, the noisy twins the rollout recorded) and the state slices, not from actor_obs.
//   mirror_joints(j) = -[j[5:10], j[0:5], j[10:15], j[15:20]]  (legs swapped, arms NOT: as written)
// grid = (env groups, 1 + copy sections, T)
// =====================================================================================================
__device__ __forceinline__ int mirror_src_joint(int j) { return j < 5 ? j + 5 : (j < 10 ? j - 5 : j); }

__global__ void __launch_bounds__(kThreads)
mirror_obs_kernel(const __grid_constant__ kbs_params P, kbs_state_view s, const float* __restrict__ computed,
                  const float* __restrict__ command, float* __restrict__ actor_obs, float* __restrict__ critic_obs,
                  float* __restrict__ command_out, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  const int64_t ld = s.ld;
  {
    const int64_t t = blockIdx.z;
    s.qpos += t * KBS_NQ * ld; s.qvel += t * KBS_NV * ld; s.sensordata += t * KBS_NSENSORDATA * ld;
    s.xpos += t * 3 * KBS_NBODY * ld;
    if (s.cinert) s.cinert += t * 10 * KBS_NBODY * ld;
    if (s.cvel) s.cvel += t * 6 * KBS_NBODY * ld;
    if (s.actuator_force) s.actuator_force += t * KBS_NUM_JOINTS * ld;
    computed += t * KBS_NUM_COMPUTED_OBS * ld;
    command += t * KBS_NUM_COMMANDS * ld;
    if (actor_obs) actor_obs += t * KBS_ACTOR_OBS * ld;
    if (critic_obs) critic_obs += t * KBS_CRITIC_OBS * ld;
    if (command_out) command_out += t * KBS_NUM_COMMANDS * ld;
  }
  if (blockIdx.y > 0) {
    // center_of_mass_inertia (.,10) * (1,1,-1,1,1,1,1,-1,1,-1); center_of_mass_velocity (.,6) * (1,-1,1,-1,1,-1)
    const int i0 = (blockIdx.y - 1) * kCopyRowsPerSection;
    for (int i = i0; i < i0 + kCopyRowsPerSection; ++i) {
      float v[4];
      if (i < 230) {
        const int c = i % 10;
        const float sg = (c == 2 || c == 7 || c == 9) ? -1.0f : 1.0f;
        kbs_ld4(s.cinert, 10 + i, ld, n0, v);
#pragma unroll
        for (int l = 0; l < 4; ++l) v[l] = v[l] * sg;
        kbs_st4(critic_obs, 80 + i, ld, n0, v);
      } else if (i < 368) {
        const int c = (i - 230) % 6;
        const float sg = (c & 1) ? -1.0f : 1.0f;
        kbs_ld4(s.cvel, 6 + (i - 230), ld, n0, v);
#pragma unroll
        for (int l = 0; l < 4; ++l) v[l] = v[l] * sg;
        kbs_st4(critic_obs, 310 + (i - 230), ld, n0, v);
      }
    }
    return;
  }
  // mirror_cmd: (vx, -vy, -wz, bh, -rx, ry, -arms)
  float c[16][4], zc[4];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    kbs_ld4(command, k, ld, n0, c[k]);
    const bool neg = (k == 1 || k == 2 || k == 4 || k >= 6);
    if (neg) {
#pragma unroll
      for (int l = 0; l < 4; ++l) c[k][l] = -c[k][l];
    }
  }
#pragma unroll
  for (int l = 0; l < 4; ++l) zc[l] = zero_cmd(c[0][l], c[1][l], c[2][l]) ? 1.0f : 0.0f;
  if (command_out) {
#pragma unroll
    for (int k = 0; k < 16; ++k) kbs_st4(command_out, k, ld, n0, c[k]);
  }
#pragma unroll 4
  for (int j = 0; j < KBS_NUM_JOINTS; ++j) {
    const int sj = mirror_src_joint(j);
    float nbj[4], nv[4], q[4], qd[4], a0[4], a1[4], c0[4], c1[4];
    kbs_ld4(computed, 20 + sj, ld, n0, nbj);
    kbs_ld4(computed, 40 + sj, ld, n0, nv);
    kbs_ld4(s.qpos, 7 + sj, ld, n0, q);
    kbs_ld4(s.qvel, 6 + sj, ld, n0, qd);
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      a0[l] = (-nbj[l] - P.joint_bias[j]) / P.joint_range[j];
      a1[l] = -nv[l] / 10.0f;
      c0[l] = (-q[l] - P.joint_bias[j]) / P.joint_range[j];
      c1[l] = -qd[l] / 10.0f;
    }
    if (actor_obs) { kbs_st4(actor_obs, j, ld, n0, a0); kbs_st4(actor_obs, 20 + j, ld, n0, a1); }
    if (critic_obs) { kbs_st4(critic_obs, j, ld, n0, c0); kbs_st4(critic_obs, 20 + j, ld, n0, c1); }
  }
  {
    // projected gravity * (1,-1,1) -> encode; gyro * (-1,1,-1)
    float npg[3][4], pg[3][4], ngy[3][4], gy[3][4], ea[5][4], ec[5][4];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      kbs_ld4(computed, 75 + k, ld, n0, npg[k]);
      kbs_ld4(computed, 69 + k, ld, n0, pg[k]);
      kbs_ld4(computed, 60 + k, ld, n0, ngy[k]);
      kbs_ld4(s.sensordata, P.sd_gyro + k, ld, n0, gy[k]);
    }
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const float ga[3] = {npg[0][l], -npg[1][l], npg[2][l]}, gc[3] = {pg[0][l], -pg[1][l], pg[2][l]};
      float oa[5], oc[5];
      encode_pg(ga, oa);
      encode_pg(gc, oc);
#pragma unroll
      for (int k = 0; k < 5; ++k) { ea[k][l] = oa[k]; ec[k][l] = oc[k]; }
      ngy[0][l] = -ngy[0][l]; ngy[2][l] = -ngy[2][l];
      gy[0][l] = -gy[0][l]; gy[2][l] = -gy[2][l];
    }
    if (actor_obs) {
      for (int k = 0; k < 5; ++k) kbs_st4(actor_obs, 40 + k, ld, n0, ea[k]);
      for (int k = 0; k < 3; ++k) kbs_st4(actor_obs, 45 + k, ld, n0, ngy[k]);
    }
    if (critic_obs) {
      for (int k = 0; k < 5; ++k) kbs_st4(critic_obs, 40 + k, ld, n0, ec[k]);
      for (int k = 0; k < 3; ++k) kbs_st4(critic_obs, 45 + k, ld, n0, gy[k]);
    }
  }
  if (actor_obs) {
    kbs_st4(actor_obs, 48, ld, n0, zc);
#pragma unroll
    for (int k = 0; k < 16; ++k) kbs_st4(actor_obs, 49 + k, ld, n0, c[k]);
  }
  if (critic_obs) {
    kbs_st4(critic_obs, 48, ld, n0, zc);
#pragma unroll
    for (int k = 0; k < 16; ++k) kbs_st4(critic_obs, 49 + k, ld, n0, c[k]);
    kbs_copy4(s.sensordata, P.sd_touch_r, critic_obs, 65, ld, n0);       // left <- right
    kbs_copy4(s.sensordata, P.sd_touch_l, critic_obs, 66, ld, n0);
    // feet_position: [fp[3:6], fp[0:3]] * (1,-1,1,1,-1,1)
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      float v[4];
      kbs_ld4(computed, 63 + (k < 3 ? k + 3 : k - 3), ld, n0, v);
      if (k % 3 == 1) {
#pragma unroll
        for (int l = 0; l < 4; ++l) v[l] = -v[l];
      }
      kbs_st4(critic_obs, 67 + k, ld, n0, v);
    }
    for (int k = 0; k < 3; ++k) kbs_copy4(s.qpos, k, critic_obs, 73 + k, ld, n0);      // base_position unchanged
    for (int k = 0; k < 4; ++k) {                                                       // base_orientation * (1,-1,-1,1)
      float v[4];
      kbs_ld4(s.qpos, 3 + k, ld, n0, v);
      if (k == 1 || k == 2) {
#pragma unroll
        for (int l = 0; l < 4; ++l) v[l] = -v[l];
      }
      kbs_st4(critic_obs, 76 + k, ld, n0, v);
    }
    for (int k = 0; k < 6; ++k) {                 // base lin vel * (1,-1,1), ang vel * (-1,1,-1)
      float v[4];
      kbs_ld4(s.qvel, k, ld, n0, v);
      if (k == 1 || k == 3 || k == 5) {
#pragma unroll
        for (int l = 0; l < 4; ++l) v[l] = -v[l];
      }
      kbs_st4(critic_obs, 448 + k, ld, n0, v);
    }
#pragma unroll 4
    for (int j = 0; j < KBS_NUM_JOINTS; ++j) {
      float f[4];
      kbs_ld4(s.actuator_force, mirror_src_joint(j), ld, n0, f);
#pragma unroll
      for (int l = 0; l < 4; ++l) f[l] = -f[l] / 4.0f;
      kbs_st4(critic_obs, 454 + j, ld, n0, f);
    }
    kbs_copy4(s.xpos, 3 * P.body_base + 2, critic_obs, 474, ld, n0);
  }
}

// mirror_joints on a [T][20][ld] array (e.g. dist.mean() of the mirrored pass, train.py:1468)
__global__ void __launch_bounds__(kThreads)
mirror_joints_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t ld, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  const int64_t t = blockIdx.z;
  const int j = blockIdx.y;
  float v[4];
  kbs_ld4(in + t * KBS_NUM_JOINTS * ld, mirror_src_joint(j), ld, n0, v);
#pragma unroll
  for (int l = 0; l < 4; ++l) v[l] = -v[l];
  kbs_st4(out + t * KBS_NUM_JOINTS * ld, j, ld, n0, v);
}

// aux_losses of PPOVariables (train.py:1462-1481): action_mirror_loss = mean_j (mean - mirror_joints(mean_m))^2 * scale_a,
// value_mirror_loss = (value - value_m)^2 * scale_c (the mean over the value's single element).  [T][.][ld] arrays;
// grid = (env groups, T).
__global__ void __launch_bounds__(kThreads)
mirror_loss_kernel(const float* __restrict__ mean, const float* __restrict__ mean_m, const float* __restrict__ value,
                   const float* __restrict__ value_m, float* __restrict__ action_loss, float* __restrict__ value_loss,
                   float scale_a, float scale_c, int64_t ld, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  const int64_t t = blockIdx.y;
  if (action_loss) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int j = 0; j < KBS_NUM_JOINTS; ++j) {
      float a[4], b[4];
      kbs_ld4(mean + t * KBS_NUM_JOINTS * ld, j, ld, n0, a);
      kbs_ld4(mean_m + t * KBS_NUM_JOINTS * ld, mirror_src_joint(j), ld, n0, b);
#pragma unroll
      for (int l = 0; l < 4; ++l) { const float d = a[l] - (-b[l]); acc[l] = acc[l] + d * d; }
    }
#pragma unroll
    for (int l = 0; l < 4; ++l) acc[l] = (acc[l] / float(KBS_NUM_JOINTS)) * scale_a;
    kbs_st4(action_loss, t, ld, n0, acc);
  }
  if (value_loss) {
    float v[4], vm[4], o[4];
    kbs_ld4(value, t, ld, n0, v);
    kbs_ld4(value_m, t, ld, n0, vm);
#pragma unroll
    for (int l = 0; l < 4; ++l) { const float d = v[l] - vm[l]; o[l] = (d * d) * scale_c; }
    kbs_st4(value_loss, t, ld, n0, o);
  }
}

// Per-episode actuator randomisation of ksim.PositionActuators (train.py:1097-1105; sampling law [U], see kbotstep.h):
// u [5][20][ld] uniforms for (kp, kd, tau_limit, action_bias, torque_bias); grid = (env groups, 20 joints).
__global__ void __launch_bounds__(kThreads)
actuator_rand_kernel(const __grid_constant__ kbs_params P, const kbs_actuator_rand_params R, const float* __restrict__ u,
                     const uint8_t* __restrict__ reset, const kbs_episode_view ep, int64_t ld, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  const int j = blockIdx.y;
  bool rs[4] = {true, true, true, true};
  if (reset) {
    const uchar4 r4 = *reinterpret_cast<const uchar4*>(reset + n0);
    rs[0] = r4.x != 0; rs[1] = r4.y != 0; rs[2] = r4.z != 0; rs[3] = r4.w != 0;
  }
  auto put = [&](float* dst, int which, float lo, float hi, float nominal) {
    if (!dst) return;
    float uu[4], o[4];
    kbs_ld4(u + int64_t(which) * KBS_NUM_JOINTS * ld, j, ld, n0, uu);
    if (reset) kbs_ld4(dst, j, ld, n0, o);
#pragma unroll
    for (int l = 0; l < 4; ++l)
      if (rs[l]) o[l] = nominal * (lo + uu[l] * (hi - lo));
    kbs_st4(dst, j, ld, n0, o);
  };
  put(const_cast<float*>(ep.kp), 0, 1.0f / R.kp_scale, R.kp_scale, P.kp[j]);
  put(const_cast<float*>(ep.kd), 1, 1.0f / R.kd_scale, R.kd_scale, P.kd[j]);
  put(const_cast<float*>(ep.tau_limit), 2, R.torque_limit_scale_low, 1.0f, P.ctrl_limit[j]);
  put(const_cast<float*>(ep.action_bias), 3, -R.action_bias_scale, R.action_bias_scale, 1.0f);
  put(const_cast<float*>(ep.torque_bias), 4, -R.torque_bias_scale, R.torque_bias_scale, 1.0f);
}

// =====================================================================================================
// Device-side randomness of a rollout (kbs_generate_rollout_noise): counter-based Philox4x32-10 (kbs_philox4x32_10).
// counter = (step lo, step hi, env group, row), key = seed: 4 x 32 bits per call = the 4 consecutive envs of a float4.
// =====================================================================================================
struct NoiseRows {
  float* base[9];        // eps_jpos, eps_jvel, eps_gyro, eps_pg, eps_action, u_switch, cmd_mode (as int32), cmd_u6, cmd_u_arms
  int rows[9];           // rows per step of each array
  int kind[9];           // 0 U(-1,1), 1 N(0,1), 2 U[0,1), 3 int 0..5
  int first[10];         // prefix sums: global row index of each array's row 0
};
__global__ void __launch_bounds__(kThreads)
rollout_noise_kernel(const __grid_constant__ NoiseRows R, uint64_t seed, int64_t step0, int64_t ld, int64_t n) {
  const int64_t grp = int64_t(blockIdx.x) * kThreads + threadIdx.x;
  const int64_t n0 = grp * 4;
  if (n0 >= n) return;
  const int gr = blockIdx.y;                       // global row
  int a = 0;
#pragma unroll
  for (int i = 1; i < 9; ++i) a += (gr >= R.first[i]) ? 1 : 0;
  if (!R.base[a]) return;
  const int row = gr - R.first[a];
  const int64_t t = blockIdx.z;
  const uint64_t step = uint64_t(step0 + t);
  const uint4 x = kbs_philox4x32_10(make_uint4(uint32_t(step), uint32_t(step >> 32), uint32_t(grp), uint32_t(gr)),
                                    make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
  const uint32_t w[4] = {x.x, x.y, x.z, x.w};
  float v[4];
  const int kind = R.kind[a];
  if (kind == 1) {
    // Box-Muller on (w0, w1) and (w2, w3): u1 in (0, 1], u2 in [0, 1)
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      const float u1 = (float(w[2 * p] >> 8) + 1.0f) * (1.0f / 16777216.0f);
      const float u2 = float(w[2 * p + 1] >> 8) * (1.0f / 16777216.0f);
      const float rr = sqrtf(-2.0f * logf(u1));
      float sn, cs;
      sincospif(2.0f * u2, &sn, &cs);
      v[2 * p] = rr * cs; v[2 * p + 1] = rr * sn;
    }
  } else {
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const float u = float(w[l] >> 8) * (1.0f / 16777216.0f);      // [0, 1)
      v[l] = kind == 0 ? 2.0f * u - 1.0f : u;
    }
  }
  float* dst = R.base[a] + (t * R.rows[a] + row) * ld + n0;
  if (kind == 3) {
    int4 m;
    m.x = min(int(v[0] * 6.0f), 5); m.y = min(int(v[1] * 6.0f), 5); m.z = min(int(v[2] * 6.0f), 5); m.w = min(int(v[3] * 6.0f), 5);
    *reinterpret_cast<int4*>(dst) = m;
  } else {
    *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// =====================================================================================================
// O12: COMDistanceObservation (train.py:509-659): >= 3 distinct contact.geom2 values -> distance between the centroid of the
// convex hull of the floor-contact points (xy; non-floor rows become the origin and stay in the set, as written) and
// subtree_com[2].xy, else -1.  Andrew's monotone chain exactly as the reference runs it (lexicographic stable sort, pop
// while cross <= 0, lower chain on the sorted order, upper chain on the reversed order, last vertex of each dropped),
// then the shoelace centroid with the mean-of-vertices fallback for |area| < 1e-12.  One thread per (env, step): the
// data-dependent loops XLA runs as while_loop inside scan live in registers / local memory here.
// grid = (env blocks, T)
// =====================================================================================================
constexpr int kMaxContacts = 32;

__global__ void __launch_bounds__(kThreads)
com_distance_kernel(const int32_t* __restrict__ geom1, const int32_t* __restrict__ geom2, const float* __restrict__ pos,
                    const float* __restrict__ com, float* __restrict__ out, int ncon, int64_t ld, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * kThreads + threadIdx.x;
  if (e >= n) return;
  const int64_t t = blockIdx.y;
  geom1 += t * ncon * ld + e; geom2 += t * ncon * ld + e; pos += t * 3 * ncon * ld + e; com += t * 3 * ld + e;
  // num_unique(contact.geom2): sort + count the changes (padding entries count like any other value: as written)
  int g[kMaxContacts];
  for (int i = 0; i < ncon; ++i) {
    const int v = geom2[i * ld];
    int j = i - 1;
    while (j >= 0 && g[j] > v) { g[j + 1] = g[j]; --j; }
    g[j + 1] = v;
  }
  int unique = ncon > 0 ? 1 : 0;
  for (int i = 1; i < ncon; ++i) unique += (g[i] != g[i - 1]) ? 1 : 0;
  if (unique < 3) { out[t * ld + e] = -1.0f; return; }
  // points, lexicographically sorted by (x, y), stable (jnp.lexsort)
  float sx[kMaxContacts], sy[kMaxContacts];
  for (int i = 0; i < ncon; ++i) {
    const bool floor = geom1[i * ld] == 0;
    const float x = floor ? pos[(3 * i) * ld] : 0.0f, y = floor ? pos[(3 * i + 1) * ld] : 0.0f;
    int j = i - 1;
    while (j >= 0 && (sx[j] > x || (sx[j] == x && sy[j] > y))) { sx[j + 1] = sx[j]; sy[j + 1] = sy[j]; --j; }
    sx[j + 1] = x; sy[j + 1] = y;
  }
  // the two chains (indices into the sorted points)
  int chain[2][kMaxContacts];
  int len[2];
  for (int c = 0; c < 2; ++c) {
    int ptr = 0;
    for (int k = 0; k < ncon; ++k) {
      const int idx = c == 0 ? k : ncon - 1 - k;
      while (ptr >= 2) {
        const int a = chain[c][ptr - 2], b = chain[c][ptr - 1];
        const float cr = (sx[b] - sx[a]) * (sy[idx] - sy[a]) - (sy[b] - sy[a]) * (sx[idx] - sx[a]);
        if (!(cr <= 0.0f)) break;
        --ptr;
      }
      chain[c][ptr++] = idx;
    }
    len[c] = ptr - 1 > 0 ? ptr - 1 : 0;          // Andrew: drop the last vertex of each chain
  }
  const int count = len[0] + len[1];
  // polygon_centroid_masked on the packed hull [lower | upper]
  float s_cross = 0.0f, s_cx = 0.0f, s_cy = 0.0f, s_mx = 0.0f, s_my = 0.0f;
  for (int i = 0; i < count; ++i) {
    const int i1 = (i + 1 < count) ? i + 1 : 0;
    const int v0 = i < len[0] ? chain[0][i] : chain[1][i - len[0]];
    const int v1 = i1 < len[0] ? chain[0][i1] : chain[1][i1 - len[0]];
    const float x = sx[v0], y = sy[v0], x1 = sx[v1], y1 = sy[v1];
    const float cr = x * y1 - x1 * y;
    s_cross = s_cross + cr;
    s_cx = s_cx + (x + x1) * cr;
    s_cy = s_cy + (y + y1) * cr;
    s_mx = s_mx + x;
    s_my = s_my + y;
  }
  const float area = 0.5f * s_cross;
  const float cnt = count > 0 ? float(count) : 1.0f;
  float cx, cy;
  if (fabsf(area) < 1e-12f) { cx = s_mx / cnt; cy = s_my / cnt; }
  else { cx = s_cx / (6.0f * area); cy = s_cy / (6.0f * area); }
  const float dx = cx - com[0], dy = cy - com[ld];
  out[t * ld + e] = sqrtf(dx * dx + dy * dy);
}

// =====================================================================================================
// PPO loss (ksim.compute_ppo_loss [U], entropy_coef train.py:1767): clipped surrogate + (clipped) value loss + entropy
// bonus, reduced to four means.  Deterministic: fixed per-thread strides, warp-shuffle + shared-memory tree per block,
// and the last block to finish (ticket counter) adds the per-block partials in block order.
// =====================================================================================================
constexpr int kLossThreads = 256;

__global__ void __launch_bounds__(kLossThreads)
ppo_loss_kernel(kbs_ppo_loss_params L, kbs_ppo_loss_io io, int64_t n, double* __restrict__ partials,
                unsigned int* __restrict__ ticket) {
  const int64_t ld = io.ld, total = io.T * ld;
  float s[4] = {0.f, 0.f, 0.f, 0.f};                 // objective, policy, value, entropy
  for (int64_t i = int64_t(blockIdx.x) * kLossThreads + threadIdx.x; i < total; i += int64_t(gridDim.x) * kLossThreads) {
    const int64_t e = i % ld;
    if (e >= n) continue;
    const float lp = io.log_probs[i], lpo = io.old_log_probs[i], adv = io.advantages[i], v = io.values[i];
    const float tgt = io.value_targets[i], ent = io.entropy[i];
    const float lr = fminf(fmaxf(lp - lpo, -L.log_clip_value), L.log_clip_value);
    const float ratio = expf(lr);
    const float pol = fminf(ratio * adv, fminf(fmaxf(ratio, 1.0f - L.clip_param), 1.0f + L.clip_param) * adv);
    const float err = tgt - v;
    float val = 0.5f * (err * err);
    if (L.use_clipped_value_loss) {
      const float vo = io.old_values[i];
      const float vc = vo + fminf(fmaxf(v - vo, -L.clip_param), L.clip_param);
      const float errc = tgt - vc;
      val = 0.5f * fmaxf(err * err, errc * errc);
    }
    const float obj = (pol - L.value_loss_coef * val) + L.entropy_coef * ent;
    if (io.per_step) io.per_step[i] = obj;
    s[0] += obj; s[1] += pol; s[2] += val; s[3] += ent;
  }
  __shared__ double red[kLossThreads / 32][4];
  __shared__ bool last;
  double d[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    d[k] = double(s[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d[k] += __shfl_down_sync(0xffffffffu, d[k], o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { for (int k = 0; k < 4; ++k) red[warp][k] = d[k]; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 0; k < 4; ++k) {
      double a = 0.0;
      for (int w = 0; w < kLossThreads / 32; ++w) a += red[w][k];
      partials[size_t(blockIdx.x) * 4 + k] = a;
    }
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last && threadIdx.x < 4) {
    __threadfence();
    double a = 0.0;
    for (unsigned b = 0; b < gridDim.x; ++b) a += partials[size_t(b) * 4 + threadIdx.x];   // block order: deterministic
    const double mean = a / (double(io.T) * double(n));
    io.out[threadIdx.x] = float(threadIdx.x == 0 ? -mean : mean);
    if (threadIdx.x == 0) *ticket = 0u;              // re-arm for the next call on this stream
  }
}

// =====================================================================================================
// UnifiedCommand train.py:724-785
// =====================================================================================================
__global__ void __launch_bounds__(kThreads)
command_kernel(const __grid_constant__ kbs_params P, const float* __restrict__ cmd_in, float* __restrict__ cmd_out,
               const float* __restrict__ u_switch, const int32_t* __restrict__ mode, const float* __restrict__ u6,
               const float* __restrict__ u_arms, const uint8_t* __restrict__ done, int64_t ld, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  float us[4] = {-1.f, -1.f, -1.f, -1.f};  // NULL u_switch: always resample (initial_command)
  if (u_switch) kbs_ld4(u_switch, 0, ld, n0, us);
  if (done) {  // episode ended: ksim draws initial_command for the new episode (SURVEY 3.2)
    const uchar4 d4 = *reinterpret_cast<const uchar4*>(done + n0);
    if (d4.x) us[0] = -1.f;
    if (d4.y) us[1] = -1.f;
    if (d4.z) us[2] = -1.f;
    if (d4.w) us[3] = -1.f;
  }
  const int4 m4 = *reinterpret_cast<const int4*>(mode + n0);
  const int md[4] = {m4.x, m4.y, m4.z, m4.w};
  float v[6][4];
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    float u[4];
    kbs_ld4(u6, k, ld, n0, u);
#pragma unroll
    for (int l = 0; l < 4; ++l) v[k][l] = P.cmd_lo[k] + u[l] * (P.cmd_hi[k] - P.cmd_lo[k]);
  }
  // slots 0..5
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    float prev[4], o[4];
    kbs_ld4(cmd_in, k, ld, n0, prev);
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const int m = md[l];
      bool on;
      if (k == 0) on = (m == 0) || (m == 3);
      else if (k == 1) on = (m == 1) || (m == 3);
      else if (k == 2) on = (m == 2) || (m == 3);
      else on = (m == 4);
      const float nw = on ? v[k][l] : 0.0f;
      o[l] = (us[l] < P.switch_prob) ? nw : prev[l];
    }
    kbs_st4(cmd_out, k, ld, n0, o);
  }
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    float u[4], prev[4], o[4];
    kbs_ld4(u_arms, k, ld, n0, u);
    kbs_ld4(cmd_in, 6 + k, ld, n0, prev);
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      // train.py:734-738: uniform() and bernoulli() share key rng_h => mask = (u < 0.5) on the same draw
      const float arm = (P.arm_lo[k] + u[l] * (P.arm_hi[k] - P.arm_lo[k])) * ((u[l] < 0.5f) ? 1.0f : 0.0f);
      const float nw = (md[l] == 3 || md[l] == 4) ? arm : 0.0f;
      o[l] = (us[l] < P.switch_prob) ? nw : prev[l];
    }
    kbs_st4(cmd_out, 6 + k, ld, n0, o);
  }
}

// =====================================================================================================
// PositionActuators.get_ctrl (ksim fork) train.py:1091-1105
// =====================================================================================================
__global__ void __launch_bounds__(kThreads)
torque_kernel(const __grid_constant__ kbs_params P, const float* __restrict__ action, const kbs_state_view s,
              const kbs_episode_view ep, float* __restrict__ ctrl, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  const int64_t ld = s.ld;
#pragma unroll 5
  for (int j = 0; j < KBS_NUM_JOINTS; ++j) {
    float a[4], q[4], qd[4], o[4];
    float kp[4] = {P.kp[j], P.kp[j], P.kp[j], P.kp[j]}, kd[4] = {P.kd[j], P.kd[j], P.kd[j], P.kd[j]};
    float lim[4] = {P.ctrl_limit[j], P.ctrl_limit[j], P.ctrl_limit[j], P.ctrl_limit[j]};
    float ab[4] = {0, 0, 0, 0}, tb[4] = {0, 0, 0, 0};
    kbs_ld4(action, j, ld, n0, a);
    kbs_ld4(s.qpos, 7 + j, ld, n0, q);
    kbs_ld4(s.qvel, 6 + j, ld, n0, qd);
    if (ep.kp) kbs_ld4(ep.kp, j, ld, n0, kp);
    if (ep.kd) kbs_ld4(ep.kd, j, ld, n0, kd);
    if (ep.tau_limit) kbs_ld4(ep.tau_limit, j, ld, n0, lim);
    if (ep.action_bias) kbs_ld4(ep.action_bias, j, ld, n0, ab);
    if (ep.torque_bias) kbs_ld4(ep.torque_bias, j, ld, n0, tb);
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const float target = ep.action_bias ? a[l] + ab[l] : a[l];
      float tau = kp[l] * (target - q[l]) - kd[l] * qd[l];
      if (ep.torque_bias) tau = tau + tb[l];
      o[l] = fminf(fmaxf(tau, -lim[l]), lim[l]);
    }
    kbs_st4(ctrl, j, ld, n0, o);
  }
}

// Per-physics-sub-step actuator path (SURVEY 8f-2; train.py:1775-1781: dt 0.004, ctrl_dt 0.02, action latency 3-10 ms,
// 5 % dropped commands; ksim engine semantics [U], see oracle position_actuator_substeps): a dropped command repeats
// the last applied action; sub-step k sees the new action once k sub_dt >= latency; PD torque on the sub-step's joint state.
// Two kernels evaluate it: all S sub-steps of recorded joint states in one launch (torque_substeps_kernel), or one sub-step
// per launch with the simulator in the loop (actuator_substep_kernel).  Both take the gains and the per-element rule from
// the two functions below, so they cannot drift apart.

// joint j's gains, limit and biases for 4 envs (nominal / zero where the episode view has no array)
struct Gains4 { float kp[4], kd[4], lim[4], ab[4], tb[4]; };
__device__ __forceinline__ void substep_gains4(const kbs_params& P, const kbs_episode_view& ep, int j, int64_t ld, int64_t n0,
                                               Gains4& g) {
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    g.kp[l] = P.kp[j]; g.kd[l] = P.kd[j]; g.lim[l] = P.ctrl_limit[j]; g.ab[l] = 0.f; g.tb[l] = 0.f;
  }
  if (ep.kp) kbs_ld4(ep.kp, j, ld, n0, g.kp);
  if (ep.kd) kbs_ld4(ep.kd, j, ld, n0, g.kd);
  if (ep.tau_limit) kbs_ld4(ep.tau_limit, j, ld, n0, g.lim);
  if (ep.action_bias) kbs_ld4(ep.action_bias, j, ld, n0, g.ab);
  if (ep.torque_bias) kbs_ld4(ep.torque_bias, j, ld, n0, g.tb);
}

// env l of 4 at sub-step time tk = k sub_dt: the latency select, PositionActuators.get_ctrl, the clamp
__device__ __forceinline__ float substep_torque(float applied, float prev, float tk, float lat, float q, float qd, const Gains4& g,
                                                int l, bool has_ab, bool has_tb) {
  const float act = (tk >= lat) ? applied : prev;
  const float target = has_ab ? act + g.ab[l] : act;
  float tau = g.kp[l] * (target - q) - g.kd[l] * qd;
  if (has_tb) tau = tau + g.tb[l];
  return fminf(fmaxf(tau, -g.lim[l]), g.lim[l]);
}

//   q_sub / qd_sub / ctrl [S][20][ld]; prev_action [20][ld] in/out
__global__ void __launch_bounds__(kThreads)
torque_substeps_kernel(const __grid_constant__ kbs_params P, const float* __restrict__ action, float* __restrict__ prev_action,
                       const float* __restrict__ u_drop, const float* __restrict__ latency, const float* __restrict__ q_sub,
                       const float* __restrict__ qd_sub, const kbs_episode_view ep, float* __restrict__ ctrl, int S, float sub_dt,
                       float drop_prob, int64_t ld, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  float ud[4], lat[4];
  kbs_ld4(u_drop, 0, ld, n0, ud);
  kbs_ld4(latency, 0, ld, n0, lat);
  const bool has_ab = ep.action_bias != nullptr, has_tb = ep.torque_bias != nullptr;
#pragma unroll 2
  for (int j = 0; j < KBS_NUM_JOINTS; ++j) {
    float a[4], pa[4], ap[4];
    Gains4 g;
    kbs_ld4(action, j, ld, n0, a);
    kbs_ld4(prev_action, j, ld, n0, pa);
    substep_gains4(P, ep, j, ld, n0, g);
#pragma unroll
    for (int l = 0; l < 4; ++l) ap[l] = (ud[l] < drop_prob) ? pa[l] : a[l];
    for (int k = 0; k < S; ++k) {
      float q[4], qd[4], o[4];
      kbs_ld4(q_sub + int64_t(k) * KBS_NUM_JOINTS * ld, j, ld, n0, q);
      kbs_ld4(qd_sub + int64_t(k) * KBS_NUM_JOINTS * ld, j, ld, n0, qd);
      const float tk = float(k) * sub_dt;
#pragma unroll
      for (int l = 0; l < 4; ++l) o[l] = substep_torque(ap[l], pa[l], tk, lat[l], q[l], qd[l], g, l, has_ab, has_tb);
      kbs_st4(ctrl + int64_t(k) * KBS_NUM_JOINTS * ld, j, ld, n0, o);
    }
    kbs_st4(prev_action, j, ld, n0, ap);
  }
}

// One sub-step of the online rollout (kbs_actuator_substep): t (the step state's index, the control step that just ran is
// t-1) and k (the actuator state's sub-step index) are read once per block.  At k = 0 the step's action is latched into
// `applied` (or prev_action where the command is dropped); ctrl = PD on this sub-step's qpos rows 7.. / qvel rows 6..; at
// k = S-1 prev_action = applied.  grid = (env groups, joint): one sub-step of a few thousand envs is ~3 MB, so one joint per
// block row gives the SMs 20x the blocks a whole-env thread would.  The last block to finish advances k (ticket, as
// step_record_kernel), so one captured launch serves every sub-step.  Out of range (t = 0, t > T, k >= S): nothing is
// written, k stays, KBS_STATUS_SUBSTEP_RANGE is set.
__global__ void __launch_bounds__(kThreads)
actuator_substep_kernel(const __grid_constant__ kbs_params P, const __grid_constant__ KbsSubstepArgs a) {
  __shared__ int64_t t_s;
  __shared__ int k_s;
  if (threadIdx.x == 0) {
    t_s = *reinterpret_cast<const volatile int64_t*>(a.t);
    k_s = *reinterpret_cast<volatile int32_t*>(a.k);
  }
  __syncthreads();
  const int64_t t = t_s;
  const int k = k_s;
  const bool in_range = t >= 1 && t <= a.T && k >= 0 && k < a.S;
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  const int j = blockIdx.y;
  if (in_range && n0 < a.n) {
    const int64_t ld = a.ld;
    const bool has_ab = a.ep.action_bias != nullptr, has_tb = a.ep.torque_bias != nullptr;
    const float tk = float(k) * a.sub_dt;
    float lat[4], pa[4], ap[4], q[4], qd[4], o[4];
    Gains4 g;
    kbs_ld4(a.latency, 0, ld, n0, lat);
    kbs_ld4(a.prev_action, j, ld, n0, pa);
    if (k == 0) {
      float ud[4], x[4];
      kbs_ld4(a.u_drop, 0, ld, n0, ud);
      kbs_ld4(a.action + (t - 1) * KBS_NUM_JOINTS * ld, j, ld, n0, x);
#pragma unroll
      for (int l = 0; l < 4; ++l) ap[l] = (ud[l] < a.drop_prob) ? pa[l] : x[l];
      kbs_st4(a.applied, j, ld, n0, ap);
    } else {
      kbs_ld4(a.applied, j, ld, n0, ap);
    }
    kbs_ld4(a.qpos, 7 + j, ld, n0, q);
    kbs_ld4(a.qvel, 6 + j, ld, n0, qd);
    substep_gains4(P, a.ep, j, ld, n0, g);
#pragma unroll
    for (int l = 0; l < 4; ++l) o[l] = substep_torque(ap[l], pa[l], tk, lat[l], q[l], qd[l], g, l, has_ab, has_tb);
    kbs_st4(a.ctrl, j, ld, n0, o);
    if (k == a.S - 1) kbs_st4(a.prev_action, j, ld, n0, ap);
  } else if (!in_range && blockIdx.x == 0 && j == 0 && threadIdx.x == 0) {
    atomicOr(a.status, unsigned(KBS_STATUS_SUBSTEP_RANGE));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(a.ticket, 1u) == gridDim.x * gridDim.y - 1) {      // every block has read k
      *a.ticket = 0u;
      if (in_range) *a.k = (k + 1 == a.S) ? 0 : k + 1;
      __threadfence();
    }
  }
}

// =====================================================================================================
// Terminations train.py:1258-1269, 817-823 (+ ksim NotUpright / EpisodeLength / done-success reduce)
// =====================================================================================================
__global__ void __launch_bounds__(kThreads)
terminate_kernel(const __grid_constant__ kbs_params P, kbs_state_view s, int32_t* __restrict__ codes,
                 uint8_t* __restrict__ done, uint8_t* __restrict__ success, float* __restrict__ pre, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  const int64_t ld = s.ld;
  {
    const int64_t t = blockIdx.y;
    s.xpos += t * 3 * KBS_NBODY * ld; s.qpos += t * KBS_NQ * ld; s.time += t * ld;
    if (codes) codes += t * 3 * ld;
    if (done) done += t * ld;
    if (success) success += t * ld;
    if (pre) pre += t * 2 * ld;
  }
  float bz[4], lz[4], rz[4], q[4][4], tm[4];
  kbs_ld4(s.xpos, 3 * P.body_base + 2, ld, n0, bz);
  kbs_ld4(s.xpos, 3 * P.body_lfoot + 2, ld, n0, lz);
  kbs_ld4(s.xpos, 3 * P.body_rfoot + 2, ld, n0, rz);
#pragma unroll
  for (int k = 0; k < 4; ++k) kbs_ld4(s.qpos, 3 + k, ld, n0, q[k]);
  kbs_ld4(s.time, 0, ld, n0, tm);
  int c0[4], c1[4], c2[4];
  float hgt[4], tilt[4];
  uchar4 d, sc;
  unsigned char* dp = reinterpret_cast<unsigned char*>(&d);
  unsigned char* sp = reinterpret_cast<unsigned char*>(&sc);
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    hgt[l] = bz[l] - fminf(lz[l], rz[l]);
    c0[l] = (hgt[l] < P.unhealthy_z) ? -1 : 0;
    float qq[4] = {q[0][l], q[1][l], q[2][l], q[3][l]};
    quat_norm_eps(qq, P.eps_quat);
    const float cz = 1.0f - 2.0f * (qq[1] * qq[1] + qq[2] * qq[2]);
    tilt[l] = acosf(fminf(fmaxf(cz, -1.0f), 1.0f));
    c1[l] = (tilt[l] > P.max_tilt) ? -1 : 0;
    c2[l] = (tm[l] > P.max_length_sec) ? 1 : 0;
    const bool dn = (c0[l] != 0) || (c1[l] != 0) || (c2[l] != 0);
    dp[l] = dn ? 1 : 0;
    sp[l] = (dn && c0[l] != -1 && c1[l] != -1 && c2[l] != -1) ? 1 : 0;
  }
  if (codes) {
    *reinterpret_cast<int4*>(codes + 0 * ld + n0) = make_int4(c0[0], c0[1], c0[2], c0[3]);
    *reinterpret_cast<int4*>(codes + 1 * ld + n0) = make_int4(c1[0], c1[1], c1[2], c1[3]);
    *reinterpret_cast<int4*>(codes + 2 * ld + n0) = make_int4(c2[0], c2[1], c2[2], c2[3]);
  }
  if (done) *reinterpret_cast<uchar4*>(done + n0) = d;
  if (success) *reinterpret_cast<uchar4*>(success + n0) = sc;
  if (pre) { kbs_st4(pre, 0, ld, n0, hgt); kbs_st4(pre, 1, ld, n0, tilt); }
}

// =====================================================================================================
// Rewards train.py:125-506, table 1224-1256.
//   reward_rot_kernel   : per env, sqrt(sum_t wz_t^2) > 1e-3  (train.py:455 reduces over TIME as written)
//   reward_terms_kernel : the 10 stateless terms, fully parallel over (t, env); emits contact/zero flags
//   reward_scan_kernel  : the 2 stateful scans (single_contact, feet_airtime) over T per env + final sum
// =====================================================================================================
__global__ void __launch_bounds__(kThreads)
reward_rot_kernel(const float* __restrict__ command, uint8_t* __restrict__ is_rot, int64_t T, int64_t ld, int64_t n) {
  const int64_t n0 = (int64_t(blockIdx.x) * kThreads + threadIdx.x) * 4;
  if (n0 >= n) return;
  float acc[4] = {0, 0, 0, 0};
  constexpr int kB = 16;   // 16 independent row loads in flight, summed in time order (the reference's reduction order)
  for (int64_t t0 = 0; t0 < T; t0 += kB) {
    float wz[kB][4];
#pragma unroll
    for (int i = 0; i < kB; ++i) kbs_ld4(command + (t0 + i < T ? t0 + i : T - 1) * KBS_NUM_COMMANDS * ld, 2, ld, n0, wz[i]);
#pragma unroll
    for (int i = 0; i < kB; ++i) {
      if (t0 + i < T) {
#pragma unroll
        for (int l = 0; l < 4; ++l) acc[l] = acc[l] + wz[i][l] * wz[i][l];
      }
    }
  }
  uchar4 o;
  o.x = sqrtf(acc[0]) > 1e-3f; o.y = sqrtf(acc[1]) > 1e-3f; o.z = sqrtf(acc[2]) > 1e-3f; o.w = sqrtf(acc[3]) > 1e-3f;
  *reinterpret_cast<uchar4*>(is_rot + n0) = o;
}

__device__ __forceinline__ float quat_dot(const float (&a)[4], const float (&b)[4]) {
  return ((a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]) + a[3] * b[3];
}

// One env-step per thread: the ~10 quaternion <-> euler conversions per env-step (IEEE atan2f / asinf / sincosf, no
// fast-math) make this kernel issue-bound, so it wants every warp slot of the SM filled (4 envs per thread left 21 warps
// per SM resident and 217 us per 4 096 x 100 launch; rows are still read as full 128-byte lines per warp).
__device__ __forceinline__ float ld1(const float* __restrict__ base, int64_t row, int64_t ld, int64_t e) {
  return __ldcs(base + row * ld + e);
}

__global__ void __launch_bounds__(kThreads, 6)
reward_terms_kernel(const __grid_constant__ kbs_params P, const kbs_traj_view tr, const uint8_t* __restrict__ is_rot,
                    float* __restrict__ total, float* __restrict__ comp, uint8_t* __restrict__ flags, int64_t n) {
  const int64_t e0 = int64_t(blockIdx.x) * kThreads + threadIdx.x;
  if (e0 >= n) return;
  const int64_t t = blockIdx.y;
  const int64_t ld = tr.state.ld;
  const float* xquat = tr.state.xquat + t * 4 * KBS_NBODY * ld;
  const float* xpos = tr.state.xpos + t * 3 * KBS_NBODY * ld;
  const float* qpos = tr.state.qpos + t * KBS_NQ * ld;
  const float* qvel = tr.state.qvel + t * KBS_NV * ld;
  const float* sd = tr.state.sensordata + t * KBS_NSENSORDATA * ld;
  const float* cmdp = tr.command + t * KBS_NUM_COMMANDS * ld;
  const float* ctrl = tr.ctrl + t * KBS_NUM_JOINTS * ld;

  // every load of the thread is issued before the first trig call: ~70 independent 4-byte loads in flight
  float c[16], bq[4], fq[2][4], v[6], pv[6], u[KBS_NUM_JOINTS], qa[10];
#pragma unroll
  for (int k = 0; k < 16; ++k) c[k] = ld1(cmdp, k, ld, e0);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    bq[k] = ld1(xquat, 4 * P.body_base + k, ld, e0);
    fq[0][k] = ld1(xquat, 4 * P.body_lfoot + k, ld, e0);
    fq[1][k] = ld1(xquat, 4 * P.body_rfoot + k, ld, e0);
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) v[k] = ld1(qvel, k, ld, e0);
  const float bz = ld1(xpos, 3 * P.body_base + 2, ld, e0);
  const float lz = ld1(xpos, 3 * P.body_lfoot + 2, ld, e0);
  const float rz = ld1(xpos, 3 * P.body_rfoot + 2, ld, e0);
  const float tl = ld1(sd, P.sd_touch_l, ld, e0);
  const float trr = ld1(sd, P.sd_touch_r, ld, e0);
  const float cd = __ldcs(tr.state.com_distance + t * ld + e0);
  const bool rot = is_rot[e0] != 0;
  bool prev_done = true;  // t = 0: edge pad, zero difference (train.py:487-494)
  if (t > 0) {
    prev_done = tr.done[(t - 1) * ld + e0] != 0;
#pragma unroll
    for (int k = 0; k < 6; ++k) pv[k] = ld1(qvel - KBS_NV * ld, k, ld, e0);
  } else {
#pragma unroll
    for (int k = 0; k < 6; ++k) pv[k] = 0.0f;
  }
#pragma unroll
  for (int j = 0; j < KBS_NUM_JOINTS; ++j) u[j] = ld1(ctrl, j, ld, e0);
#pragma unroll
  for (int k = 0; k < 10; ++k) qa[k] = ld1(qpos, 17 + k, ld, e0);

  float r[KBS_NUM_REWARDS];
  const bool zc = zero_cmd(c[0], c[1], c[2]);
  // the sums over joints first: their 36 loaded values die before the trig-heavy terms need registers
  // R5 arm_pos train.py:261-265
  {
    float err = 0.0f;
#pragma unroll
    for (int k = 0; k < 10; ++k) {
      const float d = qa[k] - (c[6 + k] + P.joint_bias[10 + k]);
      err = err + d * d;
    }
    r[4] = expf(-err / P.arm_es);
  }
  // R11 base_accel train.py:487-494
  {
    float err = 0.0f;
#pragma unroll
    for (int k = 0; k < 6; ++k) err = err + fabsf(prev_done ? 0.0f : (v[k] - pv[k]));
    r[10] = expf(-err / P.acc_es);
  }
  // R12 torque train.py:503-506
  {
    float acc = 0.0f;
#pragma unroll
    for (int j = 0; j < KBS_NUM_JOINTS; ++j) acc = acc + expf(-fabsf(u[j]) / P.torque_es);
    r[11] = zc ? acc / 20.0f : 1.0f;
  }

  float e[3];
  quat_to_euler(bq, P.eps_quat, e);
  // R1 linvel train.py:274-292
  {
    float qz[4], g[3];
    euler_to_quat(0.0f, 0.0f, e[2], qz);
    const float vc[3] = {c[0], c[1], 0.0f};
    rotate_vec(vc, qz, false, P.eps_quat, g);
    const float dx = v[0] - g[0], dy = v[1] - g[1];
    const float verr = sqrtf(dx * dx + dy * dy);
    const float err = zc ? verr : verr * verr;
    r[0] = expf(-err / P.linvel_es);
  }
  // R2 angvel train.py:301-306
  r[1] = expf(-fabsf(v[5] - c[2]) / P.angvel_es);
  // R3 roll_pitch train.py:316-334
  {
    float qxy[4], qc[4];
    euler_to_quat(e[0], e[1], 0.0f, qxy);
    euler_to_quat(c[4], c[5], 0.0f, qc);
    const float d = quat_dot(qc, qxy);
    const float qerr = 1.0f - d * d;
    r[2] = expf(-qerr / (zc ? P.rp_es_zero : P.rp_es));
  }
  // R4 base_height train.py:377-388
  {
    const float h = bz - fminf(lz - P.bh_foot_origin, rz - P.bh_foot_origin);
    r[3] = expf(-fabsf(h - (c[3] + P.bh_standard)) / P.bh_es);
  }
  // contacts train.py:139-140
  const bool cl = tl > 0.1f, cr = trr > 0.1f;
  flags[t * ld + e0] = (cl ? 1 : 0) | (cr ? 2 : 0) | (zc ? 4 : 0);
  // R7 no_contact_p train.py:161-165
  r[6] = zc ? 0.0f : ((cl || cr) ? 0.0f : 1.0f);
  // R9 feet_orient train.py:418-457
  {
    const float yaw = e[2];
    float tq[2][4], tq0[2][4];
    euler_to_quat(-kHalfPi, 0.0f, yaw - kPi, tq[0]);
    euler_to_quat(kHalfPi, 0.0f, yaw - kPi, tq[1]);
    euler_to_quat(-kHalfPi, 0.0f, 0.0f, tq0[0]);
    euler_to_quat(kHalfPi, 0.0f, 0.0f, tq0[1]);
    float rpy = 0.0f, rp = 0.0f;
#pragma unroll
    for (int f = 0; f < 2; ++f) {
      const float d = quat_dot(tq[f], fq[f]);
      rpy = rpy + (1.0f - d * d);
      float fe[3], fq0[4];
      quat_to_euler(fq[f], P.eps_quat, fe);
      euler_to_quat(fe[0], fe[1], 0.0f, fq0);
      const float d0 = quat_dot(tq0[f], fq0);
      rp = rp + (1.0f - d0 * d0);
    }
    r[8] = expf(-(rot ? rp : rpy) / P.feet_es);
  }
  // R10 com_distance train.py:466-478
  r[9] = (cd >= 0.0f) ? (zc ? expf(-cd / P.com_es) : 0.0f) : 0.0f;
  r[5] = 0.0f;  // single_contact: scan kernel
  r[7] = 0.0f;  // feet_airtime: scan kernel
  float s = 0.0f;
#pragma unroll
  for (int k = 0; k < KBS_NUM_REWARDS; ++k) s = s + P.reward_scale[k] * r[k];
  __stcs(total + t * ld + e0, s);
  if (comp) {
    float* comp_t = comp + t * KBS_NUM_REWARDS * ld;
#pragma unroll
    for (int k = 0; k < KBS_NUM_REWARDS; ++k) __stcs(comp_t + k * ld + e0, r[k]);
  }
}

// Stateful terms R6 (train.py:138-154) and R8 (train.py:197-213): sequential in T per env, exactly the
// reference's scan order (t + dt accumulated step by step in fp32, compared against grace_period).
__global__ void __launch_bounds__(kThreads)
reward_scan_kernel(const __grid_constant__ kbs_params P, const uint8_t* __restrict__ flags,
                   const uint8_t* __restrict__ done, kbs_reward_carry carry, float* __restrict__ total,
                   float* __restrict__ comp, int64_t T, int64_t ld, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * kThreads + threadIdx.x;
  if (e >= n) return;
  float t_sc = carry.t_single[e];
  float air0 = carry.airtime[e], air1 = carry.airtime[ld + e];
  bool pc0 = carry.prev_contact[e] != 0, pc1 = carry.prev_contact[ld + e] != 0;
  constexpr int kB = 16;   // the inputs of step t do not depend on the recurrence: 16 steps of loads in flight
  for (int64_t t0 = 0; t0 < T; t0 += kB) {
  unsigned fv[kB]; bool dv[kB]; float tv[kB];
#pragma unroll
  for (int i = 0; i < kB; ++i) {
    const int64_t tt = t0 + i < T ? t0 + i : T - 1;
    fv[i] = flags[tt * ld + e]; dv[i] = done[tt * ld + e] != 0; tv[i] = total[tt * ld + e];
  }
#pragma unroll
  for (int i = 0; i < kB; ++i) {
    const int64_t t = t0 + i;
    if (t >= T) break;
    const unsigned f = fv[i];
    const bool dn = dv[i];
    const bool cl = f & 1, cr = (f & 2) != 0, zc = (f & 4) != 0;
    const bool single = cl != cr;
    t_sc = single ? 0.0f : t_sc + P.ctrl_dt;
    t_sc = zc ? P.grace_period : t_sc;
    const float r6 = zc ? 1.0f : ((t_sc < P.grace_period) ? 1.0f : 0.0f);
    const bool f0 = cl && !pc0 && !dn, f1 = cr && !pc1 && !dn;
    float r8 = (air0 - P.touchdown_penalty) * (f0 ? 1.0f : 0.0f) + (air1 - P.touchdown_penalty) * (f1 ? 1.0f : 0.0f);
    r8 = zc ? 0.0f : r8;
    air0 = (cl || dn) ? 0.0f : air0 + P.ctrl_dt;
    air1 = (cr || dn) ? 0.0f : air1 + P.ctrl_dt;
    pc0 = cl; pc1 = cr;
    total[t * ld + e] = tv[i] + (P.reward_scale[5] * r6 + P.reward_scale[7] * r8);
    if (comp) {
      comp[(t * KBS_NUM_REWARDS + 5) * ld + e] = r6;
      comp[(t * KBS_NUM_REWARDS + 7) * ld + e] = r8;
    }
  }
  }
  carry.t_single[e] = t_sc;
  carry.airtime[e] = air0; carry.airtime[ld + e] = air1;
  carry.prev_contact[e] = pc0; carry.prev_contact[ld + e] = pc1;
}

// =====================================================================================================
// GAE: ksim.compute_ppo_inputs.  Block = 32 envs x 4 warps.  Time is walked backwards in chunks of kGaeChunk
// steps: all 4 warps stage the chunk (delta, gamma*lam*mask) into shared memory with coalesced row loads,
// warp 0 runs the sequential reverse scan out of shared memory, all warps store the chunk back.
// =====================================================================================================
constexpr int kGaeChunk = 32;
constexpr int kGaeEnvs = 32;

__global__ void __launch_bounds__(128)
gae_kernel(float gamma, float lam, const float* __restrict__ values, const float* __restrict__ rewards,
           const uint8_t* __restrict__ done, const uint8_t* __restrict__ success, float* __restrict__ adv,
           float* __restrict__ targets, int64_t T, int64_t ld, int64_t n) {
  __shared__ float s_delta[kGaeChunk][kGaeEnvs];
  __shared__ float s_k[kGaeChunk][kGaeEnvs];
  __shared__ float s_v[kGaeChunk][kGaeEnvs];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t e = int64_t(blockIdx.x) * kGaeEnvs + lane;
  const bool live = e < n;
  const float gl = gamma * lam;
  float a = 0.0f;  // A_{t+1}, carried by warp 0 across chunks
  for (int64_t t_hi = T; t_hi > 0; t_hi -= kGaeChunk) {
    const int64_t t_lo = (t_hi > kGaeChunk) ? t_hi - kGaeChunk : 0;
    const int len = int(t_hi - t_lo);
    for (int i = warp; i < len; i += 4) {
      const int64_t t = t_lo + i;
      float v = 0.f, vn = 0.f, r = 0.f, mask = 1.f, sc = 0.f;
      if (live) {
        v = values[t * ld + e];
        vn = (t + 1 < T) ? values[(t + 1) * ld + e] : v;
        r = rewards[t * ld + e];
        mask = done[t * ld + e] ? 0.0f : 1.0f;
        sc = success[t * ld + e] ? 1.0f : 0.0f;
      }
      const float rt = r + gamma * v * sc;
      s_delta[i][lane] = rt + gamma * vn * mask - v;
      s_k[i][lane] = gl * mask;
      s_v[i][lane] = v;
    }
    __syncthreads();
    if (warp == 0) {
      for (int i = len - 1; i >= 0; --i) {
        a = s_delta[i][lane] + s_k[i][lane] * a;
        s_delta[i][lane] = a;
      }
    }
    __syncthreads();
    if (live) {
      for (int i = warp; i < len; i += 4) {
        const int64_t t = t_lo + i;
        const float av = s_delta[i][lane];
        adv[t * ld + e] = av;
        targets[t * ld + e] = av + s_v[i][lane];
      }
    }
    __syncthreads();
  }
}

// per-trajectory advantage normalisation a / (std_t(a) + eps)  [ksim flag, unverified]
__global__ void __launch_bounds__(kThreads)
adv_norm_kernel(float eps, float* __restrict__ adv, int64_t T, int64_t ld, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * kThreads + threadIdx.x;
  if (e >= n) return;
  float s = 0.0f;
  for (int64_t t = 0; t < T; ++t) s = s + adv[t * ld + e];
  const float mean = s / float(T);
  float q = 0.0f;
  for (int64_t t = 0; t < T; ++t) { const float d = adv[t * ld + e] - mean; q = q + d * d; }
  const float sd = sqrtf(q / float(T)) + eps;
  for (int64_t t = 0; t < T; ++t) adv[t * ld + e] = adv[t * ld + e] / sd;
}

// =====================================================================================================
// convert.py:84-119 policy step marshalling (AoS <-> kernel layouts)
// =====================================================================================================
__global__ void __launch_bounds__(kThreads)
policy_pack_obs_kernel(const __grid_constant__ kbs_params P, const float* __restrict__ ja, const float* __restrict__ jv,
                       const float* __restrict__ pg, const float* __restrict__ gyro, const float* __restrict__ cmd,
                       const float* __restrict__ carry_in, int carry_w, float* __restrict__ obs, float* __restrict__ lpf,
                       int64_t ld, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * kThreads + threadIdx.x;
  if (e >= n) return;
  for (int j = 0; j < KBS_NUM_JOINTS; ++j) {
    obs[j * ld + e] = (ja[e * 20 + j] - P.joint_bias[j]) / P.joint_range[j];
    obs[(20 + j) * ld + e] = jv[e * 20 + j] / 10.0f;
    lpf[j * ld + e] = carry_in[e * carry_w + (carry_w - 20) + j];
  }
  const float g[3] = {pg[e * 3 + 0], pg[e * 3 + 1], pg[e * 3 + 2]};
  float enc[5];
  encode_pg(g, enc);
  for (int k = 0; k < 5; ++k) obs[(40 + k) * ld + e] = enc[k];
  for (int k = 0; k < 3; ++k) obs[(45 + k) * ld + e] = gyro[e * 3 + k];
  obs[48 * ld + e] = zero_cmd(cmd[e * 16 + 0], cmd[e * 16 + 1], cmd[e * 16 + 2]) ? 1.0f : 0.0f;
  for (int k = 0; k < 16; ++k) obs[(49 + k) * ld + e] = cmd[e * 16 + k];
}

// carry_flat [n][D2H + 20]  <->  AoS [depth*2][n][H]
__global__ void __launch_bounds__(256)
policy_carry_kernel(const float* __restrict__ src, float* __restrict__ dst, int d2, int H, int carry_w, int64_t n,
                    bool to_kernel_layout) {
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  const int64_t per_env = int64_t(d2) * H;
  if (idx >= n * per_env) return;
  const int64_t e = idx / per_env;
  const int rem = int(idx - e * per_env);
  const int slot = rem / H, k = rem - slot * H;
  const int64_t flat = e * carry_w + rem;
  const int64_t aos = (int64_t(slot) * n + e) * H + k;
  if (to_kernel_layout) dst[aos] = src[flat];
  else dst[flat] = src[aos];
}

__global__ void __launch_bounds__(kThreads)
policy_unpack_kernel(const float* __restrict__ lpf, const float* __restrict__ mean, float* __restrict__ carry_out,
                     int carry_w, float* __restrict__ action_out, int64_t ld, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * kThreads + threadIdx.x;
  if (e >= n) return;
  for (int j = 0; j < KBS_NUM_JOINTS; ++j) {
    carry_out[e * carry_w + (carry_w - 20) + j] = lpf[j * ld + e];
    action_out[e * 20 + j] = mean[j * ld + e];
  }
}

// =====================================================================================================
// Trajectory-wise scans of the fused rollout (recorded state: everything that does not depend on the networks is
// evaluated for all T steps up front).  One thread per env, time walked sequentially; loads are env-coalesced.
// =====================================================================================================
// UnifiedCommand over T steps: command[t+1] = (done[t] or u_switch[t] < p) ? initial_command(rand[t]) : command[t]
__device__ __forceinline__ void
command_scan_body(const kbs_params& P, int k, float* __restrict__ command /*[T+1][16][ld]*/,
                    const float* __restrict__ u_switch, const int32_t* __restrict__ mode, const float* __restrict__ u6,
                    const float* __restrict__ u_arms, const uint8_t* __restrict__ done, int64_t T, int64_t ld, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * kThreads + threadIdx.x;
  if (e >= n) return;
  // thread = (env, command row k): 16x the threads of a one-thread-per-env walk (4 096 envs alone fill only 32 SMs and
  // the kernel is pure latency).  Nothing a step reads depends on the recurrence (the new command is a function of that
  // step's mode / uniform only, train.py:768-785), so every input of 10 steps is loaded unconditionally first -- 40
  // independent loads in flight per thread, ~30 MB per 4 096 x 100 in total -- and the scan itself touches registers only.
  // (Loading the mode / uniform only at a switch, p ~ 0.014 per step, saved bytes nobody needed saved and cost two
  // dependent round trips per switch in a divergent warp: 82 us per launch.)
  float c = command[k * ld + e];
  constexpr int kB = 10;     // 40 loads in flight; keeps the combined phase_a_scans_kernel at 4 CTAs per SM (one wave)
  const float lo = k < 6 ? P.cmd_lo[k] : P.arm_lo[k - 6], hi = k < 6 ? P.cmd_hi[k] : P.arm_hi[k - 6];
  for (int64_t t0 = 0; t0 < T; t0 += kB) {
    bool sw[kB];
    int m[kB];
    float u[kB];
#pragma unroll
    for (int i = 0; i < kB; ++i) {
      const int64_t t = t0 + i < T ? t0 + i : T - 1;
      sw[i] = (done[t * ld + e] != 0) || (u_switch[t * ld + e] < P.switch_prob);
      m[i] = mode[t * ld + e];
      u[i] = k < 6 ? u6[(t * 6 + k) * ld + e] : u_arms[(t * 10 + (k - 6)) * ld + e];
    }
#pragma unroll
    for (int i = 0; i < kB; ++i) {
      const int64_t t = t0 + i;
      if (t >= T) break;
      if (sw[i]) {
        if (k < 6) {
          const float v = lo + u[i] * (hi - lo);
          bool on;
          if (k == 0) on = (m[i] == 0) || (m[i] == 3);
          else if (k == 1) on = (m[i] == 1) || (m[i] == 3);
          else if (k == 2) on = (m[i] == 2) || (m[i] == 3);
          else on = (m[i] == 4);
          c = on ? v : 0.0f;
        } else {
          const float arm = (lo + u[i] * (hi - lo)) * ((u[i] < 0.5f) ? 1.0f : 0.0f);
          c = (m[i] == 3 || m[i] == 4) ? arm : 0.0f;
        }
      }
      command[((t + 1) * KBS_NUM_COMMANDS + k) * ld + e] = c;
    }
  }
}

// Lagged projected gravity (ProjectedGravityObservation min_lag/max_lag): x_t = lag x_{t-1} + (1-lag) g_b(t), restarted at
// g_b(t) on the first step of a new episode (done[t-1]; at t = 0, done_prev[e] = the previous call's done[T-1], NULL = no
// restart).  pg_carry in/out; lagged[T][3][ld] out.
__device__ __forceinline__ void
pg_scan_body(const kbs_params& P, const float* __restrict__ sensordata, const float* __restrict__ lag_p,
               const uint8_t* __restrict__ done, const uint8_t* __restrict__ done_prev, float* __restrict__ pg_carry,
               float* __restrict__ lagged, int64_t T, int64_t ld, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * kThreads + threadIdx.x;
  if (e >= n) return;
  const float lag = lag_p ? lag_p[e] : 0.0f;
  const bool rs0 = done_prev && done_prev[e] != 0;
  float x[3] = {pg_carry[e], pg_carry[ld + e], pg_carry[2 * ld + e]};
  // the inputs of step t do not depend on the recurrence: fetch 8 steps at a time so the load latencies overlap
  constexpr int kB = 8;
  for (int64_t t0 = 0; t0 < T; t0 += kB) {
    float qv[kB][4];
    bool rsv[kB];
#pragma unroll
    for (int i = 0; i < kB; ++i) {
      const int64_t t = t0 + i < T ? t0 + i : T - 1;
      const float* sd = sensordata + (t * KBS_NSENSORDATA + P.sd_imu_quat) * ld + e;
      qv[i][0] = sd[0]; qv[i][1] = sd[ld]; qv[i][2] = sd[2 * ld]; qv[i][3] = sd[3 * ld];
      rsv[i] = t > 0 ? (done[(t - 1) * ld + e] != 0) : rs0;
    }
#pragma unroll
    for (int i = 0; i < kB; ++i) {
      const int64_t t = t0 + i;
      if (t >= T) break;
      const float q[4] = {qv[i][0], qv[i][1], qv[i][2], qv[i][3]};
      const float g[3] = {0.0f, 0.0f, -P.gravity};
      float gb[3];
      rotate_vec(g, q, true, P.eps_quat, gb);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float pv = rsv[i] ? gb[k] : x[k];
        x[k] = lag * pv + (1.0f - lag) * gb[k];
        lagged[(t * 3 + k) * ld + e] = x[k];
      }
    }
  }
  pg_carry[e] = x[0]; pg_carry[ld + e] = x[1]; pg_carry[2 * ld + e] = x[2];
}

__global__ void __launch_bounds__(kThreads)
command_scan_kernel(const __grid_constant__ kbs_params P, float* __restrict__ command, const float* __restrict__ u_switch,
                    const int32_t* __restrict__ mode, const float* __restrict__ u6, const float* __restrict__ u_arms,
                    const uint8_t* __restrict__ done, int64_t T, int64_t ld, int64_t n) {
  command_scan_body(P, blockIdx.y, command, u_switch, mode, u6, u_arms, done, T, ld, n);
}
__global__ void __launch_bounds__(kThreads)
pg_scan_kernel(const __grid_constant__ kbs_params P, const float* __restrict__ sensordata, const float* __restrict__ lag_p,
               const uint8_t* __restrict__ done, const uint8_t* __restrict__ done_prev, float* __restrict__ pg_carry,
               float* __restrict__ lagged, int64_t T, int64_t ld, int64_t n) {
  pg_scan_body(P, sensordata, lag_p, done, done_prev, pg_carry, lagged, T, ld, n);
}
// Both scans of the fused rollout's phase A in one launch (they only depend on `done`): blockIdx.y = 0..15 command rows,
// 16 = the lagged-gravity scan -- two latency-bound kernels side by side instead of back to back.
__global__ void __launch_bounds__(kThreads, 4)
phase_a_scans_kernel(const __grid_constant__ kbs_params P, float* __restrict__ command, const float* __restrict__ u_switch,
                     const int32_t* __restrict__ mode, const float* __restrict__ u6, const float* __restrict__ u_arms,
                     const uint8_t* __restrict__ done, const uint8_t* __restrict__ done_prev,
                     const float* __restrict__ sensordata, const float* __restrict__ lag_p, float* __restrict__ pg_carry,
                     float* __restrict__ lagged, int64_t T, int64_t ld, int64_t n) {
  if (blockIdx.y < KBS_NUM_COMMANDS) command_scan_body(P, blockIdx.y, command, u_switch, mode, u6, u_arms, done, T, ld, n);
  else pg_scan_body(P, sensordata, lag_p, done, done_prev, pg_carry, lagged, T, ld, n);
}

inline unsigned groups4(int64_t n) { return unsigned((((n + 3) / 4) + kThreads - 1) / kThreads); }

}  // namespace

// ---- launchers ------------------------------------------------------------------------------------
int kbs_launch_observations(kbs_handle* h, const kbs_state_view& s, const kbs_noise_view* nz,
                            const kbs_episode_view* ep, const float* command, float* pg_carry,
                            const uint8_t* pg_reset, float* computed, float* actor_obs, float* critic_obs, int64_t n,
                            cudaStream_t st, int64_t T, const float* pg_lagged, bool skip_dump, bool one_step) {
  kbs_noise_view z{};
  kbs_episode_view e{};
  if (nz) z = *nz;
  if (ep) e = *ep;
  // skip_dump: the caller reads cinert / cvel straight from the state (critic rows 80..447 stay unwritten)
  if (one_step && T == 1) {
    using S = ObsSections<true>;
    dim3 grid(groups4(n), (critic_obs && !skip_dump) ? S::kComputed + S::kCopy : S::kComputed, 1u);
    KBS_LAUNCH(h, KBS_K_OBS, st, (obs_kernel<true><<<grid, kThreads, 0, st>>>(h->p, s, z, e, command, pg_carry, pg_reset,
                                                                            pg_lagged, computed, actor_obs, critic_obs, n)));
  } else {
    using S = ObsSections<false>;
    dim3 grid(groups4(n), (critic_obs && !skip_dump) ? S::kComputed + S::kCopy : S::kComputed, unsigned(T));
    KBS_LAUNCH(h, KBS_K_OBS, st, (obs_kernel<false><<<grid, kThreads, 0, st>>>(h->p, s, z, e, command, pg_carry, pg_reset,
                                                                             pg_lagged, computed, actor_obs, critic_obs, n)));
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

static int ppo_loss_blocks(const kbs_handle* h, const kbs_ppo_loss_io& io) {
  const int64_t total = io.T * io.ld;
  int blocks = int((total + kLossThreads * 8 - 1) / (kLossThreads * 8));
  if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms;
  return blocks < 1 ? 1 : blocks;
}

int kbs_launch_ppo_loss(kbs_handle* h, const kbs_ppo_loss_params& L, const kbs_ppo_loss_io& io, int64_t n, cudaStream_t st) {
  double* partials;
  const int rc = kbs_scratch(h, [&](KbsScratch& s) { partials = s.take<double>(size_t(ppo_loss_blocks(h, io)) * 4); });
  if (rc) return rc;
  return kbs_launch_ppo_loss_at(h, L, io, n, partials, st);
}

// partials: >= 4 * 4 * num_sms doubles of caller-provided device scratch
int kbs_launch_ppo_loss_at(kbs_handle* h, const kbs_ppo_loss_params& L, const kbs_ppo_loss_io& io, int64_t n, double* partials,
                           cudaStream_t st) {
  const int blocks = ppo_loss_blocks(h, io);
  if (!h->loss_ticket) {
    KBS_CUDA_TRY(cudaMalloc(&h->loss_ticket, 256));
    KBS_CUDA_TRY(cudaMemsetAsync(h->loss_ticket, 0, 256, st));
  }
  KBS_LAUNCH(h, KBS_K_GAE, st, (ppo_loss_kernel<<<blocks, kLossThreads, 0, st>>>(L, io, n, partials, h->loss_ticket)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_com_distance(kbs_handle* h, const int32_t* geom1, const int32_t* geom2, const float* pos, const float* com,
                            float* out, int ncon, int64_t T, int64_t ld, int64_t n, cudaStream_t st) {
  if (ncon < 3 || ncon > kMaxContacts) return KBS_E_SHAPE;
  dim3 grid(unsigned((n + kThreads - 1) / kThreads), unsigned(T));
  KBS_LAUNCH(h, KBS_K_OBS, st, (com_distance_kernel<<<grid, kThreads, 0, st>>>(geom1, geom2, pos, com, out, ncon, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_mirror_obs(kbs_handle* h, const kbs_state_view& s, const float* computed, const float* command,
                          float* actor_obs, float* critic_obs, float* command_out, int64_t n, int64_t T, cudaStream_t st) {
  dim3 grid(groups4(n), critic_obs ? 1 + 368 / kCopyRowsPerSection : 1, unsigned(T));
  KBS_LAUNCH(h, KBS_K_OBS, st, (mirror_obs_kernel<<<grid, kThreads, 0, st>>>(h->p, s, computed, command, actor_obs, critic_obs,
                                                                             command_out, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_mirror_joints(kbs_handle* h, const float* in, float* out, int64_t ld, int64_t n, int64_t T, cudaStream_t st) {
  dim3 grid(groups4(n), KBS_NUM_JOINTS, unsigned(T));
  KBS_LAUNCH(h, KBS_K_OBS, st, (mirror_joints_kernel<<<grid, kThreads, 0, st>>>(in, out, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_command(kbs_handle* h, const float* cmd_in, float* cmd_out, const float* u_switch,
                       const int32_t* mode, const float* u6, const float* u_arms, const uint8_t* done, int64_t ld,
                       int64_t n, cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_COMMAND, st, (command_kernel<<<groups4(n), kThreads, 0, st>>>(h->p, cmd_in, cmd_out, u_switch,
                                                                                    mode, u6, u_arms, done, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_command_scan(kbs_handle* h, float* command, const float* u_switch, const int32_t* mode, const float* u6,
                            const float* u_arms, const uint8_t* done, int64_t T, int64_t ld, int64_t n, cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_COMMAND, st,
             (command_scan_kernel<<<dim3(unsigned((n + kThreads - 1) / kThreads), KBS_NUM_COMMANDS), kThreads, 0, st>>>(h->p, command, u_switch, mode,
                                                                                              u6, u_arms, done, T, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_phase_a_scans(kbs_handle* h, float* command, const float* u_switch, const int32_t* mode, const float* u6,
                             const float* u_arms, const uint8_t* done, const uint8_t* done_prev, const float* sensordata,
                             const float* lag, float* pg_carry, float* lagged, int64_t T, int64_t ld, int64_t n, cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_COMMAND, st,
             (phase_a_scans_kernel<<<dim3(unsigned((n + kThreads - 1) / kThreads), KBS_NUM_COMMANDS + 1), kThreads, 0, st>>>(
                 h->p, command, u_switch, mode, u6, u_arms, done, done_prev, sensordata, lag, pg_carry, lagged, T, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_pg_scan(kbs_handle* h, const float* sensordata, const float* lag, const uint8_t* done, const uint8_t* done_prev,
                       float* pg_carry, float* lagged, int64_t T, int64_t ld, int64_t n, cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_OBS, st,
             (pg_scan_kernel<<<unsigned((n + kThreads - 1) / kThreads), kThreads, 0, st>>>(h->p, sensordata, lag, done, done_prev,
                                                                                         pg_carry, lagged, T, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_torque(kbs_handle* h, const float* action, const kbs_state_view& s, const kbs_episode_view* ep,
                      float* ctrl, int64_t n, cudaStream_t st) {
  kbs_episode_view e{};
  if (ep) e = *ep;
  KBS_LAUNCH(h, KBS_K_TORQUE, st, (torque_kernel<<<groups4(n), kThreads, 0, st>>>(h->p, action, s, e, ctrl, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_mirror_loss(kbs_handle* h, const float* mean, const float* mean_m, const float* value, const float* value_m,
                           float* action_loss, float* value_loss, float scale_a, float scale_c, int64_t T, int64_t ld, int64_t n,
                           cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_ADV_NORM, st,
             (mirror_loss_kernel<<<dim3(groups4(n), unsigned(T)), kThreads, 0, st>>>(mean, mean_m, value, value_m, action_loss,
                                                                                    value_loss, scale_a, scale_c, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_actuator_rand(kbs_handle* h, const kbs_actuator_rand_params& rp, const float* u, const uint8_t* reset,
                             const kbs_episode_view& ep, int64_t ld, int64_t n, cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_TORQUE, st,
             (actuator_rand_kernel<<<dim3(groups4(n), KBS_NUM_JOINTS), kThreads, 0, st>>>(h->p, rp, u, reset, ep, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_rollout_noise(kbs_handle* h, uint64_t seed, int64_t step0, const kbs_noise_view* nz, float* eps_action, float* u_switch,
                             int32_t* cmd_mode, float* cmd_u6, float* cmd_u_arms, int64_t T, int64_t ld, int64_t n, cudaStream_t st) {
  NoiseRows R{};
  float* bases[9] = {nz ? const_cast<float*>(nz->eps_jpos) : nullptr, nz ? const_cast<float*>(nz->eps_jvel) : nullptr,
                     nz ? const_cast<float*>(nz->eps_gyro) : nullptr, nz ? const_cast<float*>(nz->eps_pg) : nullptr, eps_action, u_switch,
                     reinterpret_cast<float*>(cmd_mode), cmd_u6, cmd_u_arms};
  const int rows[9] = {20, 20, 3, 3, 20, 1, 1, 6, 10};
  const int kind[9] = {0, 0, 1, 1, 1, 2, 3, 2, 2};
  int acc = 0;
  for (int i = 0; i < 9; ++i) { R.base[i] = bases[i]; R.rows[i] = rows[i]; R.kind[i] = kind[i]; R.first[i] = acc; acc += rows[i]; }
  R.first[9] = acc;
  KBS_LAUNCH(h, KBS_K_COMMAND, st,
             (rollout_noise_kernel<<<dim3(groups4(n), unsigned(acc), unsigned(T)), kThreads, 0, st>>>(R, seed, step0, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_torque_substeps(kbs_handle* h, const float* action, float* prev_action, const float* u_drop, const float* latency,
                               const float* q_sub, const float* qd_sub, const kbs_episode_view* ep, float* ctrl, int S, float sub_dt,
                               float drop_prob, int64_t ld, int64_t n, cudaStream_t st) {
  kbs_episode_view e{};
  if (ep) e = *ep;
  KBS_LAUNCH(h, KBS_K_TORQUE, st,
             (torque_substeps_kernel<<<groups4(n), kThreads, 0, st>>>(h->p, action, prev_action, u_drop, latency, q_sub, qd_sub, e,
                                                                      ctrl, S, sub_dt, drop_prob, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_actuator_substep(kbs_handle* h, const KbsSubstepArgs& a, cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_ACTUATOR_SUBSTEP, st, (actuator_substep_kernel<<<dim3(groups4(a.n), KBS_NUM_JOINTS), kThreads, 0, st>>>(h->p, a)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_terminate(kbs_handle* h, const kbs_state_view& s, int32_t* codes, uint8_t* done, uint8_t* success,
                         float* pre, int64_t n, cudaStream_t st, int64_t T) {
  KBS_LAUNCH(h, KBS_K_TERMINATE, st,
             (terminate_kernel<<<dim3(groups4(n), unsigned(T)), kThreads, 0, st>>>(h->p, s, codes, done, success, pre, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_rewards(kbs_handle* h, const kbs_traj_view& tr, const kbs_reward_carry& carry, float* total,
                       float* components, int64_t n, cudaStream_t st) {
  const int64_t ld = tr.state.ld, T = tr.T;
  uint8_t *is_rot, *flags;   // [ld], [T][ld]
  const int rc = kbs_scratch(h, [&](KbsScratch& s) {
    is_rot = s.take<uint8_t>(size_t(ld));
    flags = s.take<uint8_t>(size_t(T) * ld);
  });
  if (rc) return rc;
  KBS_LAUNCH(h, KBS_K_REWARD_ROT, st, (reward_rot_kernel<<<groups4(n), kThreads, 0, st>>>(tr.command, is_rot, T, ld, n)));
  dim3 grid(unsigned((n + kThreads - 1) / kThreads), unsigned(T));
  KBS_LAUNCH(h, KBS_K_REWARD_TERMS, st,
             (reward_terms_kernel<<<grid, kThreads, 0, st>>>(h->p, tr, is_rot, total, components, flags, n)));
  KBS_LAUNCH(h, KBS_K_REWARD_SCAN, st,
             (reward_scan_kernel<<<unsigned((n + kThreads - 1) / kThreads), kThreads, 0, st>>>(
                 h->p, flags, tr.done, carry, total, components, T, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_gae(kbs_handle* h, const float* values, const float* rewards, const uint8_t* done,
                   const uint8_t* success, float* adv, float* targets, int64_t T, int64_t ld, int64_t n,
                   cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_GAE, st,
             (gae_kernel<<<unsigned((n + kGaeEnvs - 1) / kGaeEnvs), 128, 0, st>>>(h->p.gamma, h->p.lam, values, rewards,
                                                                                 done, success, adv, targets, T, ld, n)));
  if (h->p.normalize_advantages == 1) {
    KBS_LAUNCH(h, KBS_K_ADV_NORM, st,
               (adv_norm_kernel<<<unsigned((n + kThreads - 1) / kThreads), kThreads, 0, st>>>(h->p.adv_eps, adv, T, ld, n)));
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_policy_pack(kbs_handle* h, const float* ja, const float* jv, const float* pg, const float* gyro,
                           const float* cmd, const float* carry_in, float* obs_soa, float* carry_aos, float* lpf_soa,
                           int64_t ld, int64_t n, cudaStream_t st) {
  const int H = h->p.hidden_size, d2 = 2 * h->p.depth, cw = d2 * H + 20;
  KBS_LAUNCH(h, KBS_K_POLICY_IO, st,
             (policy_pack_obs_kernel<<<unsigned((n + kThreads - 1) / kThreads), kThreads, 0, st>>>(
                 h->p, ja, jv, pg, gyro, cmd, carry_in, cw, obs_soa, lpf_soa, ld, n)));
  const int64_t tot = n * int64_t(d2) * H;
  if (carry_aos)   // nullptr: the caller converts the flat carry records itself (tensor-core path)
    KBS_LAUNCH(h, KBS_K_POLICY_IO, st,
               (policy_carry_kernel<<<unsigned((tot + 255) / 256), 256, 0, st>>>(carry_in, carry_aos, d2, H, cw, n, true)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_policy_unpack(kbs_handle* h, const float* carry_aos, const float* lpf_soa, const float* mean_soa,
                             float* carry_out, float* action_out, int64_t ld, int64_t n, cudaStream_t st) {
  const int H = h->p.hidden_size, d2 = 2 * h->p.depth, cw = d2 * H + 20;
  const int64_t tot = n * int64_t(d2) * H;
  if (carry_aos)
    KBS_LAUNCH(h, KBS_K_POLICY_IO, st,
               (policy_carry_kernel<<<unsigned((tot + 255) / 256), 256, 0, st>>>(carry_aos, carry_out, d2, H, cw, n, false)));
  KBS_LAUNCH(h, KBS_K_POLICY_IO, st,
             (policy_unpack_kernel<<<unsigned((n + kThreads - 1) / kThreads), kThreads, 0, st>>>(
                 lpf_soa, mean_soa, carry_out, cw, action_out, ld, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// ---- the online step's record (kbs_rollout_step) -------------------------------------------------------------------------
// Moves one step's outputs into slot t of the caller's trajectories, t read from the step state, in one pass: every job is a
// contiguous run of 32-bit words (a [F][ld] block; done / success are ld bytes), copied as float4 where both ends are 16-byte
// aligned.  The command job also shifts the state's next-command rows into its current rows.  The last block to finish
// advances t and flips the state's hsb slot word, so a captured launch serves every step.
namespace {
constexpr int kStepWordsPerBlock = 4096;
__global__ void __launch_bounds__(256) step_record_kernel(const __grid_constant__ KbsStepRecord a) {
  __shared__ int64_t t_s;
  if (threadIdx.x == 0) t_s = *reinterpret_cast<volatile int64_t*>(a.t);
  __syncthreads();
  const int64_t t = t_s;
  const bool in_range = t >= 0 && t < a.T;
  if (in_range) {
    int j = 0;
    while (j + 1 < a.jobs && int(blockIdx.x) >= a.job[j + 1].block0) ++j;
    const KbsStepJob& J = a.job[j];
    const int64_t w0 = int64_t(blockIdx.x - J.block0) * kStepWordsPerBlock;
    const int64_t w1 = w0 + kStepWordsPerBlock < J.words ? w0 + kStepWordsPerBlock : J.words;
    const uint32_t* src = static_cast<const uint32_t*>(J.src);
    uint32_t* dst = static_cast<uint32_t*>(J.dst) + t * J.dst_step;
    if (J.shift) {        // command: state rows [0] -> traj[t], [1] -> traj[t + 1] and -> state rows [0]
      uint32_t* cs = const_cast<uint32_t*>(src);
      for (int64_t w = w0 + threadIdx.x; w < w1; w += blockDim.x) {
        const uint32_t c0 = cs[w], c1 = cs[J.words + w];
        dst[w] = c0; dst[J.dst_step + w] = c1; cs[w] = c1;
      }
    } else if (((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0 && (J.words & 3) == 0) {
      const uint4* s4 = reinterpret_cast<const uint4*>(src);
      uint4* d4 = reinterpret_cast<uint4*>(dst);
      for (int64_t q = w0 / 4 + threadIdx.x; q < w1 / 4; q += blockDim.x) __stcs(d4 + q, __ldcs(s4 + q));
    } else {
      for (int64_t w = w0 + threadIdx.x; w < w1; w += blockDim.x) dst[w] = src[w];
    }
  } else if (blockIdx.x == 0 && threadIdx.x == 0) {
    atomicOr(a.status, unsigned(KBS_STATUS_STEP_RANGE));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(a.ticket, 1u) == gridDim.x - 1) {       // every block has read t
      *a.ticket = 0u;
      if (in_range) *a.t = t + 1;
      if (a.hsb_slot) *a.hsb_slot ^= 1;
      __threadfence();
    }
  }
}
}  // namespace

int kbs_launch_step_record(kbs_handle* h, KbsStepRecord a, cudaStream_t st) {
  int blocks = 0;
  for (int j = 0; j < a.jobs; ++j) {
    a.job[j].block0 = blocks;
    blocks += int((a.job[j].words + kStepWordsPerBlock - 1) / kStepWordsPerBlock);
  }
  KBS_LAUNCH(h, KBS_K_STEP_RECORD, st, (step_record_kernel<<<unsigned(blocks), 256, 0, st>>>(a)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}
