// kbs_ppo_update.cu -- gradients of the PPO minibatch loss (SURVEY 8f-1; BASELINE configs[3]) and the Adam step.
//
// Replaces, for one minibatch of stored trajectories: jax.grad of ksim's PPO loss through get_ppo_variables
// (train.py:1435-1524: actor log-prob / entropy of the stored action + critic value per step, carries reset where
// done) -- i.e. back-propagation through time through both 2-layer LSTMs, the input / output projections, the actor
// head (softplus std, clamp, one-pole low-pass on the mean: a second recurrence in time) and the loss
// (ksim.compute_ppo_loss [U], kbs_ppo_loss).  Optimiser: optax.adam (train.py:1057-1063).
//
// First correct version: fp32 FFMA GEMMs (gemm_nt / split-K gemm_tn of kbs_net_simt.cu), one launch per (step, layer)
// for the recurrent part, everything that is not recurrent batched over all T x n rows.  The forward pass stores what
// the backward pass needs (activated gates, cell states, layer inputs).  Deterministic: no atomics.
#include <math.h>

#include "kbs_common.cuh"

namespace {

constexpr int kT = 256;
inline int round_up_i(int x, int m) { return (x + m - 1) / m * m; }

// env-major SoA observations [T][F][ld] -> row-major [T*n][kp] (features >= F zero)
__global__ void __launch_bounds__(kT)
soa_to_rows_kernel(const float* __restrict__ soa, int F, int64_t ld, float* __restrict__ rm, int kp, int64_t n, int64_t T) {
  const int64_t idx = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (idx >= T * n * kp) return;
  const int f = int(idx % kp);
  const int64_t row = idx / kp;
  const int64_t t = row / n, e = row - t * n;
  rm[idx] = f < F ? soa[(t * F + f) * ld + e] : 0.0f;
}

__global__ void __launch_bounds__(kT)
transpose_kernel(const float* __restrict__ in, int rows, int cols, float* __restrict__ out) {   // out[c][r] = in[r][c]
  const int64_t idx = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (idx >= int64_t(rows) * cols) return;
  const int r = int(idx / cols), c = int(idx % cols);
  out[size_t(c) * rows + r] = in[idx];
}

__device__ __forceinline__ float sigm(float x) { return 1.0f / (1.0f + expf(-x)); }

// eqx LSTMCell forward with everything the backward pass needs.  gates_pre [n][4H] (bias added).
//   ga [n][4H] = (s(i), s(f), tanh(g), s(o)); cs [n][H] = c_t; hs [n][H] = h_t (un-reset: next layer's input);
//   h_next_in / c_next_in [n][H] = the carries step t+1 reads (reset where done, train.py:1502-1506), or nullptr at t = T-1.
__global__ void __launch_bounds__(kT)
cell_fwd_save_kernel(const float* __restrict__ gates_pre, const float* __restrict__ c_in, float* __restrict__ ga,
                     float* __restrict__ cs, float* __restrict__ hs, float* __restrict__ h_next_in,
                     float* __restrict__ c_next_in, const uint8_t* __restrict__ done, int H, int64_t n) {
  const int64_t idx = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (idx >= n * H) return;
  const int64_t e = idx / H;
  const int k = int(idx - e * H);
  const float* g = gates_pre + e * 4 * H;
  const float i = sigm(g[k]), f = sigm(g[H + k]), gg = tanhf(g[2 * H + k]), o = sigm(g[3 * H + k]);
  const float c = f * c_in[idx] + i * gg;
  const float h = o * tanhf(c);
  float* a = ga + e * 4 * H;
  a[k] = i; a[H + k] = f; a[2 * H + k] = gg; a[3 * H + k] = o;
  cs[idx] = c;
  hs[idx] = h;
  if (h_next_in) {
    const bool rst = done && done[e];
    h_next_in[idx] = rst ? 0.0f : h;
    c_next_in[idx] = rst ? 0.0f : c;
  }
}

// ---- tensor-core variant of the recurrent part: the same cell math, 8 hidden units per thread, and the operands of the
// next GEMM written in the split-blocked MMA layout by the producing kernel (kbs_common.cuh) ----
__device__ __forceinline__ void ld8(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void st8(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
template <int KIND>
__device__ __forceinline__ void st8_sb(void* sb, int64_t row, int k, int K, const float (&v)[8], bool zero) {
  const float a[4] = {v[0], v[1], v[2], v[3]}, b[4] = {v[4], v[5], v[6], v[7]};
  sb_store_split8<kKbsPanelRows, KIND>(sb, row, k, K / kbs_block_k(KIND), sb_split4<KIND>(a), sb_split4<KIND>(b), zero);
}

// row-major [T][n][K] -> SB [T][np][K] (per-step panels; rows >= n of a step's last panel are left untouched)
template <int KIND>
__global__ void __launch_bounds__(kT)
rows_to_sb_kernel(const float* __restrict__ rm, char* __restrict__ sb, size_t sb_step_bytes, int K, int64_t n, int64_t T) {
  const int kq = K / 8;
  const int64_t idx = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (idx >= T * n * kq) return;
  const int g8 = int(idx % kq);
  const int64_t row = idx / kq;
  const int64_t t = row / n, e = row - t * n;
  float v[8];
  ld8(rm + row * K + g8 * 8, v);
  st8_sb<KIND>(sb + size_t(t) * sb_step_bytes, e, g8 * 8, K, v, false);
}

template <int KIND>
__global__ void __launch_bounds__(kT)
cell_fwd_save8_kernel(const float* __restrict__ gates_pre, const float* __restrict__ c_in, float* __restrict__ ga,
                      float* __restrict__ cs, float* __restrict__ hs, float* __restrict__ h_next_in,
                      float* __restrict__ c_next_in, char* __restrict__ hs_sb, char* __restrict__ h_next_in_sb,
                      const uint8_t* __restrict__ done, int H, int64_t n) {
  const int hq = H / 8;
  const int64_t idx = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (idx >= n * hq) return;
  const int64_t e = idx / hq;
  const int k = int(idx - e * hq) * 8;
  const float* g = gates_pre + e * 4 * H + k;
  float gi[8], gf[8], gg[8], go[8], ci[8], c[8], hh[8];
  ld8(g, gi); ld8(g + H, gf); ld8(g + 2 * H, gg); ld8(g + 3 * H, go); ld8(c_in + e * H + k, ci);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    gi[j] = sigm(gi[j]); gf[j] = sigm(gf[j]); gg[j] = tanhf(gg[j]); go[j] = sigm(go[j]);
    c[j] = gf[j] * ci[j] + gi[j] * gg[j];
    hh[j] = go[j] * tanhf(c[j]);
  }
  float* a = ga + e * 4 * H + k;
  st8(a, gi); st8(a + H, gf); st8(a + 2 * H, gg); st8(a + 3 * H, go);
  st8(cs + e * H + k, c);
  st8(hs + e * H + k, hh);
  st8_sb<KIND>(hs_sb, e, k, H, hh, false);
  if (h_next_in) {
    const bool rst = done && done[e];
    if (rst) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { hh[j] = 0.0f; c[j] = 0.0f; }
    }
    st8(h_next_in + e * H + k, hh);
    st8(c_next_in + e * H + k, c);
    st8_sb<KIND>(h_next_in_sb, e, k, H, hh, false);
  }
}

// dh_in / dh_rec are read with their own row strides (they live in [n][2H] GEMM outputs); dG also in SB form [np][4H]
template <int KIND>
__global__ void __launch_bounds__(kT)
cell_bwd8_kernel(const float* __restrict__ dh_in, int ld_in, const float* __restrict__ dh_rec, int ld_rec, float* __restrict__ dc_rec,
                 const float* __restrict__ ga, const float* __restrict__ cs, const float* __restrict__ c_in,
                 const uint8_t* __restrict__ done, float* __restrict__ dG, char* __restrict__ dG_sb, float gscale, int H, int64_t n) {
  const int hq = H / 8;
  const int64_t idx = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (idx >= n * hq) return;
  const int64_t e = idx / hq;
  const int k = int(idx - e * hq) * 8;
  const float keep = (done && done[e]) ? 0.0f : 1.0f;
  const float* a = ga + e * 4 * H + k;
  float i[8], f[8], g[8], o[8], c[8], ci[8], dhi[8], dhr[8], dcr[8], di[8], df[8], dg[8], dob[8];
  ld8(a, i); ld8(a + H, f); ld8(a + 2 * H, g); ld8(a + 3 * H, o);
  ld8(cs + e * H + k, c); ld8(c_in + e * H + k, ci);
  ld8(dh_in + e * ld_in + k, dhi);
  if (dh_rec) ld8(dh_rec + e * ld_rec + k, dhr);
  ld8(dc_rec + e * H + k, dcr);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float tc = tanhf(c[j]);
    const float dh = dhi[j] + (dh_rec ? keep * dhr[j] : 0.0f);
    const float dc = keep * dcr[j] + dh * o[j] * (1.0f - tc * tc);
    di[j] = dc * g[j] * i[j] * (1.0f - i[j]);
    df[j] = dc * ci[j] * f[j] * (1.0f - f[j]);
    dg[j] = dc * i[j] * (1.0f - g[j] * g[j]);
    dob[j] = dh * tc * o[j] * (1.0f - o[j]);
    dcr[j] = dc * f[j];
  }
  float* d = dG + e * 4 * H + k;
  st8(d, di); st8(d + H, df); st8(d + 2 * H, dg); st8(d + 3 * H, dob);
  st8(dc_rec + e * H + k, dcr);
  if (dG_sb) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { di[j] *= gscale; df[j] *= gscale; dg[j] *= gscale; dob[j] *= gscale; }   // into the FP16 planes' range
    st8_sb<KIND>(dG_sb, e, k, 4 * H, di, false);
    st8_sb<KIND>(dG_sb, e, H + k, 4 * H, df, false);
    st8_sb<KIND>(dG_sb, e, 2 * H + k, 4 * H, dg, false);
    st8_sb<KIND>(dG_sb, e, 3 * H + k, 4 * H, dob, false);
  }
}

// out[c] partial column sums over a chunk of rows: partial[chunk][c]
__global__ void __launch_bounds__(kT)
colsum_partial_kernel(const float* __restrict__ X, int ld, int64_t rows, int cols, int64_t rows_per_chunk, float* __restrict__ partial) {
  const int c = blockIdx.x * kT + threadIdx.x;
  if (c >= cols) return;
  const int64_t r0 = int64_t(blockIdx.y) * rows_per_chunk, r1 = (r0 + rows_per_chunk < rows) ? r0 + rows_per_chunk : rows;
  float a = 0.0f;
  for (int64_t r = r0; r < r1; ++r) a += X[r * ld + c];
  partial[size_t(blockIdx.y) * cols + c] = a;
}
__global__ void __launch_bounds__(kT)
reduce_rows_kernel(const float* __restrict__ partial, int chunks, int cols, float* __restrict__ out) {
  const int c = blockIdx.x * kT + threadIdx.x;
  if (c >= cols) return;
  float a = 0.0f;
  for (int s = 0; s < chunks; ++s) a += partial[size_t(s) * cols + c];
  out[c] = a;
}

// copy the leading [rows][cols] block of a [.][ld] matrix into a dense [rows][cols] one
__global__ void __launch_bounds__(kT)
copy_block_kernel(const float* __restrict__ src, int ld, float* __restrict__ dst, int rows, int cols) {
  const int64_t idx = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (idx >= int64_t(rows) * cols) return;
  const int r = int(idx / cols), c = int(idx % cols);
  dst[idx] = src[size_t(r) * ld + c];
}

// d min(r a, clip(r) a) / d log-prob of one transition: a dr (dr = d r / d log-prob) where the unclipped term is the minimum,
// else 0.  A non-finite advantage yields a non-finite derivative in either branch: the comparison is false for NaN, which
// used to select the clipped branch's 0 and drop the transition from the gradient silently, so the update was applied while
// the loss was NaN (jax.grad gives NaN there and ksim skips the update).  Caught by
// test_gpu_ppo_update.py::test_ppo_update_non_finite_minibatch_is_skipped.
__device__ __forceinline__ float policy_dlogp(float r, float rc, float dr, float a, bool inside) {
  return (inside || r * a < rc * a) ? a * dr : (isfinite(a) ? 0.0f : a);
}

// The same head with one WARP per env (lane j = joint j, log-prob / entropy by warp shuffles): the one-thread-per-env form
// above was 3.5 ms of an 18 ms update (512 threads walking 2 x T steps x 20 joints of libm math and strided loads).
// The steps are taken in chunks of kHC: every input of a chunk is loaded first (none depends on the filter's recurrence), then
// the chunk's steps run out of registers -- one L2 round trip per chunk instead of per step (there are only ~3 warps per SM at
// 512 envs, so nothing else hides the latency: 0.24 -> 0.07 ms per 512 x 100).  Same operations in the same order as before.
constexpr int kHC = 10;
__global__ void __launch_bounds__(128)
actor_head_fwd_bwd_warp_kernel(const __grid_constant__ kbs_params P, kbs_ppo_loss_params L, const float* __restrict__ out,
                               const float* __restrict__ actor_obs, const float* __restrict__ action,
                               const uint8_t* __restrict__ done, const float* __restrict__ lpf0, const float* __restrict__ old_lp,
                               const float* __restrict__ adv, float* __restrict__ y_s, float* __restrict__ sd_s,
                               float* __restrict__ log_prob, float* __restrict__ entropy, float* __restrict__ dout, int64_t T,
                               int64_t ld, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * 4 + (threadIdx.x >> 5);
  if (e >= n) return;                                   // whole warps leave together
  const int j = threadIdx.x & 31;
  const bool act = j < KBS_NUM_JOINTS;
  const int jj = act ? j : 0;
  constexpr float kHalfLog2Pi = 0.918938533204672742f;
  const float jb = P.joint_bias[jj];
  float y = (act && lpf0) ? lpf0[jj * ld + e] : 0.0f;
  for (int64_t t0 = 0; t0 < T; t0 += kHC) {
    float om[kHC], os[kHC], ob[kHC], ac[kHC];
    uint8_t dn[kHC];
#pragma unroll
    for (int i = 0; i < kHC; ++i) {
      const int64_t t = (t0 + i < T) ? t0 + i : T - 1;
      const float* o = out + (t * n + e) * 64;
      om[i] = o[jj];
      os[i] = o[KBS_NUM_JOINTS + jj];
      ob[i] = j >= 10 && act ? actor_obs[(t * KBS_ACTOR_OBS + 55 + (j - 10)) * ld + e] : 0.0f;
      ac[i] = action[(t * KBS_NUM_JOINTS + jj) * ld + e];
      dn[i] = done[t * ld + e];
    }
#pragma unroll
    for (int i = 0; i < kHC; ++i) {
      const int64_t t = t0 + i;
      if (t >= T) break;
      float tz = 0.0f, tl = 0.0f;
      if (act) {
        const float sraw = os[i];
        const float sp = fmaxf(sraw, 0.0f) + log1pf(expf(-fabsf(sraw)));
        const float sd = fminf((sp + P.min_std) * P.var_scale, P.max_std);
        float m = om[i] + jb;
        if (j >= 10) m = m + ob[i];
        y = y + P.lpf_alpha * (m - y);
        const int64_t so = (t * KBS_NUM_JOINTS + j) * ld + e;
        y_s[so] = y;
        sd_s[so] = sd;
        const float z = (ac[i] - y) / sd;
        tz = -0.5f * z * z - kHalfLog2Pi;
        tl = logf(sd);
      }
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) { tz += __shfl_xor_sync(0xffffffffu, tz, s); tl += __shfl_xor_sync(0xffffffffu, tl, s); }
      if (j == 0) {
        log_prob[t * ld + e] = tz - tl;
        entropy[t * ld + e] = tl + float(KBS_NUM_JOINTS) * (0.5f + kHalfLog2Pi);
      }
      if (dn[i]) y = 0.0f;
    }
  }
  __syncwarp();
  const float inv = 1.0f / (float(T) * float(n));
  float gy = 0.0f;
  for (int64_t t1 = T; t1 > 0; t1 -= kHC) {             // chunk = steps t1 - 1 down to t1 - kHC
    float lp[kHC], ol[kHC], av[kHC], sdv[kHC], yv[kHC], ac[kHC], os[kHC];
    uint8_t dn[kHC];
#pragma unroll
    for (int i = 0; i < kHC; ++i) {
      const int64_t t = (t1 - 1 - i >= 0) ? t1 - 1 - i : 0;
      const int64_t so = (t * KBS_NUM_JOINTS + jj) * ld + e;
      lp[i] = log_prob[t * ld + e];
      ol[i] = old_lp[t * ld + e];
      av[i] = adv[t * ld + e];
      dn[i] = done[t * ld + e];
      sdv[i] = sd_s[so];
      yv[i] = y_s[so];
      ac[i] = action[so];
      os[i] = out[(t * n + e) * 64 + KBS_NUM_JOINTS + jj];
    }
#pragma unroll
    for (int i = 0; i < kHC; ++i) {
      const int64_t t = t1 - 1 - i;
      if (t < 0) break;
      const float lr = lp[i] - ol[i];
      const float lrc = fminf(fmaxf(lr, -L.log_clip_value), L.log_clip_value);
      const float r = expf(lrc);
      const float a = av[i];
      const float dr = (fabsf(lr) <= L.log_clip_value) ? r : 0.0f;
      const bool inside = r >= 1.0f - L.clip_param && r <= 1.0f + L.clip_param;
      const float rc = fminf(fmaxf(r, 1.0f - L.clip_param), 1.0f + L.clip_param);
      const float dpol = policy_dlogp(r, rc, dr, a, inside);
      const float glp = -inv * dpol, gent = -inv * L.entropy_coef;
      const float keep = dn[i] ? 0.0f : 1.0f;
      float* d = dout + (t * n + e) * 64;
      if (act) {
        const float sd = sdv[i], yy = yv[i];
        const float z = (ac[i] - yy) / sd;
        const float dmu = glp * z / sd;
        const float dsd = (glp * (z * z - 1.0f) + gent) / sd;
        const float sraw = os[i];
        const float sp = fmaxf(sraw, 0.0f) + log1pf(expf(-fabsf(sraw)));
        const bool clamped = (sp + P.min_std) * P.var_scale > P.max_std;
        d[KBS_NUM_JOINTS + j] = clamped ? 0.0f : dsd * P.var_scale * sigm(sraw);
        gy = dmu + (1.0f - P.lpf_alpha) * keep * gy;
        d[j] = P.lpf_alpha * gy;
      }
      if (j < 24) d[2 * KBS_NUM_JOINTS + j] = 0.0f;
    }
  }
}

// The same head, one BLOCK (4 warps) per env: the expensive per-step math (softplus, log, exp, divisions, the joint reductions)
// does not depend on the low-pass filter's recurrence, so it runs in parallel over the steps (warp w takes steps t = w mod 4)
// around two cheap sequential scans by warp 0 (the filter forward: one FMA per step; its adjoint backward).  Every element sees
// the same operations in the same order as in the warp-per-env form: identical results; 0.115 -> 0.05 ms per 512 x 100.
// Shared memory: 3 x [T][32] floats + [T] bytes (38.5 KB at T = 100); the launcher falls back to the warp form beyond 48 KB.
__global__ void __launch_bounds__(128)
actor_head_fwd_bwd_block_kernel(const __grid_constant__ kbs_params P, kbs_ppo_loss_params L, const float* __restrict__ out,
                                const float* __restrict__ actor_obs, const float* __restrict__ action,
                                const uint8_t* __restrict__ done, const float* __restrict__ lpf0, const float* __restrict__ old_lp,
                                const float* __restrict__ adv, float* __restrict__ y_s, float* __restrict__ sd_s,
                                float* __restrict__ log_prob, float* __restrict__ entropy, float* __restrict__ dout, int64_t T,
                                int64_t ld, int64_t n) {
  extern __shared__ float hsm[];
  float* sm_y = hsm;                       // [T][32]: pre-filter mean, then the filtered mean
  float* sm_sd = hsm + T * 32;             // [T][32]
  float* sm_g = hsm + 2 * T * 32;          // [T][32]: d loss / d filtered mean (before the filter's adjoint)
  uint8_t* sm_dn = reinterpret_cast<uint8_t*>(hsm + 3 * T * 32);
  const int64_t e = blockIdx.x;
  const int w = threadIdx.x >> 5, j = threadIdx.x & 31;
  const bool act = j < KBS_NUM_JOINTS;
  const int jj = act ? j : 0;
  constexpr float kHalfLog2Pi = 0.918938533204672742f;
  const float jb = P.joint_bias[jj];
  // ---- phase 1: std and pre-filter mean of every step (kPB steps per pass: all their loads go out before the math) ----
  constexpr int kPB = 5;
  for (int64_t tb = w; tb < T; tb += 4 * kPB) {
    float o_m[kPB], o_s[kPB], o_b[kPB];
    uint8_t dn[kPB];
#pragma unroll
    for (int i = 0; i < kPB; ++i) {
      const int64_t t = (tb + 4 * i < T) ? tb + 4 * i : T - 1;
      const float* o = out + (t * n + e) * 64;
      o_m[i] = o[jj];
      o_s[i] = o[KBS_NUM_JOINTS + jj];
      o_b[i] = (act && j >= 10) ? actor_obs[(t * KBS_ACTOR_OBS + 55 + (j - 10)) * ld + e] : 0.0f;
      dn[i] = done[t * ld + e];
    }
#pragma unroll
    for (int i = 0; i < kPB; ++i) {
      const int64_t t = tb + 4 * i;
      if (t >= T) break;
      float m = 0.0f, sd = 1.0f;
      if (act) {
        const float sraw = o_s[i];
        const float sp = fmaxf(sraw, 0.0f) + log1pf(expf(-fabsf(sraw)));
        sd = fminf((sp + P.min_std) * P.var_scale, P.max_std);
        m = o_m[i] + jb;
        if (j >= 10) m = m + o_b[i];
        sd_s[(t * KBS_NUM_JOINTS + j) * ld + e] = sd;
      }
      sm_y[t * 32 + j] = m;
      sm_sd[t * 32 + j] = sd;
      if (j == 0) sm_dn[t] = dn[i];
    }
  }
  __syncthreads();
  // ---- phase 2: the filter's recurrence (done-resets included) ----
  if (w == 0 && act) {
    float y = lpf0 ? lpf0[j * ld + e] : 0.0f;
    for (int64_t t = 0; t < T; ++t) {
      const float m = sm_y[t * 32 + j];
      y = y + P.lpf_alpha * (m - y);
      sm_y[t * 32 + j] = y;
      y_s[(t * KBS_NUM_JOINTS + j) * ld + e] = y;
      if (sm_dn[t]) y = 0.0f;
    }
  }
  __syncthreads();
  // ---- phase 3: log-prob / entropy, the loss gradient, its way back through the Gaussian and softplus + clamp ----
  const float inv = 1.0f / (float(T) * float(n));
  for (int64_t tb = w; tb < T; tb += 4 * kPB) {
    float i_ac[kPB], i_ol[kPB], i_av[kPB], i_os[kPB];
#pragma unroll
    for (int i = 0; i < kPB; ++i) {
      const int64_t t = (tb + 4 * i < T) ? tb + 4 * i : T - 1;
      i_ac[i] = action[(t * KBS_NUM_JOINTS + jj) * ld + e];
      i_ol[i] = old_lp[t * ld + e];
      i_av[i] = adv[t * ld + e];
      i_os[i] = out[(t * n + e) * 64 + KBS_NUM_JOINTS + jj];
    }
#pragma unroll
    for (int i = 0; i < kPB; ++i) {
      const int64_t t = tb + 4 * i;
      if (t >= T) break;
      float tz = 0.0f, tl = 0.0f, z = 0.0f;
      const float sd = sm_sd[t * 32 + j];
      if (act) {
        z = (i_ac[i] - sm_y[t * 32 + j]) / sd;
        tz = -0.5f * z * z - kHalfLog2Pi;
        tl = logf(sd);
      }
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) { tz += __shfl_xor_sync(0xffffffffu, tz, s); tl += __shfl_xor_sync(0xffffffffu, tl, s); }
      const float lp = tz - tl;
      if (j == 0) {
        log_prob[t * ld + e] = lp;
        entropy[t * ld + e] = tl + float(KBS_NUM_JOINTS) * (0.5f + kHalfLog2Pi);
      }
      const float lr = lp - i_ol[i];
      const float lrc = fminf(fmaxf(lr, -L.log_clip_value), L.log_clip_value);
      const float r = expf(lrc);
      const float a = i_av[i];
      const float dr = (fabsf(lr) <= L.log_clip_value) ? r : 0.0f;
      const bool inside = r >= 1.0f - L.clip_param && r <= 1.0f + L.clip_param;
      const float rc = fminf(fmaxf(r, 1.0f - L.clip_param), 1.0f + L.clip_param);
      const float dpol = policy_dlogp(r, rc, dr, a, inside);
      const float glp = -inv * dpol, gent = -inv * L.entropy_coef;
      float* d = dout + (t * n + e) * 64;
      float dmu = 0.0f;
      if (act) {
        dmu = glp * z / sd;
        const float dsd = (glp * (z * z - 1.0f) + gent) / sd;
        const float sraw = i_os[i];
        const float sp = fmaxf(sraw, 0.0f) + log1pf(expf(-fabsf(sraw)));
        const bool clamped = (sp + P.min_std) * P.var_scale > P.max_std;
        d[KBS_NUM_JOINTS + j] = clamped ? 0.0f : dsd * P.var_scale * sigm(sraw);
      }
      sm_g[t * 32 + j] = dmu;
      if (j < 24) d[2 * KBS_NUM_JOINTS + j] = 0.0f;
    }
  }
  __syncthreads();
  // ---- phase 4: the filter's adjoint ----
  if (w == 0 && act) {
    float gy = 0.0f;
    for (int64_t t = T - 1; t >= 0; --t) {
      const float keep = sm_dn[t] ? 0.0f : 1.0f;
      gy = sm_g[t * 32 + j] + (1.0f - P.lpf_alpha) * keep * gy;
      dout[(t * n + e) * 64 + j] = P.lpf_alpha * gy;
    }
  }
}

// Backward half of the actor head for the persistent update path: the forward pass (rollout_persist_kernel<SAVE>) already
// produced log-prob / entropy / std / filtered mean / raw std output per step ([T][.][ld]); one warp per env (lane = joint)
// walks the steps backwards through the loss gradient, the Gaussian, softplus + clamp and the low-pass filter's recurrence
// (done-resets included).  dout [T*n][64] row-major: columns 0..19 = d loss / d mean output, 20..39 = d / d std output, rest 0.
__global__ void __launch_bounds__(128)
actor_head_bwd_warp_kernel(const __grid_constant__ kbs_params P, kbs_ppo_loss_params L, const float* __restrict__ action,
                           const uint8_t* __restrict__ done, const float* __restrict__ old_lp, const float* __restrict__ adv,
                           const float* __restrict__ y_s, const float* __restrict__ sd_s, const float* __restrict__ sraw_s,
                           const float* __restrict__ log_prob, float* __restrict__ dout, int64_t T, int64_t ld, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * 4 + (threadIdx.x >> 5);
  if (e >= n) return;
  const int j = threadIdx.x & 31;
  const bool act = j < KBS_NUM_JOINTS;
  const float inv = 1.0f / (float(T) * float(n));
  float gy = 0.0f;
  for (int64_t t = T - 1; t >= 0; --t) {
    const float lr = log_prob[t * ld + e] - old_lp[t * ld + e];
    const float lrc = fminf(fmaxf(lr, -L.log_clip_value), L.log_clip_value);
    const float r = expf(lrc);
    const float a = adv[t * ld + e];
    const float dr = (fabsf(lr) <= L.log_clip_value) ? r : 0.0f;
    const bool inside = r >= 1.0f - L.clip_param && r <= 1.0f + L.clip_param;
    const float rc = fminf(fmaxf(r, 1.0f - L.clip_param), 1.0f + L.clip_param);
    const float dpol = policy_dlogp(r, rc, dr, a, inside);
    const float glp = -inv * dpol, gent = -inv * L.entropy_coef;
    const float keep = done[t * ld + e] ? 0.0f : 1.0f;
    float* d = dout + (t * n + e) * 64;
    if (act) {
      const int64_t so = (t * KBS_NUM_JOINTS + j) * ld + e;
      const float sd = sd_s[so], yy = y_s[so];
      const float z = (action[so] - yy) / sd;
      const float dmu = glp * z / sd;
      const float dsd = (glp * (z * z - 1.0f) + gent) / sd;
      const float sraw = sraw_s[so];
      const float sp = fmaxf(sraw, 0.0f) + log1pf(expf(-fabsf(sraw)));
      const bool clamped = (sp + P.min_std) * P.var_scale > P.max_std;
      d[KBS_NUM_JOINTS + j] = clamped ? 0.0f : dsd * P.var_scale * sigm(sraw);
      gy = dmu + (1.0f - P.lpf_alpha) * keep * gy;
      d[j] = P.lpf_alpha * gy;
    }
    if (j < 24) d[2 * KBS_NUM_JOINTS + j] = 0.0f;
  }
}

// ... and of the critic head: values [T][ld] came from the forward pass
__global__ void __launch_bounds__(kT)
critic_head_bwd_kernel(kbs_ppo_loss_params L, const float* __restrict__ values, const float* __restrict__ old_values,
                       const float* __restrict__ targets, float* __restrict__ dout, int64_t T, int64_t ld, int64_t n) {
  const int64_t idx = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (idx >= T * n) return;
  const int64_t t = idx / n, e = idx - t * n;
  const float v = values[t * ld + e];
  const float tgt = targets[t * ld + e];
  const float err = tgt - v;
  float dval = -err;
  if (L.use_clipped_value_loss) {
    const float vo = old_values[t * ld + e];
    const float dv = v - vo;
    const float errc = tgt - (vo + fminf(fmaxf(dv, -L.clip_param), L.clip_param));
    if (fabsf(dv) > L.clip_param) dval = (err * err > errc * errc) ? -err : 0.0f;
  }
  float* d = dout + idx * 64;
  d[0] = L.value_loss_coef * dval / (float(T) * float(n));
#pragma unroll
  for (int j = 1; j < 64; ++j) d[j] = 0.0f;
}

// Critic head: value_t = out[t][e][0]; dout[.][0] = d loss / d value (clipped value loss), other columns zero.
__global__ void __launch_bounds__(kT)
critic_head_fwd_bwd_kernel(kbs_ppo_loss_params L, const float* __restrict__ out, const float* __restrict__ old_values,
                           const float* __restrict__ targets, float* __restrict__ values, float* __restrict__ dout, int64_t T,
                           int64_t ld, int64_t n) {
  const int64_t idx = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (idx >= T * n) return;
  const int64_t t = idx / n, e = idx - t * n;
  const float v = out[idx * 64];
  values[t * ld + e] = v;
  const float tgt = targets[t * ld + e];
  const float err = tgt - v;
  float dval = -err;                                        // d (0.5 err^2) / d v
  if (L.use_clipped_value_loss) {
    const float vo = old_values[t * ld + e];
    const float dv = v - vo;
    const float errc = tgt - (vo + fminf(fmaxf(dv, -L.clip_param), L.clip_param));
    if (fabsf(dv) > L.clip_param) dval = (err * err > errc * errc) ? -err : 0.0f;   // the clipped branch has no gradient
  }
  float* d = dout + idx * 64;
  d[0] = L.value_loss_coef * dval / (float(T) * float(n));
#pragma unroll
  for (int j = 1; j < 64; ++j) d[j] = 0.0f;
}

// Critic head of the persistent update in one pass: value = w_out . h_top + b_out (the output layer has ONE row: a GEMV, not
// the padded 64-column GEMM), the clipped value loss' gradient, dout row (column 0 = d loss / d value: the A operand of the
// dW_out GEMM) and dv [T * n] -- the backward kernel forms dh_top = dv w_out itself (rank 1), so neither `out` nor `dh_top` of
// the critic exist.  One warp per (t, env) row.
__global__ void __launch_bounds__(256)
critic_value_head_kernel(kbs_ppo_loss_params L, const float* __restrict__ h_top, const float* __restrict__ w_out,
                         const float* __restrict__ b_out, const float* __restrict__ old_values, const float* __restrict__ targets,
                         float* __restrict__ values, float* __restrict__ dout, float* __restrict__ dv, int H, int64_t T, int64_t ld,
                         int64_t n) {
  const int64_t idx = int64_t(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (idx >= T * n) return;
  const int lane = threadIdx.x & 31;
  const float* hr = h_top + idx * H;
  float acc = 0.0f;
  for (int c = lane * 4; c < H; c += 128) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(hr + c)), w = __ldg(reinterpret_cast<const float4*>(w_out + c));
    acc = fmaf(a.x, w.x, acc); acc = fmaf(a.y, w.y, acc); acc = fmaf(a.z, w.z, acc); acc = fmaf(a.w, w.w, acc);
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
  const int64_t t = idx / n, e = idx - t * n;
  const float v = acc + b_out[0];
  float dval = 0.0f;
  if (lane == 0) {
    values[t * ld + e] = v;
    const float tgt = targets[t * ld + e];
    const float err = tgt - v;
    dval = -err;                                              // d (0.5 err^2) / d v
    if (L.use_clipped_value_loss) {
      const float vo = old_values[t * ld + e];
      const float d = v - vo;
      const float errc = tgt - (vo + fminf(fmaxf(d, -L.clip_param), L.clip_param));
      if (fabsf(d) > L.clip_param) dval = (err * err > errc * errc) ? -err : 0.0f;   // the clipped branch has no gradient
    }
    dval = L.value_loss_coef * dval / (float(T) * float(n));
    dv[idx] = dval;
  }
  reinterpret_cast<float2*>(dout + idx * 64)[lane] = make_float2(dval, 0.0f);       // lanes > 0 hold 0
}

__global__ void __launch_bounds__(kT)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t count,
            float lr, float b1, float b2, float eps, float grad_scale, float bc1, float bc2) {
  const int64_t i = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (i >= count) return;
  const float gi = g[i] * grad_scale;
  const float mi = b1 * m[i] + (1.0f - b1) * gi;
  const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
  m[i] = mi; v[i] = vi;
  p[i] = p[i] - lr * (mi / bc1) / (sqrtf(vi / bc2) + eps);       // optax.scale_by_adam (eps_root = 0) then -lr
}

// optax.adamw (train.py:1064-1065) with ksim's gradient clipping folded in [U]: see kbs_adamw_step in kbotstep.h.
// norm / step_dev may be nullptr.  Every thread derives the same clip factor and bias corrections from the same device
// words, so the update is a pure elementwise map (bitwise identical on every rank).
__global__ void __launch_bounds__(kT)
adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t count,
             const kbs_adamw_params o, const float* __restrict__ norm, const long long* __restrict__ step_dev, long long step) {
  const int64_t i = int64_t(blockIdx.x) * kT + threadIdx.x;
  if (i >= count) return;
  float scale = o.grad_scale;
  if (norm) {
    const float nn = norm[0] * o.grad_scale;                     // norm of the gradient the optimiser sees
    if (!(fabsf(nn) <= 3.0e38f)) return;                         // NaN / inf: ksim skips the update, optimiser state untouched
    if (o.max_grad_norm > 0.0f && nn > o.max_grad_norm) scale = scale * (o.max_grad_norm / fmaxf(nn, 1e-6f));
  }
  const float s = float(step_dev ? step_dev[0] + 1 : step);
  // optax.scale_by_adam: decay and (1 - decay) are Python doubles rounded to fp32 separately; bias correction 1 - decay^count in fp32
  const float b1 = float(o.b1), b2 = float(o.b2), omb1 = float(1.0 - o.b1), omb2 = float(1.0 - o.b2);
  const float bc1 = 1.0f - powf(b1, s), bc2 = 1.0f - powf(b2, s);
  const float gi = g[i] * scale;
  const float mi = b1 * m[i] + omb1 * gi;
  const float vi = b2 * v[i] + omb2 * (gi * gi);
  m[i] = mi; v[i] = vi;
  const float pi = p[i];
  p[i] = pi - o.lr * ((mi / bc1) / (sqrtf(vi / bc2) + o.eps) + o.weight_decay * pi);
}
__global__ void step_advance_kernel(long long* step_dev, const float* __restrict__ norm, float grad_scale) {
  if (norm && !(fabsf(norm[0] * grad_scale) <= 3.0e38f)) return;
  step_dev[0] = step_dev[0] + 1;
}

// sum of squares in double, fixed shape: kNormBlocks blocks x kT threads, grid-stride, fixed-order tree per block, then
// one block adds the kNormBlocks partials in order
constexpr int kNormBlocks = 296;
__global__ void __launch_bounds__(kT)
sumsq_partial_kernel(const float* __restrict__ g, int64_t count, double* __restrict__ partial) {
  __shared__ double sh[kT];
  double a = 0.0;
  for (int64_t i = int64_t(blockIdx.x) * kT + threadIdx.x; i < count; i += int64_t(kNormBlocks) * kT) {
    const double x = double(g[i]);
    a += x * x;
  }
  sh[threadIdx.x] = a;
  __syncthreads();
  for (int s = kT / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}
__global__ void __launch_bounds__(kT)
sumsq_final_kernel(const double* __restrict__ partial, float* __restrict__ norm_out) {
  __shared__ double sh[kT];
  double a = 0.0;
  for (int i = threadIdx.x; i < kNormBlocks; i += kT) a += partial[i];
  sh[threadIdx.x] = a;
  __syncthreads();
  for (int s = kT / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) norm_out[0] = float(sqrt(sh[0]));
}

unsigned blocks(int64_t n) { return unsigned((n + kT - 1) / kT); }

struct NetWork {      // per-net workspace (floats), carved from the handle's scratch
  float* obs_rm; float* x0; float* out; float* dout; float* dh_top;
  float* dxh0;                           // [T*n][2H]: layer 0's (dx | dh_rec) of every step (dx feeds dW_in)
  float* dxh[KBS_MAX_DEPTH];             // [n][2H] per layer >= 1: (dx for the layer below | dh_rec for step t - 1)
  float* ga[KBS_MAX_DEPTH]; float* cs[KBS_MAX_DEPTH]; float* hs[KBS_MAX_DEPTH]; float* h_in[KBS_MAX_DEPTH]; float* c_in[KBS_MAX_DEPTH];
  float* dG[KBS_MAX_DEPTH];
  float* w_ihT[KBS_MAX_DEPTH]; float* w_hhT[KBS_MAX_DEPTH]; float* w_outT;
  // tensor-core path: the same activations as split-blocked MMA operands ([T] x per-step buffers)
  char* x0_sb; char* hs_sb[KBS_MAX_DEPTH]; char* h_in_sb[KBS_MAX_DEPTH]; char* dG_sb;
  // weight-gradient GEMMs on the tensor cores: transposed split-blocked operands (K = all T x n rows), split-K slabs
  char* tn_a; char* tn_b; float* tn_partial; float* tn_zero; char* tn_ones;
};

template <int KIND>
int run_net_k(kbs_handle* h, int net, const kbs_ppo_batch& b, const float* carry0, NetWork& w, float* gates_pre, float* dc_rec,
              float* part, int splits, int64_t n, cudaStream_t st, bool backward, const kbs_net_grads* g, bool tc) {
  const KbsNet& N = h->net[net];
  const int H = h->p.hidden_size, depth = h->p.depth;
  const int64_t T = b.T, ld = b.ld, rows = T * n;
  const int kp = round_up_i(N.num_in, 64);
  const size_t sH = size_t(n) * H;
  const size_t sbH = tc ? kbs_tc_rows_sb_bytes(h, n, H) : 0;
  int rc;
  if (!backward) {
    const float* obs = net == KBS_NET_ACTOR ? b.actor_obs : b.critic_obs;
    KBS_LAUNCH(h, KBS_K_PACK, st, (soa_to_rows_kernel<<<blocks(rows * kp), kT, 0, st>>>(obs, N.num_in, ld, w.obs_rm, kp, n, T)));
    if ((rc = kbs_simt_gemm_nt(h, w.obs_rm, kp, N.w_in, N.kin_pad, N.b_in, w.x0, H, rows, H, N.kin_pad, 0, st))) return rc;
    if (tc)
      KBS_LAUNCH(h, KBS_K_PACK, st, (rows_to_sb_kernel<KIND><<<blocks(rows * (H / 8)), kT, 0, st>>>(w.x0, w.x0_sb, sbH, H, n, T)));
    for (int l = 0; l < depth; ++l) {       // carries the first step reads: ABI layout [depth][2][n][H] or zeros
      if (carry0) {
        KBS_CUDA_TRY(cudaMemcpyAsync(w.h_in[l], carry0 + (size_t(l) * 2 + 0) * sH, sH * 4, cudaMemcpyDeviceToDevice, st));
        KBS_CUDA_TRY(cudaMemcpyAsync(w.c_in[l], carry0 + (size_t(l) * 2 + 1) * sH, sH * 4, cudaMemcpyDeviceToDevice, st));
      } else {
        KBS_CUDA_TRY(cudaMemsetAsync(w.h_in[l], 0, sH * 4, st));
        KBS_CUDA_TRY(cudaMemsetAsync(w.c_in[l], 0, sH * 4, st));
      }
      if (tc)
        KBS_LAUNCH(h, KBS_K_PACK, st, (rows_to_sb_kernel<KIND><<<blocks(n * (H / 8)), kT, 0, st>>>(w.h_in[l], w.h_in_sb[l], sbH, H, n, 1)));
    }
    for (int64_t t = 0; t < T; ++t) {
      for (int l = 0; l < depth; ++l) {
        const bool last = t + 1 == T;
        float* hn = last ? nullptr : w.h_in[l] + size_t(t + 1) * sH;
        float* cn = last ? nullptr : w.c_in[l] + size_t(t + 1) * sH;
        if (tc) {
          const char* x_sb = (l == 0 ? w.x0_sb : w.hs_sb[l - 1]) + size_t(t) * sbH;
          if ((rc = kbs_tc_gates_fwd(h, net, l, x_sb, w.h_in_sb[l] + size_t(t) * sbH, gates_pre, n, st))) return rc;
          KBS_LAUNCH(h, KBS_K_LSTM_CELL, st,
                     (cell_fwd_save8_kernel<KIND><<<blocks(n * (H / 8)), kT, 0, st>>>(
                         gates_pre, w.c_in[l] + size_t(t) * sH, w.ga[l] + size_t(t) * sH * 4, w.cs[l] + size_t(t) * sH,
                         w.hs[l] + size_t(t) * sH, hn, cn, w.hs_sb[l] + size_t(t) * sbH,
                         last ? nullptr : w.h_in_sb[l] + size_t(t + 1) * sbH, b.done + t * ld, H, n)));
        } else {
          const float* x_in = (l == 0 ? w.x0 : w.hs[l - 1]) + size_t(t) * sH;
          if ((rc = kbs_simt_gemm_nt(h, x_in, H, N.w_ih[l], H, N.b[l], gates_pre, 4 * H, n, 4 * H, H, 0, st))) return rc;
          if ((rc = kbs_simt_gemm_nt(h, w.h_in[l] + size_t(t) * sH, H, N.w_hh[l], H, nullptr, gates_pre, 4 * H, n, 4 * H, H, 1, st)))
            return rc;
          KBS_LAUNCH(h, KBS_K_LSTM_CELL, st,
                     (cell_fwd_save_kernel<<<blocks(n * H), kT, 0, st>>>(
                         gates_pre, w.c_in[l] + size_t(t) * sH, w.ga[l] + size_t(t) * sH * 4, w.cs[l] + size_t(t) * sH,
                         w.hs[l] + size_t(t) * sH, hn, cn, b.done + t * ld, H, n)));
        }
      }
    }
    if ((rc = kbs_simt_gemm_nt(h, w.hs[depth - 1], H, N.w_out, H, N.b_out, w.out, 64, rows, 64, H, 0, st))) return rc;
    KBS_LAUNCH_CHECK();
    return KBS_OK;
  }
  // ---- backward: w.dout [rows][64] holds d loss / d out ----
  if (tc) {
    if ((rc = kbs_tc_pack_bwd(h, net, st))) return rc;
  } else {
    for (int l = 0; l < depth; ++l) {
      KBS_LAUNCH(h, KBS_K_PACK, st, (transpose_kernel<<<blocks(int64_t(4) * H * H), kT, 0, st>>>(N.w_ih[l], 4 * H, H, w.w_ihT[l])));
      KBS_LAUNCH(h, KBS_K_PACK, st, (transpose_kernel<<<blocks(int64_t(4) * H * H), kT, 0, st>>>(N.w_hh[l], 4 * H, H, w.w_hhT[l])));
    }
  }
  KBS_LAUNCH(h, KBS_K_PACK, st, (transpose_kernel<<<blocks(int64_t(64) * H), kT, 0, st>>>(N.w_out, 64, H, w.w_outT)));
  if ((rc = kbs_simt_gemm_nt(h, w.dout, 64, w.w_outT, 64, nullptr, w.dh_top, H, rows, H, 64, 0, st))) return rc;
  for (int l = 0; l < depth; ++l) KBS_CUDA_TRY(cudaMemsetAsync(dc_rec + size_t(l) * sH, 0, sH * 4, st));
  // the loss is a mean over T n transitions: per-sample gradients are O(1e-2..1), dG = that / (T n).  Scale dG back up by
  // the next power of two of T n (x 16) before the FP16 split; exact, undone by the GEMM's output scale.
  float gscale = 16.0f;
  while (gscale < 16.0f * float(rows)) gscale *= 2.0f;
  for (int64_t t = T - 1; t >= 0; --t) {
    for (int l = depth - 1; l >= 0; --l) {
      // gradient wrt h_t from above: the head (top layer) or the dx half of the layer above at this step
      const float* dh_in = (l == depth - 1) ? w.dh_top + size_t(t) * sH : w.dxh[l + 1];
      const int ld_in = (l == depth - 1) ? H : 2 * H;
      // gradient wrt the carry h that step t + 1 read: the dh half of this layer's own GEMM at step t + 1
      float* dxh_next = (l == 0) ? w.dxh0 + size_t(t + 1) * sH * 2 : w.dxh[l];
      const float* dh_rec = (t + 1 < T) ? dxh_next + H : nullptr;
      float* dG = w.dG[l] + size_t(t) * sH * 4;
      float* dxh_out = (l == 0) ? w.dxh0 + size_t(t) * sH * 2 : w.dxh[l];
      if (tc) {
        KBS_LAUNCH(h, KBS_K_LSTM_CELL, st,
                   (cell_bwd8_kernel<KIND><<<blocks(n * (H / 8)), kT, 0, st>>>(dh_in, ld_in, dh_rec, 2 * H, dc_rec + size_t(l) * sH,
                                                                              w.ga[l] + size_t(t) * sH * 4, w.cs[l] + size_t(t) * sH,
                                                                              w.c_in[l] + size_t(t) * sH, b.done + t * ld, dG,
                                                                              w.dG_sb, gscale, H, n)));
        if ((rc = kbs_tc_bwd_gemm(h, net, l, w.dG_sb, dxh_out, n, 1.0f / gscale, st))) return rc;
      } else {
        KBS_LAUNCH(h, KBS_K_LSTM_CELL, st,
                   (cell_bwd8_kernel<KIND><<<blocks(n * (H / 8)), kT, 0, st>>>(dh_in, ld_in, dh_rec, 2 * H, dc_rec + size_t(l) * sH,
                                                                              w.ga[l] + size_t(t) * sH * 4, w.cs[l] + size_t(t) * sH,
                                                                              w.c_in[l] + size_t(t) * sH, b.done + t * ld, dG,
                                                                              nullptr, 1.0f, H, n)));
        if ((rc = kbs_simt_gemm_nt(h, dG, 4 * H, w.w_ihT[l], 4 * H, nullptr, dxh_out, 2 * H, n, H, 4 * H, 0, st))) return rc;
        if (t > 0 && (rc = kbs_simt_gemm_nt(h, dG, 4 * H, w.w_hhT[l], 4 * H, nullptr, dxh_out + H, 2 * H, n, H, 4 * H, 0, st)))
          return rc;
      }
    }
  }
  if (tc && (4 * H) % 128 == 0 && H % 128 == 0) {
    // ---- weight gradients on the tensor cores: dW = dG^T [x | h] etc. as split-K tcgen05 GEMMs over all T x n rows ----
    // Both operands are re-packed with K = row index (pack_tn_kernel); dG-like operands are pre-scaled by the same power of
    // two as in the recurrent GEMMs and the GEMM's output scale undoes it; every slab covers <= 3 200 rows and the slabs are
    // added in a fixed order (tn_reduce_kernel): deterministic.  Bias gradients come out of the same GEMM through a tile of
    // ones (column sum of dG).
    const KbsTnPlan plan = kbs_tc_tn_plan(h, rows);
    const float inv = 1.0f / gscale;
    KBS_CUDA_TRY(cudaMemsetAsync(w.tn_zero, 0, 1024 * sizeof(float), st));
    if ((rc = kbs_tc_ones_block(h, w.tn_ones, st))) return rc;
    for (int l = 0; l < depth; ++l) {
      const float* x_l = l == 0 ? w.x0 : w.hs[l - 1];
      const int mp = 4 * H / 128, ldc = (2 * H / 128 + 1) * 128;
      if ((rc = kbs_tc_pack_tn(h, plan, false, w.dG[l], 4 * H, 0, 4 * H, 4 * H, rows, w.tn_a, gscale, -1, st))) return rc;
      if ((rc = kbs_tc_pack_tn(h, plan, true, x_l, H, 0, H, H, rows, w.tn_b, 1.0f, -1, st))) return rc;
      if ((rc = kbs_tc_pack_tn(h, plan, true, w.h_in[l], H, 0, H, H, rows, w.tn_b + size_t(H / 128) * plan.col_bytes, 1.0f, -1, st)))
        return rc;
      if ((rc = kbs_tc_gemm_tn(h, plan, w.tn_a, mp, 4 * H, w.tn_b, 2 * H / 128, w.tn_ones, w.tn_zero, w.tn_partial, inv, st))) return rc;
      if ((rc = kbs_tc_tn_reduce(h, plan, w.tn_partial, mp, ldc, 0, 4 * H, H, g->w_ih[l], H, st))) return rc;
      if ((rc = kbs_tc_tn_reduce(h, plan, w.tn_partial, mp, ldc, H, 4 * H, H, g->w_hh[l], H, st))) return rc;
      if ((rc = kbs_tc_tn_reduce(h, plan, w.tn_partial, mp, ldc, 2 * H, 4 * H, 1, g->b[l], 1, st))) return rc;
    }
    {   // dW_in [H][num_in], db_in [H]: A = dx of layer 0, B = the observation rows with a ones column behind the last feature
      const int kpp = round_up_i(N.num_in + 1, 128), mp = H / 128;
      if ((rc = kbs_tc_pack_tn(h, plan, false, w.dxh0, 2 * H, 0, H, H, rows, w.tn_a, gscale, -1, st))) return rc;
      if ((rc = kbs_tc_pack_tn(h, plan, true, w.obs_rm, kp, 0, N.num_in, kpp, rows, w.tn_b, 1.0f, N.num_in, st))) return rc;
      if ((rc = kbs_tc_gemm_tn(h, plan, w.tn_a, mp, H, w.tn_b, kpp / 128, nullptr, w.tn_zero, w.tn_partial, inv, st))) return rc;
      if ((rc = kbs_tc_tn_reduce(h, plan, w.tn_partial, mp, kpp, 0, H, N.num_in, g->w_in, N.num_in, st))) return rc;
      if ((rc = kbs_tc_tn_reduce(h, plan, w.tn_partial, mp, kpp, N.num_in, H, 1, g->b_in, 1, st))) return rc;
    }
    {   // dW_out [num_out][H], db_out: A = d loss / d out (64 columns, rows >= num_out zero), B = top-layer output + ones tile
      const int ldc = (H / 128 + 1) * 128;
      if ((rc = kbs_tc_pack_tn(h, plan, false, w.dout, 64, 0, 64, 128, rows, w.tn_a, gscale, -1, st))) return rc;
      if ((rc = kbs_tc_pack_tn(h, plan, true, w.hs[depth - 1], H, 0, H, H, rows, w.tn_b, 1.0f, -1, st))) return rc;
      if ((rc = kbs_tc_gemm_tn(h, plan, w.tn_a, 1, N.num_out, w.tn_b, H / 128, w.tn_ones, w.tn_zero, w.tn_partial, inv, st))) return rc;
      if ((rc = kbs_tc_tn_reduce(h, plan, w.tn_partial, 1, ldc, 0, N.num_out, H, g->w_out, H, st))) return rc;
      if ((rc = kbs_tc_tn_reduce(h, plan, w.tn_partial, 1, ldc, H, N.num_out, 1, g->b_out, 1, st))) return rc;
    }
    KBS_LAUNCH_CHECK();
    return KBS_OK;
  }
  // weight gradients: sums over all (t, env) rows
  const int chunks = int((rows + 511) / 512);
  auto colsum = [&](const float* X, int ldx, int cols, float* out) {
    KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st, (colsum_partial_kernel<<<dim3(blocks(cols), chunks), kT, 0, st>>>(X, ldx, rows, cols, 512, part)));
    KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st, (reduce_rows_kernel<<<blocks(cols), kT, 0, st>>>(part, chunks, cols, out)));
  };
  float* part2 = part + size_t(chunks) * 4 * H;          // split-K partials of gemm_tn behind the column-sum partials
  for (int l = 0; l < depth; ++l) {
    const float* x_l = l == 0 ? w.x0 : w.hs[l - 1];
    if ((rc = kbs_simt_gemm_tn(h, w.dG[l], 4 * H, x_l, H, g->w_ih[l], H, 4 * H, H, rows, part2, splits, st))) return rc;
    if ((rc = kbs_simt_gemm_tn(h, w.dG[l], 4 * H, w.h_in[l], H, g->w_hh[l], H, 4 * H, H, rows, part2, splits, st))) return rc;
    colsum(w.dG[l], 4 * H, 4 * H, g->b[l]);
  }
  {
    // dW_in [H][kp] -> caller's dense [H][num_in]; dW_out [64][H] -> first num_out rows
    float* tmp = part2 + size_t(splits) * size_t(4 * H) * size_t(kp > H ? kp : H);
    if ((rc = kbs_simt_gemm_tn(h, w.dxh0, 2 * H, w.obs_rm, kp, tmp, kp, H, kp, rows, part2, splits, st))) return rc;
    KBS_LAUNCH(h, KBS_K_PACK, st, (copy_block_kernel<<<blocks(int64_t(H) * N.num_in), kT, 0, st>>>(tmp, kp, g->w_in, H, N.num_in)));
    colsum(w.dxh0, 2 * H, H, g->b_in);
    if ((rc = kbs_simt_gemm_tn(h, w.dout, 64, w.hs[depth - 1], H, tmp, H, 64, H, rows, part2, splits, st))) return rc;
    KBS_LAUNCH(h, KBS_K_PACK, st, (copy_block_kernel<<<blocks(int64_t(N.num_out) * H), kT, 0, st>>>(tmp, H, g->w_out, N.num_out, H)));
    float* bsum = tmp + size_t(64) * H;
    colsum(w.dout, 64, 64, bsum);
    KBS_CUDA_TRY(cudaMemcpyAsync(g->b_out, bsum, size_t(N.num_out) * 4, cudaMemcpyDeviceToDevice, st));
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int run_net(kbs_handle* h, int net, const kbs_ppo_batch& b, const float* carry0, NetWork& w, float* gates_pre, float* dc_rec,
            float* part, int splits, int64_t n, cudaStream_t st, bool backward, const kbs_net_grads* g) {
  const bool tc = h->p.gemm_path != KBS_GEMM_SIMT_FP32 && h->net[net].tc_image != nullptr && (h->p.hidden_size % 64) == 0;
  if (tc && kbs_tc_kind_of(h) == KBS_KIND_TF32)
    return run_net_k<KBS_KIND_TF32>(h, net, b, carry0, w, gates_pre, dc_rec, part, splits, n, st, backward, g, true);
  return run_net_k<KBS_KIND_F16>(h, net, b, carry0, w, gates_pre, dc_rec, part, splits, n, st, backward, g, tc);
}

// ---- the persistent form of kbs_ppo_grad (FP16-split datapath) ---------------------------------------------------------
// main stream: input projections (tensor core, straight from the SoA observations) -> lstm_fwd_save_kernel (ALL T steps of both
// networks' LSTM stacks, one launch; keeps operands, cell states, activated gates) -> heads (actor: FFMA GEMM + one warp per env
// through the Gaussian / low-pass filter forward and backward; critic: GEMV + value-loss gradient) -> dh_top (actor: FFMA GEMM;
// critic: rank 1, inside the backward kernel) -> bptt_persist_kernel (the whole backward recurrence of both networks, one
// launch) -> weight gradients: the four layer GEMMs read dG / x / h_in in place (dw_gemm_kernel), the input / output layers'
// through K = row re-packed operands (split-K lstm_layer_tc_kernel) -> fixed-order reductions -> loss statistics.
// side stream: whatever does not depend on the forward pass (observation re-pack, backward weight tiles, zeroed state), then the
// re-packs of what it produced, then the critic's whole weight-gradient chain beside the actor's.
// (KBS_PPO_FWD_WIDE=1: rollout_persist_kernel<SAVE> as the forward kernel; ragged n or H != 256: the layer GEMMs fall back to
// re-packed operands, transposed on the fly by the recurrence kernels.)
struct PersistWork {
  char* x_sb; char* xmid; char* hsb; float* c_hist; float* save_g; char* dG; float* dx; char* dx0; float* dc;
  float* dh_top; float* dout; float* w_outT; unsigned int* bflags;
  float* h_top_rm; float* out; unsigned int* fflags;      // narrow-tile forward: top-layer outputs, head GEMM output, counters
  char* tn_a; float* tn_partial; float* tn_zero; char* tn_ones;
  // B operands (forward-pass products) are transposed on the side stream while the backward kernel runs: one buffer each
  char* tnb_layer[KBS_MAX_DEPTH];   // [x_l | h_in_l]: 2 H / 128 tiles
  char* tnb_top;                    // top layer's outputs: H / 128 tiles
  char* tnb_obs;                    // observations + ones column: kpp / 128 tiles
  char* tna_dG[KBS_MAX_DEPTH];      // A operands: dG of each layer re-packed (by the backward kernel's transposer CTAs): 4 H / 128 panels
};

int ppo_grad_persistent(kbs_handle* h, const kbs_ppo_loss_params& L, const kbs_ppo_batch& b, const kbs_net_grads* const* grads,
                        float* log_probs, float* values, float* entropy, float* stats_out, int64_t n, cudaStream_t st) {
  const int H = h->p.hidden_size, depth = h->p.depth;
  const int64_t T = b.T, ld = b.ld, rows = T * n, np = (n + 127) / 128 * 128;
  const size_t npH = size_t(np) * H;
  const size_t sbb = kbs_tc_rows_sb_bytes(h, n, H), sb4 = kbs_tc_rows_sb_bytes(h, n, 4 * H);
  const KbsTnPlan plan = kbs_tc_tn_plan(h, T * np);
  KbsTcRolloutWs rws;
  float* osb[2]; float *y_s, *sd_s, *sraw_s, *lpf;
  double* loss_part;
  PersistWork w[2];
  int rc = kbs_scratch(h, [&](KbsScratch& s) {
    rws = kbs_tc_rollout_ws(s, h, n, 2);
    for (int k = 0; k < 2; ++k) osb[k] = s.take<float>(kbs_tc_obs_sb_floats(h, k, n, T));
    y_s = s.take<float>(size_t(T) * KBS_NUM_JOINTS * ld);
    sd_s = s.take<float>(size_t(T) * KBS_NUM_JOINTS * ld);
    sraw_s = s.take<float>(size_t(T) * KBS_NUM_JOINTS * ld);
    lpf = s.take<float>(size_t(KBS_NUM_JOINTS) * ld);
    loss_part = s.take<double>(4096);
    for (int k = 0; k < 2; ++k) {
      const size_t kpp = size_t(round_up_i(h->net[k].num_in + 1, 128));
      const size_t m_panels = size_t(4 * H / 128), b_tiles = (kpp > size_t(2 * H) ? kpp : size_t(2 * H)) / 128 + 1;
      w[k].x_sb = s.take<char>(size_t(T) * sbb);
      w[k].xmid = s.take<char>(size_t(depth) * T * sbb);
      w[k].hsb = s.take<char>(size_t(depth) * (T + 1) * sbb);
      w[k].c_hist = s.take<float>(size_t(depth) * (T + 1) * npH);
      w[k].save_g = s.take<float>(size_t(T) * depth * 4 * npH);
      w[k].dG = s.take<char>(size_t(depth) * (T + 1) * sb4);
      w[k].dx = s.take<float>(size_t(depth) * T * npH);
      w[k].dx0 = s.take<char>(size_t(T) * sbb);
      w[k].dc = s.take<float>(size_t(depth) * npH);
      w[k].dh_top = s.take<float>(size_t(rows) * H);
      w[k].dout = s.take<float>(size_t(rows) * 64);
      w[k].w_outT = s.take<float>(size_t(64) * H);
      w[k].bflags = s.take<unsigned int>(kbs_tc_bptt_flag_bytes(h, n) / 4);
      w[k].h_top_rm = s.take<float>(size_t(rows) * H);
      w[k].out = s.take<float>(size_t(rows) * 64);
      w[k].fflags = s.take<unsigned int>(kbs_tc_fwd_save_flag_bytes(h, n) / 4);
      w[k].tn_a = s.take<char>(m_panels * plan.col_bytes);
      w[k].tn_partial = s.take<float>(size_t(plan.ksplit) * m_panels * 128 * (b_tiles * 128));
      w[k].tn_zero = s.take<float>(1024);
      w[k].tn_ones = s.take<char>(4096 * sizeof(float));
      for (int l = 0; l < depth; ++l) w[k].tnb_layer[l] = s.take<char>(size_t(2 * H / 128) * plan.col_bytes);
      w[k].tnb_top = s.take<char>(size_t(H / 128) * plan.col_bytes);
      w[k].tnb_obs = s.take<char>(kpp / 128 * plan.col_bytes);
      for (int l = 0; l < depth; ++l) w[k].tna_dG[l] = s.take<char>(size_t(4 * H / 128) * plan.col_bytes);
    }
  });
  if (rc) return rc;
  // ---- forward ----
  // narrow-tile kernel (lstm_fwd_save_kernel: LSTM stacks only, heads as a batched GEMM + per-env scan afterwards) unless
  // KBS_PPO_FWD_WIDE=1 asks for rollout_persist_kernel<SAVE> (128 x 256 tiles, heads fused: the first version, kept for A/B)
  static int wide_cfg = -1;
  if (wide_cfg < 0) { const char* e = getenv("KBS_PPO_FWD_WIDE"); wide_cfg = e ? atoi(e) : 0; }
  const bool narrow = !wide_cfg && kbs_tc_fwd_save_available(h, n, T);
  // the four layer GEMMs read dG / x / h_in in place (dw_gemm_kernel) when the shapes allow: nothing is re-packed for them
  const bool dw_direct = kbs_tc_dw_direct_available(h, n);
  bool xh_transposed = false;
  const int kbH = H / 32, kb4 = 4 * H / 32;
  const int64_t kb_used = (T * np + 31) / 32;
  // ---- side stream: everything that does not depend on this call's forward pass runs beside it (the two persistent kernels
  // occupy one SM per work item of a slot -- 128 of 148 at 512 trajectories -- and the ~20 small launches below would
  // otherwise sit between them on the critical path): the observations re-packed with K = row (B operand of the dW_in GEMM),
  // W_out^T, the backward kernel's weight tiles, its zeroed carries / counters / dG(l, T), the K padding of the re-packed
  // operands.  KBS_PPO_SIDE_PACK=0 keeps one stream (A/B).
  { const int rc0 = kbs_side_stream_init(h); if (rc0) return rc0; }
  int side_pack = 1;          // read per call: a profiling pass can ask for one stream (serial per-kernel times)
  { const char* e = getenv("KBS_PPO_SIDE_PACK"); if (e) side_pack = atoi(e); }
  cudaStream_t ss = side_pack ? h->side_stream : st;
  if (side_pack) {
    KBS_CUDA_TRY(cudaEventRecord(h->ev_pre, st));
    KBS_CUDA_TRY(cudaStreamWaitEvent(ss, h->ev_pre, 0));
  }
  float gscale = 16.0f;
  while (gscale < 16.0f * float(rows)) gscale *= 2.0f;
  const bool rank1_critic = narrow && h->net[1].num_out == 1;      // the critic's output layer is one row: GEMV + rank-1 dh_top
  for (int k = 1; k >= 0; --k) {
    const KbsNet& N = h->net[k];
    const int kpp = round_up_i(N.num_in + 1, 128);
    if ((rc = kbs_tc_soa_to_tn(h, plan, k == 0 ? b.actor_obs : b.critic_obs, N.num_in, ld, n, T, kpp, true, w[k].tnb_obs, ss))) return rc;
    if (!(k == 1 && rank1_critic))
      KBS_LAUNCH(h, KBS_K_PACK, ss, (transpose_kernel<<<blocks(int64_t(64) * H), kT, 0, ss>>>(N.w_out, 64, H, w[k].w_outT)));
    if ((rc = kbs_tc_pack_bwd(h, k, ss, kbs_tc_bptt_tile(h, n)))) return rc;
    KBS_CUDA_TRY(cudaMemsetAsync(w[k].dc, 0, size_t(depth) * npH * 4, ss));
    KBS_CUDA_TRY(cudaMemsetAsync(w[k].bflags, 0, kbs_tc_bptt_flag_bytes(h, n), ss));
    for (int l = 0; l < depth; ++l)          // dG(l, T) = 0: the operand of the first backward step's recurrent GEMM
      KBS_CUDA_TRY(cudaMemsetAsync(w[k].dG + (size_t(l) * (T + 1) + T) * sb4, 0, sb4, ss));
    if (kb_used < plan.kb_total)               // K padding behind the last stored row of the re-packed dG
      for (int l = 0; l < depth; ++l)
        for (int c = 0; c < 4 * H / 128; ++c)
          KBS_CUDA_TRY(cudaMemsetAsync(w[k].tna_dG[l] + size_t(c) * plan.col_bytes + size_t(kb_used) * 16384, 0,
                                       size_t(plan.kb_total - kb_used) * 16384, ss));
    KBS_CUDA_TRY(cudaMemsetAsync(w[k].tn_zero, 0, 1024 * sizeof(float), ss));
    if ((rc = kbs_tc_ones_block(h, w[k].tn_ones, ss))) return rc;
  }
  if (side_pack) KBS_CUDA_TRY(cudaEventRecord(h->ev_lstm[0], ss));
  {
    const float* obs_soa[2] = {b.actor_obs, b.critic_obs};
    float* xsb[2] = {reinterpret_cast<float*>(w[0].x_sb), reinterpret_cast<float*>(w[1].x_sb)};
    if ((rc = kbs_tc_input_proj_all(h, 2, obs_soa, osb, xsb, ld, n, T, st, nullptr, nullptr, nullptr))) return rc;
  }
  if (narrow) {
    KbsFwdSaveArgs fa{};
    for (int k = 0; k < 2; ++k) {
      KbsFwdSaveNet& F = fa.net[k];
      F.x0 = w[k].x_sb; F.xmid = w[k].xmid; F.hsb = w[k].hsb; F.c_hist = w[k].c_hist; F.save_g = w[k].save_g;
      F.h_top_rm = w[k].h_top_rm; F.flags = w[k].fflags; F.carry0 = k == 0 ? b.actor_carry0 : b.critic_carry0;
      for (int l = 0; l < depth; ++l) F.tn_xh[l] = w[k].tnb_layer[l];
      if (kb_used < plan.kb_total)                 // K padding behind the last stored row
        for (int l = 0; l < depth; ++l)
          for (int c = 0; c < 2 * H / 128; ++c)
            KBS_CUDA_TRY(cudaMemsetAsync(w[k].tnb_layer[l] + size_t(c) * plan.col_bytes + size_t(kb_used) * 16384, 0,
                                         size_t(plan.kb_total - kb_used) * 16384, st));
    }
    fa.nets = 2; fa.n = n; fa.ld = ld; fa.T = T; fa.done = b.done; fa.tn_plan = dw_direct ? nullptr : &plan;
    fa.transposed_out = &xh_transposed;
    if ((rc = kbs_tc_fwd_save(h, fa, st))) return rc;
    // heads: out = W_out h_top + b for all T x n rows, then forward + loss gradient + backward of the head per env
    if ((rc = kbs_simt_gemm_nt(h, w[0].h_top_rm, H, h->net[0].w_out, H, h->net[0].b_out, w[0].out, 64, rows, 64, H, 0, st))) return rc;
    {
      const size_t head_smem = size_t(T) * 32 * 4 * 3 + size_t(T) + 16;
      static int block_head = -1;
      if (block_head < 0) { const char* e = getenv("KBS_PPO_HEAD_BLOCK"); block_head = e ? atoi(e) : 1; }
      if (block_head && head_smem <= 48 * 1024)
        KBS_LAUNCH(h, KBS_K_ACTOR_HEAD, st,
                   (actor_head_fwd_bwd_block_kernel<<<unsigned(n), 128, head_smem, st>>>(
                       h->p, L, w[0].out, b.actor_obs, b.action, b.done, b.lpf0, b.old_log_probs, b.advantages, y_s, sd_s, log_probs,
                       entropy, w[0].dout, T, ld, n)));
      else
        KBS_LAUNCH(h, KBS_K_ACTOR_HEAD, st,
                   (actor_head_fwd_bwd_warp_kernel<<<unsigned((n + 3) / 4), 128, 0, st>>>(
                       h->p, L, w[0].out, b.actor_obs, b.action, b.done, b.lpf0, b.old_log_probs, b.advantages, y_s, sd_s, log_probs,
                       entropy, w[0].dout, T, ld, n)));
    }
    if (rank1_critic) {
      KBS_LAUNCH(h, KBS_K_CRITIC_HEAD, st,
                 (critic_value_head_kernel<<<unsigned((rows + 7) / 8), 256, 0, st>>>(L, w[1].h_top_rm, h->net[1].w_out, h->net[1].b_out,
                                                                                    b.old_values, b.value_targets, values, w[1].dout,
                                                                                    w[1].out /*dv*/, H, T, ld, n)));
    } else {
      if ((rc = kbs_simt_gemm_nt(h, w[1].h_top_rm, H, h->net[1].w_out, H, h->net[1].b_out, w[1].out, 64, rows, 64, H, 0, st))) return rc;
      KBS_LAUNCH(h, KBS_K_CRITIC_HEAD, st,
                 (critic_head_fwd_bwd_kernel<<<blocks(rows), kT, 0, st>>>(L, w[1].out, b.old_values, b.value_targets, values, w[1].dout, T, ld, n)));
    }
  } else {
    KbsTcRolloutArgs r{};
    r.x_sb_all[0] = reinterpret_cast<float*>(w[0].x_sb); r.x_sb_all[1] = reinterpret_cast<float*>(w[1].x_sb);
    r.n = n; r.ld = ld; r.T = T; r.with_critic = true;
    r.carry[0] = const_cast<float*>(b.actor_carry0); r.carry[1] = const_cast<float*>(b.critic_carry0);
    r.done = b.done; r.actor_obs = b.actor_obs;
    // the low-pass state: a private copy of lpf0 (the kernel advances it in place)
    if (b.lpf0) KBS_CUDA_TRY(cudaMemcpyAsync(lpf, b.lpf0, size_t(KBS_NUM_JOINTS) * ld * 4, cudaMemcpyDeviceToDevice, st));
    else KBS_CUDA_TRY(cudaMemsetAsync(lpf, 0, size_t(KBS_NUM_JOINTS) * ld * 4, st));
    r.lpf = lpf;
    r.action_in = b.action; r.log_prob = log_probs; r.entropy = entropy; r.action_std = sd_s; r.mean = y_s; r.value = values;
    r.ws = rws;
    r.save = 1; r.sraw = sraw_s;
    for (int k = 0; k < 2; ++k) { r.xmid_hist[k] = w[k].xmid; r.hsb_hist[k] = w[k].hsb; r.c_hist[k] = w[k].c_hist; r.save_g[k] = w[k].save_g; }
    if ((rc = kbs_tc_rollout_recurrent(h, r, st))) return rc;
    KBS_LAUNCH(h, KBS_K_ACTOR_HEAD, st,
               (actor_head_bwd_warp_kernel<<<unsigned((n + 3) / 4), 128, 0, st>>>(h->p, L, b.action, b.done, b.old_log_probs, b.advantages,
                                                                                 y_s, sd_s, sraw_s, log_probs, w[0].dout, T, ld, n)));
    KBS_LAUNCH(h, KBS_K_CRITIC_HEAD, st,
               (critic_head_bwd_kernel<<<blocks(rows), kT, 0, st>>>(L, values, b.old_values, b.value_targets, w[1].dout, T, ld, n)));
  }
  // ---- side stream, second part: what the forward pass produced and the weight-gradient GEMMs read with K = row (the
  // top layer's outputs; [x | h_in] of every layer unless the forward kernel re-packed them itself), while the backward
  // kernel runs; joined before the GEMMs ----
  if (side_pack) {
    KBS_CUDA_TRY(cudaEventRecord(h->ev_lstm[1], st));
    KBS_CUDA_TRY(cudaStreamWaitEvent(ss, h->ev_lstm[1], 0));
  }
  for (int k = 1; k >= 0; --k) {
    for (int l = 0; l < depth && !xh_transposed && !dw_direct; ++l) {
      const char* x_hist = l == 0 ? w[k].x_sb : w[k].xmid + size_t(l - 1) * T * sbb;
      if ((rc = kbs_tc_sb_to_tn(h, plan, true, x_hist, sbb, kbH, 0, kbH, n, T, w[k].tnb_layer[l], ss))) return rc;
      if ((rc = kbs_tc_sb_to_tn(h, plan, true, w[k].hsb + size_t(l) * (T + 1) * sbb, sbb, kbH, 0, kbH, n, T,
                                w[k].tnb_layer[l] + size_t(H / 128) * plan.col_bytes, ss)))
        return rc;
    }
    if (narrow) {
      if ((rc = kbs_tc_pack_tn(h, plan, true, w[k].h_top_rm, H, 0, H, H, rows, w[k].tnb_top, 1.0f, -1, ss, n, np))) return rc;
    } else if ((rc = kbs_tc_sb_to_tn(h, plan, true, w[k].xmid + size_t(depth - 1) * T * sbb, sbb, kbH, 0, kbH, n, T, w[k].tnb_top, ss))) {
      return rc;
    }
    // A operand of the dW_out GEMM: d loss / d out (row-major, K' = t np + env)
    if ((rc = kbs_tc_pack_tn(h, plan, false, w[k].dout, 64, 0, 64, 128, rows, w[k].tn_a, gscale, -1, ss, n, np))) return rc;
  }
  if (side_pack) KBS_CUDA_TRY(cudaEventRecord(h->ev_head[0], ss));
  // ---- backward recurrence ----
  if (side_pack) KBS_CUDA_TRY(cudaStreamWaitEvent(st, h->ev_lstm[0], 0));        // join: W_out^T, backward weight tiles, zeroed state
  KbsBpttArgs ba{};
  for (int k = 0; k < 2; ++k) {
    KbsBpttNet& B = ba.net[k];
    if (k == 1 && rank1_critic) {
      B.dh_top = nullptr; B.dv = w[1].out; B.w_out = h->net[1].w_out;
    } else {
      if ((rc = kbs_simt_gemm_nt(h, w[k].dout, 64, w[k].w_outT, 64, nullptr, w[k].dh_top, H, rows, H, 64, 0, st))) return rc;
      B.dh_top = w[k].dh_top;
    }
    B.dG = w[k].dG; B.save_g = w[k].save_g; B.c_hist = w[k].c_hist; B.dx = w[k].dx; B.dx0 = w[k].dx0;
    B.dc = w[k].dc; B.flags = w[k].bflags;
    for (int l = 0; l < depth; ++l) B.tn_dG[l] = w[k].tna_dG[l];
  }
  ba.nets = 2; ba.n = n; ba.ld = ld; ba.T = T; ba.done = b.done; ba.gscale = gscale;
  bool dG_transposed = false;
  ba.tn_plan = dw_direct ? nullptr : &plan; ba.transposed_out = &dG_transposed;
  if ((rc = kbs_tc_bptt(h, ba, st))) return rc;
  if (side_pack) KBS_CUDA_TRY(cudaStreamWaitEvent(st, h->ev_head[0], 0));       // join: the B operands are ready
  // ---- weight gradients: the two networks' GEMM chains are independent (own operands, own partial slabs): the critic's
  // runs on the side stream beside the actor's, so the small launches of one (dW_in / dW_out: 32-128 CTAs, the fixed-order
  // reductions) fill the SMs the other leaves idle; the critic's gradients are final first (ppo.py starts its all-reduce) ----
  const float inv = 1.0f / gscale;
  if (side_pack) {
    KBS_CUDA_TRY(cudaEventRecord(h->ev_head[1], st));
    KBS_CUDA_TRY(cudaStreamWaitEvent(ss, h->ev_head[1], 0));
  }
  for (int k = 1; k >= 0; --k) {
    const KbsNet& N = h->net[k];
    const kbs_net_grads* g = grads[k];
    cudaStream_t sk = k == 1 ? ss : st;
    for (int l = 0; l < depth; ++l) {
      const int mp = 4 * H / 128, ldc = (2 * H / 128 + 1) * 128;
      if (dw_direct) {
        const char* x_hist = l == 0 ? w[k].x_sb : w[k].xmid + size_t(l - 1) * T * sbb;
        if ((rc = kbs_tc_dw_direct(h, plan, w[k].dG + size_t(l) * (T + 1) * sb4, x_hist, w[k].hsb + size_t(l) * (T + 1) * sbb, n, T,
                                   w[k].tn_partial, inv, sk)))
          return rc;
      } else {
        if (!dG_transposed &&
            (rc = kbs_tc_sb_to_tn(h, plan, false, w[k].dG + size_t(l) * (T + 1) * sb4, sb4, kb4, 0, kb4, n, T, w[k].tna_dG[l], sk)))
          return rc;
        if ((rc = kbs_tc_gemm_tn(h, plan, w[k].tna_dG[l], mp, 4 * H, w[k].tnb_layer[l], 2 * H / 128, w[k].tn_ones, w[k].tn_zero,
                                 w[k].tn_partial, inv, sk)))
          return rc;
      }
      {
        const int sg3[3][3] = {{0, H, H}, {H, H, H}, {2 * H, 1, 1}};
        float* const dst3[3] = {g->w_ih[l], g->w_hh[l], g->b[l]};
        if ((rc = kbs_tc_tn_reduce_multi(h, plan, w[k].tn_partial, mp, ldc, 4 * H, 3, sg3, dst3, sk))) return rc;
      }
    }
    {   // dW_out, db_out: A = d loss / d out (packed on the side stream above), B = the top layer's outputs + ones tile
      const int ldc = (H / 128 + 1) * 128;
      if ((rc = kbs_tc_gemm_tn(h, plan, w[k].tn_a, 1, N.num_out, w[k].tnb_top, H / 128, w[k].tn_ones, w[k].tn_zero, w[k].tn_partial, inv, sk)))
        return rc;
      const int sg2[2][3] = {{0, H, H}, {H, 1, 1}};
      float* const dst2[2] = {g->w_out, g->b_out};
      if ((rc = kbs_tc_tn_reduce_multi(h, plan, w[k].tn_partial, 1, ldc, N.num_out, 2, sg2, dst2, sk))) return rc;
    }
    {   // dW_in, db_in
      const int kpp = round_up_i(N.num_in + 1, 128), mp = H / 128;
      if ((rc = kbs_tc_sb_to_tn(h, plan, false, w[k].dx0, sbb, kbH, 0, kbH, n, T, w[k].tn_a, sk))) return rc;
      if ((rc = kbs_tc_gemm_tn(h, plan, w[k].tn_a, mp, H, w[k].tnb_obs, kpp / 128, nullptr, w[k].tn_zero, w[k].tn_partial, inv, sk))) return rc;
      const int sg2[2][3] = {{0, N.num_in, N.num_in}, {N.num_in, 1, 1}};
      float* const dst2[2] = {g->w_in, g->b_in};
      if ((rc = kbs_tc_tn_reduce_multi(h, plan, w[k].tn_partial, mp, kpp, H, 2, sg2, dst2, sk))) return rc;
    }
    if (k == 1) {
      if (h->ev_critic_ready) KBS_CUDA_TRY(cudaEventRecord(h->ev_critic_ready, sk));   // the critic's gradients are final
      if (side_pack) KBS_CUDA_TRY(cudaEventRecord(h->ev_chunk[0], ss));
    }
  }
  if (side_pack) KBS_CUDA_TRY(cudaStreamWaitEvent(st, h->ev_chunk[0], 0));        // join: both networks' gradients are final
  {
    kbs_ppo_loss_io io{};
    io.log_probs = log_probs; io.old_log_probs = b.old_log_probs; io.advantages = b.advantages; io.values = values;
    io.old_values = b.old_values; io.value_targets = b.value_targets; io.entropy = entropy; io.out = stats_out;
    io.T = T; io.ld = ld;
    if ((rc = kbs_launch_ppo_loss_at(h, L, io, n, loss_part, st))) return rc;
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// ---- minibatches of the update phase (kbs_minibatch_permutation, kbs_shuffle_minibatches) ------------------------------------

// One CTA: Philox key of every env, bitonic sort of (key << 32) | e over the next power of two (padding = ~0, sorts last)
// in shared memory.  All threads read *pass_dev before the first barrier; thread 0 advances it after.
constexpr int kPermThreads = 1024;
__global__ void __launch_bounds__(kPermThreads)
minibatch_permutation_kernel(uint64_t seed, long long* __restrict__ pass_dev, int64_t env0, int32_t* __restrict__ perm, int n,
                             int np2) {
  extern __shared__ unsigned long long sk[];
  const unsigned long long pass = (unsigned long long)pass_dev[0];
  const uint2 key = make_uint2(uint32_t(seed), uint32_t(seed >> 32));
  for (int e = threadIdx.x; e < np2; e += kPermThreads) {
    unsigned long long v = ~0ull;
    if (e < n) {
      const uint4 x = kbs_philox4x32_10(make_uint4(uint32_t(pass), uint32_t(pass >> 32), uint32_t(env0 + e), 0xFFFFFFFFu), key);
      v = ((unsigned long long)x.x << 32) | unsigned(e);
    }
    sk[e] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) pass_dev[0] = (long long)(pass + 1);
  for (int k = 2; k <= np2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < np2 / 2; i += kPermThreads) {
        const int lo = 2 * i - (i & (j - 1)), hi = lo + j;
        const unsigned long long a = sk[lo], b = sk[hi];
        if ((a > b) == ((lo & k) == 0)) { sk[lo] = b; sk[hi] = a; }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < n; i += kPermThreads) perm[i] = int32_t(uint32_t(sk[i]));
}

// The SoA fields of a rollout, as one list of rows: array a has rows[a] rows ([T][F] flattened) of n values at stride ld in
// src, written as [num_batches][rows][bs] to dst.
struct ShuffleRows {
  const char* src[9];
  char* dst[9];
  int64_t first[10];     // prefix sums of the arrays' row counts
  int esize[9];          // 4 = float, 1 = u8
};
constexpr int kShufThreads = 256;
// one CTA per source row: stage the row's n values in shared memory (coalesced), then write its num_batches contiguous
// bs-wide segments, 4 output columns per thread (bs % 4 == 0: the 4 columns are in one segment)
__global__ void __launch_bounds__(kShufThreads)
shuffle_rows_kernel(const __grid_constant__ ShuffleRows R, const int32_t* __restrict__ perm, int64_t ld, int n, int bs) {
  extern __shared__ float4 srow4[];
  const int64_t g = blockIdx.x;
  int a = 0;
#pragma unroll
  for (int i = 1; i < 9; ++i) a += (g >= R.first[i]) ? 1 : 0;
  const int64_t r = g - R.first[a], rows = R.first[a + 1] - R.first[a];
  const int es = R.esize[a];
  const int n16 = n * es / 16, n4 = n * es / 4;      // row bytes / 16 (float) or / 4 (u8; n % 4 == 0, ld % 4 == 0)
  if (es == 4) {
    const float4* s = reinterpret_cast<const float4*>(R.src[a] + r * ld * 4);
    for (int i = threadIdx.x; i < n16; i += kShufThreads) srow4[i] = __ldcs(s + i);
  } else {
    const uint32_t* s = reinterpret_cast<const uint32_t*>(R.src[a] + r * ld);
    uint32_t* d = reinterpret_cast<uint32_t*>(srow4);
    for (int i = threadIdx.x; i < n4; i += kShufThreads) d[i] = s[i];
  }
  __syncthreads();
  const float* srow = reinterpret_cast<const float*>(srow4);
  const uint8_t* srow_b = reinterpret_cast<const uint8_t*>(srow4);
  for (int k = threadIdx.x * 4; k < n; k += kShufThreads * 4) {
    const int4 p = *reinterpret_cast<const int4*>(perm + k);
    const int idx[4] = {p.x, p.y, p.z, p.w};
    const int b = k / bs, j = k - b * bs;
    const int64_t o = (int64_t(b) * rows + r) * bs + j;
    if (es == 4) {
      float v[4];
#pragma unroll
      for (int l = 0; l < 4; ++l) v[l] = (unsigned(idx[l]) < unsigned(n)) ? srow[idx[l]] : __int_as_float(0x7FC00000);
      *reinterpret_cast<float4*>(R.dst[a] + o * 4) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
      uchar4 v;
      v.x = (unsigned(idx[0]) < unsigned(n)) ? srow_b[idx[0]] : 0;
      v.y = (unsigned(idx[1]) < unsigned(n)) ? srow_b[idx[1]] : 0;
      v.z = (unsigned(idx[2]) < unsigned(n)) ? srow_b[idx[2]] : 0;
      v.w = (unsigned(idx[3]) < unsigned(n)) ? srow_b[idx[3]] : 0;
      *reinterpret_cast<uchar4*>(R.dst[a] + o) = v;
    }
  }
}

// carries [D2][n][H] -> [num_batches][D2][bs][H], one warp per H-float row; blockIdx.y = net
__global__ void __launch_bounds__(kShufThreads)
shuffle_carry_kernel(const float* __restrict__ src0, float* __restrict__ dst0, const float* __restrict__ src1, float* __restrict__ dst1,
                     const int32_t* __restrict__ perm, int n, int bs, int d2, int H) {
  const float* src = blockIdx.y ? src1 : src0;
  float* dst = blockIdx.y ? dst1 : dst0;
  if (!src) return;
  const int64_t o = int64_t(blockIdx.x) * (kShufThreads / 32) + (threadIdx.x >> 5);
  if (o >= int64_t(n) * d2) return;
  const int lane = threadIdx.x & 31;
  const int64_t per_b = int64_t(d2) * bs;
  const int b = int(o / per_b), rem = int(o - b * per_b), s = rem / bs, j = rem - s * bs;
  const int e = perm[b * bs + j];
  float4* d = reinterpret_cast<float4*>(dst + o * H);
  if (unsigned(e) < unsigned(n)) {
    const float4* sr = reinterpret_cast<const float4*>(src + (int64_t(s) * n + e) * H);
    for (int i = lane; i < H / 4; i += 32) d[i] = __ldcs(sr + i);
  } else {
    const float q = __int_as_float(0x7FC00000);
    for (int i = lane; i < H / 4; i += 32) d[i] = make_float4(q, q, q, q);
  }
}

// shared-memory opt-in of both kernels for the largest n_envs, once per handle (not a call to make during graph capture)
int minibatch_attr(kbs_handle* h) {
  if (h->minibatch_attr_set) return KBS_OK;
  KBS_CUDA_TRY(cudaFuncSetAttribute(minibatch_permutation_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    KBS_MAX_PERMUTATION_ENVS * int(sizeof(unsigned long long))));
  KBS_CUDA_TRY(cudaFuncSetAttribute(shuffle_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    KBS_MAX_PERMUTATION_ENVS * int(sizeof(float))));
  h->minibatch_attr_set = true;
  return KBS_OK;
}

}  // namespace

int kbs_launch_minibatch_permutation(kbs_handle* h, uint64_t seed, int64_t* pass_dev, int64_t env0, int32_t* perm, int64_t n,
                                     cudaStream_t st) {
  int np2 = 2;
  while (np2 < n) np2 <<= 1;
  const size_t smem = size_t(np2) * sizeof(unsigned long long);
  if (int rc = minibatch_attr(h)) return rc;
  static_assert(sizeof(long long) == sizeof(int64_t), "pass counter width");
  KBS_LAUNCH(h, KBS_K_PERMUTATION, st,
             (minibatch_permutation_kernel<<<1, kPermThreads, smem, st>>>(seed, reinterpret_cast<long long*>(pass_dev), env0, perm,
                                                                          int(n), np2)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_shuffle_minibatches(kbs_handle* h, const int32_t* perm, const kbs_ppo_batch& src, const kbs_ppo_minibatches& dst,
                                   int64_t n, cudaStream_t st) {
  const int64_t T = src.T;
  ShuffleRows R{};
  const void* s[9] = {src.actor_obs, src.critic_obs, src.action, src.done, src.old_log_probs, src.advantages, src.value_targets,
                      src.old_values, src.lpf0};
  void* d[9] = {dst.actor_obs, dst.critic_obs, dst.action, dst.done, dst.old_log_probs, dst.advantages, dst.value_targets,
                dst.old_values, dst.lpf0};
  const int64_t rows[9] = {T * KBS_ACTOR_OBS, T * KBS_CRITIC_OBS, T * KBS_NUM_JOINTS, T, T, T, T, T, s[8] ? KBS_NUM_JOINTS : 0};
  R.first[0] = 0;
  for (int a = 0; a < 9; ++a) {
    R.src[a] = static_cast<const char*>(s[a]);
    R.dst[a] = static_cast<char*>(d[a]);
    R.esize[a] = a == 3 ? 1 : 4;
    R.first[a + 1] = R.first[a] + rows[a];
  }
  const size_t smem = size_t(n) * sizeof(float);
  if (int rc = minibatch_attr(h)) return rc;
  const int bs = int(dst.batch_size);
  KBS_LAUNCH(h, KBS_K_SHUFFLE, st,
             (shuffle_rows_kernel<<<unsigned(R.first[9]), kShufThreads, smem, st>>>(R, perm, src.ld, int(n), bs)));
  if (src.actor_carry0 || src.critic_carry0) {
    const int d2 = 2 * h->p.depth, H = h->p.hidden_size;
    const unsigned gx = unsigned((n * d2 + kShufThreads / 32 - 1) / (kShufThreads / 32));
    KBS_LAUNCH(h, KBS_K_SHUFFLE, st,
               (shuffle_carry_kernel<<<dim3(gx, 2), kShufThreads, 0, st>>>(src.actor_carry0, dst.actor_carry0, src.critic_carry0,
                                                                          dst.critic_carry0, perm, int(n), bs, d2, H)));
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

extern "C" {

int kbs_ppo_grad(kbs_handle* h, const kbs_ppo_loss_params* params, const kbs_ppo_batch* b, const kbs_net_grads* actor,
                 const kbs_net_grads* critic, float* log_probs, float* values, float* entropy, float* stats_out, int64_t n,
                 void* stream) {
  if (!h || !params || !b || !actor || !critic || !log_probs || !values || !entropy || !stats_out) return KBS_E_NULL;
  if (!b->actor_obs || !b->critic_obs || !b->action || !b->done || !b->old_log_probs || !b->advantages || !b->value_targets ||
      !b->old_values)
    return KBS_E_NULL;
  if (b->T <= 0 || n <= 0 || b->ld < n || (b->ld & 3)) return KBS_E_SHAPE;
  for (int k = 0; k < 2; ++k)
    if (!h->net[k].packed) return KBS_E_STATE;
  { const int rc0 = kbs_enter(h); if (rc0) return rc0; }
  cudaStream_t st = (cudaStream_t)stream;
  {
    // FP16-split datapath: the persistent form (2 launches for the whole forward + backward recurrence); KBS_PPO_PER_STEP=1
    // keeps the per-step launch sequence below (A/B, and the cross-check of the persistent kernels)
    const char* e = getenv("KBS_PPO_PER_STEP");
    if (!(e && atoi(e)) && h->p.gemm_path == KBS_GEMM_TC_2XF16 && h->p.depth <= 2 && kbs_tc_bptt_available(h, n, b->T)) {
      const kbs_net_grads* gr[2] = {actor, critic};
      return ppo_grad_persistent(h, *params, *b, gr, log_probs, values, entropy, stats_out, n, st);
    }
  }
  const int H = h->p.hidden_size, depth = h->p.depth;
  const int64_t T = b->T, ld = b->ld, rows = T * n;
  const size_t sH = size_t(n) * H;
  const int splits = 16;   // 8 x 2 x 16 = 256 CTAs of the large-tile weight-gradient GEMM: two per SM (128 registers)
  const int chunks = int((rows + 511) / 512);
  const int kp_max = round_up_i(KBS_CRITIC_OBS, 64);
  const bool tc = h->p.gemm_path != KBS_GEMM_SIMT_FP32;
  const size_t part_f = size_t(chunks) * 4 * H + size_t(splits) * size_t(4 * H) * size_t(kp_max) + size_t(H) * kp_max + 64 * H + 4096;
  float* gates_pre[2]; float* dc_rec[2]; float* part[2]; float *y_s, *sd_s;
  NetWork w[2];
  int rc = kbs_scratch(h, [&](KbsScratch& s) {
    for (int k = 0; k < 2; ++k) {            // per net: actor and critic run concurrently on two streams
      gates_pre[k] = s.take<float>(sH * 4);
      dc_rec[k] = s.take<float>(size_t(depth) * sH);
      part[k] = s.take<float>(part_f);
    }
    y_s = s.take<float>(size_t(T) * KBS_NUM_JOINTS * ld);
    sd_s = s.take<float>(size_t(T) * KBS_NUM_JOINTS * ld);
    for (int k = 0; k < 2; ++k) {
      const size_t kp = size_t(round_up_i(h->net[k].num_in, 64));
      w[k].obs_rm = s.take<float>(size_t(rows) * kp);
      w[k].x0 = s.take<float>(size_t(rows) * H);
      w[k].dh_top = s.take<float>(size_t(rows) * H);
      w[k].dxh0 = s.take<float>(size_t(rows) * 2 * H);
      w[k].out = s.take<float>(size_t(rows) * 64);
      w[k].dout = s.take<float>(size_t(rows) * 64);
      for (int l = 0; l < depth; ++l) {
        w[k].dxh[l] = s.take<float>(sH * 2);
        w[k].ga[l] = s.take<float>(size_t(rows) * 4 * H);
        w[k].dG[l] = s.take<float>(size_t(rows) * 4 * H);
        w[k].cs[l] = s.take<float>(size_t(rows) * H);
        w[k].hs[l] = s.take<float>(size_t(rows) * H);
        w[k].h_in[l] = s.take<float>(size_t(rows) * H);
        w[k].c_in[l] = s.take<float>(size_t(rows) * H);
        w[k].w_ihT[l] = s.take<float>(size_t(4) * H * H);
        w[k].w_hhT[l] = s.take<float>(size_t(4) * H * H);
      }
      w[k].w_outT = s.take<float>(size_t(64) * H);
      if (tc) {
        const size_t sbH = kbs_tc_rows_sb_bytes(h, n, H), sb4H = kbs_tc_rows_sb_bytes(h, n, 4 * H);
        w[k].x0_sb = s.take<char>(size_t(T) * sbH);
        for (int l = 0; l < depth; ++l) {
          w[k].hs_sb[l] = s.take<char>(size_t(T) * sbH);
          w[k].h_in_sb[l] = s.take<char>(size_t(T) * sbH);
        }
        w[k].dG_sb = s.take<char>(sb4H);
        const KbsTnPlan plan = kbs_tc_tn_plan(h, rows);
        const size_t m_panels = size_t(4 * H / 128), b_tiles = size_t((int(kp) > 2 * H ? int(kp) : 2 * H) / 128 + 1);
        w[k].tn_a = s.take<char>(m_panels * plan.col_bytes);
        w[k].tn_b = s.take<char>(b_tiles * plan.col_bytes);
        w[k].tn_partial = s.take<float>(size_t(plan.ksplit) * m_panels * 128 * (b_tiles * 128));
        w[k].tn_zero = s.take<float>(1024);
        w[k].tn_ones = s.take<char>(4096 * sizeof(float));
      }
    }
  });
  if (rc) return rc;
  // The two networks share nothing until the loss statistics: the critic runs on the handle's side stream, forked from
  // and joined into the caller's stream with events (capturable: the whole call can be replayed as one CUDA graph).
  { const int rc0 = kbs_side_stream_init(h); if (rc0) return rc0; }
  cudaStream_t sc = h->side_stream;
  KBS_CUDA_TRY(cudaEventRecord(h->ev_pre, st));
  KBS_CUDA_TRY(cudaStreamWaitEvent(sc, h->ev_pre, 0));
  // forward with saved activations
  if ((rc = run_net(h, KBS_NET_ACTOR, *b, b->actor_carry0, w[0], gates_pre[0], dc_rec[0], part[0], splits, n, st,
                    false, nullptr)))
    return rc;
  if ((rc = run_net(h, KBS_NET_CRITIC, *b, b->critic_carry0, w[1], gates_pre[1], dc_rec[1], part[1], splits, n, sc,
                    false, nullptr)))
    return rc;
  // heads: outputs, loss gradient wrt the head outputs
  KBS_LAUNCH(h, KBS_K_ACTOR_HEAD, st,
             (actor_head_fwd_bwd_warp_kernel<<<unsigned((n + 3) / 4), 128, 0, st>>>(
                 h->p, *params, w[0].out, b->actor_obs, b->action, b->done, b->lpf0, b->old_log_probs, b->advantages, y_s, sd_s,
                 log_probs, entropy, w[0].dout, T, ld, n)));
  KBS_LAUNCH(h, KBS_K_CRITIC_HEAD, sc,
             (critic_head_fwd_bwd_kernel<<<blocks(rows), kT, 0, sc>>>(*params, w[1].out, b->old_values, b->value_targets, values,
                                                                      w[1].dout, T, ld, n)));
  // critic backward on the side stream
  if ((rc = run_net(h, KBS_NET_CRITIC, *b, nullptr, w[1], gates_pre[1], dc_rec[1], part[1], splits, n, sc, true, critic)))
    return rc;
  KBS_CUDA_TRY(cudaEventRecord(h->ev_head[0], sc));
  if ((rc = run_net(h, KBS_NET_ACTOR, *b, nullptr, w[0], gates_pre[0], dc_rec[0], part[0], splits, n, st, true, actor)))
    return rc;
  KBS_CUDA_TRY(cudaStreamWaitEvent(st, h->ev_head[0], 0));       // join: values + critic gradients are complete
  if (h->ev_critic_ready) KBS_CUDA_TRY(cudaEventRecord(h->ev_critic_ready, st));
  // loss statistics (same kernel as kbs_ppo_loss; partials in the actor's reduction scratch, free again by now)
  {
    kbs_ppo_loss_io io{};
    io.log_probs = log_probs; io.old_log_probs = b->old_log_probs; io.advantages = b->advantages; io.values = values;
    io.old_values = b->old_values; io.value_targets = b->value_targets; io.entropy = entropy; io.out = stats_out;
    io.T = T; io.ld = ld;
    if ((rc = kbs_launch_ppo_loss_at(h, *params, io, n, reinterpret_cast<double*>(part[0]), st))) return rc;
  }
  return KBS_OK;
}

int kbs_adam_step(kbs_handle* h, float* param, const float* grad, float* m, float* v, int64_t count, float lr, float b1, float b2,
                  float eps, float grad_scale, int64_t step, void* stream) {
  if (!h || !param || !grad || !m || !v) return KBS_E_NULL;
  if (count <= 0 || step <= 0) return KBS_E_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  const float bc1 = 1.0f - powf(b1, float(step)), bc2 = 1.0f - powf(b2, float(step));
  KBS_LAUNCH(h, KBS_K_ADV_NORM, st, (adam_kernel<<<blocks(count), kT, 0, st>>>(param, grad, m, v, count, lr, b1, b2, eps, grad_scale, bc1, bc2)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_adamw_step(kbs_handle* h, float* param, const float* grad, float* m, float* v, int64_t count, const kbs_adamw_params* o,
                   const float* grad_norm, int64_t* step_dev, int64_t step, void* stream) {
  if (!h || !param || !grad || !m || !v || !o) return KBS_E_NULL;
  if (count <= 0 || (!step_dev && step <= 0)) return KBS_E_SHAPE;
  if (!(o->b1 >= 0.0 && o->b1 < 1.0) || !(o->b2 >= 0.0 && o->b2 < 1.0) || !(o->eps >= 0.0f)) return KBS_E_PARAM;
  cudaStream_t st = (cudaStream_t)stream;
  static_assert(sizeof(long long) == sizeof(int64_t), "step counter width");
  long long* sd = reinterpret_cast<long long*>(step_dev);
  KBS_LAUNCH(h, KBS_K_ADV_NORM, st, (adamw_kernel<<<blocks(count), kT, 0, st>>>(param, grad, m, v, count, *o, grad_norm, sd, (long long)step)));
  if (sd) KBS_LAUNCH(h, KBS_K_ADV_NORM, st, (step_advance_kernel<<<1, 1, 0, st>>>(sd, grad_norm, o->grad_scale)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_ppo_grad_set_events(kbs_handle* h, void* critic_ready) {
  if (!h) return KBS_E_NULL;
  h->ev_critic_ready = (cudaEvent_t)critic_ready;
  return KBS_OK;
}

int kbs_grad_norm(kbs_handle* h, const float* grad, int64_t count, float* norm_out, void* stream) {
  if (!h || !grad || !norm_out) return KBS_E_NULL;
  if (count <= 0) return KBS_E_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  if (!h->norm_partial) KBS_CUDA_TRY(cudaMalloc(&h->norm_partial, sizeof(double) * kNormBlocks));
  KBS_LAUNCH(h, KBS_K_ADV_NORM, st, (sumsq_partial_kernel<<<kNormBlocks, kT, 0, st>>>(grad, count, h->norm_partial)));
  KBS_LAUNCH(h, KBS_K_ADV_NORM, st, (sumsq_final_kernel<<<1, kT, 0, st>>>(h->norm_partial, norm_out)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

}  // extern "C"
