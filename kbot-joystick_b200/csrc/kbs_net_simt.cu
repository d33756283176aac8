// kbs_net_simt.cu -- fp32 FFMA datapath for the actor/critic trunk (input_proj -> depth x LSTMCell ->
// output_proj, train.py:913-922, 993-1002) plus the actor / critic heads shared by both datapaths.
// This is the exact-fp32 path (summation order aside); the tcgen05 3xTF32 path lives in kbs_net_tc.cu.
#include <math.h>

#include "kbs_common.cuh"

namespace {

constexpr int BM = 64, BN = 64, BK = 16, PAD = 4;

// C[m][n] (+)= sum_k A(m,k) W[n][k] + bias[n].   A: row-major [M][lda] or SoA [K][lda] (env contiguous).
// W: [Npad][ldw] row-major, Npad % 64 == 0, K % 16 == 0 (zero padded by the pack step).
// gridDim.z walks a time axis: A += z * a_tstride, C += z * c_tstride (floats).
template <bool A_SOA>
__global__ void __launch_bounds__(256)
gemm_nt_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ W, int ldw,
               const float* __restrict__ bias, float* __restrict__ C, int ldc, int64_t M, int K, int Kvalid,
               int accumulate, int64_t a_tstride = 0, int64_t c_tstride = 0) {
  A += int64_t(blockIdx.z) * a_tstride;
  C += int64_t(blockIdx.z) * c_tstride;
  __shared__ __align__(16) float As[BK][BM + PAD];
  __shared__ __align__(16) float Ws[BK][BN + PAD];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int64_t m0 = int64_t(blockIdx.x) * BM;
  const int n0 = blockIdx.y * BN;
  float acc[4][4] = {};

  for (int k0 = 0; k0 < K; k0 += BK) {
    if (A_SOA) {
      const int k = tid >> 4, m4 = (tid & 15) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (k0 + k < Kvalid && m0 + m4 < M) v = *reinterpret_cast<const float4*>(A + int64_t(k0 + k) * lda + m0 + m4);
      *reinterpret_cast<float4*>(&As[k][m4]) = v;
    } else {
      const int r = tid >> 2, kq = (tid & 3) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m0 + r < M) v = *reinterpret_cast<const float4*>(A + (m0 + r) * lda + k0 + kq);
      As[kq + 0][r] = v.x; As[kq + 1][r] = v.y; As[kq + 2][r] = v.z; As[kq + 3][r] = v.w;
    }
    {
      const int r = tid >> 2, kq = (tid & 3) * 4;
      const float4 v = *reinterpret_cast<const float4*>(W + int64_t(n0 + r) * ldw + k0 + kq);
      Ws[kq + 0][r] = v.x; Ws[kq + 1][r] = v.y; Ws[kq + 2][r] = v.z; Ws[kq + 3][r] = v.w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Ws[k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
  if (bias) bb = *reinterpret_cast<const float4*>(bias + n0 + tx * 4);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + ty * 4 + i;
    if (m >= M) continue;
    float4* cp = reinterpret_cast<float4*>(C + m * ldc + n0 + tx * 4);
    float4 o = make_float4(acc[i][0] + bb.x, acc[i][1] + bb.y, acc[i][2] + bb.z, acc[i][3] + bb.w);
    if (accumulate) { const float4 c = *cp; o.x += c.x; o.y += c.y; o.z += c.z; o.w += c.w; }
    *cp = o;
  }
}

// C[m][n] = sum_k A[k][m] B[k][n] over k in [k0, k1) of this split (gridDim.z splits; partial z goes to C + z * M * ldc).
// A: [K][lda] (M columns), B: [K][ldb] (N columns), both read along their contiguous axis.  M % 64 == 0, N % 64 == 0.
// Used by the PPO update for the weight gradients dW = dG^T X summed over (t, env).
__global__ void __launch_bounds__(256)
gemm_tn_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb, float* __restrict__ C, int ldc,
               int M, int64_t K) {
  __shared__ __align__(16) float As[BK][BM + PAD];
  __shared__ __align__(16) float Bs[BK][BN + PAD];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int64_t per = (K + gridDim.z - 1) / gridDim.z;
  const int64_t kb = int64_t(blockIdx.z) * per, ke = (kb + per < K) ? kb + per : K;
  C += size_t(blockIdx.z) * size_t(M) * ldc;
  float acc[4][4] = {};
  for (int64_t k0 = kb; k0 < ke; k0 += BK) {
    const int k = tid >> 4, c4 = (tid & 15) * 4;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (k0 + k < ke) {
      a = *reinterpret_cast<const float4*>(A + (k0 + k) * lda + m0 + c4);
      b = *reinterpret_cast<const float4*>(B + (k0 + k) * ldb + n0 + c4);
    }
    *reinterpret_cast<float4*>(&As[k][c4]) = a;
    *reinterpret_cast<float4*>(&Bs[k][c4]) = b;
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 av4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 bv4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float av[4] = {av4.x, av4.y, av4.z, av4.w}, bv[4] = {bv4.x, bv4.y, bv4.z, bv4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
    *reinterpret_cast<float4*>(C + size_t(m0 + ty * 4 + i) * ldc + n0 + tx * 4) =
        make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
}

// Large-tile variant of gemm_tn for the weight-gradient GEMMs of the PPO update (K = T x n ~ 5e4): 128 x 128 x 16 tiles,
// 8 x 8 outputs per thread (two 4-wide strips per axis), global loads of slab k+1 issued before the FMAs of slab k
// (register staging + double-buffered shared memory: one barrier per slab).  M % 128 == 0, N % 128 == 0.
constexpr int LBM = 128, LBN = 128;
__global__ void __launch_bounds__(256, 2)
gemm_tn_large_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb, float* __restrict__ C, int ldc,
                     int M, int64_t K) {
  __shared__ __align__(16) float As[2][BK][LBM];
  __shared__ __align__(16) float Bs[2][BK][LBN];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;                    // 16 x 16 threads; thread owns rows ty*4 + {0..3, 64..67}, cols likewise
  const int m0 = blockIdx.x * LBM, n0 = blockIdx.y * LBN;
  const int64_t per = ((K + gridDim.z - 1) / gridDim.z + BK - 1) / BK * BK;
  const int64_t kb = int64_t(blockIdx.z) * per, ke = (kb + per < K) ? kb + per : K;
  C += size_t(blockIdx.z) * size_t(M) * ldc;
  // loader mapping: 16 k-rows x 128 columns = 512 float4 per operand, 2 per thread
  const int lk = tid >> 5, lc = (tid & 31) * 4;              // k rows lk and lk + 8
  float acc[8][8] = {};
  float4 ra[2], rb[2];
  auto gload = [&](int64_t k0) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int64_t k = k0 + lk + 8 * h;
      ra[h] = rb[h] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (k < ke) {
        ra[h] = *reinterpret_cast<const float4*>(A + k * lda + m0 + lc);
        rb[h] = *reinterpret_cast<const float4*>(B + k * ldb + n0 + lc);
      }
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      *reinterpret_cast<float4*>(&As[buf][lk + 8 * h][lc]) = ra[h];
      *reinterpret_cast<float4*>(&Bs[buf][lk + 8 * h][lc]) = rb[h];
    }
  };
  if (kb < ke) {
    gload(kb);
    sstore(0);
  }
  __syncthreads();
  int buf = 0;
  for (int64_t k0 = kb; k0 < ke; k0 += BK) {
    const bool more = k0 + BK < ke;
    if (more) gload(k0 + BK);
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (more) sstore(buf ^ 1);
    __syncthreads();
    buf ^= 1;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    float* row = C + size_t(m) * ldc + n0;
    *reinterpret_cast<float4*>(row + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    *reinterpret_cast<float4*>(row + 64 + tx * 4) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
  }
}

// out[i] = sum_s partial[s][i]  (fixed order: deterministic)
__global__ void __launch_bounds__(256)
reduce_splits_kernel(const float* __restrict__ partial, float* __restrict__ out, int64_t count, int splits) {
  const int64_t i = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (i >= count) return;
  float a = 0.0f;
  for (int s = 0; s < splits; ++s) a += partial[size_t(s) * count + i];
  out[i] = a;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// eqx LSTMCell: i,f,g,o = split(lin, 4); c' = s(f) c + s(i) tanh(g); h' = s(o) tanh(c').
// gates [n][4H] (bias already added).  h_next: un-reset output for the next layer; carry_h/c: reset where done
// (train.py:1502-1506).
__global__ void __launch_bounds__(256)
lstm_cell_kernel(const float* __restrict__ gates, float* __restrict__ carry_h, float* __restrict__ carry_c,
                 float* __restrict__ h_next, const uint8_t* __restrict__ done, int H, int64_t n) {
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  const int hq = H / 4;
  if (idx >= n * hq) return;
  const int64_t e = idx / hq;
  const int k = int(idx - e * hq) * 4;
  const float* g = gates + e * 4 * H + k;
  const float4 gi = *reinterpret_cast<const float4*>(g);
  const float4 gf = *reinterpret_cast<const float4*>(g + H);
  const float4 gg = *reinterpret_cast<const float4*>(g + 2 * H);
  const float4 go = *reinterpret_cast<const float4*>(g + 3 * H);
  const float4 c4 = *reinterpret_cast<const float4*>(carry_c + e * H + k);
  const float iv[4] = {gi.x, gi.y, gi.z, gi.w}, fv[4] = {gf.x, gf.y, gf.z, gf.w};
  const float gv[4] = {gg.x, gg.y, gg.z, gg.w}, ov[4] = {go.x, go.y, go.z, go.w};
  const float cv[4] = {c4.x, c4.y, c4.z, c4.w};
  float hn[4], cn[4];
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    cn[l] = sigmoidf_(fv[l]) * cv[l] + sigmoidf_(iv[l]) * tanhf(gv[l]);
    hn[l] = sigmoidf_(ov[l]) * tanhf(cn[l]);
  }
  *reinterpret_cast<float4*>(h_next + e * H + k) = make_float4(hn[0], hn[1], hn[2], hn[3]);
  const bool rst = done && done[e];
  *reinterpret_cast<float4*>(carry_h + e * H + k) = rst ? make_float4(0, 0, 0, 0) : make_float4(hn[0], hn[1], hn[2], hn[3]);
  *reinterpret_cast<float4*>(carry_c + e * H + k) = rst ? make_float4(0, 0, 0, 0) : make_float4(cn[0], cn[1], cn[2], cn[3]);
}

// Actor head, train.py:924-939 + distrax MultivariateNormalDiag (log_prob / entropy / sample / mode).
// One thread per env; reads out[n][ldo] row-major, writes env-major SoA (coalesced across the warp).
__global__ void __launch_bounds__(128)
actor_head_kernel(const __grid_constant__ kbs_params P, const float* __restrict__ out, int ldo,
                  const float* __restrict__ obs, int64_t ld, float* __restrict__ lpf, const float* __restrict__ eps,
                  const float* __restrict__ action_in, const uint8_t* __restrict__ done, kbs_actor_out o, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * 128 + threadIdx.x;
  if (e >= n) return;
  const float* row = out + e * ldo;
  float v[KBS_ACTOR_OUT];
#pragma unroll
  for (int k = 0; k < KBS_ACTOR_OUT; k += 4) {
    const float4 t = *reinterpret_cast<const float4*>(row + k);
    v[k] = t.x; v[k + 1] = t.y; v[k + 2] = t.z; v[k + 3] = t.w;
  }
  const bool rst = done && done[e];
  float s_z = 0.0f, s_log = 0.0f;
  constexpr float kHalfLog2Pi = 0.918938533204672742f;
#pragma unroll
  for (int j = 0; j < KBS_NUM_JOINTS; ++j) {
    // std = clip((softplus(s) + min_std) * var_scale, max=max_std)
    const float sraw = v[KBS_NUM_JOINTS + j];
    const float sp = fmaxf(sraw, 0.0f) + log1pf(expf(-fabsf(sraw)));
    const float sd = fminf((sp + P.min_std) * P.var_scale, P.max_std);
    // mean = out + JOINT_BIASES + [0 x 10, obs[-10:]]   (obs slots 55..64 = arm command)
    float m = v[j] + P.joint_bias[j];
    m = m + ((j >= 10) ? obs[(55 + (j - 10)) * ld + e] : 0.0f);
    // ksim.lowpass_one_pole: y' = y + alpha (x - y)
    const float y = lpf[j * ld + e];
    const float yn = y + P.lpf_alpha * (m - y);
    lpf[j * ld + e] = rst ? 0.0f : yn;
    float a = yn;                                       // mode()
    if (eps) a = yn + sd * eps[j * ld + e];             // sample(seed)
    const float a_eval = action_in ? action_in[j * ld + e] : a;
    const float z = (a_eval - yn) / sd;
    s_z = s_z + (-0.5f * z * z - kHalfLog2Pi);
    s_log = s_log + logf(sd);
    if (o.action) o.action[j * ld + e] = a;
    if (o.mean) o.mean[j * ld + e] = yn;
    if (o.std) o.std[j * ld + e] = sd;
  }
  if (o.log_prob) o.log_prob[e] = s_z - s_log;
  if (o.entropy) o.entropy[e] = s_log + float(KBS_NUM_JOINTS) * (0.5f + kHalfLog2Pi);
}

__global__ void __launch_bounds__(128)
critic_head_kernel(const float* __restrict__ out, int ldo, float* __restrict__ value, int64_t n) {
  const int64_t e = int64_t(blockIdx.x) * 128 + threadIdx.x;
  if (e < n) value[e] = out[e * ldo];
}

// zero-padded copy [rows][cols] -> [rows_pad][cols_pad]
__global__ void pad_copy_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols, int rows_pad,
                                int cols_pad) {
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= int64_t(rows_pad) * cols_pad) return;
  const int r = int(idx / cols_pad), c = int(idx % cols_pad);
  dst[idx] = (r < rows && c < cols) ? src[int64_t(r) * cols + c] : 0.0f;
}

int pad_copy(kbs_handle* h, const float* src, float** dst, int rows, int cols, int rows_pad, int cols_pad,
             cudaStream_t st) {
  // shapes are fixed per handle (hidden size, depth, net): a re-pack after a weight update reuses the allocation, so the
  // device pointers stay stable (CUDA graphs captured over them stay valid)
  if (!*dst) KBS_CUDA_TRY(cudaMalloc(dst, sizeof(float) * size_t(rows_pad) * cols_pad));
  const int64_t tot = int64_t(rows_pad) * cols_pad;
  KBS_LAUNCH(h, KBS_K_PACK, st,
             (pad_copy_kernel<<<unsigned((tot + 255) / 256), 256, 0, st>>>(src, *dst, rows, cols, rows_pad, cols_pad)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

}  // namespace

int kbs_simt_pack(kbs_handle* h, int net, const kbs_net_weights* w, cudaStream_t st) {
  KbsNet& N = h->net[net];
  const int H = h->p.hidden_size;
  N.num_in = (net == KBS_NET_ACTOR) ? KBS_ACTOR_OBS : KBS_CRITIC_OBS;
  N.num_out = (net == KBS_NET_ACTOR) ? KBS_ACTOR_OUT : 1;
  N.kin_pad = round_up(N.num_in, 16);
  N.nout_pad = 64;
  int rc;
  if ((rc = pad_copy(h, w->w_in, &N.w_in, H, N.num_in, H, N.kin_pad, st))) return rc;
  if ((rc = pad_copy(h, w->b_in, &N.b_in, 1, H, 1, H, st))) return rc;
  for (int l = 0; l < h->p.depth; ++l) {
    if ((rc = pad_copy(h, w->w_ih[l], &N.w_ih[l], 4 * H, H, 4 * H, H, st))) return rc;
    if ((rc = pad_copy(h, w->w_hh[l], &N.w_hh[l], 4 * H, H, 4 * H, H, st))) return rc;
    if ((rc = pad_copy(h, w->b[l], &N.b[l], 1, 4 * H, 1, 4 * H, st))) return rc;
  }
  if ((rc = pad_copy(h, w->w_out, &N.w_out, N.num_out, H, N.nout_pad, H, st))) return rc;
  if ((rc = pad_copy(h, w->b_out, &N.b_out, 1, N.num_out, 1, N.nout_pad, st))) return rc;
  N.packed = true;
  return KBS_OK;
}

// ---- plain fp32 GEMM launchers for the PPO update (kbs_ppo_update.cu) ----
// C[M][ldc] (+)= A[M][lda] . W[Npad][ldw]^T + bias; batch > 1 walks gridDim.z with the given strides (floats)
int kbs_simt_gemm_nt(kbs_handle* h, const float* A, int64_t lda, const float* W, int ldw, const float* bias, float* C, int ldc,
                     int64_t M, int Npad, int K, int accumulate, cudaStream_t st, int batch, int64_t a_ts, int64_t c_ts) {
  if (Npad % BN || K % BK) return KBS_E_SHAPE;
  const unsigned mb = unsigned((M + BM - 1) / BM);
  KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
             (gemm_nt_kernel<false><<<dim3(mb, Npad / BN, batch), 256, 0, st>>>(A, lda, W, ldw, bias, C, ldc, M, K, K, accumulate,
                                                                                a_ts, c_ts)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// C[M][ldc] = sum_k A[k][0..M) x B[k][0..N): split-K over `splits` partial buffers (partials: splits x M x ldc floats),
// reduced in a fixed order
int kbs_simt_gemm_tn(kbs_handle* h, const float* A, int lda, const float* B, int ldb, float* C, int ldc, int M, int N, int64_t K,
                     float* partials, int splits, cudaStream_t st) {
  if (M % BM || N % BN || ldc < N) return KBS_E_SHAPE;
  if (M % LBM == 0 && N % LBN == 0)
    KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
               (gemm_tn_large_kernel<<<dim3(M / LBM, N / LBN, splits), 256, 0, st>>>(A, lda, B, ldb, partials, ldc, M, K)));
  else
    KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
               (gemm_tn_kernel<<<dim3(M / BM, N / BN, splits), 256, 0, st>>>(A, lda, B, ldb, partials, ldc, M, K)));
  const int64_t count = int64_t(M) * ldc;
  KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
             (reduce_splits_kernel<<<unsigned((count + 255) / 256), 256, 0, st>>>(partials, C, count, splits)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

KbsSimtTrunkWs kbs_simt_trunk_ws(KbsScratch& s, const kbs_handle* h, int64_t n) {
  const size_t nH = size_t(n) * h->p.hidden_size;
  return {s.take<float>(nH), s.take<float>(4 * nH), s.take<float>(nH)};   // braced list: taken left to right
}

// out_rowmajor: [n][nout_pad = 64]
int kbs_simt_trunk(kbs_handle* h, int net, const float* obs_soa, int64_t ld, float* carry, const uint8_t* done,
                   float* out_rm, const KbsSimtTrunkWs& ws, int64_t n, cudaStream_t st) {
  const KbsNet& N = h->net[net];
  if (!N.packed) return KBS_E_STATE;
  const int H = h->p.hidden_size;
  float* x = ws.x; float* gates = ws.gates; float* hbuf = ws.hbuf;
  const unsigned mb = unsigned((n + BM - 1) / BM);
  KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
             (gemm_nt_kernel<true><<<dim3(mb, H / BN), 256, 0, st>>>(obs_soa, ld, N.w_in, N.kin_pad, N.b_in, x, H, n,
                                                                    N.kin_pad, N.num_in, 0)));
  const float* in = x;
  for (int l = 0; l < h->p.depth; ++l) {
    float* ch = carry + (size_t(l) * 2 + 0) * size_t(n) * H;
    float* cc = carry + (size_t(l) * 2 + 1) * size_t(n) * H;
    KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
               (gemm_nt_kernel<false><<<dim3(mb, 4 * H / BN), 256, 0, st>>>(in, H, N.w_ih[l], H, N.b[l], gates, 4 * H, n, H,
                                                                           H, 0)));
    KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
               (gemm_nt_kernel<false><<<dim3(mb, 4 * H / BN), 256, 0, st>>>(ch, H, N.w_hh[l], H, nullptr, gates, 4 * H, n,
                                                                           H, H, 1)));
    const int64_t tot = n * (H / 4);
    KBS_LAUNCH(h, KBS_K_LSTM_CELL, st,
               (lstm_cell_kernel<<<unsigned((tot + 255) / 256), 256, 0, st>>>(gates, ch, cc, hbuf, done, H, n)));
    in = hbuf;
  }
  KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
             (gemm_nt_kernel<false><<<dim3(mb, N.nout_pad / BN), 256, 0, st>>>(in, H, N.w_out, H, N.b_out, out_rm,
                                                                              N.nout_pad, n, H, H, 0)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// input_proj / output_proj alone (used by the tensor-core trunk around its LSTM stack)
int kbs_simt_in_proj(kbs_handle* h, int net, const float* obs_soa, int64_t ld, float* x_rm, int64_t n, cudaStream_t st) {
  const KbsNet& N = h->net[net];
  if (!N.packed) return KBS_E_STATE;
  const int H = h->p.hidden_size;
  const unsigned mb = unsigned((n + BM - 1) / BM);
  KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
             (gemm_nt_kernel<true><<<dim3(mb, H / BN), 256, 0, st>>>(obs_soa, ld, N.w_in, N.kin_pad, N.b_in, x_rm, H, n,
                                                                    N.kin_pad, N.num_in, 0)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_simt_out_proj(kbs_handle* h, int net, const float* h_rm, float* out_rm, int64_t n, cudaStream_t st) {
  const KbsNet& N = h->net[net];
  if (!N.packed) return KBS_E_STATE;
  const int H = h->p.hidden_size;
  const unsigned mb = unsigned((n + BM - 1) / BM);
  KBS_LAUNCH(h, KBS_K_GEMM_SIMT, st,
             (gemm_nt_kernel<false><<<dim3(mb, N.nout_pad / BN), 256, 0, st>>>(h_rm, H, N.w_out, H, N.b_out, out_rm,
                                                                              N.nout_pad, n, H, H, 0)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_actor_head(kbs_handle* h, const float* out_rm, int ldo, const float* obs_soa, int64_t ld, float* lpf,
                          const float* eps, const float* action_in, const uint8_t* done, const kbs_actor_out& o,
                          int64_t n, cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_ACTOR_HEAD, st,
             (actor_head_kernel<<<unsigned((n + 127) / 128), 128, 0, st>>>(h->p, out_rm, ldo, obs_soa, ld, lpf, eps,
                                                                          action_in, done, o, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_launch_critic_head(kbs_handle* h, const float* out_rm, int ldo, float* value, int64_t n, cudaStream_t st) {
  KBS_LAUNCH(h, KBS_K_CRITIC_HEAD, st,
             (critic_head_kernel<<<unsigned((n + 127) / 128), 128, 0, st>>>(out_rm, ldo, value, n)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}
