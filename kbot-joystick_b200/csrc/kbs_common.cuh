// kbs_common.cuh -- shared definitions for libkbotstep (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kbotstep.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libkbotstep is written for sm_100a (B200) only"
#endif

#define KBS_CUDA_TRY(expr)                      \
  do {                                          \
    cudaError_t _e = (expr);                    \
    if (_e != cudaSuccess) return (int)_e;      \
  } while (0)

#define KBS_LAUNCH_CHECK()                      \
  do {                                          \
    cudaError_t _e = cudaPeekAtLastError();     \
    if (_e != cudaSuccess) return (int)_e;      \
  } while (0)

// Packed network held by the handle.
struct KbsNet {
  bool packed = false;
  int num_in = 0, num_out = 0;  // logical sizes (65/40, 475/1)
  int kin_pad = 0;              // num_in rounded up to 16
  int nout_pad = 0;             // num_out rounded up to 64 (SIMT) / 16 (TC)
  // fp32 copies in eqx [out][in] layout, K padded (SIMT path + source for the TC pack)
  float* w_in = nullptr;   // [H][kin_pad]
  float* b_in = nullptr;   // [H]
  float* w_ih[KBS_MAX_DEPTH] = {nullptr, nullptr, nullptr, nullptr};  // [4H][H]
  float* w_hh[KBS_MAX_DEPTH] = {nullptr, nullptr, nullptr, nullptr};  // [4H][H]
  float* b[KBS_MAX_DEPTH] = {nullptr, nullptr, nullptr, nullptr};     // [4H]
  float* w_out = nullptr;  // [nout_pad][H]
  float* b_out = nullptr;  // [nout_pad]
  // tcgen05 path: one contiguous image of UMMA-ready operand tiles (see kbs_net_tc.cu)
  float* tc_image = nullptr;
  size_t tc_image_floats = 0;
  float* tc_bwd_image = nullptr;   // PPO update: [W_ih | W_hh] transposed per layer as MMA operand (kbs_tc_pack_bwd), 128-column tiles
  float* tc_bwd_image64 = nullptr; // ... and in the 64-column tiles of bptt_persist_kernel
  float* tc_fwd8_image = nullptr;  // LSTM weights in 128-column tiles of 8-unit groups (lstm_fwd_save_kernel, FP16 kind)
};

// kernel ids of the per-kernel CUDA-event profiler (kbs_profile_*): one id per __global__ of the library
enum KbsKernelId {
  KBS_K_OBS = 0, KBS_K_COMMAND, KBS_K_TORQUE, KBS_K_TERMINATE, KBS_K_REWARD_ROT, KBS_K_REWARD_TERMS, KBS_K_REWARD_SCAN,
  KBS_K_GAE, KBS_K_ADV_NORM, KBS_K_POLICY_IO, KBS_K_GEMM_SIMT, KBS_K_LSTM_CELL, KBS_K_ACTOR_HEAD, KBS_K_CRITIC_HEAD,
  KBS_K_PACK, KBS_K_LSTM_TC, KBS_K_PROJ_TC, KBS_K_ROLLOUT_TC, KBS_K_BPTT_TC, KBS_K_GEMM_TN, KBS_K_PACK_TN, KBS_K_TN_REDUCE,
  KBS_K_STEP_RECORD, KBS_K_ACTUATOR_SUBSTEP, KBS_K_PERMUTATION, KBS_K_SHUFFLE, KBS_K_COUNT
};
static_assert(KBS_K_COUNT == KBS_NUM_KERNEL_IDS, "kbotstep.h KBS_NUM_KERNEL_IDS");
constexpr int kKbsProfMaxPairs = 8192;
constexpr int kKbsMaxChunks = 8;

struct kbs_handle {
  kbs_params p;
  int device = 0;
  int num_sms = 148;
  KbsNet net[2];
  // scratch, grown on demand (never during stream capture: warm up first)
  float* scratch = nullptr;
  size_t scratch_floats = 0;
  int64_t launches = 0;
  // per-kernel event profiler (off by default; bench.py turns it on for a dedicated pass)
  bool prof_on = false;
  int prof_n = 0;
  cudaEvent_t* prof_ev = nullptr;   // 2 * kKbsProfMaxPairs events, created on first enable
  int8_t* prof_id = nullptr;        // kernel id of each pair
  // debug: per-CTA phase stamps of one LSTM launch inside kbs_rollout (kbs_debug_tc_trace_attach)
  // side stream of the fused rollout (heads overlap the next step's LSTM launches); forked/joined with events
  cudaStream_t side_stream = nullptr;
  cudaStream_t aux_stream = nullptr;          // chunked observation / input-projection phase of the fused rollout
  cudaEvent_t ev_pre = nullptr, ev_chunk[8] = {};
  cudaEvent_t ev_lstm[2] = {nullptr, nullptr}, ev_head[2] = {nullptr, nullptr};
  double* norm_partial = nullptr;             // kbs_grad_norm: per-block partial sums of squares
  unsigned int* loss_ticket = nullptr;        // "last block" counter of ppo_loss_kernel
  unsigned int* persist_status = nullptr;     // device health word (KBS_STATUS_*): sticky, OR-accumulated by the kernels
  unsigned int* status_host = nullptr;        // pinned host copy, refreshed by an async D2H after the fused entry points' kernels
  bool tc_attr_set = false;                   // cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: once per handle
  bool head_attr_set = false;
  bool bptt_attr_set = false;
  bool fwd_save_attr_set = false;
  bool dw_attr_set = false;
  bool minibatch_attr_set = false;            // kbs_minibatch_permutation / kbs_shuffle_minibatches shared-memory opt-in
  cudaEvent_t ev_critic_ready = nullptr;      // caller's event (kbs_ppo_grad_set_events): recorded when the critic's gradients are final
  bool scratch_locked = false;                // kbs_scratch_lock: growing the scratch is an error (a CUDA graph holds pointers)
  long long* trace_buf = nullptr;
  int64_t trace_step = -1;
  int trace_layer = 0;
};

// Wraps one kernel launch: counts it and, when profiling, brackets it with events on the launch stream.
struct KbsLaunchScope {
  kbs_handle* h; cudaStream_t st; int slot;
  KbsLaunchScope(kbs_handle* h_, int id, cudaStream_t st_) : h(h_), st(st_), slot(-1) {
    h->launches++;
    if (h->prof_on && h->prof_n < kKbsProfMaxPairs) {
      slot = h->prof_n++;
      h->prof_id[slot] = (int8_t)id;
      cudaEventRecord(h->prof_ev[2 * slot], st);
    }
  }
  ~KbsLaunchScope() { if (slot >= 0) cudaEventRecord(h->prof_ev[2 * slot + 1], st); }
};
#define KBS_LAUNCH(h, id, st, ...) do { KbsLaunchScope _ls((h), (id), (st)); __VA_ARGS__; } while (0)

int kbs_side_stream_init(kbs_handle* h);   // kbs_api.cu: lazily creates side_stream + events (returns cudaError_t)
// device health word (kbs_api.cu): allocate on first use; enqueue its copy to the pinned host word behind the kernels of a
// fused entry point; entry check = wrong current device or a sticky status -> error code
int kbs_status_init(kbs_handle* h);
int kbs_status_publish(kbs_handle* h, cudaStream_t st);
int kbs_enter(kbs_handle* h);
// scratch management (kbs_api.cu): grows the handle's allocation (KBS_E_STATE while kbs_scratch_lock holds it)
int kbs_scratch_reserve(kbs_handle* h, size_t floats);

// Bump allocator over the handle's scratch.  An entry point states its layout once, as code that only takes pieces (no
// launches, no branches on which pass it is in); kbs_scratch runs it with a null base to add up the total, grows the
// scratch to that, and runs it again on the real base to hand out the pointers.  Every piece is rounded up to 256 bytes.
struct KbsScratch {
  char* base;
  size_t bytes = 0;
  template <class T> T* take(size_t count) {
    T* p = base ? reinterpret_cast<T*>(base + bytes) : nullptr;
    bytes += (count * sizeof(T) + 255) / 256 * 256;
    return p;
  }
};
template <class Layout>
int kbs_scratch(kbs_handle* h, Layout&& layout) {
  KbsScratch size{nullptr};
  layout(size);
  if (const int rc = kbs_scratch_reserve(h, size.bytes / sizeof(float))) return rc;
  KbsScratch s{reinterpret_cast<char*>(h->scratch)};
  layout(s);
  return KBS_OK;
}

// ---- stage launchers implemented across the translation units -------------------------------------
// kbs_elementwise.cu
int kbs_launch_observations(kbs_handle* h, const kbs_state_view& s, const kbs_noise_view* nz,
                            const kbs_episode_view* ep, const float* command, float* pg_carry,
                            const uint8_t* pg_reset, float* computed, float* actor_obs, float* critic_obs, int64_t n,
                            cudaStream_t st, int64_t T = 1, const float* pg_lagged = nullptr, bool skip_dump = false,
                            bool one_step = false);   // one_step (T = 1): the launch shape of kbs_rollout_step
int kbs_launch_ppo_loss(kbs_handle* h, const kbs_ppo_loss_params& L, const kbs_ppo_loss_io& io, int64_t n, cudaStream_t st);
int kbs_launch_ppo_loss_at(kbs_handle* h, const kbs_ppo_loss_params& L, const kbs_ppo_loss_io& io, int64_t n, double* partials,
                           cudaStream_t st);
int kbs_launch_com_distance(kbs_handle* h, const int32_t* geom1, const int32_t* geom2, const float* pos, const float* com,
                            float* out, int ncon, int64_t T, int64_t ld, int64_t n, cudaStream_t st);
int kbs_launch_mirror_obs(kbs_handle* h, const kbs_state_view& s, const float* computed, const float* command,
                          float* actor_obs, float* critic_obs, float* command_out, int64_t n, int64_t T, cudaStream_t st);
int kbs_launch_mirror_joints(kbs_handle* h, const float* in, float* out, int64_t ld, int64_t n, int64_t T, cudaStream_t st);
int kbs_launch_command(kbs_handle* h, const float* cmd_in, float* cmd_out, const float* u_switch,
                       const int32_t* mode, const float* u6, const float* u_arms, const uint8_t* done, int64_t ld,
                       int64_t n, cudaStream_t st);
int kbs_launch_command_scan(kbs_handle* h, float* command, const float* u_switch, const int32_t* mode, const float* u6,
                            const float* u_arms, const uint8_t* done, int64_t T, int64_t ld, int64_t n, cudaStream_t st);
int kbs_launch_phase_a_scans(kbs_handle* h, float* command, const float* u_switch, const int32_t* mode, const float* u6,
                             const float* u_arms, const uint8_t* done, const uint8_t* done_prev, const float* sensordata,
                             const float* lag, float* pg_carry, float* lagged, int64_t T, int64_t ld, int64_t n, cudaStream_t st);
int kbs_launch_pg_scan(kbs_handle* h, const float* sensordata, const float* lag, const uint8_t* done, const uint8_t* done_prev,
                       float* pg_carry, float* lagged, int64_t T, int64_t ld, int64_t n, cudaStream_t st);
int kbs_launch_torque(kbs_handle* h, const float* action, const kbs_state_view& s, const kbs_episode_view* ep,
                      float* ctrl, int64_t n, cudaStream_t st);
int kbs_launch_torque_substeps(kbs_handle* h, const float* action, float* prev_action, const float* u_drop, const float* latency,
                               const float* q_sub, const float* qd_sub, const kbs_episode_view* ep, float* ctrl, int S, float sub_dt,
                               float drop_prob, int64_t ld, int64_t n, cudaStream_t st);
int kbs_launch_mirror_loss(kbs_handle* h, const float* mean, const float* mean_m, const float* value, const float* value_m,
                           float* action_loss, float* value_loss, float scale_a, float scale_c, int64_t T, int64_t ld, int64_t n,
                           cudaStream_t st);
int kbs_launch_actuator_rand(kbs_handle* h, const kbs_actuator_rand_params& rp, const float* u, const uint8_t* reset,
                             const kbs_episode_view& ep, int64_t ld, int64_t n, cudaStream_t st);
int kbs_launch_rollout_noise(kbs_handle* h, uint64_t seed, int64_t step0, const kbs_noise_view* nz, float* eps_action, float* u_switch,
                             int32_t* cmd_mode, float* cmd_u6, float* cmd_u_arms, int64_t T, int64_t ld, int64_t n, cudaStream_t st);
int kbs_launch_terminate(kbs_handle* h, const kbs_state_view& s, int32_t* codes, uint8_t* done, uint8_t* success,
                         float* pre, int64_t n, cudaStream_t st, int64_t T = 1);
int kbs_launch_rewards(kbs_handle* h, const kbs_traj_view& tr, const kbs_reward_carry& carry, float* total,
                       float* components, int64_t n, cudaStream_t st);
int kbs_launch_gae(kbs_handle* h, const float* values, const float* rewards, const uint8_t* done,
                   const uint8_t* success, float* adv, float* targets, int64_t T, int64_t ld, int64_t n,
                   cudaStream_t st);
int kbs_launch_policy_pack(kbs_handle* h, const float* ja, const float* jv, const float* pg, const float* gyro,
                           const float* cmd, const float* carry_in, float* obs_soa, float* carry_aos, float* lpf_soa,
                           int64_t ld, int64_t n, cudaStream_t st);
int kbs_launch_policy_unpack(kbs_handle* h, const float* carry_aos, const float* lpf_soa, const float* mean_soa,
                             float* carry_out, float* action_out, int64_t ld, int64_t n, cudaStream_t st);
// the online step's record into slot t (kbs_rollout_step): jobs of 32-bit words, dst advanced by t * dst_step words;
// shift = the command job (src = the state's [2][16][ld] rows, words = 16 ld; dst = the [T+1] trajectory)
struct KbsStepJob { const void* src; void* dst; int64_t words, dst_step; int shift, block0; };
constexpr int kKbsStepMaxJobs = 24;
struct KbsStepRecord {
  KbsStepJob job[kKbsStepMaxJobs]; int jobs;
  int64_t T; int64_t* t; int* hsb_slot; unsigned int* ticket; unsigned int* status;
};
int kbs_launch_step_record(kbs_handle* h, KbsStepRecord a, cudaStream_t st);
// one physics sub-step of the online rollout (kbs_actuator_substep): t from the step state, k / ticket / prev_action /
// applied from the actuator state; action = the [T][20][ld] trajectory
struct KbsSubstepArgs {
  const float* action; int64_t T; const int64_t* t;
  int32_t* k; unsigned int* ticket; float* prev_action; float* applied;
  const float* u_drop; const float* latency; const float* qpos; const float* qvel; kbs_episode_view ep; float* ctrl;
  int S; float sub_dt, drop_prob; int64_t ld, n; unsigned int* status;
};
int kbs_launch_actuator_substep(kbs_handle* h, const KbsSubstepArgs& a, cudaStream_t st);
// kbs_ppo_update.cu: the update phase's minibatch construction (arguments validated by the entry points in kbs_api.cu)
int kbs_launch_minibatch_permutation(kbs_handle* h, uint64_t seed, int64_t* pass_dev, int64_t env0, int32_t* perm, int64_t n,
                                     cudaStream_t st);
int kbs_launch_shuffle_minibatches(kbs_handle* h, const int32_t* perm, const kbs_ppo_batch& src, const kbs_ppo_minibatches& dst,
                                   int64_t n, cudaStream_t st);

// kbs_net_simt.cu : fp32 FFMA datapath
int kbs_simt_pack(kbs_handle* h, int net, const kbs_net_weights* w, cudaStream_t st);
struct KbsSimtTrunkWs { float* x; float* gates; float* hbuf; };   // [n][H], [n][4H], [n][H]
KbsSimtTrunkWs kbs_simt_trunk_ws(KbsScratch& s, const kbs_handle* h, int64_t n);
int kbs_simt_trunk(kbs_handle* h, int net, const float* obs_soa, int64_t ld, float* carry, const uint8_t* done,
                   float* out_rowmajor /*[n][nout_pad]*/, const KbsSimtTrunkWs& ws, int64_t n, cudaStream_t st);

int kbs_simt_gemm_nt(kbs_handle* h, const float* A, int64_t lda, const float* W, int ldw, const float* bias, float* C, int ldc,
                     int64_t M, int Npad, int K, int accumulate, cudaStream_t st, int batch = 1, int64_t a_ts = 0, int64_t c_ts = 0);
int kbs_simt_gemm_tn(kbs_handle* h, const float* A, int lda, const float* B, int ldb, float* C, int ldc, int M, int N, int64_t K,
                     float* partials, int splits, cudaStream_t st);
int kbs_simt_in_proj(kbs_handle* h, int net, const float* obs_soa, int64_t ld, float* x_rm, int64_t n, cudaStream_t st);
int kbs_simt_out_proj(kbs_handle* h, int net, const float* h_rm, float* out_rm, int64_t n, cudaStream_t st);

// kbs_net_tc.cu : tcgen05 3xTF32 datapath
int kbs_tc_pack(kbs_handle* h, int net, cudaStream_t st);
// workspace of kbs_tc_lstm_stack: x_sb ping/pong [2], h_sb [depth][2 (in, out)] x act SB; fb [depth][c, h] x np*H
struct KbsTcStackWs { char* x_sb; char* h_sb; float* fb; };
KbsTcStackWs kbs_tc_stack_ws(KbsScratch& s, const kbs_handle* h, int64_t n);
int kbs_tc_lstm_stack(kbs_handle* h, int net, const float* x_rm, float* carry, const uint8_t* done, float* out_h_rm,
                      const KbsTcStackWs& ws, int64_t n, bool carry_sb_valid, cudaStream_t st);
// workspace of kbs_tc_rollout_recurrent, per net: hsb, xmid [depth][2] x act SB; h2rm [2 parity][n][H]; fb [depth][c, h] x np*H;
// flags [depth + 1][panels]
struct KbsTcRolloutWs { char* hsb[2]; char* xmid[2]; float* h2rm[2]; float* fb[2]; unsigned int* flags[2]; };
KbsTcRolloutWs kbs_tc_rollout_ws(KbsScratch& s, const kbs_handle* h, int64_t n, int nets);
// recurrent phase of the fused rollout (kbs_net_tc.cu)
struct KbsTcRolloutArgs {
  int64_t n, ld, T;
  bool with_critic;
  const float* x_sb_all[2];   // [T] x kbs_tc_sb_floats SB input-projection outputs per net (actor, critic)
  bool x_is_obs[2];           // x_sb_all[k] holds the packed observations: the projection is folded into layer 0
                              // (set by kbs_tc_input_proj_all(.., r_out); persistent kernel only)
  float* carry[2];            // ABI carries [depth][2][n][H]
  // carry_ld != 0 (persistent kernel only): the carries are rows of a flat per-env record instead (convert.py carry
  // [n][depth*2*H + 20]): element (slot = 2 * layer + {h, c}, env e, unit k) at carry[net][e * carry_ld + slot * H + k],
  // read from carry[] and written to carry_out[] (nullptr = in place).
  int64_t carry_ld;
  float* carry_out[2];
  const uint8_t* done;        // [T][ld]
  const float* actor_obs;     // [T][65][ld]
  float* lpf;                 // [20][ld]
  const float* eps_action;    // [T][20][ld] or nullptr
  const float* qpos;          // [T][27][ld]
  const float* qvel;          // [T][26][ld]
  kbs_episode_view ep;
  float* action; float* log_prob; float* ctrl; float* value;   // action / ctrl may be nullptr (PPO-variable pass)
  const float* action_in;     // [T][20][ld] stored actions whose log-prob is wanted, or nullptr (log-prob of own sample)
  float* entropy;             // [T][ld] or nullptr
  float* action_std;          // [T][20][ld] or nullptr
  float* mean;                // [T][20][ld] dist.mean() or nullptr (persistent kernel only)
  // save != 0 (forward pass of the PPO update; FP16-split persistent kernel only): every step keeps its operands and
  // activations for the backward pass -- xmid_hist [depth][T] x sb, hsb_hist [depth][T + 1] x sb, c_hist [depth][T + 1] x np*H,
  // save_g [T][depth][4] x np*H, sraw [T][20][ld]; carry[] may be nullptr (zeros); the final carries are not written back.
  int save;
  char* xmid_hist[2]; char* hsb_hist[2]; float* c_hist[2]; float* save_g[2]; float* sraw;
  KbsTcRolloutWs ws;          // kbs_tc_rollout_ws for (with_critic ? 2 : 1) nets
  // res_hsb_slot != nullptr (kbs_rollout_step, T = 1, persistent kernel only): the carries are resident in a step state in
  // the kernel's own layouts -- per net hsb [depth][2] x sb and fb [depth][c, h] x np*H, and the device word naming the hsb
  // slot this launch reads -- so nothing is converted on either side; carry[] is not read
  char* res_hsb[2]; float* res_fb[2]; const int* res_hsb_slot;
  int64_t chunk_len;          // > 0: before step t with t % chunk_len == 0, wait for chunk_events[t / chunk_len]
  cudaEvent_t* chunk_events;  //      (the input projections of that chunk of steps, produced on another stream)
};
// the online step's resident carries of one net (kbs_net_tc.cu): pieces of the caller's step state, carved like scratch
struct KbsTcStepNet { char* hsb; float* fb; };
KbsTcStepNet kbs_tc_step_net(KbsScratch& s, const kbs_handle* h, int64_t n);
int kbs_tc_step_carry(kbs_handle* h, float* carry, const KbsTcStepNet& w, int64_t n, bool to_state, cudaStream_t st);
int64_t kbs_tc_sb_floats(const kbs_handle* h, int64_t n);
int64_t kbs_tc_obs_sb_floats(const kbs_handle* h, int net, int64_t n, int64_t T);
// cinert / cvel != nullptr: the critic's privileged dump (features 80..447) is read from the recorded state
// ([T][240][ld] / [T][144][ld]) instead of obs_soa[critic]
int kbs_tc_input_proj_all(kbs_handle* h, int nets, const float* const* obs_soa, float* const* obs_sb, float* const* x_sb_all,
                          int64_t ld, int64_t n, int64_t T, cudaStream_t st, const float* cinert = nullptr,
                          const float* cvel = nullptr, struct KbsTcRolloutArgs* r_out = nullptr);
bool kbs_tc_fused_input(const kbs_handle* h, int net, int64_t n, int64_t T, int nets);
int kbs_tc_rollout_recurrent(kbs_handle* h, const KbsTcRolloutArgs& r, cudaStream_t st);
// true when kbs_tc_rollout_recurrent will take the persistent kernel for this shape (all T steps in one launch)
bool kbs_tc_persistent_available(const kbs_handle* h, int64_t n, int64_t T, int nets);
int kbs_tc_debug_trace(kbs_handle* h, long long* trace_out, const KbsTcRolloutWs& ws, int64_t n, cudaStream_t st);
// tensor-core GEMMs of the PPO update
int kbs_tc_gates_fwd(kbs_handle* h, int net, int layer, const void* x_sb, const void* h_sb, float* gates_out, int64_t n,
                     cudaStream_t st);
int kbs_tc_pack_bwd(kbs_handle* h, int net, cudaStream_t st, int tile = 128);
int kbs_tc_bptt_tile(const kbs_handle* h, int64_t n);   // tile width kbs_tc_bptt will use for n trajectories (64 | 128): pack for it
int kbs_tc_bwd_gemm(kbs_handle* h, int net, int layer, const void* dG_sb, float* out, int64_t n, float out_scale, cudaStream_t st);
size_t kbs_tc_rows_sb_bytes(const kbs_handle* h, int64_t n, int K);
// weight-gradient GEMMs C = A^T B over K = all stored rows (split-K tcgen05; operands = transposed split-blocked buffers)
struct KbsTnPlan { int kb_split, ksplit, kb_total; size_t col_bytes; };
KbsTnPlan kbs_tc_tn_plan(const kbs_handle* h, int64_t rows);
int kbs_tc_pack_tn(kbs_handle* h, const KbsTnPlan& plan, bool b_operand, const float* src, int64_t ld, int col0, int ncols,
                   int ncols_pad, int64_t rows, char* dst, float scale, int ones_col, cudaStream_t st, int64_t n_step = 0,
                   int64_t np_step = 0);
int kbs_tc_gemm_tn(kbs_handle* h, const KbsTnPlan& plan, const char* a_t, int m_panels, int m_valid, const char* b_t, int n_tiles,
                   const char* ones_blk, const float* zero_bias, float* partial, float out_scale, cudaStream_t st);
int kbs_tc_ones_block(kbs_handle* h, char* blk, cudaStream_t st);
// the same operands from the per-step split-blocked buffers the persistent kernels keep (K' = t np + row), FP16 kind:
// source K blocks [blk0, blk0 + nblk) of every step -> nblk / 4 panels (A) or tiles (B) at dst
int kbs_tc_sb_to_tn(kbs_handle* h, const KbsTnPlan& plan, bool b_operand, const char* src, size_t step_bytes, int kb_src, int blk0,
                    int nblk, int64_t n, int64_t T, char* dst, cudaStream_t st);
int kbs_tc_soa_to_tn(kbs_handle* h, const KbsTnPlan& plan, const float* soa, int F, int64_t ld, int64_t n, int64_t T, int ncols_pad,
                     bool ones, char* dst, cudaStream_t st);
// the four big weight-gradient GEMMs of an update straight from the kept per-step operands (dw_gemm_kernel: MN-major UMMA
// operands, no K = row re-pack); partial = the K-major GEMM's slabs [ksplit][4H][2H + 128]
bool kbs_tc_dw_direct_available(const kbs_handle* h, int64_t n);
int kbs_tc_dw_direct(kbs_handle* h, const KbsTnPlan& plan, const char* dG, const char* x_hist, const char* h_hist, int64_t n, int64_t T,
                     float* partial, float out_scale, cudaStream_t st);
// backward recurrence of the PPO update as one persistent kernel (bptt_persist_kernel)
struct KbsBpttNet {
  char* dG; const float* save_g; const float* c_hist; const float* dh_top; float* dx; char* dx0; float* dc; unsigned int* flags;
  char* tn_dG[KBS_MAX_DEPTH];      // optional: per layer, the K = row re-pack of dG (written by the kernel's transposer CTAs)
  const float* dv; const float* w_out;   // dh_top == nullptr: one-row output layer, dh_top = dv [T * n] x w_out [H] (rank 1)
};
struct KbsBpttArgs {
  KbsBpttNet net[2]; int nets; int64_t n, ld, T; const uint8_t* done; float gscale;
  const KbsTnPlan* tn_plan;        // with tn_dG: layout of the re-packed operands
  bool* transposed_out;            // set to whether the kernel re-packed dG itself (enough idle SMs) or the caller has to
};
// forward recurrence of the PPO update (lstm_fwd_save_kernel): LSTM stacks only, everything kept for the backward pass
struct KbsFwdSaveNet {
  const char* x0; char* xmid; char* hsb; float* c_hist; float* save_g; float* h_top_rm; unsigned int* flags;
  const float* carry0;             // ABI [depth][2][n][H] or nullptr (zeros)
  char* tn_xh[KBS_MAX_DEPTH];      // optional: per layer, the K = row re-pack of [x | h_in] (B operand of the dW GEMMs)
};
struct KbsFwdSaveArgs {
  KbsFwdSaveNet net[2]; int nets; int64_t n, ld, T; const uint8_t* done;
  const KbsTnPlan* tn_plan; bool* transposed_out;
};
size_t kbs_tc_fwd_save_flag_bytes(const kbs_handle* h, int64_t n);
bool kbs_tc_fwd_save_available(const kbs_handle* h, int64_t n, int64_t T);
int kbs_tc_fwd_save(kbs_handle* h, const KbsFwdSaveArgs& f, cudaStream_t st);
size_t kbs_tc_bptt_flag_bytes(const kbs_handle* h, int64_t n);
bool kbs_tc_bptt_available(const kbs_handle* h, int64_t n, int64_t T);
int kbs_tc_bptt(kbs_handle* h, const KbsBpttArgs& a, cudaStream_t st);
int kbs_tc_tn_reduce(kbs_handle* h, const KbsTnPlan& plan, const float* partial, int m_panels, int ldc, int col0, int nrows,
                     int ncols, float* dst, int ld_dst, cudaStream_t st);
int kbs_tc_tn_reduce_multi(kbs_handle* h, const KbsTnPlan& plan, const float* partial, int m_panels, int ldc, int nrows, int nseg,
                           const int (*seg)[3], float* const* dst, cudaStream_t st);
int kbs_tc_kind_of(const kbs_handle* h);
int kbs_tc_debug_gates(kbs_handle* h, int net, int layer, const float* x_rm, const float* h_rm, float* gates_out,
                       float* ws, int64_t n, cudaStream_t st);

// heads (kbs_net_simt.cu): consume out_rowmajor
int kbs_launch_actor_head(kbs_handle* h, const float* out_rm, int ldo, const float* obs_soa, int64_t ld, float* lpf,
                          const float* eps, const float* action_in, const uint8_t* done, const kbs_actor_out& o,
                          int64_t n, cudaStream_t st);
int kbs_launch_critic_head(kbs_handle* h, const float* out_rm, int ldo, float* value, int64_t n, cudaStream_t st);

// ---- device helpers ---------------------------------------------------------------------------------
__device__ __forceinline__ void kbs_ld4(const float* __restrict__ base, int64_t row, int64_t ld, int64_t n0,
                                        float (&v)[4]) {
  const float4 t = __ldcs(reinterpret_cast<const float4*>(base + row * ld + n0));
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void kbs_st4(float* __restrict__ base, int64_t row, int64_t ld, int64_t n0,
                                        const float (&v)[4]) {
  __stcs(reinterpret_cast<float4*>(base + row * ld + n0), make_float4(v[0], v[1], v[2], v[3]));
}
__device__ __forceinline__ void kbs_copy4(const float* __restrict__ src, int64_t srow, float* __restrict__ dst,
                                          int64_t drow, int64_t ld, int64_t n0) {
  __stcs(reinterpret_cast<float4*>(dst + drow * ld + n0),
         __ldcs(reinterpret_cast<const float4*>(src + srow * ld + n0)));
}

constexpr int kKbsPanelRows = 128;   // rows of an activation panel (UMMA M)
// ---- "SB" split-blocked operand format of the tcgen05 datapath (see kbs_net_tc.cu) -----------------------------------
// An fp32 value travels as two tensor-core-exact planes:  KIND_TF32: hi = rn_tf32(x), lo = rn_tf32(x - hi)  (2 x 4 B)
//                                                          KIND_F16 : hi = rn_f16(x),  lo = rn_f16((x - hi) * 2^11) (2 x 2 B)
// A "chunk" is 16 bytes of consecutive K (4 tf32 / 8 f16 elements); a block = 4 chunks; layout of one panel (R rows):
//   [k-block][hi|lo][chunk 0..3][row 0..R-1][16 B]   == UMMA canonical K-major SWIZZLE_NONE (LBO = R*16 B, SBO = 128 B)
enum { KBS_KIND_TF32 = 0, KBS_KIND_F16 = 1 };
constexpr float kKbsF16LoScale = 2048.0f;   // 2^11
inline __host__ __device__ constexpr int kbs_chunk_elems(int kind) { return kind == KBS_KIND_TF32 ? 4 : 8; }
inline __host__ __device__ constexpr int kbs_block_k(int kind) { return 4 * kbs_chunk_elems(kind); }   // 16 / 32
// bytes of an SB buffer holding rows x K (rows padded to panels, K to blocks by the caller)
inline size_t kbs_sb_bytes(int64_t rows_padded, int K) { return size_t(rows_padded) * size_t(K) * 2 * 4; }   // tf32
inline size_t kbs_sb_bytes_kind(int kind, int64_t rows_padded, int K) {
  return size_t(rows_padded) * size_t(K) * 2 * (kind == KBS_KIND_TF32 ? 4 : 2);
}
#ifdef __CUDACC__
#include <cuda_fp16.h>
__device__ __forceinline__ float tf32_rn(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
// float(a) + c rounded once to fp32: sm_100's mixed-precision add (one FHADD, no separate f16 -> f32 conversion)
__device__ __forceinline__ float kbs_add_f16_f32(__half a, float c) {
  float d;
  asm("add.rn.f32.f16 %0, %1, %2;" : "=f"(d) : "h"(__half_as_ushort(a)), "f"(c));
  return d;
}
// byte offset of the 16-byte chunk holding (row, k) in plane `part`
// WB = weight-block variant: [k-block][chunk][hi|lo][row][16 B], i.e. the hi and lo rows of one k-chunk are adjacent, so
// ONE N = 2R descriptor (LBO = 2R*16 B) presents [W_hi | W_lo] to the tensor core and x_hi . [W_hi | W_lo]^T comes out of a
// single instruction (A is streamed from shared memory once instead of twice).
template <int R, int KIND, bool WB = false>
__device__ __forceinline__ size_t sb_chunk_offset(int64_t row, int k, int kblocks, int part) {
  constexpr int E = kbs_chunk_elems(KIND);
  const int64_t panel = row / R;
  const int r = int(row - panel * R);
  const int b = k / (4 * E), kc = (k / E) & 3;
  if (WB) return ((((size_t(panel) * kblocks + b) * 4 + kc) * 2 + part) * size_t(R) + size_t(r)) * 16;
  return ((((size_t(panel) * kblocks + b) * 2 + part) * 4 + kc) * size_t(R) + size_t(r)) * 16;
}
// split 4 consecutive K values into the (hi, lo) planes: 16 B each for TF32, 8 B each for F16
struct KbsSplit4 { uint4 hi, lo; };   // F16 uses .x/.y only
template <int KIND>
__device__ __forceinline__ KbsSplit4 sb_split4(const float (&x)[4]) {
  KbsSplit4 s;
  if (KIND == KBS_KIND_TF32) {
    float h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { h[i] = tf32_rn(x[i]); l[i] = tf32_rn(x[i] - h[i]); }
    s.hi = make_uint4(__float_as_uint(h[0]), __float_as_uint(h[1]), __float_as_uint(h[2]), __float_as_uint(h[3]));
    s.lo = make_uint4(__float_as_uint(l[0]), __float_as_uint(l[1]), __float_as_uint(l[2]), __float_as_uint(l[3]));
  } else {
    // hi = fp16(x), and lo = (x - hi) 2^11 is taken from that same fp16 value (hi - x is exact in fp32), so lo carries the
    // whole residual at every magnitude: within fp16's normal range (|x| >= 2^-14) hi keeps 11 significant bits; below it hi
    // is a multiple of 2^-24, the subnormal spacing.  A hi rounded to 11 bits in fp32 and only then converted would round a
    // second time below 2^-14, up to 2^-25 that neither plane holds.  The split's error is <= 2^-22 |x| + 2^-36 (the last
    // term: lo's own rounding in fp16's subnormal range).  The f32 -> f16 conversions run on the quarter-rate XU pipe shared
    // with ex2/rcp, so they are issued packed (cvt.rn.f16x2.f32); hi - x is one mixed-precision add (kbs_add_f16_f32).
    const __half2 h01 = __floats2half2_rn(x[0], x[1]), h23 = __floats2half2_rn(x[2], x[3]);
    const float d0 = kbs_add_f16_f32(__low2half(h01), -x[0]), d1 = kbs_add_f16_f32(__high2half(h01), -x[1]);
    const float d2 = kbs_add_f16_f32(__low2half(h23), -x[2]), d3 = kbs_add_f16_f32(__high2half(h23), -x[3]);
    const __half2 l01 = __floats2half2_rn(d0 * -kKbsF16LoScale, d1 * -kKbsF16LoScale);
    const __half2 l23 = __floats2half2_rn(d2 * -kKbsF16LoScale, d3 * -kKbsF16LoScale);
    s.hi = make_uint4(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23), 0u, 0u);
    s.lo = make_uint4(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23), 0u, 0u);
  }
  return s;
}
template <int R, int KIND, bool WB = false>
__device__ __forceinline__ void sb_store_split(void* __restrict__ sb, int64_t row, int k, int kblocks, const KbsSplit4& s) {
  char* base = reinterpret_cast<char*>(sb);
  if (KIND == KBS_KIND_TF32) {
    *reinterpret_cast<uint4*>(base + sb_chunk_offset<R, KIND, WB>(row, k, kblocks, 0)) = s.hi;
    *reinterpret_cast<uint4*>(base + sb_chunk_offset<R, KIND, WB>(row, k, kblocks, 1)) = s.lo;
  } else {
    const int sub = (k & 4) * 2;   // byte offset of the half-chunk inside the 16-byte chunk
    *reinterpret_cast<uint2*>(base + sb_chunk_offset<R, KIND, WB>(row, k, kblocks, 0) + sub) = make_uint2(s.hi.x, s.hi.y);
    *reinterpret_cast<uint2*>(base + sb_chunk_offset<R, KIND, WB>(row, k, kblocks, 1) + sub) = make_uint2(s.lo.x, s.lo.y);
  }
}
// 8 consecutive K values (k % 8 == 0) from two splits: FP16 kind = ONE 16-byte chunk per plane; zero = store zeros
template <int R, int KIND>
__device__ __forceinline__ void sb_store_split8(void* __restrict__ sb, int64_t row, int k, int kblocks, const KbsSplit4& a,
                                                const KbsSplit4& b, bool zero) {
  char* base = reinterpret_cast<char*>(sb);
  const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
  if (KIND == KBS_KIND_TF32) {
    *reinterpret_cast<uint4*>(base + sb_chunk_offset<R, KIND>(row, k, kblocks, 0)) = zero ? z4 : a.hi;
    *reinterpret_cast<uint4*>(base + sb_chunk_offset<R, KIND>(row, k, kblocks, 1)) = zero ? z4 : a.lo;
    *reinterpret_cast<uint4*>(base + sb_chunk_offset<R, KIND>(row, k + 4, kblocks, 0)) = zero ? z4 : b.hi;
    *reinterpret_cast<uint4*>(base + sb_chunk_offset<R, KIND>(row, k + 4, kblocks, 1)) = zero ? z4 : b.lo;
  } else {
    *reinterpret_cast<uint4*>(base + sb_chunk_offset<R, KIND>(row, k, kblocks, 0)) =
        zero ? z4 : make_uint4(a.hi.x, a.hi.y, b.hi.x, b.hi.y);
    *reinterpret_cast<uint4*>(base + sb_chunk_offset<R, KIND>(row, k, kblocks, 1)) =
        zero ? z4 : make_uint4(a.lo.x, a.lo.y, b.lo.x, b.lo.y);
  }
}
// FP16-split operands must stay finite and below the largest half (65504): anything else would silently become inf in the
// hi plane.  Callers OR the per-thread result over the warp and set KBS_STATUS_F16_RANGE in the handle's health word.
template <int KIND, int NV>
__device__ __forceinline__ bool sb_out_of_range(const float (&x)[NV]) {
  if (KIND != KBS_KIND_F16) return false;
  float m = 0.0f;
#pragma unroll
  for (int i = 0; i < NV; ++i) m = fmaxf(m, fabsf(x[i]));      // fmaxf drops NaNs: test them separately
  bool bad = !(m < 65504.0f);
#pragma unroll
  for (int i = 0; i < NV; ++i) bad = bad || (x[i] != x[i]);
  return bad;
}
__device__ __forceinline__ void sb_flag_range(unsigned int* status, bool bad) {
  if (bad && status) atomicOr(status, unsigned(KBS_STATUS_F16_RANGE));       // rare: a predicated-off branch otherwise
}
// store 4 consecutive K values (k % 4 == 0)
template <int R, int KIND, bool WB = false>
__device__ __forceinline__ void sb_store4(void* __restrict__ sb, int64_t row, int k, int kblocks, const float (&x)[4]) {
  sb_store_split<R, KIND, WB>(sb, row, k, kblocks, sb_split4<KIND>(x));
}
// Counter-based Philox4x32-10 (Salmon et al., SC'11): 128-bit counter c, 64-bit key k -> 4 x 32 random bits.  Shared by the
// rollout noise (kbs_generate_rollout_noise) and the minibatch permutation (kbs_minibatch_permutation), whose counters are
// disjoint: the permutation's fourth counter word is 0xFFFFFFFF, which no rollout-noise row index reaches.
__device__ __forceinline__ uint4 kbs_philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
  }
  return c;
}
#endif  // __CUDACC__

static inline bool kbs_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
