// kbs_net_tc.cu -- tcgen05 (5th-gen tensor core) datapath of the LSTM trunk, fp32-accurate by 3xTF32.
//
// One kernel = one LSTM layer-step for a 128-env tile x 64 hidden units (all four gates):
//     gates[128][256] = [x | h_prev][128][2H] . Wcat[256][2H]^T          (tcgen05.mma kind::tf32, fp32 accum in TMEM)
//     epilogue: + bias, c' = s(f) c + s(i) tanh(g), h' = s(o) tanh(c')   (eqx LSTMCell, train.py:889-893, 919)
// Every fp32 operand x is carried as a pair of TF32-representable planes hi = rn_tf32(x), lo = rn_tf32(x - hi) and the
// product is accumulated as hi.hi + hi.lo + lo.hi (the lo.lo term is below 2^-22 relative): three MMAs per K-step,
// |error| ~ fp32 rounding, which is what the 1e-5 parity bound needs (SURVEY F7).
// MEASURED (tools/tc_accum_probe.py, profiles/r01_tc_accumulation.md): tcgen05 adds each MMA's K=8 partial sum to the
// fp32 accumulator with TRUNCATION (round toward zero), ~0.6 ulp of bias per instruction.  The small hi.lo / lo.hi
// terms therefore go to their OWN accumulator (TMEM columns 256..511) and meet the hi.hi sum in the epilogue with a
// round-to-nearest FADD: 64 instead of 192 truncations on the O(1) accumulator, and no small term is truncated away.
//
// Operand layout ("SB" = split-blocked): 128-row panels (A) / 256-column gate tiles (B), K cut into blocks of 16; a
// block holds [hi|lo][4 k-chunks of 16 B][rows][4 floats] -- exactly the UMMA canonical K-major SWIZZLE_NONE layout
// (8-row x 16-byte core matrices, SBO = 128 B between 8-row groups, LBO = rows*16 B between k-chunks), so one
// cp.async.bulk per operand per stage lands it in shared memory ready for the tensor core, no tensor map needed.
// Weights are packed once (kbs_weights_pack); activations are written in SB form by the producing epilogue.
#include <math.h>
#include <cuda.h>
#include <stdlib.h>

#include "kbs_common.cuh"

namespace {

constexpr int kPanelRows = 128;          // UMMA M
constexpr int kTileCols = 128;           // UMMA N: 32 hidden units x 4 gates (gate-interleaved), or 128 plain columns (proj)
constexpr int kUnitsPerTile = 32;
// One pipeline stage = one SB block of each operand = 4 chunks of 16 B along K (2 MMA k-steps): K = 16 for TF32
// operands, 32 for F16 operands -- the BYTES (and therefore all shared-memory offsets / descriptors) are identical.
#ifndef KBS_STAGES
#define KBS_STAGES 6
#endif
constexpr int kStages = KBS_STAGES;
constexpr int kABlockBytes = 2 * 4 * kPanelRows * 16;   // [hi|lo][4 chunks][128 rows][16 B] = 16 KB
constexpr int kBBlockBytes = 2 * 4 * kTileCols * 16;    // 16 KB
constexpr int kStageBytes = kABlockBytes + kBBlockBytes;   // 32 KB
static_assert(kABlockBytes == kBBlockBytes, "the two producer lanes copy equal-sized blocks");
// Persistent CTA (one per SM) walking a list of (net, panel, tile) items.  TMEM holds TWO accumulator sets
// {hi.hi sum | correction sum} x 128 columns, so the epilogue of item j (TMEM -> cell math -> state stores) overlaps the
// MMAs of item j+1 -- with 256-column tiles both accumulators filled TMEM and the epilogue (as long as the FP16 K loop,
// profiles/r01_tc_kernel_phases.md) ran serially after it.
// warp 0 = MMA issuer (+ TMEM allocation); warps 1..3 = bulk-copy producers (lane 0; one thread can start a stage only
// every ~735 cycles, profiles/r01_bulk_copy_microbench.md); warps 4..11 = epilogue (2 per TMEM lane quarter).
// MEASURED (tools/tc_trace.py per-stage stamps): one thread issues a tcgen05.mma only every ~108 cycles, which hides
// behind a 128-cycle N = 256 instruction but not behind a 64-cycle N = 128 one -- so THREE threads issue, two MMAs per
// stage each: warp 0 the hi.hi MMAs (main set), warps 1 / 2 the lo.hi + hi.lo MMAs of k-step 0 / 1 (correction set).
// All three commit to the stage's empty barrier; warp 2's first MMA of an item is ordered after warp 1's (which
// zero-initialises the correction set) with tcgen05.fence + an mbarrier.
constexpr int kIssuers = 3;
constexpr int kProducers = 2;
constexpr int kEpiWarps = 8;
constexpr int kThreadsTC = 32 * (kIssuers + kProducers + kEpiWarps);
constexpr int kMaxBias = 1024;           // 4H floats per net (H <= 256)
constexpr int kSmemBytes = kStages * kStageBytes + 2 * kMaxBias * 4 + 256 /*barriers*/ + 1024 /*align*/;

// ---- PTX wrappers -----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// one lane of a converged warp; the surrounding code stays warp-uniform, so the compiler keeps descriptors / addresses
// in uniform registers instead of moving them there (R2UR) for every tcgen05 instruction
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// UMMA shared-memory descriptor, K-major, SWIZZLE_NONE (cute::UMMA::SmemDescriptor: addr>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout_type=0 [61,64)).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return uint64_t((saddr >> 4) & 0x3FFFu) | (uint64_t((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         (uint64_t((sbo_bytes >> 4) & 0x3FFFu) << 32) | (uint64_t(1) << 46);
}
// instruction descriptor: D = F32 (1<<4), A = B = TF32 (2<<7, 2<<10), both K-major, N>>3 at [17,23), M>>4 at [24,29)
// (F16 operands: format code 0, kind::f16, K = 16 per instruction)
template <int N>
__host__ __device__ constexpr uint32_t idesc_tf32() { return (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(N >> 3) << 17) | (uint32_t(kPanelRows >> 4) << 24); }
template <int N>
__host__ __device__ constexpr uint32_t idesc_f16() { return (1u << 4) | (0u << 7) | (0u << 10) | (uint32_t(N >> 3) << 17) | (uint32_t(kPanelRows >> 4) << 24); }

template <int KIND, int N>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  if (KIND == KBS_KIND_TF32) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc_tf32<N>()), "r"(accumulate) : "memory");
  } else {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc_f16<N>()), "r"(accumulate) : "memory");
  }
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
      "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]),
        "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]),
        "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Epilogue activations on the SFU: ex2.approx / rcp.approx are accurate to ~2^-22 relative, i.e. sigma and tanh carry
// an ABSOLUTE error below 4e-7 -- under the ~1e-6 the truncating tensor-core accumulation already costs -- at ~6
// instructions instead of ~25 for expf/tanhf + IEEE division (the epilogue was ~20 % of the kernel).
__device__ __forceinline__ float fast_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigmoidf_(float x) {
  return fast_rcp(1.0f + fast_ex2(-1.4426950408889634f * x));          // 1 / (1 + e^-x); e^-x -> inf gives 0
}
// s(a) * tanh(b) with ONE reciprocal: (1 - e_b) / ((1 + e_a)(1 + e_b)), e_a = e^-a (may be +inf -> 0), e_b = e^-2|b| <= 1
__device__ __forceinline__ float sig_mul_tanh(float a, float b) {
  const float ea = fast_ex2(-1.4426950408889634f * a);
  const float eb = fast_ex2(-2.885390081777927f * fabsf(b));
  return copysignf((1.0f - eb) * fast_rcp((1.0f + ea) * (1.0f + eb)), b);
}

__device__ __forceinline__ float tanhf_(float x) {
  const float e = fast_ex2(-2.885390081777927f * fabsf(x));            // e^-2|x| <= 1
  return copysignf((1.0f - e) * fast_rcp(1.0f + e), x);
}

// fp32 "FB" blocked layout of a [rows][H] state matrix: [panel][H/4][128 rows][4 floats] -- a thread that owns one row
// reads/writes 16 B at consecutive addresses across the warp (the row-major ABI layout costs one sector per lane).
__device__ __forceinline__ size_t fb_offset(int64_t row, int k, int H) {
  const int64_t panel = row / kPanelRows;
  const int r = int(row - panel * kPanelRows);
  return ((size_t(panel) * (H / 4) + (k >> 2)) * kPanelRows + r) * 4;   // floats
}

// ---- the layer kernel -----------------------------------------------------------------------------------------------
enum { MODE_LSTM = 0, MODE_PROJ = 1, MODE_RAW = 2, MODE_PROJ_SOA = 3, MODE_PLAIN = 4 };   // PLAIN: fp32 row-major [n][ldo] output
constexpr int kSoaWarps = 4;             // MODE_PROJ_SOA: warps 1..4 build the activation stage in shared memory, one row per thread
struct LayerArgs {
  const char* x_sb;       // A blocks, first K segment: [panels][kb_x] blocks (layer input / observation rows)
  const char* h_sb_in;    // A blocks, second K segment: [panels][kb_h] blocks (h_{t-1}, reset where done_{t-1}); kb_h may be 0
  const char* w_sb;       // B blocks: [tiles][kb_x + kb_h]
  const float* bias_t;    // [tiles][128] bias in tile-column order
  float* c;               // LSTM: cell carry in/out (reset where done), fp32 "FB" blocked layout (fb_offset)
  float* h_carry;         // LSTM: hidden carry out (reset where done), FB layout
  char* h_sb_out;         // LSTM: SB recurrent state out (reset where done); must NOT alias h_sb_in
  char* x_next_sb;        // LSTM: SB input of the next layer (un-reset) or nullptr.  PROJ: SB output [rows][H]
  float* h_next_rm;       // LSTM: [n][H] row-major un-reset output (last layer) or nullptr
  float* raw;             // RAW: [n][4H] pre-activation gates in eqx order (i,f,g,o)
  const uint8_t* done;    // [n] or nullptr
  long long* trace;       // debug: per-CTA clock64 stamps [ctas][8] or nullptr
  int64_t n;              // valid rows (LSTM/RAW: envs; PROJ: T * padded envs, all rows valid)
  int H, kb_x, kb_h, mode;
  int panels, tiles;      // work items of this net = panels x tiles (panels = 0: net unused)
  int dbg;                // profiling only (KBS_TC_EPI_DEBUG): 1 = linear instead of sigmoid/tanh, 2 = no state stores
  // MODE_PROJ_SOA: the A operand is built from env-major SoA observations [T][F][ld] by software producers (no packed
  // staging buffer): rows = T x n_pad, row -> (t, env); features >= F and envs >= n_env are zero.  cinert / cvel != nullptr:
  // features 80..447 come straight from the recorded state (critic's privileged dump, train.py:1405-1413).
  const float* soa; const float* cinert; const float* cvel;
  int F; int64_t soa_ld, n_env, n_pad;
  int ldo;                // MODE_PLAIN: row stride of `raw` (floats)
  float oscale;           // MODE_PLAIN: output multiplier (power of two: undoes the operand pre-scaling of small gradients)
  unsigned int* status;   // health word: KBS_STATUS_F16_RANGE when a projection output leaves the FP16-split range (or nullptr)
  // split-K (MODE_PLAIN, the weight-gradient GEMMs of the PPO update: K = all T x n stored rows): the K blocks of a panel /
  // tile are cut into `ksplit` runs of kb_x blocks, one work item each, every run into its own output slab
  // (raw + ks * raw_split_stride) -- a fixed-order reduction kernel adds the slabs (no atomics: bitwise reproducible, and a
  // run stays short enough for the tensor core's truncating accumulation).  kb_stride = K blocks between consecutive
  // panels / tiles of the operands (0 = kb_x + kb_h, the unsplit layout).
  int ksplit, kb_stride;
  size_t raw_split_stride;
  // ones tile: B tile index `ones_tile` (>= 0) is not read from w_sb but is the single block `ones_block` for every K
  // block: column 0 = 1.0, the rest 0 -- its output column 0 is the column sum of A (the bias gradients).
  int ones_tile;
  const char* ones_block;
};
struct LayerArgs2 { LayerArgs net[2]; };   // actor / critic share one launch

struct WorkItem { int net, panel, tile, ks; };
__host__ __device__ __forceinline__ int net_items(const LayerArgs& a) { return a.panels * a.tiles * (a.ksplit > 1 ? a.ksplit : 1); }
__device__ __forceinline__ WorkItem decode_item(const LayerArgs2& args, int item) {
  const int n0 = net_items(args.net[0]);
  WorkItem w;
  w.net = item >= n0 ? 1 : 0;
  int r = item - (w.net ? n0 : 0);
  const int tiles = args.net[w.net].tiles;
  const int per_split = args.net[w.net].panels * tiles;
  w.ks = r / per_split;         // split-K: the items of one K run are adjacent (its A / B blocks are shared through L2)
  r -= w.ks * per_split;
  w.panel = r / tiles;          // consecutive items share the activation panel (L2 reuse of A across its tiles)
  w.tile = r - w.panel * tiles;
  return w;
}

template <int KIND>
__global__ void __launch_bounds__(kThreadsTC, 1) lstm_layer_tc_kernel(const __grid_constant__ LayerArgs2 args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* bias_s = reinterpret_cast<float*>(smem + kStages * kStageBytes);                 // [2 nets][kMaxBias]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes + 2 * kMaxBias * 4);
  uint64_t* full = bars;                      // [kStages]  bulk copies landed
  uint64_t* empty = bars + kStages;           // [kStages]  MMAs have read the stage
  uint64_t* acc_full = bars + 2 * kStages;    // [2]        accumulator set complete
  uint64_t* acc_empty = acc_full + 2;         // [2]        epilogue has pulled the set into registers
  uint64_t* corr_init = acc_empty + 2;        // [2]        warp 1 has issued the zero-initialising correction MMA of the set
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(corr_init + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_items = net_items(args.net[0]) + net_items(args.net[1]);
  long long* tr = args.net[0].trace ? args.net[0].trace + size_t(blockIdx.x) * 8 : nullptr;
  if (tr && threadIdx.x == 0) tr[0] = clock64();
  // CTA 0 only: per-stage stamps of the first 64 stages: [0] producer saw empty, [1] producer issued, [2] MMA saw full,
  // [3] MMA issued + committed
  long long* tr2 = (args.net[0].trace && blockIdx.x == 0) ? args.net[0].trace + size_t(gridDim.x) * 8 : nullptr;
  long long* tr3 = args.net[0].trace ? args.net[0].trace + size_t(gridDim.x) * 8 + 256 + 2 * blockIdx.x : nullptr;   // globaltimer ns
  if (tr3 && threadIdx.x == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); tr3[0] = (long long)gt; }

  if (threadIdx.x == 0) {
    const bool soa_mode = args.net[0].mode == MODE_PROJ_SOA;    // full[s]: the weight copy's expect_tx arrive + one arrive per row warp
    for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], soa_mode ? 1 + kSoaWarps : 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], kEpiWarps); mbar_init(&corr_init[b], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {   // TMEM: 2 accumulator sets x {hi.hi | correction} x 128 fp32 columns = all 512 columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (tr && threadIdx.x == 0) tr[1] = clock64();    // setup done
  // Programmatic dependent launch: the next launch in the stream may start its prologue on SMs this grid has left;
  // every thread that touches memory written by the previous grid executes griddepcontrol.wait first (pdl_wait).
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (args.net[0].mode == MODE_PROJ_SOA && warp >= 1 && warp <= kSoaWarps) {
    // ===== software producers of the fused input projection: thread = one row (t, env) of the 128-row panel.  Per stage
    // (K = 32 features) it reads 32 SoA rows at its env (a warp reads 32 consecutive envs: coalesced), splits them into
    // the hi / lo planes and writes four 16-byte chunks per plane into the stage in UMMA layout; generic-proxy stores
    // are made visible to the tensor core with fence.proxy.async before the warp arrives on full[s].  Warp 1's lane 0
    // also issues the stage's weight block as a bulk copy.  Saves the packed staging buffer's write + read. =====
    const int pw = warp - 1, r = pw * 32 + lane;
    asm volatile("griddepcontrol.wait;" ::: "memory");       // the observations come from the previous grid
    uint32_t g = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const WorkItem w = decode_item(args, item);
      const LayerArgs& a = args.net[w.net];
      const int64_t row = int64_t(w.panel) * kPanelRows + r;
      const int64_t t = row / a.n_pad, e = row - t * a.n_pad;
      const bool valid = e < a.n_env;
      const char* wb = a.w_sb + size_t(w.tile) * a.kb_x * kBBlockBytes;
      constexpr int kE = kbs_chunk_elems(KIND);             // features per 16-byte chunk: 8 (FP16) / 4 (TF32)
      for (int b = 0; b < a.kb_x; ++b, ++g) {
        const int s = g % kStages;
        float x[4 * kE];
#pragma unroll
        for (int i = 0; i < 4 * kE; ++i) {
          const int f = b * (4 * kE) + i;
          x[i] = 0.0f;
          if (valid && f < a.F) {
            const float* p;
            if (a.cinert && f >= 80 && f < 448) {
              const int c = f - 80;
              p = c < 230 ? a.cinert + (t * (10 * KBS_NBODY) + 10 + c) * a.soa_ld : a.cvel + (t * (6 * KBS_NBODY) + 6 + (c - 230)) * a.soa_ld;
            } else {
              p = a.soa + (t * a.F + f) * a.soa_ld;
            }
            x[i] = __ldcs(p + e);
          }
        }
        // NOTE (historical path, KBS_PROJ_FUSED=1 only): generic stores this close behind the reader's tcgen05.commit can
        // race with the tail of its operand reads -- input_proj_fused_kernel waits one stage longer for that reason.
        mbar_wait(&empty[s], ((g / kStages) & 1) ^ 1);
        uint8_t* sa = smem + size_t(s) * kStageBytes;
        if (pw == 0 && lane == 0) {
          mbar_expect_tx(&full[s], kBBlockBytes);
          bulk_g2s(sa + kABlockBytes, wb + size_t(b) * kBBlockBytes, kBBlockBytes, &full[s]);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {                        // chunk c of the block: [part][chunk][row][16 B]
          uint4 hi, lo;
          if (KIND == KBS_KIND_F16) {
            const float x0[4] = {x[8 * c], x[8 * c + 1], x[8 * c + 2], x[8 * c + 3]};
            const float x1[4] = {x[8 * c + 4], x[8 * c + 5], x[8 * c + 6], x[8 * c + 7]};
            const KbsSplit4 s0 = sb_split4<KIND>(x0), s1 = sb_split4<KIND>(x1);
            hi = make_uint4(s0.hi.x, s0.hi.y, s1.hi.x, s1.hi.y);
            lo = make_uint4(s0.lo.x, s0.lo.y, s1.lo.x, s1.lo.y);
          } else {
            const float x0[4] = {x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]};
            const KbsSplit4 s0 = sb_split4<KIND>(x0);
            hi = s0.hi; lo = s0.lo;
          }
          *reinterpret_cast<uint4*>(sa + c * 2048 + r * 16) = hi;
          *reinterpret_cast<uint4*>(sa + 8192 + c * 2048 + r * 16) = lo;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);
      }
    }
  } else if (args.net[0].mode != MODE_PROJ_SOA && warp >= kIssuers && warp < kIssuers + kProducers) {
    if (lane < 2) {
      // ===== producers: global stage g belongs to producer warp g % kProducers.  MEASURED (tools/bulk_copy_bench3.cu): a
      // cp.async.bulk blocks its issuing thread ~530 cycles (16 KB), so the two operand copies of a stage are issued by
      // TWO lanes in one instruction (lane 0: activation block, lane 1: weight block) instead of back to back.
      uint32_t g = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const WorkItem w = decode_item(args, item);
        const LayerArgs& a = args.net[w.net];
        const int kb_x = a.kb_x, kb_total = a.kb_x + a.kb_h;
        const int kbs = a.kb_stride ? a.kb_stride : kb_total;          // split-K: blocks between panels / tiles
        const char* xa = a.x_sb + (size_t(w.panel) * (a.kb_stride ? a.kb_stride : kb_x) + size_t(w.ks) * kb_x) * kABlockBytes;
        const char* ha = a.h_sb_in + size_t(w.panel) * a.kb_h * kABlockBytes;
        const bool ones = a.ones_block != nullptr && w.tile == a.ones_tile;
        const char* wb = ones ? a.ones_block : a.w_sb + (size_t(w.tile) * kbs + size_t(w.ks) * kb_total) * kBBlockBytes;
        for (int b = 0; b < kb_total; ++b, ++g) {
          if (int(g % kProducers) != warp - kIssuers) continue;
          const int s = g % kStages;
          const uint32_t cp_bytes = (a.dbg & 16) ? 16u : uint32_t(kABlockBytes);   // dbg 16: token copies (MMA-rate probe)
          if (lane == 0) {
            if (g < kProducers) asm volatile("griddepcontrol.wait;" ::: "memory");   // activations come from the previous grid
            mbar_wait(&empty[s], ((g / kStages) & 1) ^ 1);
            if (tr2 && g < 64) tr2[g] = clock64();
            mbar_expect_tx(&full[s], 2 * cp_bytes);
          }
          __syncwarp(0x3);
          uint8_t* sa = smem + size_t(s) * kStageBytes;
          const char* src = lane == 0 ? ((b < kb_x) ? xa + size_t(b) * kABlockBytes : ha + size_t(b - kb_x) * kABlockBytes)
                                      : wb + (ones ? size_t(0) : size_t(b) * kBBlockBytes);
          bulk_g2s(sa + lane * kABlockBytes, src, cp_bytes, &full[s]);    // kABlockBytes == kBBlockBytes
          if (tr2 && g < 64 && lane == 0) tr2[64 + g] = clock64();
        }
      }
    }
    __syncwarp();                        // reconverge before the CTA barrier (bar.sync is warp-aligned)
  } else if (warp < kIssuers) {
    if (warp == 0) {
      // ===== MMA issuer (whole warp runs the loop; one elected lane issues; warps 1, 2 idle).  Per k-step two instructions:
      // x_hi . [W_hi | W_lo]^T as ONE N = 256 MMA into [main | correction] columns, x_lo . W_hi^T as an N = 128 MMA into
      // the correction columns; one commit per stage.  MEASURED (tools/stage_pipe_bench.cu): every tcgen05 instruction
      // costs the issue path ~110-128 cycles whoever issues it, so three warps with three commits per stage were no
      // faster than one thread with one -- and one thread fixes the accumulation order (bitwise reproducible). =====
      uint32_t g = 0;
      int j = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++j) {
        const WorkItem w = decode_item(args, item);
        const LayerArgs& a = args.net[w.net];
        const int kb_total = a.kb_x + a.kb_h;
        const int buf = j & 1;
        mbar_wait(&acc_empty[buf], ((j >> 1) & 1) ^ 1);     // the epilogue of item j-2 has drained this set
        tc_fence_after();
        const uint32_t d_main = tmem_base + buf * (2 * kTileCols), d_corr = d_main + kTileCols;
        for (int b = 0; b < kb_total; ++b, ++g) {
          const int s = g % kStages;
          mbar_wait(&full[s], (g / kStages) & 1);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + size_t(s) * kStageBytes);
          const uint32_t sb = sa + kABlockBytes;
          // A block [part][chunk][128 rows][16 B]: part stride 8 KB, chunk stride 2 KB, k-step (2 chunks) 4 KB.
          // B block [chunk][hi|lo][128 rows][16 B]: chunk stride 4 KB (LBO), k-step 8 KB; hi rows then lo rows = one
          // 256-row operand.
          const uint64_t a_hi = umma_desc(sa, 2048, 128), a_lo = umma_desc(sa + 8192, 2048, 128);
          const uint64_t b_all = umma_desc(sb, 4096, 128);
          if (elect_one()) {
            if (tr && g == 0) tr[2] = clock64();        // first stage landed
            if (tr2 && g < 64) tr2[128 + g] = clock64();
            umma<KIND, 2 * kTileCols>(d_main, a_hi, b_all, b != 0);
            umma<KIND, kTileCols>(d_corr, a_lo, b_all, 1);
            umma<KIND, 2 * kTileCols>(d_main, a_hi + (4096 >> 4), b_all + (8192 >> 4), 1);
            umma<KIND, kTileCols>(d_corr, a_lo + (4096 >> 4), b_all + (8192 >> 4), 1);
            umma_commit(&empty[s]);          // frees the stage when these MMAs have read it
            if (tr2 && g < 64) tr2[192 + g] = clock64();
          }
          __syncwarp();
        }
        if (elect_one()) {
          umma_commit(&acc_full[buf]);       // accumulator set complete
          if (tr && j == 0) tr[3] = clock64();
        }
        __syncwarp();
      }
    }
  } else {
    // ===== epilogue: warp%4 selects the TMEM lane quarter, (warp-4)/4 the half of the tile's 128 columns =====
    // the whole bias vector of each net (<= 4 KB) goes to shared memory; only the epilogue warps wait for it (named
    // barrier 1), the issuers and producers are already running
    {
      const int et = threadIdx.x - 32 * (kIssuers + kProducers);
      for (int k = 0; k < 2; ++k) {
        const int nb = args.net[k].panels ? args.net[k].tiles * kTileCols : 0;
        for (int i = et * 4; i < nb; i += 32 * kEpiWarps * 4)
          *reinterpret_cast<float4*>(bias_s + k * kMaxBias + i) = *reinterpret_cast<const float4*>(args.net[k].bias_t + i);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
      asm volatile("griddepcontrol.wait;" ::: "memory");    // state / done / outputs belong to the previous grid until here
    }
    const int q4 = warp & 3, c2 = (warp - kIssuers - kProducers) >> 2;
    const int r = q4 * 32 + lane;
    constexpr float kCorr = (KIND == KBS_KIND_F16) ? (1.0f / kKbsF16LoScale) : 1.0f;   // lo planes are scaled by 2^11
    constexpr int kBlk = kbs_block_k(KIND);
    int j = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++j) {
      const WorkItem w = decode_item(args, item);
      const LayerArgs& a = args.net[w.net];
      const int H = a.H, kb_out = H / kBlk;
      const int buf = j & 1;
      const int64_t R = int64_t(w.panel) * kPanelRows + r;
      const bool live = R < a.n;
      // tile column layout (LSTM): [half c2][gate i,f,g,o][16 units]; this thread: 16 units x 4 gates = 64 columns
      const int u0 = w.tile * kUnitsPerTile + c2 * 16;          // first hidden unit of this thread
      float4 cpre[4];                                           // c_{t-1}, fetched while the MMAs of this item run
      if (a.mode == MODE_LSTM && live) {
#pragma unroll
        for (int q = 0; q < 4; ++q) cpre[q] = *reinterpret_cast<const float4*>(a.c + fb_offset(R, u0 + q * 4, H));
      }
      const bool rst = a.mode == MODE_LSTM && live && a.done && a.done[R];
      mbar_wait(&acc_full[buf], (j >> 1) & 1);
      tc_fence_after();
      if (tr && j == 0 && threadIdx.x == 32 * (kIssuers + kProducers)) tr[4] = clock64();
      const uint32_t tq = tmem_base + (uint32_t(q4 * 32) << 16) + uint32_t(buf * (2 * kTileCols) + c2 * 64);
      float v[64];
      {
        float cr[32];
        tmem_ld32(tq, v);
        tmem_ld32(tq + 32, v + 32);
        tmem_ld32(tq + kTileCols, cr);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] += kCorr * cr[i];
        tmem_ld32(tq + kTileCols + 32, cr);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) v[32 + i] += kCorr * cr[i];
      }
      // the accumulator set is in registers: hand it back to the MMA issuer before doing the math
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
      const float* bs = bias_s + w.net * kMaxBias + w.tile * kTileCols + c2 * 64;
#pragma unroll
      for (int i = 0; i < 64; ++i) v[i] += bs[i];
      if (!live) continue;
      if (a.mode == MODE_PROJ || a.mode == MODE_PROJ_SOA) {
        const int col0 = w.tile * kTileCols + c2 * 64;
        if (col0 < H) {
          sb_flag_range(a.status, sb_out_of_range<KIND, 64>(v));
#pragma unroll
          for (int i = 0; i < 64; i += 4) {
            const float o[4] = {v[i], v[i + 1], v[i + 2], v[i + 3]};
            sb_store4<kPanelRows, KIND>(a.x_next_sb, R, col0 + i, kb_out, o);
          }
        }
      } else if (a.mode == MODE_PLAIN) {
        float* o = a.raw + size_t(w.ks) * a.raw_split_stride + R * a.ldo + w.tile * kTileCols + c2 * 64;
#pragma unroll
        for (int i = 0; i < 64; i += 4)
          *reinterpret_cast<float4*>(o + i) = make_float4(a.oscale * v[i], a.oscale * v[i + 1], a.oscale * v[i + 2], a.oscale * v[i + 3]);
      } else if (a.mode == MODE_RAW) {
        float* g = a.raw + R * 4 * H + u0;
#pragma unroll
        for (int gate = 0; gate < 4; ++gate)
#pragma unroll
          for (int i = 0; i < 16; i += 4)
            *reinterpret_cast<float4*>(g + gate * H + i) =
                make_float4(v[gate * 16 + i], v[gate * 16 + i + 1], v[gate * 16 + i + 2], v[gate * 16 + i + 3]);
      } else {
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
          const float4 c4 = cpre[i >> 2];
          const float cv[4] = {c4.x, c4.y, c4.z, c4.w};
          float hn[4], cn[4], cr[4];
#pragma unroll
          for (int l = 0; l < 4; ++l) {
            const float gi = v[i + l], gf = v[16 + i + l], gg = v[32 + i + l], go = v[48 + i + l];
            // c' = s(f) c + s(i) tanh(g);  h' = s(o) tanh(c')   (eqx LSTMCell)
            if (a.dbg & 1) { cn[l] = gf * cv[l] + gi * gg; hn[l] = go * cn[l]; }
            else {
              cn[l] = sigmoidf_(gf) * cv[l] + sig_mul_tanh(gi, gg);
              hn[l] = sig_mul_tanh(go, cn[l]);
            }
            cr[l] = rst ? 0.0f : cn[l];
          }
          if ((a.dbg & 2) && hn[0] != 12345.0f) continue;
          KbsSplit4 sp = sb_split4<KIND>(hn);               // one split serves the next layer (un-reset) ...
          if (a.x_next_sb) sb_store_split<kPanelRows, KIND>(a.x_next_sb, R, u0 + i, kb_out, sp);
          if (a.h_next_rm) *reinterpret_cast<float4*>(a.h_next_rm + R * H + u0 + i) = make_float4(hn[0], hn[1], hn[2], hn[3]);
          if (rst) { sp.hi = make_uint4(0u, 0u, 0u, 0u); sp.lo = sp.hi; hn[0] = hn[1] = hn[2] = hn[3] = 0.0f; }
          sb_store_split<kPanelRows, KIND>(a.h_sb_out, R, u0 + i, kb_out, sp);   // ... and the recurrent input (reset)
          *reinterpret_cast<float4*>(a.c + fb_offset(R, u0 + i, H)) = make_float4(cr[0], cr[1], cr[2], cr[3]);
          *reinterpret_cast<float4*>(a.h_carry + fb_offset(R, u0 + i, H)) = make_float4(hn[0], hn[1], hn[2], hn[3]);
        }
      }
      if (tr && j == 0 && threadIdx.x == 32 * (kIssuers + kProducers)) tr[7] = clock64();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tr && threadIdx.x == 0) { tr[5] = clock64(); unsigned sm; asm("mov.u32 %0, %%smid;" : "=r"(sm)); tr[6] = sm; }
  if (tr3 && threadIdx.x == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); tr3[1] = (long long)gt; }
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

// ---- fused output head of the rollout (FFMA: N = 40 / 1 is far below a tensor-core tile) ----------------------------
// blockIdx.y = 0: actor  out = W_out h2 + b (train.py:922) -> std/mean/bias/low-pass/sample/log-prob (train.py:924-939,
//                 1564, distrax MVN-diag) -> PD torque (train.py:1091-1105), all for 32 envs per block;
// blockIdx.y = 1: critic value = w_out . h2 + b (train.py:1002).
struct HeadArgs {
  const float* h2[2];        // [n][H] row-major top-layer output (un-reset), actor / critic
  const float* w_out[2];     // [64][H] zero-padded row-major
  const float* b_out[2];     // [64]
  const float* arm_cmd;      // actor_obs rows 55..64 of this step: [10][ld]
  float* lpf;                // [20][ld] in/out
  const float* eps;          // [20][ld] or nullptr (mode)
  const uint8_t* done;       // [ld] or nullptr
  const float* q;            // qpos rows 7.. [20][ld]
  const float* qd;           // qvel rows 6.. [20][ld]
  kbs_episode_view ep;
  float* action; float* log_prob; float* ctrl; float* value;   // [20][ld], [ld], [20][ld] or nullptr, [ld]
  // stored-transition mode of _ppo_scan_fn (train.py:1443-1452, 1486-1487): log-prob of action_in, entropy, stddev
  const float* action_in;    // [20][ld] or nullptr
  float* entropy;            // [ld] or nullptr
  float* std;                // [20][ld] or nullptr
  int64_t n, ld;
  int H;
};
constexpr int kHeadEnvs = 32;

__global__ void __launch_bounds__(128)
rollout_head_kernel(const __grid_constant__ kbs_params P, const __grid_constant__ HeadArgs a) {
  extern __shared__ __align__(16) float hsm[];
  const int H = a.H, hs = H + 4;                 // row stride keeps float4 alignment and spreads banks
  float* h_s = hsm;                              // [32][H + 4]
  float* w_s = hsm + kHeadEnvs * hs;             // [40][H]
  float* out_s = w_s + KBS_ACTOR_OUT * H;        // [32][41]
  float* part = out_s + kHeadEnvs * 41;          // [4][32][2]
  const int net = blockIdx.y;
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int64_t e0 = int64_t(blockIdx.x) * kHeadEnvs;
  const int nout = net == 0 ? KBS_ACTOR_OUT : 1;
  // The per-joint inputs of the head / torque math do not depend on the GEMM: fetch them first so their L2/HBM latency
  // hides under the staging and the out-projection (ncu: the kernel was long-scoreboard bound, FMA pipe 10 % active).
  const int64_t e = e0 + lane;
  const bool live = e < a.n;
  const int64_t ld = a.ld;
  float in_lpf[5], in_eps[5], in_arm[5], in_ain[5], in_q[5], in_qd[5], in_kp[5], in_kd[5], in_lim[5], in_ab[5], in_tb[5];
  bool rst = false;
  if (net == 0 && live) {
    rst = a.done && a.done[e];
#pragma unroll
    for (int jj = 0; jj < 5; ++jj) {
      const int j = 5 * g + jj;
      const int64_t o = j * ld + e;
      in_lpf[jj] = a.lpf[o];
      in_eps[jj] = a.eps ? a.eps[o] : 0.0f;
      in_arm[jj] = (j >= 10) ? a.arm_cmd[(j - 10) * ld + e] : 0.0f;
      in_ain[jj] = a.action_in ? a.action_in[o] : 0.0f;
      if (a.ctrl) {
        in_q[jj] = a.q[o]; in_qd[jj] = a.qd[o];
        in_kp[jj] = a.ep.kp ? a.ep.kp[o] : P.kp[j];
        in_kd[jj] = a.ep.kd ? a.ep.kd[o] : P.kd[j];
        in_lim[jj] = a.ep.tau_limit ? a.ep.tau_limit[o] : P.ctrl_limit[j];
        in_ab[jj] = a.ep.action_bias ? a.ep.action_bias[o] : 0.0f;
        in_tb[jj] = a.ep.torque_bias ? a.ep.torque_bias[o] : 0.0f;
      }
    }
  }
  // stage h2 tile and W_out with cp.async: all ~36 16-byte requests of a thread are in flight at once
  for (int i = threadIdx.x; i < kHeadEnvs * (H / 4); i += 128) {
    const int r = i / (H / 4), c4 = i % (H / 4);
    float* dst = h_s + r * hs + c4 * 4;
    if (e0 + r < a.n) {
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(a.h2[net] + (e0 + r) * H + c4 * 4)
                   : "memory");
    } else {
      *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  for (int i = threadIdx.x; i < nout * (H / 4); i += 128)
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(w_s + i * 4)), "l"(a.w_out[net] + i * 4) : "memory");
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();
  if (net == 1) {
    // critic: 4 warps split K, fixed-order combine
    float s = 0.0f;
    const int kq = H / 4;
    for (int k = g * kq; k < (g + 1) * kq; k += 4) {
      const float4 hv = *reinterpret_cast<const float4*>(h_s + lane * hs + k);
      const float4 wv = *reinterpret_cast<const float4*>(w_s + k);
      s = fmaf(hv.x, wv.x, s); s = fmaf(hv.y, wv.y, s); s = fmaf(hv.z, wv.z, s); s = fmaf(hv.w, wv.w, s);
    }
    part[g * 32 + lane] = s;
    __syncthreads();
    if (g == 0 && live) a.value[e] = ((part[lane] + part[32 + lane]) + (part[64 + lane] + part[96 + lane])) + a.b_out[1][0];
    return;
  }
  // actor: thread (env = lane, outputs 10g .. 10g+9)
  {
    float acc[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) acc[i] = 0.0f;
    const float* wr = w_s + (10 * g) * H;
    for (int k = 0; k < H; k += 4) {
      const float4 hv = *reinterpret_cast<const float4*>(h_s + lane * hs + k);
#pragma unroll
      for (int i = 0; i < 10; ++i) {
        const float4 wv = *reinterpret_cast<const float4*>(wr + i * H + k);
        acc[i] = fmaf(hv.x, wv.x, acc[i]); acc[i] = fmaf(hv.y, wv.y, acc[i]);
        acc[i] = fmaf(hv.z, wv.z, acc[i]); acc[i] = fmaf(hv.w, wv.w, acc[i]);
      }
    }
#pragma unroll
    for (int i = 0; i < 10; ++i) out_s[lane * 41 + 10 * g + i] = acc[i] + a.b_out[0][10 * g + i];
  }
  __syncthreads();
  // head: thread (env = lane, joints 5g .. 5g+4); all global accesses are env-contiguous rows
  float s_z = 0.0f, s_log = 0.0f;
  constexpr float kHalfLog2Pi = 0.918938533204672742f;
  if (live) {
#pragma unroll
    for (int jj = 0; jj < 5; ++jj) {
      const int j = 5 * g + jj;
      const int64_t o = j * ld + e;
      const float sraw = out_s[lane * 41 + KBS_NUM_JOINTS + j];
      const float sp = fmaxf(sraw, 0.0f) + log1pf(expf(-fabsf(sraw)));
      const float sd = fminf((sp + P.min_std) * P.var_scale, P.max_std);
      float m = out_s[lane * 41 + j] + P.joint_bias[j];
      m = m + in_arm[jj];
      const float y = in_lpf[jj];
      const float yn = y + P.lpf_alpha * (m - y);
      a.lpf[o] = rst ? 0.0f : yn;
      float act = yn;
      if (a.eps) act = yn + sd * in_eps[jj];
      const float a_eval = a.action_in ? in_ain[jj] : act;
      const float z = (a_eval - yn) / sd;
      s_z = s_z + (-0.5f * z * z - kHalfLog2Pi);
      s_log = s_log + logf(sd);
      if (a.action) a.action[o] = act;
      if (a.std) a.std[o] = sd;
      if (!a.ctrl) continue;
      // PositionActuators.get_ctrl
      const float target = a.ep.action_bias ? __fadd_rn(act, in_ab[jj]) : act;
      float tau = __fsub_rn(__fmul_rn(in_kp[jj], __fsub_rn(target, in_q[jj])), __fmul_rn(in_kd[jj], in_qd[jj]));
      if (a.ep.torque_bias) tau = __fadd_rn(tau, in_tb[jj]);
      a.ctrl[o] = fminf(fmaxf(tau, -in_lim[jj]), in_lim[jj]);
    }
  }
  part[(g * 32 + lane) * 2] = s_z;
  part[(g * 32 + lane) * 2 + 1] = s_log;
  __syncthreads();
  if (g == 0 && live) {
    float z = 0.0f, l = 0.0f;
#pragma unroll
    for (int w = 0; w < 4; ++w) { z = z + part[(w * 32 + lane) * 2]; l = l + part[(w * 32 + lane) * 2 + 1]; }
    if (a.log_prob) a.log_prob[e] = z - l;
    if (a.entropy) a.entropy[e] = l + float(KBS_NUM_JOINTS) * (0.5f + kHalfLog2Pi);
  }
}

// ---- persistent recurrence kernel: ALL T control steps of the rollout in ONE launch --------------------------------------
// One CTA per SM walks a static, globally ordered list of work items; there is no kernel boundary between steps or
// layers.  Item kinds: LSTM (net, layer l, step t, 128-env panel, 128-column gate tile) -- the same datapath as
// lstm_layer_tc_kernel -- and HEAD (net, step t, panel): out = W_out h_top on the tensor core (W_out zero-padded to one
// 128-column tile), then in the epilogue the whole actor head for the row's env (std / mean / low-pass / sample /
// log-prob / entropy / PD torque, train.py:922-939, 1091-1105, 1564) or the critic value (train.py:1002).
// Order: "slot" s holds layer l at step s - l and the head at step s - depth (a wavefront: everything in a slot depends
// only on earlier slots), items of a slot are panel-major so the ~17 CTAs that share a panel's activations run together.
// Dependencies between CTAs travel through monotone completion counters in global memory, one per (net, layer | head,
// panel): every epilogue warp adds 1 after its stores (fence + red), so "layer l of step t is complete for panel p" is
// counter >= (t + 1) * tiles * kEpiWarps.  The producer lane polls the (at most three) counters an item needs before
// its first bulk copy, then publishes the item's sequence number in shared memory for the epilogue warps (which read
// the cell state with L2-coherent loads).  All CTAs are co-resident (cooperative launch, grid <= SM count) and every
// CTA takes its items in the global order, so the earliest unfinished item can always run: no deadlock.  Polling is
// bounded: after ~2^22 polls a CTA records an error in `status` and stops waiting.
constexpr int kPMaxDepth = 2;            // bias table in shared memory: [2 nets][kPMaxDepth][4H] + head [2][128]
constexpr int kPBiasFloats = 2 * kPMaxDepth * kMaxBias + 2 * 256;
constexpr int kEpiWarpsP = 16;
constexpr int kIssuersP = 1;
constexpr int kProducersP = 1;           // one 16 KB + one 32 KB request per 878-cycle stage: one warp keeps up
constexpr int kThreadsP = 32 * (kIssuersP + kProducersP + kEpiWarpsP + 2);   // + dependency poller warp + publisher warp = 640
constexpr int kPHeadPartFloats = 4 * kPanelRows * 2;
// Tile of the persistent kernel: 128 envs x 256 gate columns (64 hidden units).  MEASURED (tools/stage_pipe_bench.cu): one
// thread issues a tcgen05.mma only every ~110-128 cycles whatever its size, and a tcgen05.commit costs about as much, so
// only N = 256 instructions (128 tensor cycles each) keep the tensor pipe busy: 3 x N = 256 per k-step (hi.hi -> main,
// lo.hi + hi.lo -> correction) = 878 cycles per stage against 768 of tensor work, where the N = 128 tile ran at 643-720
// cycles for 384.  Main + correction of one tile fill the 512 TMEM columns: single-buffered, the epilogue pulls the
// accumulators into registers and hands TMEM back before doing the cell math.
constexpr int kTileColsP = 256;
constexpr int kUnitsPerTileP = kTileColsP / 4;
constexpr int kBBlockBytesP = 2 * 4 * kTileColsP * 16;          // [chunk][hi|lo][256 rows][16 B] = 32 KB
constexpr int kStageBytesP = kABlockBytes + kBBlockBytesP;      // 48 KB
constexpr int kStagesP = 4;              // power of two that divides every item's stage count (8 or 16 at H = 256).  A ring of
                                         // 8 half-stages (24 KB, one k-step, 3 MMAs + commit each) measured the same 20.6 K
                                         // cycles per item: the extra commits eat what the finer ring gives.
constexpr int kPSmemBytes = kStagesP * kStageBytesP + (kPBiasFloats + kPHeadPartFloats) * 4 + 256 /*barriers*/ + 1024 /*align*/;

struct PNet {
  const char* x_sb_all;            // [T] x x0_stride: layer-0 inputs -- the input projection of every step (kb_x0 = H / block
                                   // K), or, for a net whose input projection is folded into layer 0 (kbs_tc_fused_input),
                                   // the packed observations themselves (kb_x0 = padded input width / block K)
  size_t x0_stride;                // bytes per step of x_sb_all
  int kb_x0;                       // K blocks of the layer-0 input operand
  char* hsb;                       // [depth][2] x sbb: recurrent SB state (reset where done); step t reads parity
                                   // (t + *hsb_slot) & 1
  char* xmid;                      // [depth][2] x sbb: un-reset SB output of layer l at step t (parity t & 1)
  float* fb;                       // [depth][c, h] x np*H: fp32 FB state
  const char* w_sb[kPMaxDepth];
  const float* bias_t[kPMaxDepth];
  const char* w_head;              // [128][H] SB, rows >= num_out zero
  const float* bias_head;          // [128]
  unsigned int* flags;             // [depth + 1][panels] completion counters (zeroed before the launch)
  // SAVE instantiation (forward pass of the PPO update, kbs_ppo_grad): nothing is ping-ponged, every step keeps its
  // operands and activations for the backward pass --
  //   xmid [depth][T] x sbb, hsb [depth][T + 1] x sbb (slot t = what step t reads), c_hist [depth][T + 1] x np*H (FB; slot t =
  //   the cell state step t reads, i.e. reset where done_{t-1}), save_g [T][depth][4 gates i,f,g,o] x np*H (FB, activated).
  float* c_hist;
  float* save_g;
};
struct PArgs {
  PNet net[2];
  int nets, depth, H, panels, tiles;
  int gpanels;                     // panels per group of the item order (p_decode); = panels: one group
  int64_t n, ld, T;
  size_t sbb;
  const uint8_t* done;             // [T][ld] or nullptr
  // head I/O (time-major SoA, env contiguous); see HeadArgs
  const float* arm_cmd;            // actor_obs + 55 * ld, stride KBS_ACTOR_OBS * ld per step
  float* lpf;
  const float* eps;                // stride 20 * ld
  const float* q; const float* qd; // qpos + 7 * ld (stride KBS_NQ * ld), qvel + 6 * ld (stride KBS_NV * ld)
  kbs_episode_view ep;
  float* action; float* log_prob; float* ctrl; float* value;
  const float* action_in; float* entropy; float* std;
  float* mean;                     // [T][20][ld] dist.mean() = the low-pass-filtered mean (mirror loss), or nullptr
  float* sraw;                     // [T][20][ld] pre-softplus std output of the actor head (backward pass of the update), or nullptr
  int hist;                        // 1 = SAVE instantiation: per-step buffers, no write-after-read dependencies
  int dbg;                         // profiling only (KBS_PERSIST_DBG): 1 = ignore dependencies (wrong results, timing probe)
  unsigned int* status;            // != 0: a dependency wait timed out (bug / lost CTA)
  const int* hsb_slot;             // device 0 / 1 or nullptr (= 0): the hsb slot step 0 reads.  The online step (T = 1,
                                   // kbs_rollout_step) keeps hsb resident and flips this word after every launch, so a
                                   // replayed launch finds its input where the previous one left it
  long long* trace;                // per CTA [8]: total cycles, poller wait cycles, items, issuer wait-for-stage cycles,
                                   // epilogue cycles in LSTM / head items, epilogue wait-for-accumulator, issuer wait-for-TMEM
};

struct PItem { int kind, net, layer, panel, tile; int t; bool valid; };
// Global item order: panel GROUP (gpanels consecutive panels of both nets), then slot, then (net, panel, layer | head, tile).
// A group runs its whole T-step wavefront before the next group starts (panels are independent): the h / x / c working set
// in flight is gpanels x nets x ~1.5 MB instead of every panel's (96 MB at 4 096 envs: it cycled through the 126 MB L2 once
// per control step, and every activation store of the rollout went to HBM and back: 9 GB per launch against ~1 GB algorithmic).
__device__ __forceinline__ PItem p_decode(const PArgs& a, int g) {
  const int lt = a.depth * a.tiles, per_panel = lt + 1, per_net = a.gpanels * per_panel, C = a.nets * per_net;
  const int per_group = (int(a.T) + a.depth) * C;
  const int grp = g / per_group;
  g -= grp * per_group;
  const int s = g / C;
  int i = g - s * C;
  PItem it;
  it.net = i / per_net; i -= it.net * per_net;
  const int pl = i / per_panel;
  it.panel = grp * a.gpanels + pl;
  const int q = i - pl * per_panel;
  if (q < lt) { it.kind = 0; it.layer = q / a.tiles; it.tile = q - it.layer * a.tiles; it.t = s - it.layer; }
  else { it.kind = 1; it.layer = a.depth; it.tile = 0; it.t = s - a.depth; }
  it.valid = it.t >= 0 && it.t < int(a.T) && it.panel < a.panels;
  return it;
}
__device__ __forceinline__ unsigned int ld_volatile_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Blocks until the counters item `it` depends on have reached their targets; returns cycles spent.  Bounded in WALL-CLOCK
// time (globaltimer: independent of the SM clock): after kPWaitTimeoutNs without progress the CTA records
// KBS_STATUS_TIMEOUT_* in the health word and -- like every other CTA that then sees the word set -- stops waiting
// altogether (`drain`): the launch finishes quickly with garbage results instead of hanging the GPU, and the entry point
// that launched it reports KBS_E_DEVICE at the next call (kbs_enter).
constexpr unsigned long long kPWaitTimeoutNs = 2000000000ull;
__device__ __forceinline__ long long p_wait_deps(const PArgs& a, const PItem& it, bool& drain) {
  if (drain) return 0;
  const PNet& N = a.net[it.net];
  const unsigned int full_l = unsigned(a.tiles * kEpiWarpsP), full_h = unsigned(kEpiWarpsP);
  const unsigned int* fp[3]; unsigned int tg[3]; int nd = 0;
  const unsigned int t = unsigned(it.t);
  if (it.kind == 0) {
    const int l = it.layer;
    if (t >= 1) { fp[nd] = N.flags + l * a.panels + it.panel; tg[nd++] = t * full_l; }              // h_{t-1}, c_{t-1}
    if (l >= 1) { fp[nd] = N.flags + (l - 1) * a.panels + it.panel; tg[nd++] = (t + 1) * full_l; }  // x_t from layer l-1
    if (t >= 2 && !a.hist) {   // xmid[l][t & 1] was last read by the consumer of this layer's output at step t - 2
      fp[nd] = N.flags + (l + 1) * a.panels + it.panel;
      tg[nd++] = (t - 1) * (l + 1 == a.depth ? full_h : full_l);
    }
  } else {
    fp[nd] = N.flags + (a.depth - 1) * a.panels + it.panel; tg[nd++] = (t + 1) * full_l;            // h_top of step t
    if (t >= 1) { fp[nd] = N.flags + a.depth * a.panels + it.panel; tg[nd++] = t * full_h; }       // lpf of step t-1
  }
  if (nd == 0) return 0;
  for (int i = nd; i < 3; ++i) { fp[i] = fp[0]; tg[i] = 0u; }   // fixed three independent loads per poll
  const long long c0 = clock64();
  unsigned int polls = 0;
  unsigned long long t0 = 0;
  while (true) {
    const unsigned int v0 = ld_volatile_u32(fp[0]), v1 = ld_volatile_u32(fp[1]), v2 = ld_volatile_u32(fp[2]);
    if (v0 >= tg[0] && v1 >= tg[1] && v2 >= tg[2]) break;
    if ((++polls & 1023u) == 0u) {
      if (ld_volatile_u32(a.status) & 3u) { drain = true; break; }          // another CTA gave up: drain
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > kPWaitTimeoutNs) { atomicOr(a.status, 1u + unsigned(it.kind)); drain = true; break; }
    }
  }
  __threadfence();                                            // acquire: the counted stores are visible
  return clock64() - c0;
}

template <int KIND, bool SAVE>
__global__ void __launch_bounds__(kThreadsP, 1)
rollout_persist_kernel(const __grid_constant__ kbs_params P, const __grid_constant__ PArgs args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* bias_s = reinterpret_cast<float*>(smem + kStagesP * kStageBytesP);   // [net][layer][kMaxBias] then head [net][256]
  float* bias_head_s = bias_s + 2 * kPMaxDepth * kMaxBias;
  float* head_part = bias_s + kPBiasFloats;                                 // [4 joint groups][128 rows][2]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStagesP * kStageBytesP + (kPBiasFloats + kPHeadPartFloats) * 4);
  uint64_t* full = bars;
  uint64_t* empty = bars + kStagesP;
  uint64_t* acc_full = bars + 2 * kStagesP;
  uint64_t* acc_empty = acc_full + 2;
  uint64_t* corr_init = acc_empty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(corr_init + 2);
  volatile int* dep_seq = reinterpret_cast<volatile int*>(tmem_slot + 1);   // items whose dependencies are satisfied
  unsigned int* epi_done = reinterpret_cast<unsigned int*>(tmem_slot + 2);  // epilogue warps that have stored their share (monotone)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int per_slot = args.nets * args.gpanels * (args.depth * args.tiles + 1);
  const int n_g = ((args.panels + args.gpanels - 1) / args.gpanels) * (int(args.T) + args.depth) * per_slot;
  const int H = args.H;
  const int hslot = (!SAVE && args.hsb_slot) ? *args.hsb_slot : 0;
  constexpr int kBlk = kbs_block_k(KIND);
  const int kb = H / kBlk;
  long long* tr = args.trace ? args.trace + size_t(blockIdx.x) * 16 : nullptr;
  const long long t_start = clock64();
  unsigned long long gt_start = 0;
  if (tr && threadIdx.x == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_start));

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStagesP; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], kEpiWarpsP);
    }
    *dep_seq = 0;
    *epi_done = 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kIssuersP + kProducersP + kEpiWarpsP + 1) {
    if (lane == 0) {
      // ===== publisher: the gpu-scope fence that makes an item's stores visible costs ~2 K cycles of store-ack latency.
      // The epilogue warps therefore only signal "stored" in shared memory (release.cta) and move on; this thread
      // observes all 16 signals (acquire.cta), fences at gpu scope -- cumulative over everything it has observed, the
      // same pattern as bar.sync + one thread's __threadfence() in a grid barrier -- and bumps the item's counter =====
      int j = 0;
      for (int gi = blockIdx.x; gi < n_g; gi += gridDim.x) {
        const PItem it = p_decode(args, gi);
        if (!it.valid) continue;
        ++j;
        const unsigned int want = unsigned(j) * kEpiWarpsP;
        unsigned int seen;
        do {
          asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(seen) : "r"(smem_u32(epi_done)) : "memory");
        } while (seen < want);
        __threadfence();
        atomicAdd(args.net[it.net].flags + it.layer * args.panels + it.panel, unsigned(kEpiWarpsP));
      }
    }
    __syncwarp();
  } else if (warp == kIssuersP + kProducersP + kEpiWarpsP) {
    if (lane == 0) {
      // ===== dependency poller: runs ahead of the producers through the item list, so the L2 round trips of the
      // counter polls and the fence stay off the load pipeline's critical path; publishes "items 0..j-1 may start" =====
      int j = 0;
      long long waited = 0;
      bool drain = false;
      for (int gi = blockIdx.x; gi < n_g; gi += gridDim.x) {
        const PItem it = p_decode(args, gi);
        if (!it.valid) continue;
        if (!(args.dbg & 1)) waited += p_wait_deps(args, it, drain);
        *dep_seq = ++j;
      }
      if (tr) { tr[1] = waited; tr[2] = j; }
    }
    __syncwarp();
  } else if (warp >= kIssuersP && warp < kIssuersP + kProducersP) {
    if (lane < 2) {
      // ===== producers (see lstm_layer_tc_kernel): lane 0 = activation block, lane 1 = weight block of the stage =====
      uint32_t g = 0;
      int j = 0;
      long long pw[3] = {0, 0, 0};
      for (int gi = blockIdx.x; gi < n_g; gi += gridDim.x) {
        const PItem it = p_decode(args, gi);
        if (!it.valid) continue;
        const PNet& N = args.net[it.net];
        const int kb_x = (it.kind == 0 && it.layer == 0) ? N.kb_x0 : kb;
        const int kb_total = it.kind == 0 ? kb_x + kb : kb;
        size_t poff = size_t(it.panel) * kb * kABlockBytes;
        if (args.dbg & 8) poff = size_t(blockIdx.x % args.panels) * kb * kABlockBytes;   // probe: no two CTAs share a panel at a time
        const char* xa; const char* ha; const char* wb;
        if (it.kind == 0) {
          const size_t xs = SAVE ? size_t(it.layer - 1) * size_t(args.T) + size_t(it.t) : size_t((it.layer - 1) * 2 + (it.t & 1));
          const size_t hs = SAVE ? size_t(it.layer) * size_t(args.T + 1) + size_t(it.t) : size_t(it.layer * 2 + ((it.t + hslot) & 1));
          xa = it.layer == 0 ? N.x_sb_all + size_t(it.t) * N.x0_stride + poff / kb * kb_x : N.xmid + xs * args.sbb + poff;
          ha = N.hsb + hs * args.sbb + poff;
          wb = N.w_sb[it.layer] + size_t((args.dbg & 16) ? (blockIdx.x + it.t) % args.tiles : it.tile) * kb_total * kBBlockBytesP;
        } else {
          xa = N.xmid + (SAVE ? size_t(args.depth - 1) * size_t(args.T) + size_t(it.t) : size_t((args.depth - 1) * 2 + (it.t & 1))) * args.sbb + poff;
          ha = xa;
          wb = N.w_head;
        }
        ++j;
        bool need_dep = true;        // lane 0: the item's dependency wait + proxy fence, taken just before its first activation copy
        for (int b = 0; b < kb_total; ++b, ++g) {
          const int s = g % kStagesP;
          // probes: 32 = token weight copies, 128 = no weight request at all, 256 = half-size activation request
          const uint32_t wbytes = (args.dbg & 128) ? 0u : (args.dbg & 32) ? 16u : uint32_t(kBBlockBytesP);
          const uint32_t abytes = (args.dbg & 256) ? uint32_t(kABlockBytes / 2) : uint32_t(kABlockBytes);
          long long p0 = 0, p1 = 0;
          if (lane == 0) {
            if (tr) p0 = clock64();
            mbar_wait(&empty[s], ((g / kStagesP) & 1) ^ 1);
            if (tr) p1 = clock64();
            mbar_expect_tx(&full[s], abytes + wbytes);
          }
          __syncwarp(0x3);
          uint8_t* sa = smem + size_t(s) * kStageBytesP;
          const char* src = lane == 0 ? ((b < kb_x) ? xa + size_t(b) * kABlockBytes : ha + size_t(b - kb_x) * kABlockBytes)
                                      : wb + size_t(b) * kBBlockBytesP;
          // the weight block needs no dependency: lane 1 issues it at once, while lane 0 (first stage of the item only) waits
          // for the poller's go-ahead and orders the other CTAs' generic stores before its bulk copy
          if (lane == 0 && need_dep) {
            const long long d0 = tr ? clock64() : 0;
            while (*dep_seq < j) { }
            __threadfence_block();
            asm volatile("fence.proxy.async;" ::: "memory");
            if (tr) pw[2] += clock64() - d0;
            need_dep = false;
          }
          if (lane == 0 || wbytes) bulk_g2s(sa + lane * kABlockBytes, src, lane == 0 ? abytes : wbytes, &full[s]);
          if (tr && lane == 0) { pw[0] += p1 - p0; pw[1] += clock64() - p1; }
        }
      }
      if (tr && lane == 0 && warp == kIssuersP) { tr[12] = pw[0]; tr[13] = pw[1]; tr[14] = pw[2]; }
    }
    __syncwarp();
  } else if (warp < kIssuersP) {
    // ===== MMA issuer (warp 0; warps 1, 2 idle here).  A power-of-two ring with the stage loop unrolled over it (stage index,
    // barrier addresses and parities are compile-time / one register) and descriptors = one 64-bit add from a base keep
    // the issuing thread's own instruction stream short. =====
    // One thread issues everything, in order: per stage 2 k-steps x (x_hi.W_hi -> main, x_lo.W_hi -> correction,
    // x_hi.W_lo -> correction), all N = 256, and ONE tcgen05.commit (three issuing warps = three commits per stage were
    // slower: every tcgen05 instruction costs the issue path ~110 cycles).  In-order issue from one thread also fixes
    // the accumulation order: results are bitwise reproducible run to run.
    int j = 0;
    uint32_t ph = 0;                              // parity of the full[] barriers: flips after every pass over the ring
    long long waited = 0, waited_acc = 0;
    {
      const uint32_t smem_base = smem_u32(smem);
      const uint64_t a_hi = umma_desc(smem_base, 2048, 128);                      // A block [part][chunk][128 rows][16 B]
      const uint64_t a_lo = a_hi + (8192 >> 4);
      const uint64_t b_hi = umma_desc(smem_base + kABlockBytes, 8192, 128);       // B block [chunk][hi|lo][256 rows][16 B]
      const uint64_t b_lo = b_hi + (4096 >> 4);
      constexpr uint64_t kStageDesc = uint64_t(kStageBytesP) >> 4;                // descriptor address units are 16 B
      constexpr uint64_t kAStep = 4096 >> 4, kBStep = 16384 >> 4;                 // k-step (2 chunks) strides
      for (int gi = blockIdx.x; gi < n_g; gi += gridDim.x) {
        const PItem it = p_decode(args, gi);
        if (!it.valid) continue;
        const int kb_total = it.kind == 0 ? ((it.layer == 0 ? args.net[it.net].kb_x0 : kb) + kb) : kb;
        const long long e0 = tr ? clock64() : 0;
        mbar_wait(&acc_empty[0], (j & 1) ^ 1);    // the epilogue of the previous item has pulled the accumulators
        if (tr) waited_acc += clock64() - e0;
        tc_fence_after();
        const uint32_t d_main = tmem_base, d_corr = tmem_base + kTileColsP;
        for (int b0 = 0; b0 < kb_total; b0 += kStagesP) {
#pragma unroll
          for (int st = 0; st < kStagesP; ++st) {
            const long long w0 = tr ? clock64() : 0;
            mbar_wait(&full[st], ph);
            if (tr) waited += clock64() - w0;
            tc_fence_after();
            const uint64_t so = st * kStageDesc;
            if (elect_one()) {
              if (!(args.dbg & 64)) {
                const uint32_t acc = (b0 | st) != 0;
                umma<KIND, kTileColsP>(d_main, a_hi + so, b_hi + so, acc);
                umma<KIND, kTileColsP>(d_corr, a_lo + so, b_hi + so, acc);
                umma<KIND, kTileColsP>(d_corr, a_hi + so, b_lo + so, 1);
                umma<KIND, kTileColsP>(d_main, a_hi + so + kAStep, b_hi + so + kBStep, 1);
                umma<KIND, kTileColsP>(d_corr, a_lo + so + kAStep, b_hi + so + kBStep, 1);
                umma<KIND, kTileColsP>(d_corr, a_hi + so + kAStep, b_lo + so + kBStep, 1);
              }
              umma_commit(&empty[st]);            // frees the stage when the MMAs issued so far have read it
            }
            __syncwarp();
          }
          ph ^= 1;
        }
        if (elect_one()) umma_commit(&acc_full[0]);
        __syncwarp();
        ++j;
      }
      if (tr && lane == 0) { tr[3] = waited; tr[7] = waited_acc; }
    }
  } else {
    // ===== epilogue: 16 warps; warp % 4 = TMEM lane quarter (rows), grp = the other two bits = which 16 of the tile's 64
    // hidden units (LSTM items: columns [grp][gate i,f,g,o][16 units]) or which 5 of the 20 joints (actor head items).
    const int ew = warp - kIssuersP - kProducersP;
    {
      const int et = threadIdx.x - 32 * (kIssuersP + kProducersP);
      for (int k = 0; k < args.nets; ++k) {
        for (int l = 0; l < args.depth; ++l)
          for (int i = et * 4; i < 4 * H; i += 32 * kEpiWarpsP * 4)
            *reinterpret_cast<float4*>(bias_s + (k * kPMaxDepth + l) * kMaxBias + i) =
                *reinterpret_cast<const float4*>(args.net[k].bias_t[l] + i);
        if (et < kTileColsP) bias_head_s[k * kTileColsP + et] = args.net[k].bias_head[et];
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarpsP) : "memory");
    }
    const int q4 = warp & 3, grp = ew >> 2;
    const int r = q4 * 32 + lane;
    constexpr float kCorr = (KIND == KBS_KIND_F16) ? (1.0f / kKbsF16LoScale) : 1.0f;
    const int64_t ld = args.ld;
    const int colq = grp * 64;                   // this thread's 16 columns of gate g start at colq + 16 g
    int j = 0;
    long long epi_cyc[2] = {0, 0}, epi_wait = 0, ph[4] = {0, 0, 0, 0};
    for (int gi = blockIdx.x; gi < n_g; gi += gridDim.x) {
      const PItem it = p_decode(args, gi);
      if (!it.valid) continue;
      const PNet& N = args.net[it.net];
      const int64_t R = int64_t(it.panel) * kPanelRows + r;
      const bool live = R < args.n;
      const int u0 = it.tile * kUnitsPerTileP + grp * 16;
      // dependencies of this item are satisfied once the poller says so (acquire through shared memory)
      while (*dep_seq < j + 1) { }
      __threadfence_block();
      const size_t npH = size_t(args.panels) * kPanelRows * H;
      float* cst = SAVE ? N.c_hist + (size_t(it.layer) * size_t(args.T + 1) + size_t(it.kind == 0 ? it.t : 0)) * npH
                        : N.fb + size_t(it.layer) * 2 * npH;                                 // c this step reads (kind 0 only)
      float* cdst = SAVE ? cst + npH : cst;                                                 // ... and the one it writes
      float4 cpre[4];
      if (it.kind == 0 && live) {
#pragma unroll
        for (int q = 0; q < 4; ++q) cpre[q] = __ldcg(reinterpret_cast<const float4*>(cst + fb_offset(R, u0 + q * 4, H)));
      }
      const uint8_t* done_t = args.done ? args.done + size_t(it.t) * ld : nullptr;
      const bool rst = live && done_t && done_t[R];
      bool published = false;                   // SAVE: LSTM items signal before their (unread) activation stores
      const long long ew0 = tr ? clock64() : 0;
      mbar_wait(&acc_full[0], j & 1);
      const long long ew1 = tr ? clock64() : 0;
      tc_fence_after();
      const uint32_t tq = tmem_base + (uint32_t(q4 * 32) << 16) + uint32_t(colq);
      if (it.kind == 0) {
        float v[64];
#pragma unroll
        for (int g4 = 0; g4 < 4; ++g4) {
          float cr[16];
          tmem_ld16(tq + 16 * g4, v + 16 * g4);
          tmem_ld16(tq + kTileColsP + 16 * g4, cr);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) v[16 * g4 + i] += kCorr * cr[i];
        }
        // the accumulators are in registers: hand TMEM back to the MMA issuer before doing the math
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[0]);
        if (tr) ph[0] += clock64() - ew1;
        const float* bs = bias_s + (it.net * kPMaxDepth + it.layer) * kMaxBias + it.tile * kTileColsP + colq;
#pragma unroll
        for (int i = 0; i < 64; ++i) v[i] += bs[i];
        if (live && !(args.dbg & 2)) {
          char* x_out = N.xmid + (SAVE ? size_t(it.layer) * size_t(args.T) + size_t(it.t) : size_t(it.layer * 2 + (it.t & 1))) * args.sbb;
          char* h_out = N.hsb + (SAVE ? size_t(it.layer) * size_t(args.T + 1) + size_t(it.t + 1)
                                      : size_t(it.layer * 2 + ((it.t + 1 + hslot) & 1))) * args.sbb;
          float* h_carry = (!SAVE && it.t == int(args.T) - 1) ? cst + npH : nullptr;
          // 8 hidden units = exactly one 16-byte SB chunk per plane (FP16 kind): every store below is a full 16 B per
          // lane, 512 contiguous bytes per warp (8-byte half-chunk stores cost the operand pipeline 2.5 K cycles per item)
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            float hn[8], cn[8];
            if (SAVE) {
              // the backward pass wants the four activated gates: evaluate them separately and keep them (FB layout)
              float ai[8], af[8], ag[8], ao[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int u = hf * 8 + i;
                const float cprev = (&cpre[u >> 2].x)[u & 3];
                ai[i] = sigmoidf_(v[u]); af[i] = sigmoidf_(v[16 + u]); ag[i] = tanhf_(v[32 + u]); ao[i] = sigmoidf_(v[48 + u]);
                cn[i] = af[i] * cprev + ai[i] * ag[i];
                hn[i] = ao[i] * tanhf_(cn[i]);
                if (rst) cn[i] = 0.0f;
              }
              // the activated gates replace the pre-activations in v[]: they are stored AFTER the item is published (nothing
              // in this launch reads them; the next step is waiting for h and c)
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int u = hf * 8 + i;
                v[u] = ai[i]; v[16 + u] = af[i]; v[32 + u] = ag[i]; v[48 + u] = ao[i];
              }
            } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int u = hf * 8 + i;
              const float cprev = (&cpre[u >> 2].x)[u & 3];
              const float gi_ = v[u], gf = v[16 + u], gg = v[32 + u], go = v[48 + u];
              // c' = s(f) c + s(i) tanh(g);  h' = s(o) tanh(c')   (eqx LSTMCell)
              cn[i] = sigmoidf_(gf) * cprev + sig_mul_tanh(gi_, gg);
              hn[i] = sig_mul_tanh(go, cn[i]);
              if (rst) cn[i] = 0.0f;
            }
            }
            if (!((args.dbg & 4) && hn[0] != 12345.0f)) {
              const int uu = u0 + hf * 8;
              const float h0[4] = {hn[0], hn[1], hn[2], hn[3]}, h1[4] = {hn[4], hn[5], hn[6], hn[7]};
              const KbsSplit4 s0 = sb_split4<KIND>(h0), s1 = sb_split4<KIND>(h1);   // one split serves both consumers
              sb_store_split8<kPanelRows, KIND>(x_out, R, uu, kb, s0, s1, false);   // next layer / head input (un-reset)
              sb_store_split8<kPanelRows, KIND>(h_out, R, uu, kb, s0, s1, rst);     // recurrent input (reset where done)
              *reinterpret_cast<float4*>(cdst + fb_offset(R, uu, H)) = make_float4(cn[0], cn[1], cn[2], cn[3]);
              *reinterpret_cast<float4*>(cdst + fb_offset(R, uu + 4, H)) = make_float4(cn[4], cn[5], cn[6], cn[7]);
              if (h_carry) {
                const float z = rst ? 0.0f : 1.0f;
                *reinterpret_cast<float4*>(h_carry + fb_offset(R, uu, H)) = make_float4(z * hn[0], z * hn[1], z * hn[2], z * hn[3]);
                *reinterpret_cast<float4*>(h_carry + fb_offset(R, uu + 4, H)) = make_float4(z * hn[4], z * hn[5], z * hn[6], z * hn[7]);
              }
            }
          }
        }
        if (SAVE) {
          // publish now (h, x, c are stored), then keep the activated gates for the backward pass
          __syncwarp();
          if (lane == 0) asm volatile("red.release.cta.shared::cta.add.u32 [%0], 1;" ::"r"(smem_u32(epi_done)) : "memory");
          published = true;
          if (live && !(args.dbg & 2)) {
            float* sg = N.save_g + (size_t(it.t) * args.depth + it.layer) * 4 * npH;
#pragma unroll
            for (int gate = 0; gate < 4; ++gate)
#pragma unroll
              for (int q = 0; q < 4; ++q)
                *reinterpret_cast<float4*>(sg + gate * npH + fb_offset(R, u0 + 4 * q, H)) =
                    make_float4(v[16 * gate + 4 * q], v[16 * gate + 4 * q + 1], v[16 * gate + 4 * q + 2], v[16 * gate + 4 * q + 3]);
          }
        }
      } else {
        // head item: "gate" 0 columns = mean rows, "gate" 1 columns = std rows of joints 5 grp .. 5 grp + 4 (pack_head_weights_kernel)
        float v[16];
        {
          float cr[16];
          tmem_ld8(tq, v); tmem_ld8(tq + 16, v + 8);
          tmem_ld8(tq + kTileColsP, cr); tmem_ld8(tq + kTileColsP + 16, cr + 8);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] += kCorr * cr[i];
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[0]);
        const float* bs = bias_head_s + it.net * kTileColsP + colq;
        const int64_t e = R;
        const size_t t = size_t(it.t);
        float s_z = 0.0f, s_log = 0.0f;
        if (it.net == 1) {
          if (live && grp == 0) args.value[t * ld + e] = v[0] + bs[0];
        } else {
          constexpr float kHalfLog2Pi = 0.918938533204672742f;
          if (live) {
            const int j0 = 5 * grp;
            float in_lpf[5], in_eps[5], in_arm[5], in_ain[5], in_q[5], in_qd[5], in_kp[5], in_kd[5], in_lim[5], in_ab[5], in_tb[5];
#pragma unroll
            for (int jj = 0; jj < 5; ++jj) {            // every input of the 5 joints first: one L2 round trip, not five
              const int jn = j0 + jj;
              const int64_t o = jn * ld + e;
              in_lpf[jj] = __ldcg(args.lpf + o);
              in_eps[jj] = args.eps ? __ldg(args.eps + t * KBS_NUM_JOINTS * ld + o) : 0.0f;
              in_arm[jj] = (jn >= 10) ? __ldg(args.arm_cmd + t * KBS_ACTOR_OBS * ld + (jn - 10) * ld + e) : 0.0f;
              in_ain[jj] = args.action_in ? __ldg(args.action_in + t * KBS_NUM_JOINTS * ld + o) : 0.0f;
              if (args.ctrl) {
                in_q[jj] = __ldg(args.q + t * KBS_NQ * ld + o);
                in_qd[jj] = __ldg(args.qd + t * KBS_NV * ld + o);
                in_kp[jj] = args.ep.kp ? __ldg(args.ep.kp + o) : P.kp[jn];
                in_kd[jj] = args.ep.kd ? __ldg(args.ep.kd + o) : P.kd[jn];
                in_lim[jj] = args.ep.tau_limit ? __ldg(args.ep.tau_limit + o) : P.ctrl_limit[jn];
                in_ab[jj] = args.ep.action_bias ? __ldg(args.ep.action_bias + o) : 0.0f;
                in_tb[jj] = args.ep.torque_bias ? __ldg(args.ep.torque_bias + o) : 0.0f;
              }
            }
#pragma unroll
            for (int jj = 0; jj < 5; ++jj) {
              const int jn = j0 + jj;
              const int64_t o = jn * ld + e;
              const float sraw = v[8 + jj] + bs[16 + jj];
              const float sp = fmaxf(sraw, 0.0f) + log1pf(expf(-fabsf(sraw)));
              const float sd = fminf((sp + P.min_std) * P.var_scale, P.max_std);
              float m = (v[jj] + bs[jj]) + P.joint_bias[jn];
              m = m + in_arm[jj];
              const float y = in_lpf[jj];
              const float yn = y + P.lpf_alpha * (m - y);
              args.lpf[o] = rst ? 0.0f : yn;
              float act = yn;
              if (args.eps) act = yn + sd * in_eps[jj];
              const float a_eval = args.action_in ? in_ain[jj] : act;
              const float z = (a_eval - yn) / sd;
              s_z = s_z + (-0.5f * z * z - kHalfLog2Pi);
              s_log = s_log + logf(sd);
              if (args.action) args.action[t * KBS_NUM_JOINTS * ld + o] = act;
              if (args.std) args.std[t * KBS_NUM_JOINTS * ld + o] = sd;
              if (args.mean) args.mean[t * KBS_NUM_JOINTS * ld + o] = yn;
              if (SAVE && args.sraw) args.sraw[t * KBS_NUM_JOINTS * ld + o] = sraw;
              if (args.ctrl) {                         // PositionActuators.get_ctrl (train.py:1091-1105)
                const float target = args.ep.action_bias ? __fadd_rn(act, in_ab[jj]) : act;
                float tau = __fsub_rn(__fmul_rn(in_kp[jj], __fsub_rn(target, in_q[jj])), __fmul_rn(in_kd[jj], in_qd[jj]));
                if (args.ep.torque_bias) tau = __fadd_rn(tau, in_tb[jj]);
                args.ctrl[t * KBS_NUM_JOINTS * ld + o] = fminf(fmaxf(tau, -in_lim[jj]), in_lim[jj]);
              }
            }
          }
          // log-prob / entropy: the four joint groups of a row meet in shared memory (fixed order: deterministic)
          head_part[(grp * kPanelRows + r) * 2] = s_z;
          head_part[(grp * kPanelRows + r) * 2 + 1] = s_log;
          asm volatile("bar.sync %0, 128;" ::"r"(2 + q4) : "memory");
          if (grp == 0 && live) {
            float z = 0.0f, l = 0.0f;
#pragma unroll
            for (int w = 0; w < 4; ++w) { z = z + head_part[(w * kPanelRows + r) * 2]; l = l + head_part[(w * kPanelRows + r) * 2 + 1]; }
            if (args.log_prob) args.log_prob[t * ld + e] = z - l;
            if (args.entropy) args.entropy[t * ld + e] = l + float(KBS_NUM_JOINTS) * (0.5f + kHalfLog2Pi);
          }
          asm volatile("bar.sync %0, 128;" ::"r"(2 + q4) : "memory");   // head_part may be rewritten by the next head item
        }
      }
      // publish: this warp's share of the item is in global memory
      const long long ew2 = tr ? clock64() : 0;
      __syncwarp();
      long long ewf = 0;
      if (lane == 0 && !published) {
        asm volatile("red.release.cta.shared::cta.add.u32 [%0], 1;" ::"r"(smem_u32(epi_done)) : "memory");
        if (tr) ewf = clock64();
      }
      if (tr) { const long long ew3 = clock64(); epi_cyc[it.kind] += ew3 - ew1; epi_wait += ew1 - ew0; if (it.kind == 0) { ph[1] += ew2 - ew1; ph[2] += ew3 - ew2; ph[3] += ewf - ew2; } }
      ++j;
    }
    if (tr && threadIdx.x == 32 * (kIssuersP + kProducersP)) { tr[4] = epi_cyc[0]; tr[5] = epi_cyc[1]; tr[6] = epi_wait; tr[8] = ph[0]; tr[9] = ph[1]; tr[10] = ph[2]; tr[11] = ph[3]; }
  }
  tc_fence_before();
  __syncthreads();
  if (tr && threadIdx.x == 0) {
    unsigned long long gt_end;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_end));
    tr[0] = clock64() - t_start;
    tr[15] = (long long)(gt_end - gt_start);      // ns: SM clock under load = tr[0] / tr[15] GHz
  }
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

// ---- persistent BPTT kernel: the backward recurrence of the PPO update in ONE launch -----------------------------------------
// Replaces, for one minibatch: the T x depth x {cell_bwd8_kernel launch + lstm_layer_tc_kernel(MODE_PLAIN) launch} sequence of
// kbs_ppo_grad (jax.grad through xax.scan(_ppo_scan_fn), train.py:1435-1524).  Same scaffolding as rollout_persist_kernel (one
// CTA per SM, wavefront of work items, monotone completion counters in global memory, poller / publisher warps).  Items, per
// (net, layer l, step s, 128-env panel, 128-column tile):
//   H tile: acc = dG(l, s+1) . W_hh  (the gradient reaching h_s through the recurrence; K = 4H)   -- tensor core
//           epilogue = the LSTM cell's backward at step s for the tile's 128 hidden units: dh = dh_in + keep_s acc,
//           dc = keep_s dc_rec + dh o (1 - tanh^2 c_s), gate gradients -> dG(l, s) written as the (pre-scaled) split operand
//           of the next GEMMs, dc_rec <- dc f.  dh_in = dx(l+1, s) from the layer above, or the head's gradient (top layer).
//   X tile: dx(l, s) = dG(l, s) . W_ih  (gradient wrt the layer's input): fp32 for the layer below, or, for layer 0, the
//           split operand the input-projection weight gradient is built from.
// Slot order: H(l, s) in slot (T-1-s) + 2 (depth-1-l), X(l, s) one slot later (it needs dG(l, s) = both H tiles), and
// H(l-1, s) one slot after that (it needs dx(l, s)); dG(l, T) is a zero operand, so step T-1 is a regular item.
// The weight gradients are NOT accumulated here: dG / x / h are kept for every step and contracted over all T x n rows
// by the split-K GEMMs (kbs_tc_gemm_tn).
// Tile = 128 envs x kBT = 64 output columns.  MEASURED (tools/ppo_trace.py, 512 trajectories): with one item per CTA and slot
// the kernel is bound by what ONE SM can pull from L2 (~60 B/clk): an item streams its whole dG panel (128 x 4H, 512 KB) plus
// its weight tile, 1 MB at 128 columns.  Narrow tiles put more SMs (128 instead of 64 per slot) on the same slot: 768 KB per
// item, and half the epilogue per thread.  (MMA issue is not the limit here: 2 instructions per k-step either way.)
// BT = 128 is a second instantiation kept for A/B (kbs_tc_bptt_tile).
constexpr int kBT = 64;                                   // the narrow tile (and the width kbs_tc_pack_bwd's second image is for)
template <int BT> struct BTile {
  static constexpr int kBBlockBytes = 2 * 4 * BT * 16;               // [chunk][hi|lo][BT rows][16 B] = 8 / 16 KB
  static constexpr int kStageBytes = kABlockBytes + kBBlockBytes;    // 24 / 32 KB
  static constexpr int kStages = BT == 64 ? 8 : 6;
  static constexpr int kSmemBytes = kStages * kStageBytes + 256 /*barriers*/ + 1024 /*align*/;
};
constexpr int kBEpiWarps = 16;
constexpr int kBThreads = 32 * (1 + 1 + kBEpiWarps + 2);
struct BNet {
  const char* w_bwd[kPMaxDepth];   // per layer: 2 H/128 tiles of 128 output columns of [dx | dh], K = 4H (pack_bwd_weights_kernel)
  char* dG;                        // [depth][T + 1] x sb4: slot s = dG(l, s) (scaled by gscale); slot T = zeros (memset by the host)
  const float* save_g;             // forward pass: [T][depth][4] x np*H activated gates (FB)
  const float* c_hist;             // forward pass: [depth][T + 1] x np*H (FB): slot s = the cell state step s read
  const float* dh_top;             // [T * n][H] row-major: gradient wrt the top layer's output (from the output head)
  const float* dv;                 // instead of dh_top for a one-row output layer (the critic): d loss / d out [T * n] ...
  const float* w_out;              // ... and that row [H]: dh_top = dv w_out is formed in the epilogue
  float* dx;                       // [depth][T] x np*H (FB): gradient wrt the input of layer l >= 1 at step s
  char* dx0;                       // [T] x sbb: the same for layer 0, as split operand (scaled by gscale)
  float* dc;                       // [depth] x np*H (FB): gradient wrt the cell carry, running (zeroed by the host)
  unsigned int* flags;             // [depth][2 (H, X)][panels] completion counters (zeroed by the host)
  char* tn_dG[kPMaxDepth];         // n_tctas > 0: per layer, dG re-packed with K = t np + row (A^T operand of the dW GEMMs)
};
struct BArgs {
  BNet net[2];
  int nets, depth, H, panels;
  int64_t n, ld, T;
  size_t sbb, sb4;                 // bytes of one [np][H] / [np][4H] split operand
  const uint8_t* done;             // [T][ld]
  float gscale, inv_gscale;
  unsigned int* status;
  int dbg;
  long long* trace;                // per CTA [16]: see tools/ppo_trace.py
  // tn != 0: the X tiles re-pack dG on the fly into the K = row operand layout of the weight-gradient GEMMs (sb_to_tn_kernel's
  // job: 0.85 ms of separate launches and 1.7 GB of HBM traffic after this kernel).  The dG panel an X tile multiplies
  // passes through its shared memory anyway; while the MMAs of the item run, the (idle) epilogue warps transpose the stages
  // -- the th X tiles of a panel take every th-th K block each -- and write them out.  MEASURED alternative: 12 / 20 extra
  // "transposer" CTAs chasing the completion counters were too slow (10.6 / 7.9 ms per update instead of 6.3).
  int tn, tn_kb_total;
  size_t tn_col_bytes;
};
struct BItem { int kind, net, layer, panel, tile, s; bool valid; };
template <int BT>
__device__ __forceinline__ BItem b_decode(const BArgs& a, int g) {
  const int th = a.H / BT;                      // tiles per half of the [dx | dh] output
  const int per_panel = a.depth * 2 * th, per_net = a.panels * per_panel, C = a.nets * per_net;
  const int sigma = g / C;
  int i = g - sigma * C;
  BItem it;
  it.net = i / per_net; i -= it.net * per_net;
  it.panel = i / per_panel;
  const int q = i - it.panel * per_panel;
  it.layer = q / (2 * th);
  const int k = q - it.layer * 2 * th;
  it.kind = k >= th ? 1 : 0;
  it.tile = k - it.kind * th;
  const int base = sigma - 2 * (a.depth - 1 - it.layer);
  it.s = int(a.T) - 1 - base + it.kind;
  it.valid = base >= 0 && it.s >= 0 && it.s <= int(a.T) - 1;
  return it;
}
template <int BT>
__device__ __forceinline__ long long b_wait_deps(const BArgs& a, const BItem& it, bool& drain) {
  if (drain) return 0;
  const long long c0 = clock64();
  const BNet& N = a.net[it.net];
  const unsigned int per = unsigned((a.H / BT) * kBEpiWarps);
  const unsigned int* fp[2]; unsigned int tg[2]; int nd = 0;
  const unsigned int T = unsigned(a.T), s = unsigned(it.s);
  const int l = it.layer;
  if (it.kind == 0) {
    if (s + 1 < T) { fp[nd] = N.flags + (l * 2 + 0) * a.panels + it.panel; tg[nd++] = (T - 1 - s) * per; }          // dG(l, s+1), dc
    if (l + 1 < a.depth) { fp[nd] = N.flags + ((l + 1) * 2 + 1) * a.panels + it.panel; tg[nd++] = (T - s) * per; }  // dx(l+1, s)
  } else {
    fp[nd] = N.flags + (l * 2 + 0) * a.panels + it.panel; tg[nd++] = (T - s) * per;                                 // dG(l, s)
  }
  if (nd == 0) return 0;
  if (nd == 1) { fp[1] = fp[0]; tg[1] = 0u; }
  unsigned int polls = 0;
  unsigned long long t0 = 0;
  while (true) {
    const unsigned int v0 = ld_volatile_u32(fp[0]), v1 = ld_volatile_u32(fp[1]);
    if (v0 >= tg[0] && v1 >= tg[1]) break;
    if ((++polls & 1023u) == 0u) {
      if (ld_volatile_u32(a.status) & 3u) { drain = true; break; }
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > kPWaitTimeoutNs) { atomicOr(a.status, unsigned(KBS_STATUS_TIMEOUT_LSTM)); drain = true; break; }
    }
  }
  __threadfence();
  return clock64() - c0;
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// The forward pass's saves of an H tile (4 activated gates + the cell state the step read: 5 x 16 units per thread) come from
// HBM (1 GB per update: far beyond L2).  They are known long before the item can start, so the epilogue warps request them
// one item ahead: by the time the accumulators are ready the lines sit in L2 (~2 K cycles of DRAM latency per batch of
// loads otherwise, four batches in a row on the critical path of every backward step).
template <int BT>
__device__ __forceinline__ void b_prefetch_saves(const BArgs& a, const BItem& it, int r, int grp, size_t npH) {
  if (it.kind != 0) return;
  const BNet& N = a.net[it.net];
  const int64_t R = int64_t(it.panel) * kPanelRows + r;
  if (R >= a.n) return;
  const int u0 = it.tile * BT + grp * (BT / 4);
  const float* sg = N.save_g + (size_t(it.s) * a.depth + it.layer) * 4 * npH;
  const float* cin = N.c_hist + (size_t(it.layer) * size_t(a.T + 1) + size_t(it.s)) * npH;
#pragma unroll
  for (int q = 0; q < BT / 16; ++q) {
    const size_t o = fb_offset(R, u0 + 4 * q, a.H);
    prefetch_l2(sg + o); prefetch_l2(sg + npH + o); prefetch_l2(sg + 2 * npH + o); prefetch_l2(sg + 3 * npH + o);
    prefetch_l2(cin + o);
  }
}

__device__ __forceinline__ void b_ld8fb(const float* base, int64_t R, int u, int H, float (&o)[8], bool coherent) {
  const float4* p0 = reinterpret_cast<const float4*>(base + fb_offset(R, u, H));
  const float4* p1 = reinterpret_cast<const float4*>(base + fb_offset(R, u + 4, H));
  const float4 a = coherent ? __ldcg(p0) : __ldg(p0), b = coherent ? __ldcg(p1) : __ldg(p1);
  o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}
template <int KIND, int BT>
__global__ void __launch_bounds__(kBThreads, 1) bptt_persist_kernel(const __grid_constant__ BArgs args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BTile<BT>::kStages * BTile<BT>::kStageBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + BTile<BT>::kStages;
  uint64_t* acc_full = bars + 2 * BTile<BT>::kStages;     // [2]
  uint64_t* acc_empty = acc_full + 2;           // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  volatile int* dep_seq = reinterpret_cast<volatile int*>(tmem_slot + 1);
  unsigned int* epi_done = reinterpret_cast<unsigned int*>(tmem_slot + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int H = args.H, th = H / BT;
  const int per_slot = args.nets * args.panels * args.depth * 2 * th;
  const int n_g = (int(args.T) + 2 * (args.depth - 1) + 1) * per_slot;
  constexpr int kBlk = kbs_block_k(KIND);
  const int kb4 = 4 * H / kBlk;                  // K blocks of every item
  const size_t npH = size_t(args.panels) * kPanelRows * H;
  long long* tr = args.trace ? args.trace + size_t(blockIdx.x) * 16 : nullptr;
  const long long t_start = clock64();
  unsigned long long gt_start = 0;
  if (tr && threadIdx.x == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_start));

  if (threadIdx.x == 0) {
    // empty[s]: the MMA commit, + (tn) the four epilogue warps that look at the stage for the on-the-fly re-pack
    for (int s = 0; s < BTile<BT>::kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], args.tn ? 5 : 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], kBEpiWarps); }
    *dep_seq = 0;
    *epi_done = 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_cc = int(gridDim.x);

  if (warp == 2 + kBEpiWarps + 1) {
    if (lane == 0) {
      // ===== publisher (see rollout_persist_kernel) =====
      int j = 0;
      for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
        const BItem it = b_decode<BT>(args, gi);
        if (!it.valid) continue;
        ++j;
        const unsigned int want = unsigned(j) * kBEpiWarps;
        unsigned int seen;
        do {
          asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(seen) : "r"(smem_u32(epi_done)) : "memory");
        } while (seen < want);
        __threadfence();
        atomicAdd(args.net[it.net].flags + (it.layer * 2 + it.kind) * args.panels + it.panel, unsigned(kBEpiWarps));
      }
    }
    __syncwarp();
  } else if (warp == 2 + kBEpiWarps) {
    if (lane == 0) {
      // ===== dependency poller =====
      int j = 0;
      bool drain = false;
      long long waited = 0;
      for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
        const BItem it = b_decode<BT>(args, gi);
        if (!it.valid) continue;
        if (!(args.dbg & 1)) waited += b_wait_deps<BT>(args, it, drain);
        *dep_seq = ++j;
      }
      if (tr) { tr[1] = waited; tr[2] = j; }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane < 2) {
      // ===== producers: lane 0 = the dG block (activation side), lane 1 = the weight block of the stage =====
      uint32_t g = 0;
      int j = 0;
      for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
        const BItem it = b_decode<BT>(args, gi);
        if (!it.valid) continue;
        const BNet& N = args.net[it.net];
        const int slot = it.s + (it.kind == 0 ? 1 : 0);
        const char* xa = N.dG + (size_t(it.layer) * size_t(args.T + 1) + size_t(slot)) * args.sb4 + size_t(it.panel) * kb4 * kABlockBytes;
        const char* wb = N.w_bwd[it.layer] + size_t(it.kind == 0 ? th + it.tile : it.tile) * kb4 * BTile<BT>::kBBlockBytes;
        ++j;
        bool need_dep = true;
        for (int b = 0; b < kb4; ++b, ++g) {
          const int s = g % BTile<BT>::kStages;
          if (lane == 0) {
            mbar_wait(&empty[s], ((g / BTile<BT>::kStages) & 1) ^ 1);
            mbar_expect_tx(&full[s], uint32_t(kABlockBytes + BTile<BT>::kBBlockBytes));
          }
          __syncwarp(0x3);
          uint8_t* sa = smem + size_t(s) * BTile<BT>::kStageBytes;
          if (lane == 0 && need_dep) {
            while (*dep_seq < j) { }
            __threadfence_block();
            asm volatile("fence.proxy.async;" ::: "memory");
            need_dep = false;
          }
          const char* src = lane == 0 ? xa + size_t(b) * kABlockBytes : wb + size_t(b) * BTile<BT>::kBBlockBytes;
          bulk_g2s(sa + lane * kABlockBytes, src, lane == 0 ? uint32_t(kABlockBytes) : uint32_t(BTile<BT>::kBBlockBytes), &full[s]);
        }
      }
    }
    __syncwarp();
  } else if (warp == 0) {
    // ===== MMA issuer: per k-step  dG_hi . [W_hi | W_lo]^T (N = 256: main | correction columns) + dG_lo . W_hi^T (N = 128) =====
    uint32_t g = 0;
    int j = 0;
    long long w_full = 0, w_acc = 0;
    for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
      const BItem it = b_decode<BT>(args, gi);
      if (!it.valid) continue;
      const int buf = j & 1;
      const long long e0 = tr ? clock64() : 0;
      mbar_wait(&acc_empty[buf], ((j >> 1) & 1) ^ 1);
      if (tr) w_acc += clock64() - e0;
      tc_fence_after();
      const uint32_t d_main = tmem_base + buf * (2 * BT), d_corr = d_main + BT;
      for (int b = 0; b < kb4; ++b, ++g) {
        const int s = g % BTile<BT>::kStages;
        const long long f0 = tr ? clock64() : 0;
        mbar_wait(&full[s], (g / BTile<BT>::kStages) & 1);
        if (tr) w_full += clock64() - f0;
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + size_t(s) * BTile<BT>::kStageBytes);
        const uint32_t sb = sa + kABlockBytes;
        const uint64_t a_hi = umma_desc(sa, 2048, 128), a_lo = umma_desc(sa + 8192, 2048, 128);
        // B block [chunk][hi|lo][BT rows][16 B]: chunk stride (LBO) 2 BT 16 B, k-step (2 chunks) twice that
        const uint64_t b_all = umma_desc(sb, 2 * BT * 16, 128);
        constexpr uint64_t kBStep = uint64_t(4 * BT * 16) >> 4;
        if (elect_one()) {
          umma<KIND, 2 * BT>(d_main, a_hi, b_all, b != 0);
          umma<KIND, BT>(d_corr, a_lo, b_all, 1);
          umma<KIND, 2 * BT>(d_main, a_hi + (4096 >> 4), b_all + kBStep, 1);
          umma<KIND, BT>(d_corr, a_lo + (4096 >> 4), b_all + kBStep, 1);
          umma_commit(&empty[s]);
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(&acc_full[buf]);
      __syncwarp();
      ++j;
    }
    if (tr && lane == 0) { tr[3] = w_full; tr[4] = w_acc; }
  } else {
    // ===== epilogue: 16 warps; warp % 4 = TMEM lane quarter (rows), grp = which 16 of the tile's 64 columns (hidden units).
    // The accumulators are pulled 8 columns at a time, right where they are used (TMEM is double-buffered and a CTA rarely
    // has a second item in the same slot, so holding the buffer through the epilogue costs nothing and keeps the register
    // footprint of a batch -- 7 x 8 operands -- below the spill line). =====
    const int ew = warp - 2;
    const int q4 = warp & 3, grp = ew >> 2;
    const int r = q4 * 32 + lane;
    constexpr float kCorr = (KIND == KBS_KIND_F16) ? (1.0f / kKbsF16LoScale) : 1.0f;
    const int64_t ld = args.ld;
    int j = 0;
    bool bad = false;
    uint32_t gstage = 0;                  // ring position of the current item's first stage (as the producer / issuer count)
    {   // the first item's saves
      for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
        const BItem it0 = b_decode<BT>(args, gi);
        if (it0.valid) { b_prefetch_saves<BT>(args, it0, r, grp, npH); break; }
      }
    }
    for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
      const BItem it = b_decode<BT>(args, gi);
      if (!it.valid) continue;
      {   // request the NEXT item's saves now: a whole item of lead time
        for (int gn = gi + n_cc; gn < n_g; gn += n_cc) {
          const BItem itn = b_decode<BT>(args, gn);
          if (itn.valid) { b_prefetch_saves<BT>(args, itn, r, grp, npH); break; }
        }
      }
      const BNet& N = args.net[it.net];
      const int64_t R = int64_t(it.panel) * kPanelRows + r;
      const bool live = R < args.n;
      const int buf = j & 1;
      const int u0 = it.tile * BT + grp * (BT / 4);         // first of this thread's 16 units (columns of the half)
      while (*dep_seq < j + 1) { }
      __threadfence_block();
      const size_t s = size_t(it.s);
      const float keep = (live && it.kind == 0 && args.done[s * ld + R]) ? 0.0f : 1.0f;
      const float* sg = N.save_g + (s * args.depth + it.layer) * 4 * npH;
      const float* cin = N.c_hist + (size_t(it.layer) * size_t(args.T + 1) + s) * npH;
      float* dcp = N.dc + size_t(it.layer) * npH;
      const bool top = it.layer + 1 == args.depth;
      const float* dxu = top ? N.dh_top + (s * size_t(args.n) + size_t(live ? R : 0)) * H
                             : N.dx + (size_t(it.layer + 1) * size_t(args.T) + s) * npH;
      char* dGo = N.dG + (size_t(it.layer) * size_t(args.T + 1) + s) * args.sb4;
      if (args.tn) {
        // ring slot st belongs to warp group st % 4 (= grp): wait until the stage has landed, re-pack it if this X tile owns
        // the K block, release it (every stage gets exactly four such arrivals, whoever owns it)
        for (int b = 0; b < kb4; ++b) {
          const uint32_t g = gstage + uint32_t(b);
          const int st = int(g % BTile<BT>::kStages);
          if ((st & 3) != grp) continue;            // by ring slot: the same warps watch every phase of a barrier (see lstm_fwd_save_kernel)
          mbar_wait(&full[st], (g / BTile<BT>::kStages) & 1);
          if (it.kind == 1 && (b % th) == it.tile) {
            const uint8_t* sa = smem + size_t(st) * BTile<BT>::kStageBytes;       // A block [hi|lo][chunk][128 rows][16 B]
            const int cm = (ew & 3) * 32 + lane;                        // one of the block's 128 core matrices (8 rows x 8 K)
            const int r8 = cm & 15, c = (cm >> 4) & 3, plane = cm >> 6;
            const uint8_t* sp = sa + ((size_t(plane) * 4 + c) * kPanelRows + size_t(r8) * 8) * 16;
            uint4 in[8];
#pragma unroll
            for (int rr = 0; rr < 8; ++rr) {
              in[rr] = *reinterpret_cast<const uint4*>(sp + rr * 16);
              if (int64_t(it.panel) * kPanelRows + r8 * 8 + rr >= args.n) in[rr] = make_uint4(0u, 0u, 0u, 0u);
            }
            const int64_t kp = (int64_t(it.s) * args.panels + it.panel) * kPanelRows + r8 * 8;    // K' of the chunk's first row
            const int64_t kbq = kp / 32;
            const int cq = int((kp / 8) & 3);
            const int j0 = b * 32 + c * 8;                                                        // operand row of its first K value
            char* dp = N.tn_dG[it.layer] + size_t(j0 / kTileCols) * args.tn_col_bytes +
                       (((size_t(kbq) * 2 + plane) * 4 + cq) * kTileCols + size_t(j0 % kTileCols)) * 16;
#pragma unroll
            for (int i8 = 0; i8 < 8; ++i8) {
              const unsigned sel = (i8 & 1) ? 0x7632u : 0x5410u;
              uint4 o;
              o.x = __byte_perm((&in[0].x)[i8 >> 1], (&in[1].x)[i8 >> 1], sel);
              o.y = __byte_perm((&in[2].x)[i8 >> 1], (&in[3].x)[i8 >> 1], sel);
              o.z = __byte_perm((&in[4].x)[i8 >> 1], (&in[5].x)[i8 >> 1], sel);
              o.w = __byte_perm((&in[6].x)[i8 >> 1], (&in[7].x)[i8 >> 1], sel);
              *reinterpret_cast<uint4*>(dp + size_t(i8) * 16) = o;
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[st]);
        }
        gstage += uint32_t(kb4);
      }
      // H tile: the forward pass's saves of the first 8 units are requested before the wait for the accumulator (they depend on
      // nothing of this kernel): their L2 round trip runs under the item's MMAs instead of behind them
      float qi[8], gf[8], gg[8], go[8], ci[8];
      const bool hk = it.kind == 0 && live;
      if (hk) {
        b_ld8fb(sg, R, u0, H, qi, false); b_ld8fb(sg + npH, R, u0, H, gf, false); b_ld8fb(sg + 2 * npH, R, u0, H, gg, false);
        b_ld8fb(sg + 3 * npH, R, u0, H, go, false); b_ld8fb(cin, R, u0, H, ci, false);
      }
      mbar_wait(&acc_full[buf], (j >> 1) & 1);
      tc_fence_after();
      const uint32_t tq = tmem_base + (uint32_t(q4 * 32) << 16) + uint32_t(buf * (2 * BT) + grp * (BT / 4));
#pragma unroll 1
      for (int c8 = 0; c8 < BT / 32; ++c8) {
        const int u = u0 + 8 * c8;
        float v[8];
        {
          float cr[8];
          tmem_ld8(tq + 8 * c8, v);
          tmem_ld8(tq + BT + 8 * c8, cr);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] += kCorr * cr[i];
        }
        if (!live) continue;
        if (it.kind == 1) {
          // ---- X tile: dx(l, s) ----
          if (it.layer == 0) {
            char* dst = N.dx0 + s * args.sbb;                  // stays scaled: it is the A^T operand of the dW_in GEMM
            const float x0[4] = {v[0], v[1], v[2], v[3]}, x1[4] = {v[4], v[5], v[6], v[7]};
            bad = bad || sb_out_of_range<KIND, 4>(x0) || sb_out_of_range<KIND, 4>(x1);
            sb_store_split8<kPanelRows, KIND>(dst, R, u, H / kBlk, sb_split4<KIND>(x0), sb_split4<KIND>(x1), false);
          } else {
            float* dst = N.dx + (size_t(it.layer) * size_t(args.T) + s) * npH;
            const float g = args.inv_gscale;
            *reinterpret_cast<float4*>(dst + fb_offset(R, u, H)) = make_float4(g * v[0], g * v[1], g * v[2], g * v[3]);
            *reinterpret_cast<float4*>(dst + fb_offset(R, u + 4, H)) = make_float4(g * v[4], g * v[5], g * v[6], g * v[7]);
          }
          continue;
        }
        // ---- H tile: the cell's backward at step s for units u .. u + 7 ----
        float dhi[8], dcr[8];
        if (c8 > 0) {
          b_ld8fb(sg, R, u, H, qi, false); b_ld8fb(sg + npH, R, u, H, gf, false); b_ld8fb(sg + 2 * npH, R, u, H, gg, false);
          b_ld8fb(sg + 3 * npH, R, u, H, go, false); b_ld8fb(cin, R, u, H, ci, false);
        }
        b_ld8fb(dcp, R, u, H, dcr, true);
        if (top && N.dv) {
          const float d = __ldg(N.dv + s * size_t(args.n) + size_t(R));
          const float4 a = __ldg(reinterpret_cast<const float4*>(N.w_out + u)), b = __ldg(reinterpret_cast<const float4*>(N.w_out + u + 4));
          dhi[0] = d * a.x; dhi[1] = d * a.y; dhi[2] = d * a.z; dhi[3] = d * a.w;
          dhi[4] = d * b.x; dhi[5] = d * b.y; dhi[6] = d * b.z; dhi[7] = d * b.w;
        } else if (top) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(dxu + u)), b = __ldg(reinterpret_cast<const float4*>(dxu + u + 4));
          dhi[0] = a.x; dhi[1] = a.y; dhi[2] = a.z; dhi[3] = a.w; dhi[4] = b.x; dhi[5] = b.y; dhi[6] = b.z; dhi[7] = b.w;
        } else {
          b_ld8fb(dxu, R, u, H, dhi, true);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float c = gf[i] * ci[i] + qi[i] * gg[i];                 // c_s, as the forward pass formed it
          const float tc = tanhf_(c);
          const float dh = dhi[i] + keep * (args.inv_gscale * v[i]);
          const float dc = keep * dcr[i] + dh * go[i] * (1.0f - tc * tc);
          dcr[i] = dc * gf[i];
          const float di = args.gscale * (dc * gg[i] * qi[i] * (1.0f - qi[i]));
          const float df = args.gscale * (dc * ci[i] * gf[i] * (1.0f - gf[i]));
          const float dg = args.gscale * (dc * qi[i] * (1.0f - gg[i] * gg[i]));
          const float dob = args.gscale * (dh * tc * go[i] * (1.0f - go[i]));
          qi[i] = di; gf[i] = df; gg[i] = dg; go[i] = dob;              // the gate gradients replace the gates
        }
        *reinterpret_cast<float4*>(dcp + fb_offset(R, u, H)) = make_float4(dcr[0], dcr[1], dcr[2], dcr[3]);
        *reinterpret_cast<float4*>(dcp + fb_offset(R, u + 4, H)) = make_float4(dcr[4], dcr[5], dcr[6], dcr[7]);
        auto st8 = [&](int gate, const float (&x)[8]) {
          const float x0[4] = {x[0], x[1], x[2], x[3]}, x1[4] = {x[4], x[5], x[6], x[7]};
          bad = bad || sb_out_of_range<KIND, 4>(x0) || sb_out_of_range<KIND, 4>(x1);
          sb_store_split8<kPanelRows, KIND>(dGo, R, gate * H + u, 4 * H / kBlk, sb_split4<KIND>(x0), sb_split4<KIND>(x1), false);
        };
        st8(0, qi); st8(1, gf); st8(2, gg); st8(3, go);
      }
      // the accumulator buffer goes back to the MMA issuer, then the item is published
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&acc_empty[buf]);
        asm volatile("red.release.cta.shared::cta.add.u32 [%0], 1;" ::"r"(smem_u32(epi_done)) : "memory");
      }
      ++j;
    }
    sb_flag_range(args.status, bad);
  }
  tc_fence_before();
  __syncthreads();
  if (tr && threadIdx.x == 0) {
    unsigned long long gt_end;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_end));
    tr[0] = clock64() - t_start;
    tr[15] = (long long)(gt_end - gt_start);
  }
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}

// ---- persistent forward kernel of the PPO update (SAVE pass): narrow tiles -------------------------------------------------
// The forward recurrence of kbs_ppo_grad at minibatch size (512 trajectories = 4 panels): rollout_persist_kernel<SAVE> with
// its 128 x 256 tiles put 64 LSTM items in a slot and each SM streamed 768 KB per item from L2 at the ~60 B/clk one SM gets
// (34.7 K cycles per slot, tools/ppo_trace.py).  This kernel is the same wavefront with 128 x 128 tiles (32 hidden units x 4
// gates, 8-unit column groups): 128 items per slot on 128 SMs, 512 KB per item, 8 units per epilogue thread.  It computes the
// LSTM stacks only -- the output heads of the update are one batched GEMM + a per-env scan afterwards (the low-pass filter's
// recurrence does not feed the LSTMs) -- and keeps for the backward pass: the per-step operands (xmid / hsb), the cell states,
// the activated gates, the top layer's outputs (row-major, for the head GEMM), and (tn) the K = row re-pack of [x | h_in],
// the B operand of the weight-gradient GEMMs, written from the stages in shared memory while the MMAs run.
constexpr int kSStages = 6;
constexpr int kSSmemBytes = kSStages * kStageBytes + 2 * kMaxBias * kPMaxDepth * 4 + 256 /*barriers*/ + 1024 /*align*/;
constexpr int kSEpiWarps = 16;
constexpr int kSThreads = 32 * (1 + 1 + kSEpiWarps + 2);
constexpr int kSGU = 8;                     // units per column group: tile column = grp * 32 + gate * 8 + uu
struct SNet {
  const char* x0; size_t x0_stride;        // [T] x x0_stride: layer-0 inputs (the input projection of every step)
  char* xmid;                              // [depth][T] x sbb: un-reset output of layer l at step t
  char* hsb;                               // [depth][T + 1] x sbb: slot t = the hidden state step t reads (reset where done)
  float* c_hist;                           // [depth][T + 1] x np*H (FB): slot t = the cell state step t reads
  float* save_g;                           // [T][depth][4] x np*H (FB): activated gates i, f, g, o
  float* h_top_rm;                         // [T * n][H] row-major: the top layer's outputs (head GEMM)
  const char* w[kPMaxDepth];               // per layer: H / 32 tiles of 128 gate columns (8-unit groups), K = 2H, WB blocks
  const float* bias[kPMaxDepth];           // [4H] in tile-column order
  unsigned int* flags;                     // [depth][panels] completion counters (zeroed by the host)
  char* tn_xh[kPMaxDepth];                 // tn: per layer, [x | h_in] re-packed with K = t np + row (2 H / 128 tiles, WB blocks)
};
struct SArgs {
  SNet net[2];
  int nets, depth, H, panels;
  int64_t n, ld, T;
  size_t sbb;
  const uint8_t* done;                     // [T][ld]
  unsigned int* status;
  int dbg, tn, tn_kb_total;
  size_t tn_col_bytes;
};
struct SItem { int net, layer, panel, tile, t; bool valid; };
__device__ __forceinline__ SItem s_decode(const SArgs& a, int g) {
  const int tiles = a.H / 32;
  const int per_panel = a.depth * tiles, per_net = a.panels * per_panel, C = a.nets * per_net;
  const int sigma = g / C;
  int i = g - sigma * C;
  SItem it;
  it.net = i / per_net; i -= it.net * per_net;
  it.panel = i / per_panel;
  const int q = i - it.panel * per_panel;
  it.layer = q / tiles;
  it.tile = q - it.layer * tiles;
  it.t = sigma - it.layer;
  it.valid = it.t >= 0 && it.t < int(a.T);
  return it;
}
__device__ __forceinline__ void s_wait_deps(const SArgs& a, const SItem& it, bool& drain) {
  if (drain) return;
  const SNet& N = a.net[it.net];
  const unsigned int per = unsigned((a.H / 32) * kSEpiWarps);
  const unsigned int* fp[2]; unsigned int tg[2]; int nd = 0;
  const unsigned int t = unsigned(it.t);
  if (t >= 1) { fp[nd] = N.flags + it.layer * a.panels + it.panel; tg[nd++] = t * per; }                 // h_{t-1}, c_{t-1}
  if (it.layer >= 1) { fp[nd] = N.flags + (it.layer - 1) * a.panels + it.panel; tg[nd++] = (t + 1) * per; }   // x_t
  if (nd == 0) return;
  if (nd == 1) { fp[1] = fp[0]; tg[1] = 0u; }
  unsigned int polls = 0;
  unsigned long long t0 = 0;
  while (true) {
    const unsigned int v0 = ld_volatile_u32(fp[0]), v1 = ld_volatile_u32(fp[1]);
    if (v0 >= tg[0] && v1 >= tg[1]) break;
    if ((++polls & 1023u) == 0u) {
      if (ld_volatile_u32(a.status) & 3u) { drain = true; break; }
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > kPWaitTimeoutNs) { atomicOr(a.status, unsigned(KBS_STATUS_TIMEOUT_LSTM)); drain = true; break; }
    }
  }
  __threadfence();
}

template <int KIND>
__global__ void __launch_bounds__(kSThreads, 1) lstm_fwd_save_kernel(const __grid_constant__ SArgs args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* bias_s = reinterpret_cast<float*>(smem + kSStages * kStageBytes);          // [net][layer][kMaxBias]
  uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + 2 * kPMaxDepth * kMaxBias);
  uint64_t* full = bars;
  uint64_t* empty = bars + kSStages;
  uint64_t* acc_full = bars + 2 * kSStages;     // [2]
  uint64_t* acc_empty = acc_full + 2;           // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  volatile int* dep_seq = reinterpret_cast<volatile int*>(tmem_slot + 1);
  unsigned int* epi_done = reinterpret_cast<unsigned int*>(tmem_slot + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int H = args.H, tiles = H / 32;
  const int per_slot = args.nets * args.panels * args.depth * tiles;
  const int n_g = (int(args.T) + args.depth - 1) * per_slot;
  constexpr int kBlk = kbs_block_k(KIND);
  const int kb = H / kBlk;                       // K blocks of each half ([x | h]) of an item
  const size_t npH = size_t(args.panels) * kPanelRows * H;
  const int n_cc = int(gridDim.x);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kSStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], args.tn ? 5 : 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], kSEpiWarps); }
    *dep_seq = 0;
    *epi_done = 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 2 + kSEpiWarps + 1) {
    if (lane == 0) {
      // ===== publisher (see rollout_persist_kernel) =====
      int j = 0;
      for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
        const SItem it = s_decode(args, gi);
        if (!it.valid) continue;
        ++j;
        const unsigned int want = unsigned(j) * kSEpiWarps;
        unsigned int seen;
        do {
          asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(seen) : "r"(smem_u32(epi_done)) : "memory");
        } while (seen < want);
        __threadfence();
        atomicAdd(args.net[it.net].flags + it.layer * args.panels + it.panel, unsigned(kSEpiWarps));
      }
    }
    __syncwarp();
  } else if (warp == 2 + kSEpiWarps) {
    if (lane == 0) {
      // ===== dependency poller =====
      int j = 0;
      bool drain = false;
      for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
        const SItem it = s_decode(args, gi);
        if (!it.valid) continue;
        if (!(args.dbg & 1)) s_wait_deps(args, it, drain);
        *dep_seq = ++j;
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane < 2) {
      // ===== producers: lane 0 = the activation block ([x | h_in]), lane 1 = the weight block of the stage =====
      uint32_t g = 0;
      int j = 0;
      for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
        const SItem it = s_decode(args, gi);
        if (!it.valid) continue;
        const SNet& N = args.net[it.net];
        const size_t poff = size_t(it.panel) * kb * kABlockBytes;
        const char* xa = it.layer == 0 ? N.x0 + size_t(it.t) * N.x0_stride + poff
                                       : N.xmid + (size_t(it.layer - 1) * size_t(args.T) + size_t(it.t)) * args.sbb + poff;
        const char* ha = N.hsb + (size_t(it.layer) * size_t(args.T + 1) + size_t(it.t)) * args.sbb + poff;
        const char* wb = N.w[it.layer] + size_t(it.tile) * (2 * kb) * kBBlockBytes;
        ++j;
        bool need_dep = true;
        for (int b = 0; b < 2 * kb; ++b, ++g) {
          const int s = g % kSStages;
          if (lane == 0) {
            mbar_wait(&empty[s], ((g / kSStages) & 1) ^ 1);
            mbar_expect_tx(&full[s], uint32_t(kABlockBytes + kBBlockBytes));
          }
          __syncwarp(0x3);
          uint8_t* sa = smem + size_t(s) * kStageBytes;
          if (lane == 0 && need_dep) {
            while (*dep_seq < j) { }
            __threadfence_block();
            asm volatile("fence.proxy.async;" ::: "memory");
            need_dep = false;
          }
          const char* src = lane == 0 ? (b < kb ? xa + size_t(b) * kABlockBytes : ha + size_t(b - kb) * kABlockBytes)
                                      : wb + size_t(b) * kBBlockBytes;
          bulk_g2s(sa + lane * kABlockBytes, src, uint32_t(kABlockBytes), &full[s]);      // kABlockBytes == kBBlockBytes
        }
      }
    }
    __syncwarp();
  } else if (warp == 0) {
    // ===== MMA issuer: per k-step  a_hi . [W_hi | W_lo]^T (N = 256: main | correction columns) + a_lo . W_hi^T (N = 128) =====
    uint32_t g = 0;
    int j = 0;
    for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
      const SItem it = s_decode(args, gi);
      if (!it.valid) continue;
      const int buf = j & 1;
      mbar_wait(&acc_empty[buf], ((j >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_main = tmem_base + buf * (2 * kTileCols), d_corr = d_main + kTileCols;
      for (int b = 0; b < 2 * kb; ++b, ++g) {
        const int s = g % kSStages;
        mbar_wait(&full[s], (g / kSStages) & 1);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + size_t(s) * kStageBytes);
        const uint32_t sb = sa + kABlockBytes;
        const uint64_t a_hi = umma_desc(sa, 2048, 128), a_lo = umma_desc(sa + 8192, 2048, 128);
        const uint64_t b_all = umma_desc(sb, 4096, 128);
        if (elect_one()) {
          umma<KIND, 2 * kTileCols>(d_main, a_hi, b_all, b != 0);
          umma<KIND, kTileCols>(d_corr, a_lo, b_all, 1);
          umma<KIND, 2 * kTileCols>(d_main, a_hi + (4096 >> 4), b_all + (8192 >> 4), 1);
          umma<KIND, kTileCols>(d_corr, a_lo + (4096 >> 4), b_all + (8192 >> 4), 1);
          umma_commit(&empty[s]);
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(&acc_full[buf]);
      __syncwarp();
      ++j;
    }
  } else {
    // ===== epilogue: 16 warps; warp % 4 = TMEM lane quarter (rows), grp = which 8 of the tile's 32 hidden units =====
    const int ew = warp - 2;
    {
      const int et = threadIdx.x - 64;
      for (int k = 0; k < args.nets; ++k)
        for (int l = 0; l < args.depth; ++l)
          for (int i = et * 4; i < 4 * H; i += 32 * kSEpiWarps * 4)
            *reinterpret_cast<float4*>(bias_s + (k * kPMaxDepth + l) * kMaxBias + i) =
                *reinterpret_cast<const float4*>(args.net[k].bias[l] + i);
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kSEpiWarps) : "memory");
    }
    const int q4 = warp & 3, grp = ew >> 2;
    const int r = q4 * 32 + lane;
    constexpr float kCorr = (KIND == KBS_KIND_F16) ? (1.0f / kKbsF16LoScale) : 1.0f;
    const int64_t ld = args.ld;
    int j = 0;
    uint32_t gstage = 0;
    for (int gi = blockIdx.x; gi < n_g; gi += n_cc) {
      const SItem it = s_decode(args, gi);
      if (!it.valid) continue;
      const SNet& N = args.net[it.net];
      const int64_t R = int64_t(it.panel) * kPanelRows + r;
      const bool live = R < args.n;
      const int buf = j & 1;
      const int u0 = it.tile * 32 + grp * kSGU;               // first of this thread's 8 hidden units
      while (*dep_seq < j + 1) { }
      __threadfence_block();
      const size_t t = size_t(it.t);
      const float* cin = N.c_hist + (size_t(it.layer) * size_t(args.T + 1) + t) * npH;
      float4 c0, c1;
      if (live) {
        c0 = __ldcg(reinterpret_cast<const float4*>(cin + fb_offset(R, u0, H)));
        c1 = __ldcg(reinterpret_cast<const float4*>(cin + fb_offset(R, u0 + 4, H)));
      }
      const bool rst = live && args.done[t * ld + R];
      if (args.tn) {
        // on-the-fly re-pack of the item's [x | h_in] stages (see bptt_persist_kernel): ring slot st belongs to warp group st % 4
        for (int b = 0; b < 2 * kb; ++b) {
          const uint32_t g = gstage + uint32_t(b);
          const int st = int(g % kSStages);
          // ownership by ring SLOT, not by stage number: a barrier must always be watched by the same warps, which then see
          // every one of its phases in order -- a parity wait on a barrier that is still a whole phase behind returns at once
          // (kSStages = 6 is not a multiple of 4: owners by stage number read slots that had not landed yet, ~1 in 400 panels)
          if ((st & 3) != grp) continue;
          mbar_wait(&full[st], (g / kSStages) & 1);
          if ((b % tiles) == it.tile) {
            const uint8_t* sa = smem + size_t(st) * kStageBytes;
            const int cm = (ew & 3) * 32 + lane;
            const int r8 = cm & 15, c = (cm >> 4) & 3, plane = cm >> 6;
            const uint8_t* sp = sa + ((size_t(plane) * 4 + c) * kPanelRows + size_t(r8) * 8) * 16;
            uint4 in[8];
#pragma unroll
            for (int rr = 0; rr < 8; ++rr) {
              in[rr] = *reinterpret_cast<const uint4*>(sp + rr * 16);
              if (int64_t(it.panel) * kPanelRows + r8 * 8 + rr >= args.n) in[rr] = make_uint4(0u, 0u, 0u, 0u);
            }
            const int64_t kp = (int64_t(it.t) * args.panels + it.panel) * kPanelRows + r8 * 8;
            const int64_t kbq = kp / 32;
            const int cq = int((kp / 8) & 3);
            const int j0 = b * 32 + c * 8;                      // column of [x | h_in]: x blocks first, then h blocks
            char* dp = N.tn_xh[it.layer] + size_t(j0 / kTileCols) * args.tn_col_bytes +
                       (((size_t(kbq) * 4 + cq) * 2 + plane) * kTileCols + size_t(j0 % kTileCols)) * 16;    // WB block layout
#pragma unroll
            for (int i8 = 0; i8 < 8; ++i8) {
              const unsigned sel = (i8 & 1) ? 0x7632u : 0x5410u;
              uint4 o;
              o.x = __byte_perm((&in[0].x)[i8 >> 1], (&in[1].x)[i8 >> 1], sel);
              o.y = __byte_perm((&in[2].x)[i8 >> 1], (&in[3].x)[i8 >> 1], sel);
              o.z = __byte_perm((&in[4].x)[i8 >> 1], (&in[5].x)[i8 >> 1], sel);
              o.w = __byte_perm((&in[6].x)[i8 >> 1], (&in[7].x)[i8 >> 1], sel);
              *reinterpret_cast<uint4*>(dp + size_t(i8) * 16) = o;
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[st]);
        }
        gstage += uint32_t(2 * kb);
      }
      mbar_wait(&acc_full[buf], (j >> 1) & 1);
      tc_fence_after();
      const uint32_t tq = tmem_base + (uint32_t(q4 * 32) << 16) + uint32_t(buf * (2 * kTileCols) + grp * 32);
      float v[32];
      {
        float cr[32];
        tmem_ld32(tq, v);
        tmem_ld32(tq + kTileCols, cr);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] += kCorr * cr[i];
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
      const float* bs = bias_s + (it.net * kPMaxDepth + it.layer) * kMaxBias + it.tile * kTileCols + grp * 32;
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] += bs[i];
      if (live) {
        float hn[8], cn[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float cprev = i < 4 ? (&c0.x)[i] : (&c1.x)[i - 4];
          const float ai = sigmoidf_(v[i]), af = sigmoidf_(v[8 + i]), ag = tanhf_(v[16 + i]), ao = sigmoidf_(v[24 + i]);
          cn[i] = af * cprev + ai * ag;                           // c' = s(f) c + s(i) tanh(g)   (eqx LSTMCell)
          hn[i] = ao * tanhf_(cn[i]);                             // h' = s(o) tanh(c')
          if (rst) cn[i] = 0.0f;
          v[i] = ai; v[8 + i] = af; v[16 + i] = ag; v[24 + i] = ao;   // the activated gates, kept for the backward pass
        }
        const float h0[4] = {hn[0], hn[1], hn[2], hn[3]}, h1[4] = {hn[4], hn[5], hn[6], hn[7]};
        const KbsSplit4 s0 = sb_split4<KIND>(h0), s1 = sb_split4<KIND>(h1);
        char* x_out = N.xmid + (size_t(it.layer) * size_t(args.T) + t) * args.sbb;
        char* h_out = N.hsb + (size_t(it.layer) * size_t(args.T + 1) + t + 1) * args.sbb;
        float* cdst = N.c_hist + (size_t(it.layer) * size_t(args.T + 1) + t + 1) * npH;
        sb_store_split8<kPanelRows, KIND>(h_out, R, u0, kb, s0, s1, rst);      // what step t + 1 reads (reset where done)
        *reinterpret_cast<float4*>(cdst + fb_offset(R, u0, H)) = make_float4(cn[0], cn[1], cn[2], cn[3]);
        *reinterpret_cast<float4*>(cdst + fb_offset(R, u0 + 4, H)) = make_float4(cn[4], cn[5], cn[6], cn[7]);
        sb_store_split8<kPanelRows, KIND>(x_out, R, u0, kb, s0, s1, false);    // what the layer above reads (un-reset)
        if (it.layer + 1 == args.depth) {
          float* hr = N.h_top_rm + (t * size_t(args.n) + size_t(R)) * H + u0;
          *reinterpret_cast<float4*>(hr) = make_float4(hn[0], hn[1], hn[2], hn[3]);
          *reinterpret_cast<float4*>(hr + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
        }
      }
      // publish (h, c, x are stored), then keep the activated gates: nothing in this launch reads them
      __syncwarp();
      if (lane == 0) asm volatile("red.release.cta.shared::cta.add.u32 [%0], 1;" ::"r"(smem_u32(epi_done)) : "memory");
      if (live) {
        float* sg = N.save_g + (t * args.depth + it.layer) * 4 * npH;
#pragma unroll
        for (int gate = 0; gate < 4; ++gate) {
          *reinterpret_cast<float4*>(sg + gate * npH + fb_offset(R, u0, H)) = make_float4(v[8 * gate], v[8 * gate + 1], v[8 * gate + 2], v[8 * gate + 3]);
          *reinterpret_cast<float4*>(sg + gate * npH + fb_offset(R, u0 + 4, H)) =
              make_float4(v[8 * gate + 4], v[8 * gate + 5], v[8 * gate + 6], v[8 * gate + 7]);
        }
      }
      ++j;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}

// ---- input projection straight from the env-major SoA observations ("async" form of MODE_PROJ_SOA) -------------------------
// x = W_in o + b_in for all T x n rows, written as the SB operand of LSTM layer 0, WITHOUT the packed staging buffer:
// pack_soa_sb_kernel (read 1.9 KB + write 1.9 KB per critic row) followed by the MODE_PROJ launch (read it again, 128-column
// tiles: two items per panel) cost 0.33 + 0.33 ms per 4 096 x 100 rollout for ~0.2 ms of HBM traffic.  Here one CTA per SM
// walks the 128-row panels; per K block (32 features; 16 for TF32):
//   warp 1    raw producer: one 2-D TMA tensor request per stage = 32 feature rows x 128 envs (features 80..447 of the
//             critic come straight from the recorded cinert / cvel arrays, train.py:1405-1413), 4-deep ring: ~48 KB of HBM
//             reads in flight per SM (the register-staged MODE_PROJ_SOA had ~16 KB: 4x slower);
//   warp 2    weight producer: the 32 KB W_in block (one 256-column tile = all H outputs, L2-resident) into the operand ring;
//   warps 12-19  converters, two sets of 4 warps on alternate stages: thread = env row; 32 floats from the raw stage
//             (conflict-free column reads) -> hi / lo split -> the A block in UMMA layout -> fence.proxy.async -> arrive;
//   warp 0    MMA issuer: the persistent kernel's scheme (3 x N = 256 MMAs per k-step, main + correction accumulators);
//   warps 4-11   epilogue: TMEM -> + bias -> split -> SB stores (16-byte chunks, 512 B per warp).
// Requires H == 256 (one tile).  KBS_PROJ_STAGED=1 restores pack + MODE_PROJ.
constexpr int kFStagesRaw = 4, kFStagesOp = 3;
constexpr int kFRawBytes = 32 * kPanelRows * 4;                  // 32 feature rows x 128 envs x 4 B = 16 KB
constexpr int kFOpBytes = kABlockBytes + 2 * 4 * 256 * 16;       // A block 16 KB + B block [chunk][hi|lo][256 rows][16 B] 32 KB
constexpr int kFThreads = 640;
constexpr int kFConvWarp0 = 12, kFConvWarps = 8, kFEpiWarp0 = 4, kFEpiWarps = 8;
constexpr int kFSmemBytes = kFStagesRaw * kFRawBytes + kFStagesOp * kFOpBytes + 256 * 4 + 256 /*barriers*/ + 1024 /*align*/;

constexpr int kFMaxBlocks = 32;
struct FProjArgs {
  // K blocks of the projection in the order the kernel walks them: block b = kFeat consecutive feature ROWS of one source
  // array starting at blk_row0[b] (within a step), the first blk_nvalid[b] of them real (the rest -- the unwritten dump
  // slots of the critic's SoA buffer, rows of the next step, rows past the array -- are masked to zero by the converters
  // and meet zero weights).  Sources: 0 = observations [T][F][ld], 1 = cinert [T][240][ld], 2 = cvel [T][144][ld]
  // (features 80..447 of the critic are cinert[1:] | cvel[1:], train.py:1405-1413).  The weight tile is packed in the same
  // K order (pack_proj_weights_kmap_kernel).
  CUtensorMap tmap[3];     // 2-D {ld envs, T * rows per step} fp32, box {128 envs, kFeat rows}
  int rows_per_step[3];
  signed char blk_src[kFMaxBlocks];
  short blk_row0[kFMaxBlocks];
  short blk_nvalid[kFMaxBlocks];
  int kb, H;
  int64_t n, n_pad;
  const char* w_sb;        // [kb] x 32 KB blocks, WB layout, 256 columns
  const float* bias;       // [256]
  char* x_sb;              // out [T] x sbb
  size_t sbb;
  int items;               // T * n_pad / 128
  unsigned int* status;    // health word: KBS_STATUS_F16_RANGE when an input or an output leaves the FP16-split range
  int dbg;                 // profiling only (KBS_FPROJ_DBG): 1 converters skip load + split, 2 no MMAs, 4 no raw copies,
                           // 8 no epilogue stores
  long long* trace;        // per CTA [16] at trace + (148 + blockIdx.x) * 16: total cycles, items, then wait cycles of
                           // raw producer (raw_empty), weight producer (empty), converter warp 12 (raw_full, empty),
                           // issuer (full, acc_empty), epilogue warp 4 (acc_full)
};

template <int KIND>
__global__ void __launch_bounds__(kFThreads, 1) input_proj_fused_kernel(const __grid_constant__ FProjArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* raw = smem;
  uint8_t* op = smem + kFStagesRaw * kFRawBytes;
  float* bias_s = reinterpret_cast<float*>(op + kFStagesOp * kFOpBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + 256);
  uint64_t* raw_full = bars;                       // [kFStagesRaw] feature rows landed
  uint64_t* raw_empty = raw_full + kFStagesRaw;    // [kFStagesRaw] converters have the values in registers
  uint64_t* full = raw_empty + kFStagesRaw;        // [kFStagesOp]  A block written + W block landed
  uint64_t* empty = full + kFStagesOp;             // [kFStagesOp]  MMAs have read the stage
  uint64_t* acc_full = empty + kFStagesOp;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  constexpr int kE = kbs_chunk_elems(KIND), kFeat = 4 * kE;      // features per 16-byte chunk / per K block
  constexpr int kBlk = kbs_block_k(KIND);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ppt = int(a.n_pad / kPanelRows);                     // panels per step

  if (threadIdx.x == 0) {
    for (int s = 0; s < kFStagesRaw; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], kFConvWarps / 2); }
    for (int s = 0; s < kFStagesOp; ++s) { mbar_init(&full[s], 1 + kFConvWarps / 2); mbar_init(&empty[s], 1); }
    mbar_init(acc_full, 1); mbar_init(acc_empty, kFEpiWarps);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  long long* tr = a.trace ? a.trace + size_t(148 + blockIdx.x) * 16 : nullptr;
  const long long t_start = clock64();
#define FTR_WAIT(slot, stmt) do { if (tr) { const long long w0_ = clock64(); stmt; tw[slot] += clock64() - w0_; } else { stmt; } } while (0)
  long long tw[2] = {0, 0};

  if (warp == 1) {
    // ===== raw producer: ONE 2-D TMA request per stage = the block's kFeat feature rows x the panel's 128 envs (16 KB,
    // box rows land as [feature][env] fp32).  MEASURED (tools/fproj_probe.py): the same rows as 32 separate 512-byte
    // cp.async.bulk requests cost the SM ~48 cycles each whichever warps issue them = 1.5 K cycles per stage (the MMAs
    // need 880), and as cp.async (LDGSTS) 16-byte pieces the kernel was slower still.  Out-of-range envs / rows are
    // zero-filled by the TMA unit, so every stage expects the full box. =====
    if (lane == 0) {
      uint32_t g = 0;
      for (int item = blockIdx.x; item < a.items; item += gridDim.x) {
        const int t = item / ppt, e0 = (item % ppt) * kPanelRows;
        for (int b = 0; b < a.kb; ++b, ++g) {
          const int sr = g % kFStagesRaw;
          const int src = a.blk_src[b];
          FTR_WAIT(0, mbar_wait(&raw_empty[sr], ((g / kFStagesRaw) & 1) ^ 1));
          mbar_expect_tx(&raw_full[sr], (a.dbg & 4) ? 0u : uint32_t(kFeat * kPanelRows * 4));
          if (!(a.dbg & 4)) {
            const int c1 = t * a.rows_per_step[src] + a.blk_row0[b];
            asm volatile(
                "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                    smem_u32(raw + size_t(sr) * kFRawBytes)),
                "l"(reinterpret_cast<uint64_t>(&a.tmap[src])), "r"(e0), "r"(c1), "r"(smem_u32(&raw_full[sr]))
                : "memory");
          }
        }
      }
      if (tr) tr[2] = tw[0];
    }
    __syncwarp();
  } else if (warp == 2) {
    // ===== weight producer =====
    if (lane == 0) {
      uint32_t g = 0;
      for (int item = blockIdx.x; item < a.items; item += gridDim.x) {
        for (int b = 0; b < a.kb; ++b, ++g) {
          const int s = g % kFStagesOp;
          FTR_WAIT(0, mbar_wait(&empty[s], ((g / kFStagesOp) & 1) ^ 1));
          mbar_expect_tx(&full[s], uint32_t(kFOpBytes - kABlockBytes));
          bulk_g2s(op + size_t(s) * kFOpBytes + kABlockBytes, a.w_sb + size_t(b) * (kFOpBytes - kABlockBytes),
                   uint32_t(kFOpBytes - kABlockBytes), &full[s]);
        }
      }
      if (tr) tr[3] = tw[0];
    }
    __syncwarp();
  } else if (warp >= kFConvWarp0 && warp < kFConvWarp0 + kFConvWarps) {
    // ===== converters: two sets of 4 warps on ALTERNATE stages; thread = env row of the panel, whole K block.  MEASURED:
    // one set of 4 (or 8 half-block) warps on every stage is busy ~1.1-1.4 K cycles per stage (load, split, store, proxy
    // fence, barrier round trips: a latency chain) against 880 cycles of MMA issue; two stages in flight hide it. =====
    const int cw = warp - kFConvWarp0;
    const int set = cw >> 2;
    const int r = (cw & 3) * 32 + lane;
    uint32_t g = 0;
    bool bad = false;                                   // an input outside the FP16-split range (raw physical quantities)
    for (int item = blockIdx.x; item < a.items; item += gridDim.x) {
      const int64_t e0 = int64_t(item % ppt) * kPanelRows;
      const bool valid = e0 + r < a.n;
      for (int b = 0; b < a.kb; ++b, ++g) {
        if (int(g & 1) != set) continue;
        const int sr = g % kFStagesRaw, s = g % kFStagesOp;
        FTR_WAIT(0, mbar_wait(&raw_full[sr], (g / kFStagesRaw) & 1));
        const float* rf = reinterpret_cast<const float*>(raw + size_t(sr) * kFRawBytes) + r;
        const int nv = int(a.blk_nvalid[b]);
        float x[kFeat];
#pragma unroll
        for (int i = 0; i < kFeat; ++i) x[i] = (valid && i < nv && !(a.dbg & 1)) ? rf[i * kPanelRows] : 0.0f;
        bad = bad || sb_out_of_range<KIND, kFeat>(x);
        __syncwarp();
        if (lane == 0) mbar_arrive(&raw_empty[sr]);
        // Stage g reuses the operand slot of stage g - 3.  Its generic-proxy stores land ~50 cycles after the barrier flips,
        // and MEASURED (tools/fproj_stress.py, 3xTF32 operands, whose converters outrun the MMAs and sit on this wait):
        // releasing them on empty[s] -- the tcgen05.commit of stage g - 3 -- gave one wrong 32-row x 1-stage contribution
        // in ~3 % of the launches (0 / 384 with the wait below): the commit's arrival does not cover the tail of the
        // operand reads against a writer this fast (the bulk copies of the other kernels arrive >= 1 us later and never
        // see it).  So a slot is rewritten only after the commit of stage g - 2: commits complete in order, which puts a
        // whole stage of MMA time between the last read and the first store.
        if (g >= 2) { const uint32_t gp = g - 2; FTR_WAIT(1, mbar_wait(&empty[gp % kFStagesOp], (gp / kFStagesOp) & 1)); }
        uint8_t* sa = op + size_t(s) * kFOpBytes;
        if (!(a.dbg & 1))
#pragma unroll
        for (int c = 0; c < 4; ++c) {                        // chunk c of the block: [part][chunk][row][16 B]
          uint4 hi, lo;
          if (KIND == KBS_KIND_F16) {
            const float x0[4] = {x[(8 * c) % kFeat], x[(8 * c + 1) % kFeat], x[(8 * c + 2) % kFeat], x[(8 * c + 3) % kFeat]};
            const float x1[4] = {x[(8 * c + 4) % kFeat], x[(8 * c + 5) % kFeat], x[(8 * c + 6) % kFeat], x[(8 * c + 7) % kFeat]};
            const KbsSplit4 s0 = sb_split4<KIND>(x0), s1 = sb_split4<KIND>(x1);
            hi = make_uint4(s0.hi.x, s0.hi.y, s1.hi.x, s1.hi.y);
            lo = make_uint4(s0.lo.x, s0.lo.y, s1.lo.x, s1.lo.y);
          } else {
            const float x0[4] = {x[(4 * c) % kFeat], x[(4 * c + 1) % kFeat], x[(4 * c + 2) % kFeat], x[(4 * c + 3) % kFeat]};
            const KbsSplit4 s0 = sb_split4<KIND>(x0);
            hi = s0.hi; lo = s0.lo;
          }
          *reinterpret_cast<uint4*>(sa + c * 2048 + r * 16) = hi;
          *reinterpret_cast<uint4*>(sa + 8192 + c * 2048 + r * 16) = lo;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);
      }
    }
    sb_flag_range(a.status, bad);
    if (tr && warp == kFConvWarp0 && lane == 0) { tr[4] = tw[0]; tr[5] = tw[1]; }
  } else if (warp == 0) {
    // ===== MMA issuer =====
    uint32_t g = 0;
    int j = 0;
    for (int item = blockIdx.x; item < a.items; item += gridDim.x, ++j) {
      FTR_WAIT(1, mbar_wait(acc_empty, (j & 1) ^ 1));
      tc_fence_after();
      const uint32_t d_main = tmem_base, d_corr = tmem_base + 256;
      for (int b = 0; b < a.kb; ++b, ++g) {
        const int s = g % kFStagesOp;
        FTR_WAIT(0, mbar_wait(&full[s], (g / kFStagesOp) & 1));
        tc_fence_after();
        const uint32_t sa = smem_u32(op + size_t(s) * kFOpBytes);
        const uint64_t a_hi = umma_desc(sa, 2048, 128), a_lo = a_hi + (8192 >> 4);
        const uint64_t b_hi = umma_desc(sa + kABlockBytes, 8192, 128), b_lo = b_hi + (4096 >> 4);
        constexpr uint64_t kAStep = 4096 >> 4, kBStep = 16384 >> 4;
        if (elect_one()) {
          const uint32_t acc = b != 0;
          if (!(a.dbg & 2)) {
          umma<KIND, 256>(d_main, a_hi, b_hi, acc);
          umma<KIND, 256>(d_corr, a_lo, b_hi, acc);
          umma<KIND, 256>(d_corr, a_hi, b_lo, 1);
          umma<KIND, 256>(d_main, a_hi + kAStep, b_hi + kBStep, 1);
          umma<KIND, 256>(d_corr, a_lo + kAStep, b_hi + kBStep, 1);
          umma<KIND, 256>(d_corr, a_hi + kAStep, b_lo + kBStep, 1);
          }
          umma_commit(&empty[s]);
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(acc_full);
      __syncwarp();
    }
    if (tr && lane == 0) { tr[6] = tw[0]; tr[7] = tw[1]; tr[1] = j; }
  } else if (warp >= kFEpiWarp0 && warp < kFEpiWarp0 + kFEpiWarps) {
    // ===== epilogue: warp % 4 = TMEM lane quarter, (warp - 4) / 4 = which 128 of the 256 output columns =====
    const int et = threadIdx.x - 32 * kFEpiWarp0;
    bias_s[et] = a.bias[et];
    asm volatile("bar.sync 1, %0;" ::"n"(32 * kFEpiWarps) : "memory");
    const int q4 = warp & 3, half = (warp - kFEpiWarp0) >> 2;
    const int r = q4 * 32 + lane;
    constexpr float kCorr = (KIND == KBS_KIND_F16) ? (1.0f / kKbsF16LoScale) : 1.0f;
    int j = 0;
    for (int item = blockIdx.x; item < a.items; item += gridDim.x, ++j) {
      const int64_t t = item / ppt, R = int64_t(item % ppt) * kPanelRows + r;
      char* xo = a.x_sb + size_t(t) * a.sbb;
      FTR_WAIT(0, mbar_wait(acc_full, j & 1));
      tc_fence_after();
      const uint32_t tq = tmem_base + (uint32_t(q4 * 32) << 16) + uint32_t(half * 128);
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        // 32 output columns per pass: all four TMEM loads are in flight before the wait; after the last pass's loads the
        // accumulators are in registers and TMEM goes back to the MMA issuer before the split + stores
        float v[32], cr[32];
        tmem_ld16(tq + cc * 32, v);
        tmem_ld16(tq + cc * 32 + 16, v + 16);
        tmem_ld16(tq + 256 + cc * 32, cr);
        tmem_ld16(tq + 256 + cc * 32 + 16, cr + 16);
        tmem_ld_wait();
        if (cc == 3) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(acc_empty);
        }
        const float* bs = bias_s + half * 128 + cc * 32;
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = (v[i] + kCorr * cr[i]) + bs[i];
        sb_flag_range(a.status, sb_out_of_range<KIND, 32>(v));
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          const float x0[4] = {v[8 * c8], v[8 * c8 + 1], v[8 * c8 + 2], v[8 * c8 + 3]};
          const float x1[4] = {v[8 * c8 + 4], v[8 * c8 + 5], v[8 * c8 + 6], v[8 * c8 + 7]};
          if (!(a.dbg & 8))
          sb_store_split8<kPanelRows, KIND>(xo, R, half * 128 + cc * 32 + c8 * 8, a.H / kBlk, sb_split4<KIND>(x0), sb_split4<KIND>(x1),
                                            false);
        }
      }
    }
    if (tr && warp == kFEpiWarp0 && lane == 0) tr[8] = tw[0];
  }
#undef FTR_WAIT
  tc_fence_before();
  __syncthreads();
  if (tr && threadIdx.x == 0) tr[0] = clock64() - t_start;
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}

// ---- packing kernels ------------------------------------------------------------------------------------------------
// eqx LSTMCell weights [4H][H] x2 + bias [4H]  ->  gate-interleaved SB tiles (hi/lo) + interleaved bias.
// tile j (128 columns = 32 hidden units), column c = half * 64 + gate * 16 + uu  ->  unit = 32 j + 16 half + uu:
// an epilogue thread that owns 16 units finds their i, f, g, o pre-activations in 64 CONSECUTIVE TMEM columns.
template <int KIND, int TILE, int GU = 16>
__global__ void __launch_bounds__(256)
pack_lstm_weights_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh, const float* __restrict__ b,
                         char* __restrict__ w_sb, float* __restrict__ bias_t, int H, int Kx, int ldx) {
  // w_ih: [4H][ldx] with Kx (<= ldx) columns used -- eqx weight_ih (Kx = ldx = H), or the layer-0 weight with the input
  // projection folded in (fuse_input_weights_kernel: Kx = padded observation width)
  const int kq = (Kx + H) / 4;
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= int64_t(4 * H) * kq) return;
  const int col_g = int(idx / kq);                        // global packed column: tile * TILE + c
  const int k = int(idx % kq) * 4;
  const int tile = col_g / TILE, c = col_g % TILE;
  const int grp = c / (4 * GU), gate = (c % (4 * GU)) / GU, uu = c % GU;      // [GU-unit group][gate i,f,g,o][unit]
  const int u = tile * (TILE / 4) + grp * GU + uu;
  const int row = gate * H + u;                           // eqx row (i,f,g,o blocks of H)
  const float* src = (k < Kx) ? w_ih + size_t(row) * ldx + k : w_hh + size_t(row) * H + (k - Kx);
  const float x[4] = {src[0], src[1], src[2], src[3]};
  sb_store4<TILE, KIND, true>(w_sb, col_g, k, (Kx + H) / kbs_block_k(KIND), x);
  if (k == 0) bias_t[col_g] = b[row];
}

// Input projection folded into LSTM layer 0 (persistent kernel): gates = W_ih (W_in o + b_in) + W_hh h + b
//   = (W_ih W_in) o + W_hh h + (W_ih b_in + b).  wf [4H][Kf] = W_ih W_in (columns >= num_in zero), bf [4H]; sums in
// double, rounded once to fp32 (the reference rounds x = W_in o + b_in to fp32 first: the two forms differ at the 1e-7
// level, inside the 1e-5 tolerance; the oracle keeps the reference's two-step form).
__global__ void __launch_bounds__(256)
fuse_input_weights_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_in, int ld_in, int num_in,
                          const float* __restrict__ b_in, const float* __restrict__ b, float* __restrict__ wf,
                          float* __restrict__ bf, int H, int Kf) {
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= int64_t(4 * H) * (Kf + 1)) return;
  const int row = int(idx / (Kf + 1)), k = int(idx % (Kf + 1));
  const float* wr = w_ih + size_t(row) * H;
  double acc = 0.0;
  if (k == Kf) {
    for (int j = 0; j < H; ++j) acc += double(wr[j]) * double(b_in[j]);
    bf[row] = float(acc + double(b[row]));
  } else {
    if (k < num_in)
      for (int j = 0; j < H; ++j) acc += double(wr[j]) * double(w_in[size_t(j) * ld_in + k]);
    wf[size_t(row) * Kf + k] = float(acc);
  }
}

// eqx Linear weight [H][ldw] (K zero-padded to ldw) -> ceil(H/128) SB tiles of 128 plain columns (rows >= H zero), K padded to Kp.
template <int KIND, int TILE = kTileCols>
__global__ void __launch_bounds__(256)
pack_proj_weights_kernel(const float* __restrict__ w, int ldw, const float* __restrict__ b, char* __restrict__ w_sb,
                         float* __restrict__ bias_t, int H, int Kp, int cols) {
  const int kq = Kp / 4;
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= int64_t(cols) * kq) return;
  const int col = int(idx / kq), k = int(idx % kq) * 4;
  float x[4] = {0.f, 0.f, 0.f, 0.f};
  if (col < H) {
#pragma unroll
    for (int i = 0; i < 4; ++i) x[i] = (k + i < ldw) ? w[size_t(col) * ldw + k + i] : 0.0f;
  }
  sb_store4<TILE, KIND, true>(w_sb, col, k, Kp / kbs_block_k(KIND), x);
  if (k == 0) bias_t[col] = col < H ? b[col] : 0.0f;
}

// W_in as ONE 256-column tile in the K order input_proj_fused_kernel walks: K index kk = block kk / kf, row j = kk % kf of
// the block -> eqx input column fbase[block] + j, or a zero weight for a masked row (j >= nvalid[block]).
struct FPackLayout {
  int kb;
  int fbase[kFMaxBlocks];
  short nvalid[kFMaxBlocks];
};
template <int KIND>
__global__ void __launch_bounds__(256)
pack_proj_weights_kmap_kernel(const float* __restrict__ w, int ldw, const float* __restrict__ b, const __grid_constant__ FPackLayout L,
                              char* __restrict__ w_sb, float* __restrict__ bias_t, int H, int Kq) {
  constexpr int kf = kbs_block_k(KIND);
  const int kq = Kq / 4;
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= int64_t(256) * kq) return;
  const int col = int(idx / kq), k = int(idx % kq) * 4;
  float x[4] = {0.f, 0.f, 0.f, 0.f};
  if (col < H) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int blk = (k + i) / kf, j = (k + i) % kf;
      x[i] = j < L.nvalid[blk] ? w[size_t(col) * ldw + L.fbase[blk] + j] : 0.0f;
    }
  }
  sb_store4<256, KIND, true>(w_sb, col, k, Kq / kf, x);
  if (k == 0) bias_t[col] = col < H ? b[col] : 0.0f;
}

// Output head of the persistent rollout kernel: eqx Linear weight [num_out][H] -> ONE 256-column SB tile whose columns
// follow the epilogue's thread map: column c = grp * 64 + gate * 16 + uu; joint group grp holds joints 5 grp .. 5 grp + 4
// in uu = 0..4: gate 0 = mean row (joint), gate 1 = std row (20 + joint); all else zero.  The critic (num_out = 1)
// lands in column 0.
template <int KIND>
__global__ void __launch_bounds__(256)
pack_head_weights_kernel(const float* __restrict__ w, const float* __restrict__ b, char* __restrict__ w_sb,
                         float* __restrict__ bias_t, int H, int num_out) {
  const int kq = H / 4;
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= int64_t(kTileColsP) * kq) return;
  const int col = int(idx / kq), k = int(idx % kq) * 4;
  const int grp = col / 64, gate = (col % 64) / 16, uu = col % 16;
  int row = -1;
  if (gate < 2 && uu < 5) row = gate * KBS_NUM_JOINTS + grp * 5 + uu;
  if (row >= num_out) row = -1;
  float x[4] = {0.f, 0.f, 0.f, 0.f};
  if (row >= 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) x[i] = w[size_t(row) * H + k + i];
  }
  sb_store4<kTileColsP, KIND, true>(w_sb, col, k, H / kbs_block_k(KIND), x);
  if (k == 0) bias_t[col] = row >= 0 ? b[row] : 0.0f;
}

// ABI row-major [n][H] <-> FB blocked state.  to_fb: rows >= n of the last panel are zero-filled.
__global__ void __launch_bounds__(256)
fb_convert_kernel(float* __restrict__ rm, float* __restrict__ fb, int64_t n, int64_t n_pad, int H, int to_fb) {
  const int hq = H / 4;
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= n_pad * hq) return;
  const int64_t panel = idx / (int64_t(kPanelRows) * hq);
  const int rem = int(idx - panel * int64_t(kPanelRows) * hq);
  const int kc = rem / kPanelRows, r = rem % kPanelRows;
  const int64_t row = panel * kPanelRows + r;
  float4* f = reinterpret_cast<float4*>(fb + fb_offset(row, kc * 4, H));
  if (to_fb) {
    *f = row < n ? *reinterpret_cast<const float4*>(rm + row * H + kc * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
  } else if (row < n) {
    *reinterpret_cast<float4*>(rm + row * H + kc * 4) = *f;
  }
}

// row-major [n][K] fp32 -> SB (A operand, 128-row panels).  Rows >= n of the last panel are zero-filled.
template <int KIND>
__global__ void __launch_bounds__(256)
pack_rows_sb_kernel(const float* __restrict__ src, int64_t ld, char* __restrict__ sb, int64_t n, int64_t n_pad, int K) {
  const int kq = K / 4;
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= n_pad * kq) return;
  // consecutive threads -> consecutive rows of the same 4-wide K group: coalesced SB stores
  const int64_t panel = idx / (int64_t(kPanelRows) * kq);
  const int rem = int(idx - panel * int64_t(kPanelRows) * kq);
  const int kc = rem / kPanelRows, r = rem % kPanelRows;
  const int64_t row = panel * kPanelRows + r;
  float x[4] = {0.f, 0.f, 0.f, 0.f};
  if (row < n) {
    const float4 v = *reinterpret_cast<const float4*>(src + row * ld + kc * 4);
    x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
  }
  sb_store4<kPanelRows, KIND>(sb, row, kc * 4, K / kbs_block_k(KIND), x);
}

// All ABI carry <-> kernel layout conversions of one rollout call as ONE launch (blockIdx.y = job): the 8 + 8 separate
// fb_convert / pack_rows launches around the persistent kernel were pure launch latency (~6 us each, 4 MB moved).
//   mode 0: row-major [n][H] -> SB (h, A operand);  mode 1: row-major -> FB (c);  mode 2: FB -> row-major.
struct CarryJobs {
  float* rm[8];
  void* blk[8];
  int mode[8];
  int64_t ld_rm;     // row stride of the row-major side (H for the ABI carries, the record width for flat carries)
  unsigned int* status;   // health word (FP16-split range of the caller's hidden carries)
};
// Both sides coalesced: a block moves a 32-row x 32-group tile (group = 8 consecutive units = 32 B) through shared
// memory -- on the row-major side a warp touches 1 KB of ONE row (flat carry records are 4 KB apart: one row per lane
// fetched half-used sectors at 3.1 TB/s), on the blocked side 512 B of one 16-byte chunk column (lane = row).
template <int KIND>
__global__ void __launch_bounds__(256)
carry_convert_kernel(const __grid_constant__ CarryJobs J, int64_t n, int64_t n_pad, int H) {
  __shared__ float4 tile[2][32][33];
  const int j = blockIdx.y;
  const int kgs = H / 8, kt = (kgs + 31) / 32;
  const int64_t rb = blockIdx.x / kt;
  const int kg0 = int(blockIdx.x - rb * kt) * 32;
  const int64_t row0 = rb * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* rm = J.rm[j];
  const int mode = J.mode[j];
  const int64_t ldr = J.ld_rm;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  if (mode != 2) {
    for (int rr = warp; rr < 32; rr += 8) {
      const int64_t row = row0 + rr;
      const int kg = kg0 + lane;
      float4 a = z, b = z;
      if (row < n && kg < kgs) {
        const float4* p = reinterpret_cast<const float4*>(rm + row * ldr + kg * 8);
        a = __ldcs(p); b = __ldcs(p + 1);
      }
      tile[0][rr][lane] = a; tile[1][rr][lane] = b;
    }
    __syncthreads();
    const int64_t row = row0 + lane;                  // < n_pad: rows >= n carry zeros
    for (int kk = warp; kk < 32 && kg0 + kk < kgs; kk += 8) {
      const int kg = kg0 + kk;
      const float4 a = tile[0][lane][kk], b = tile[1][lane][kk];
      if (mode == 1) {
        float* fb = static_cast<float*>(J.blk[j]);
        *reinterpret_cast<float4*>(fb + fb_offset(row, kg * 8, H)) = a;
        *reinterpret_cast<float4*>(fb + fb_offset(row, kg * 8 + 4, H)) = b;
      } else {
        const float x0[4] = {a.x, a.y, a.z, a.w}, x1[4] = {b.x, b.y, b.z, b.w};
        sb_flag_range(J.status, sb_out_of_range<KIND, 4>(x0) || sb_out_of_range<KIND, 4>(x1));
        sb_store_split8<kPanelRows, KIND>(J.blk[j], row, kg * 8, H / kbs_block_k(KIND), sb_split4<KIND>(x0), sb_split4<KIND>(x1),
                                          false);
      }
    }
  } else {
    const float* fb = static_cast<const float*>(J.blk[j]);
    const int64_t row = row0 + lane;
    for (int kk = warp; kk < 32 && kg0 + kk < kgs; kk += 8) {
      const int kg = kg0 + kk;
      tile[0][lane][kk] = *reinterpret_cast<const float4*>(fb + fb_offset(row, kg * 8, H));
      tile[1][lane][kk] = *reinterpret_cast<const float4*>(fb + fb_offset(row, kg * 8 + 4, H));
    }
    __syncthreads();
    for (int rr = warp; rr < 32; rr += 8) {
      const int64_t r2 = row0 + rr;
      const int kg = kg0 + lane;
      if (r2 < n && kg < kgs) {
        float4* p = reinterpret_cast<float4*>(rm + r2 * ldr + kg * 8);
        __stcs(p, tile[0][rr][lane]); __stcs(p + 1, tile[1][rr][lane]);
      }
    }
  }
}

// env-major SoA observations [T][F][ld] -> SB rows [T * n_pad][Kp] (features beyond F and envs beyond n zero-filled).
// thread = (t, panel, 8-feature group, row): reads 8 SoA rows at one env (coalesced over envs) and writes one full
// 16-byte chunk per plane (FP16 kind; two per plane for TF32): 512 contiguous bytes per warp and store instruction.
// Critic shortcut (cinert != nullptr): features 80..447 are the privileged dump cinert[1:] (230) | cvel[1:] (138)
// (train.py:1405-1413) -- they are read straight from the recorded state, so the observation kernel never writes them
// to the SoA buffer and this kernel never reads them back (saves 2 x 1.5 KB of HBM traffic per env-step).
template <int KIND>
__global__ void __launch_bounds__(256)
pack_soa_sb_kernel(const float* __restrict__ soa, int F, int64_t ld, char* __restrict__ sb, int64_t n, int64_t n_pad,
                   int Kp, int64_t T, const float* __restrict__ cinert, const float* __restrict__ cvel,
                   unsigned int* __restrict__ status) {
  const int kq = Kp / 8;
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  const int64_t rows = T * n_pad;
  if (idx >= rows * kq) return;
  const int64_t panel = idx / (int64_t(kPanelRows) * kq);          // global panel over (t, env panel)
  const int rem = int(idx - panel * int64_t(kPanelRows) * kq);
  const int kc = rem / kPanelRows, r = rem % kPanelRows;
  const int64_t row = panel * kPanelRows + r;
  const int64_t t = row / n_pad, e = row - t * n_pad;
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int f = kc * 8 + i;
    x[i] = 0.0f;
    if (e < n && f < F) {
      const float* p;
      if (cinert && f >= 80 && f < 448) {
        const int c = f - 80;
        p = c < 230 ? cinert + (t * (10 * KBS_NBODY) + 10 + c) * ld : cvel + (t * (6 * KBS_NBODY) + 6 + (c - 230)) * ld;
      } else {
        p = soa + (t * F + f) * ld;
      }
      x[i] = __ldcs(p + e);
    }
  }
  sb_flag_range(status, sb_out_of_range<KIND, 8>(x));
  const float x0[4] = {x[0], x[1], x[2], x[3]}, x1[4] = {x[4], x[5], x[6], x[7]};
  sb_store_split8<kPanelRows, KIND>(sb, row, kc * 8, Kp / kbs_block_k(KIND), sb_split4<KIND>(x0), sb_split4<KIND>(x1), false);
}

// ---- operands of the weight-gradient GEMMs (C = A^T B over K = all stored rows) ---------------------------------------------
// fp32 row-major src [rows][ld], columns [col0, col0 + ncols)  ->  TRANSPOSED split-blocked operand: operand "row" = source
// column j (128 per panel / tile), K = source row.  One thread = one 16-byte chunk per plane: E consecutive source rows of
// one column (lanes = consecutive columns: coalesced reads of a row, 512 contiguous bytes per store instruction).
// Source rows >= rows (K padding) and columns >= ncols (panel padding) are zero; column `ones_col` (>= 0) is the constant 1
// (its product with A^T is A's column sum).  WB: B-operand block layout [chunk][hi|lo][row][16 B], else [hi|lo][chunk][row][16 B].
template <int KIND, bool WB>
__global__ void __launch_bounds__(256)
pack_tn_kernel(const float* __restrict__ src, int64_t ld, int col0, int ncols, int ncols_pad, int64_t rows, int kb_total,
               char* __restrict__ dst, float scale, int ones_col, unsigned int* __restrict__ status, int64_t n_step, int64_t np_step) {
  constexpr int E = kbs_chunk_elems(KIND);
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  const int64_t chunks = int64_t(kb_total) * 4;
  if (idx >= chunks * ncols_pad) return;
  const int j = int(idx % ncols_pad);
  const int64_t kc = idx / ncols_pad;
  const int64_t r0 = kc * E;
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = 0.0f;
  // np_step != 0: K' = t np_step + e addresses source row t n_step + e (e < n_step; the rest of a step's panel padding is
  // zero) -- the K indexing of the per-step operands the persistent kernels keep
  // (a chunk of E <= 8 consecutive K' never straddles a step: np_step is a multiple of 128)
  const int64_t t_c = np_step ? r0 / np_step : 0, e_c = np_step ? r0 - t_c * np_step : 0;
  auto src_row = [&](int64_t k) -> int64_t {
    if (np_step == 0) return k < rows ? k : -1;
    const int64_t e = e_c + (k - r0);
    return (e < n_step && t_c * n_step + e < rows) ? t_c * n_step + e : -1;
  };
  if (j < ncols) {
#pragma unroll
    for (int i = 0; i < E; ++i) {
      const int64_t sr = src_row(r0 + i);
      if (sr >= 0) x[i] = __ldcs(src + sr * ld + col0 + j) * scale;
    }
  } else if (j == ones_col) {
#pragma unroll
    for (int i = 0; i < E; ++i)
      if (src_row(r0 + i) >= 0) x[i] = 1.0f;
  }
  sb_flag_range(status, sb_out_of_range<KIND, 8>(x));
  uint4 hi, lo;
  const float x0[4] = {x[0], x[1], x[2], x[3]};
  const KbsSplit4 s0 = sb_split4<KIND>(x0);
  if (KIND == KBS_KIND_F16) {
    const float x1[4] = {x[4], x[5], x[6], x[7]};
    const KbsSplit4 s1 = sb_split4<KIND>(x1);
    hi = make_uint4(s0.hi.x, s0.hi.y, s1.hi.x, s1.hi.y);
    lo = make_uint4(s0.lo.x, s0.lo.y, s1.lo.x, s1.lo.y);
  } else {
    hi = s0.hi; lo = s0.lo;
  }
  *reinterpret_cast<uint4*>(dst + sb_chunk_offset<kTileCols, KIND, WB>(j, int(r0), kb_total, 0)) = hi;
  *reinterpret_cast<uint4*>(dst + sb_chunk_offset<kTileCols, KIND, WB>(j, int(r0), kb_total, 1)) = lo;
}

// The same operand from what the persistent kernels keep: per-step split-blocked buffers [T] x step_bytes, each [np rows][K]
// K-major (kb_src K blocks per 128-row panel).  One thread = one core matrix of one plane: 8 rows x 8 consecutive K values
// (128 contiguous bytes) -> transposed in registers -> 8 operand rows (features) x one 16-byte chunk of 8 consecutive K' =
// t np + row (128 contiguous bytes again).  The planes are copied as they are (no re-split: the GEMM sees bit-identical
// operand values).  Rows >= n of a step (panel padding: never written by the producers) become zero.  FP16 kind only.
template <bool WB>
__global__ void __launch_bounds__(256)
sb_to_tn_kernel(const char* __restrict__ src, size_t step_bytes, int kb_src, int blk0, int nblk, int64_t n, int panels, int64_t T,
                char* __restrict__ dst, int kb_total, size_t col_bytes) {
  // one block = one plane of one K block of one panel of one step: 4 chunks x 128 rows x 16 B = 8 KB, contiguous in the source.
  // It is staged in shared memory with coalesced 16-byte loads; each thread then gathers the 8 rows of one (chunk, 8-row
  // group, K value) -- the transposed 16-byte chunk -- and stores it: 8 consecutive threads write 128 contiguous bytes.
  // (The first version moved a whole core matrix per thread through registers: 128-byte strides between the lanes of every
  // load and store, 1.1 TB/s at 8 192 trajectories; this one is bound by HBM.)
  __shared__ uint4 tile[4 * kPanelRows];
  int64_t q = blockIdx.x;
  const int plane = int(q & 1); q >>= 1;
  const int b = int(q % nblk); q /= nblk;
  const int pnl = int(q % panels);
  const int64_t t = q / panels;
  const char* sp = src + size_t(t) * step_bytes + (((size_t(pnl) * kb_src + size_t(blk0 + b)) * 2 + plane) * 4) * kPanelRows * 16;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int o = threadIdx.x + 256 * k;                         // [chunk][row]
    const int row = o & (kPanelRows - 1);
    uint4 v = __ldcs(reinterpret_cast<const uint4*>(sp) + o);
    if (int64_t(pnl) * kPanelRows + row >= n) v = make_uint4(0u, 0u, 0u, 0u);
    tile[o] = v;
  }
  __syncthreads();
  const unsigned short* th = reinterpret_cast<const unsigned short*>(tile);
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int o = threadIdx.x + 256 * k;
    const int i = o & 7, r8 = (o >> 3) & 15, c = o >> 7;
    const unsigned short* hp = th + (size_t(c) * kPanelRows + size_t(r8) * 8) * 8 + i;     // row rr at + rr * 8 halves
    uint4 out;
    out.x = uint32_t(hp[0]) | (uint32_t(hp[8]) << 16);
    out.y = uint32_t(hp[16]) | (uint32_t(hp[24]) << 16);
    out.z = uint32_t(hp[32]) | (uint32_t(hp[40]) << 16);
    out.w = uint32_t(hp[48]) | (uint32_t(hp[56]) << 16);
    const int64_t kp = (t * panels + pnl) * kPanelRows + r8 * 8;          // K' of the chunk's first row
    const int64_t kbq = kp / 32;
    const int cq = int((kp / 8) & 3);
    const int j = b * 32 + c * 8 + i;                                       // operand row
    char* dp = dst + size_t(j / kTileCols) * col_bytes;
    const int rowj = j % kTileCols;
    const size_t off = WB ? (((size_t(kbq) * 4 + cq) * 2 + plane) * kTileCols + rowj) * 16
                          : (((size_t(kbq) * 2 + plane) * 4 + cq) * kTileCols + rowj) * 16;
    *reinterpret_cast<uint4*>(dp + off) = out;
  }
}

// ... and from env-major SoA observations [T][F][ld] (K' = t np + env; envs >= n zero; column F = ones when `ones`): the B
// operand of the input-projection weight gradient.  Lanes run along the envs (coalesced reads).  FP16 kind only.
__global__ void __launch_bounds__(256)
soa_to_tn_kernel(const float* __restrict__ soa, int F, int64_t ld, int64_t n, int64_t np, int64_t T, int ncols_pad, int ones,
                 char* __restrict__ dst, int kb_total, size_t col_bytes, unsigned int* __restrict__ status) {
  // block = 32 features x 64 envs of one step, through shared memory: loads run along the envs (256 contiguous bytes per
  // feature row), stores along the features (512 contiguous bytes per warp) -- the first version stored along the envs:
  // 16-byte pieces 4 KB apart, 26 ms for the critic's observations at 8 192 trajectories.
  __shared__ float tile[32][65];
  const int64_t e0 = int64_t(blockIdx.x) * 64;
  const int f0 = blockIdx.y * 32;
  const int64_t t = blockIdx.z;
  for (int o = threadIdx.x; o < 32 * 64; o += 256) {
    const int f = f0 + (o >> 6);
    const int64_t e = e0 + (o & 63);
    float v = 0.0f;
    if (e < n) {
      if (f < F) v = __ldcs(soa + (t * F + f) * ld + e);
      else if (ones && f == F) v = 1.0f;
    }
    tile[o >> 6][o & 63] = v;
  }
  __syncthreads();
  const int jl = threadIdx.x & 31, kc = threadIdx.x >> 5;      // feature (lane), 8-env chunk of the block
  const int j = f0 + jl;
  if (j >= ncols_pad) return;
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = tile[jl][kc * 8 + i];
  sb_flag_range(status, sb_out_of_range<KBS_KIND_F16, 8>(x));
  const float x0[4] = {x[0], x[1], x[2], x[3]}, x1[4] = {x[4], x[5], x[6], x[7]};
  const KbsSplit4 s0 = sb_split4<KBS_KIND_F16>(x0), s1 = sb_split4<KBS_KIND_F16>(x1);
  const int64_t kp = t * np + e0 + kc * 8;
  if (e0 + kc * 8 >= np) return;
  char* dp = dst + size_t(j / kTileCols) * col_bytes;
  *reinterpret_cast<uint4*>(dp + sb_chunk_offset<kTileCols, KBS_KIND_F16, true>(j % kTileCols, int(kp), kb_total, 0)) =
      make_uint4(s0.hi.x, s0.hi.y, s1.hi.x, s1.hi.y);
  *reinterpret_cast<uint4*>(dp + sb_chunk_offset<kTileCols, KBS_KIND_F16, true>(j % kTileCols, int(kp), kb_total, 1)) =
      make_uint4(s0.lo.x, s0.lo.y, s1.lo.x, s1.lo.y);
}

// one B block whose column 0 is the constant 1 (hi plane) and everything else 0: the "ones tile" of the TN GEMMs
template <int KIND>
__global__ void __launch_bounds__(256) ones_block_kernel(char* __restrict__ blk) {
  const int idx = blockIdx.x * 256 + threadIdx.x;                 // one 16-byte chunk each: 2 * 4 * 128 chunks
  if (idx >= 2 * 4 * kTileCols) return;
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  // WB block layout [chunk][hi|lo][row][16 B]: row 0 of the hi plane of every chunk = ones
  const int row = idx % kTileCols, part = (idx / kTileCols) & 1;
  if (row == 0 && part == 0) {
    if (KIND == KBS_KIND_F16) { const uint32_t o = 0x3C003C00u; v = make_uint4(o, o, o, o); }
    else { const uint32_t o = __float_as_uint(1.0f); v = make_uint4(o, o, o, o); }
  }
  *reinterpret_cast<uint4*>(blk + size_t(idx) * 16) = v;
}

// dst[r][c] = sum_s partial[s][r][col0 + c]   (s in order: deterministic)
__global__ void __launch_bounds__(256)
tn_reduce_kernel(const float* __restrict__ partial, int ksplit, size_t split_stride, int ldc, int col0, int nrows, int ncols,
                 float* __restrict__ dst, int ld_dst) {
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= int64_t(nrows) * ncols) return;
  const int r = int(idx / ncols), c = int(idx % ncols);
  const float* p = partial + size_t(r) * ldc + col0 + c;
  float a = 0.0f;
  for (int sidx = 0; sidx < ksplit; ++sidx) a += p[size_t(sidx) * split_stride];
  dst[size_t(r) * ld_dst + c] = a;
}

// the same for up to three column ranges of the slabs at once (w_ih | w_hh | bias of a layer: one pass instead of three launches)
struct TnSegs { int col0[3], ncols[3], ld_dst[3]; float* dst[3]; int nseg, total_cols; };
__global__ void __launch_bounds__(256)
tn_reduce_multi_kernel(const float* __restrict__ partial, int ksplit, size_t split_stride, int ldc, int nrows, TnSegs sg) {
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= int64_t(nrows) * sg.total_cols) return;
  const int r = int(idx / sg.total_cols);
  int c = int(idx % sg.total_cols), k = 0;
  while (k + 1 < sg.nseg && c >= sg.ncols[k]) { c -= sg.ncols[k]; ++k; }
  const float* p = partial + size_t(r) * ldc + sg.col0[k] + c;
  float a = 0.0f;
  for (int sidx = 0; sidx < ksplit; ++sidx) a += p[size_t(sidx) * split_stride];
  sg.dst[k][size_t(r) * sg.ld_dst[k] + c] = a;
}

inline int64_t pad_rows(int64_t n) { return (n + kPanelRows - 1) / kPanelRows * kPanelRows; }
inline int round_up_i(int x, int m) { return (x + m - 1) / m * m; }

// persistent launch: one CTA per SM (or per item if there are fewer items)
template <int KIND>
cudaError_t launch_layer_k(const LayerArgs2& a2, int num_sms, cudaStream_t st) {
  const int items = net_items(a2.net[0]) + net_items(a2.net[1]);
  const int grid = items < num_sms ? items : num_sms;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreadsTC);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // see griddepcontrol.* in the kernel
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, lstm_layer_tc_kernel<KIND>, a2);
}
inline cudaError_t launch_layer(const kbs_handle* h, int kind, const LayerArgs2& a2, cudaStream_t st) {
  return kind == KBS_KIND_TF32 ? launch_layer_k<KBS_KIND_TF32>(a2, h->num_sms, st) : launch_layer_k<KBS_KIND_F16>(a2, h->num_sms, st);
}

}  // namespace

// ---- host side --------------------------------------------------------------------------------------------------------
static inline int tc_kind(const kbs_handle* h) { return h->p.gemm_path == KBS_GEMM_TC_2XF16 ? KBS_KIND_F16 : KBS_KIND_TF32; }
static inline int proj_kp(const kbs_handle* h, int net) {       // input width padded to whole K blocks
  return round_up_i(h->net[net].num_in, kbs_block_k(tc_kind(h)));
}
// tc_image of one net (bytes): per layer [w_sb (4H x 2H SB) | bias_t (4H floats)], then proj [w_sb (256 x Kp SB) | bias (256)]
static size_t layer_image_bytes(const kbs_handle* h) {
  const int H = h->p.hidden_size;
  return kbs_sb_bytes_kind(tc_kind(h), 4 * H, 2 * H) + size_t(4 * H) * 4;
}
static inline int proj_cols(const kbs_handle* h) { return round_up_i(h->p.hidden_size, kTileCols); }
static size_t proj_image_bytes(const kbs_handle* h, int net) {
  return kbs_sb_bytes_kind(tc_kind(h), proj_cols(h), proj_kp(h, net)) + size_t(proj_cols(h)) * 4;
}
static inline char* layer_w(const kbs_handle* h, int net, int l) {
  return reinterpret_cast<char*>(h->net[net].tc_image) + layer_image_bytes(h) * l;
}
static inline float* layer_bias(const kbs_handle* h, int net, int l) {
  const int H = h->p.hidden_size;
  return reinterpret_cast<float*>(layer_w(h, net, l) + kbs_sb_bytes_kind(tc_kind(h), 4 * H, 2 * H));
}
static inline char* proj_w(const kbs_handle* h, int net) { return layer_w(h, net, h->p.depth); }
static inline float* proj_bias(const kbs_handle* h, int net) {
  return reinterpret_cast<float*>(proj_w(h, net) + kbs_sb_bytes_kind(tc_kind(h), proj_cols(h), proj_kp(h, net)));
}
// persistent rollout kernel: the same LSTM weights in 256-column tiles (image P), then the output head: W_out zero-padded
// to one 256-column tile [256][H] SB + bias [256]
static inline char* layer_w_p(const kbs_handle* h, int net, int l) {
  return proj_w(h, net) + proj_image_bytes(h, net) + layer_image_bytes(h) * l;
}
static inline float* layer_bias_p(const kbs_handle* h, int net, int l) {
  const int H = h->p.hidden_size;
  return reinterpret_cast<float*>(layer_w_p(h, net, l) + kbs_sb_bytes_kind(tc_kind(h), 4 * H, 2 * H));
}
static size_t head_image_bytes(const kbs_handle* h) {
  return kbs_sb_bytes_kind(tc_kind(h), kTileColsP, h->p.hidden_size) + size_t(kTileColsP) * 4;
}
static inline char* head_w(const kbs_handle* h, int net) { return layer_w_p(h, net, h->p.depth); }
static inline float* head_bias(const kbs_handle* h, int net) {
  return reinterpret_cast<float*>(head_w(h, net) + kbs_sb_bytes_kind(tc_kind(h), kTileColsP, h->p.hidden_size));
}
// Layer 0 with the input projection folded in (persistent kernel, see fuse_input_weights_kernel): the observation operand
// is padded to a multiple of 4 K blocks (the kernel's stage ring); worth it when that is narrower than H (actor: 65 ->
// 128 < 256; critic: 475 -> 512 > 256, keeps its projection launch).  Image F: [wf fp32 | bf | w_sb | bias_t].
static inline int fused_kp(const kbs_handle* h, int net) { return round_up_i(h->net[net].num_in, 4 * kbs_block_k(tc_kind(h))); }
static inline bool fused_shape(const kbs_handle* h, int net) { return fused_kp(h, net) < h->p.hidden_size; }
static size_t fused_image_bytes(const kbs_handle* h, int net) {
  if (!fused_shape(h, net)) return 0;
  const int H = h->p.hidden_size, Kf = fused_kp(h, net);
  return size_t(4 * H) * Kf * 4 + size_t(4 * H) * 4 + kbs_sb_bytes_kind(tc_kind(h), 4 * H, Kf + H) + size_t(4 * H) * 4;
}
static inline float* fused_wf(const kbs_handle* h, int net) {
  return reinterpret_cast<float*>(head_w(h, net) + head_image_bytes(h));
}
static inline float* fused_bf(const kbs_handle* h, int net) { return fused_wf(h, net) + size_t(4 * h->p.hidden_size) * fused_kp(h, net); }
static inline char* fused_w(const kbs_handle* h, int net) { return reinterpret_cast<char*>(fused_bf(h, net) + 4 * h->p.hidden_size); }
static inline float* fused_bias(const kbs_handle* h, int net) {
  return reinterpret_cast<float*>(fused_w(h, net) + kbs_sb_bytes_kind(tc_kind(h), 4 * h->p.hidden_size, fused_kp(h, net) + h->p.hidden_size));
}
// Images Q0 / Q1: W_in as ONE 256-column tile for input_proj_fused_kernel (H == 256 only), in the kernel's K-block order.
//   layout 0 (plain): the net's SoA observation rows 0 .. Kp-1 in order;
//   layout 1 (critic with the privileged dump read from the recorded state): obs rows 0..79 | cinert rows 10..239 |
//            cvel rows 6..143 | obs rows 448..474, each region padded to whole K blocks (masked rows, zero weights).
// Per image: [w_sb (256 x Kq SB, WB layout) | bias (256)].
struct FLayout {
  int kb = 0;
  signed char src[kFMaxBlocks];
  short row0[kFMaxBlocks], nvalid[kFMaxBlocks];
  int fbase[kFMaxBlocks];      // eqx input column of the block's first row
};
static inline bool projq_shape(const kbs_handle* h) { return h->p.hidden_size == 256; }
static FLayout projq_layout(const kbs_handle* h, int net, int which) {
  FLayout L;
  const int kf = kbs_block_k(tc_kind(h)), F = h->net[net].num_in;
  auto region = [&](int src, int start, int count, int f_base) {
    for (int i = 0; i * kf < count; ++i) {
      const int b = L.kb++;
      L.src[b] = (signed char)src; L.row0[b] = short(start + i * kf);
      L.nvalid[b] = short(count - i * kf < kf ? count - i * kf : kf);
      L.fbase[b] = f_base + i * kf;
    }
  };
  if (which == 1) { region(0, 0, 80, 0); region(1, 10, 230, 80); region(2, 6, 138, 310); region(0, 448, F - 448, 448); }
  else region(0, 0, F, 0);
  return L;
}
static inline bool projq_has_dump_layout(const kbs_handle* h, int net) { return h->net[net].num_in == KBS_CRITIC_OBS; }
static inline int projq_kq(const kbs_handle* h, int net, int which) {
  const int kf = kbs_block_k(tc_kind(h)), F = h->net[net].num_in;
  auto up = [&](int c) { return (c + kf - 1) / kf * kf; };
  return which == 1 ? up(80) + up(230) + up(138) + up(F - 448) : up(F);
}
static size_t projq_image_bytes1(const kbs_handle* h, int net, int which) {
  const int Kq = projq_kq(h, net, which);
  return kbs_sb_bytes_kind(tc_kind(h), 256, Kq) + size_t(256) * 4;
}
static size_t projq_image_bytes(const kbs_handle* h, int net) {
  if (!projq_shape(h)) return 0;
  return projq_image_bytes1(h, net, 0) + (projq_has_dump_layout(h, net) ? projq_image_bytes1(h, net, 1) : 0);
}
static inline char* projq_w(const kbs_handle* h, int net, int which) {
  char* base = reinterpret_cast<char*>(fused_wf(h, net)) + fused_image_bytes(h, net);
  return which ? base + projq_image_bytes1(h, net, 0) : base;
}
static inline float* projq_bias(const kbs_handle* h, int net, int which) {
  return reinterpret_cast<float*>(projq_w(h, net, which) + kbs_sb_bytes_kind(tc_kind(h), 256, projq_kq(h, net, which)));
}

typedef CUresult (*KbsTensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                         const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                         CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static KbsTensorMapEncodeFn tensor_map_encode_fn() {
  static KbsTensorMapEncodeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<KbsTensorMapEncodeFn>(p);
  }
  return fn;
}
// 2-D fp32 tensor {ld envs (inner), rows}, box {128 envs, box_rows}; out-of-range elements read as zero
static bool encode_rows_map(CUtensorMap* m, const float* base, int64_t ld, int64_t rows, int box_rows) {
  KbsTensorMapEncodeFn fn = tensor_map_encode_fn();
  if (!fn || !base) return false;
  const cuuint64_t gdim[2] = {cuuint64_t(ld), cuuint64_t(rows)};
  const cuuint64_t gstride[1] = {cuuint64_t(ld) * 4};
  const cuuint32_t box[2] = {cuuint32_t(kPanelRows), cuuint32_t(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
static inline bool persist_shape_ok(const kbs_handle* h) {
  const int H = h->p.hidden_size;
  return H % kUnitsPerTileP == 0 && h->p.depth <= kPMaxDepth && H <= kMaxBias / 4 &&
         (H / kbs_block_k(tc_kind(h))) % 4 == 0;
}

int kbs_tc_pack(kbs_handle* h, int net, cudaStream_t st) {
  KbsNet& N = h->net[net];
  const int H = h->p.hidden_size, kind = tc_kind(h);
  if (H % kUnitsPerTile) return KBS_E_SHAPE;
  if (!h->tc_attr_set) {      // per device (context), so per handle: a handle on another GPU of the same process needs its own opt-in
    KBS_CUDA_TRY(cudaFuncSetAttribute(lstm_layer_tc_kernel<KBS_KIND_TF32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    KBS_CUDA_TRY(cudaFuncSetAttribute(lstm_layer_tc_kernel<KBS_KIND_F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    KBS_CUDA_TRY((cudaFuncSetAttribute(rollout_persist_kernel<KBS_KIND_TF32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmemBytes)));
    KBS_CUDA_TRY((cudaFuncSetAttribute(rollout_persist_kernel<KBS_KIND_F16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmemBytes)));
    KBS_CUDA_TRY((cudaFuncSetAttribute(rollout_persist_kernel<KBS_KIND_F16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmemBytes)));
    KBS_CUDA_TRY(cudaFuncSetAttribute(input_proj_fused_kernel<KBS_KIND_TF32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFSmemBytes));
    KBS_CUDA_TRY(cudaFuncSetAttribute(input_proj_fused_kernel<KBS_KIND_F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFSmemBytes));
    h->tc_attr_set = true;
  }
  const size_t bytes = 2 * layer_image_bytes(h) * h->p.depth + proj_image_bytes(h, net) + head_image_bytes(h) +
                       fused_image_bytes(h, net) + projq_image_bytes(h, net);
  N.tc_image_floats = (bytes + 3) / 4;
  if (!N.tc_image) KBS_CUDA_TRY(cudaMalloc(&N.tc_image, bytes));      // fixed size per handle: re-packs keep the pointer
  for (int l = 0; l < h->p.depth; ++l) {
    const int64_t total = int64_t(4 * H) * (2 * H / 4);
    const unsigned gb = unsigned((total + 255) / 256);
    if (kind == KBS_KIND_TF32)
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_lstm_weights_kernel<KBS_KIND_TF32, kTileCols><<<gb, 256, 0, st>>>(
                                        N.w_ih[l], N.w_hh[l], N.b[l], layer_w(h, net, l), layer_bias(h, net, l), H, H, H)));
    else
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_lstm_weights_kernel<KBS_KIND_F16, kTileCols><<<gb, 256, 0, st>>>(
                                        N.w_ih[l], N.w_hh[l], N.b[l], layer_w(h, net, l), layer_bias(h, net, l), H, H, H)));
    if (kind == KBS_KIND_F16 && H % 32 == 0) {     // 128-column tiles in 8-unit groups: lstm_fwd_save_kernel (PPO update)
      if (!N.tc_fwd8_image) KBS_CUDA_TRY(cudaMalloc(&N.tc_fwd8_image, layer_image_bytes(h) * h->p.depth));
      char* w8 = reinterpret_cast<char*>(N.tc_fwd8_image) + layer_image_bytes(h) * l;
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_lstm_weights_kernel<KBS_KIND_F16, kTileCols, kSGU><<<gb, 256, 0, st>>>(
                                        N.w_ih[l], N.w_hh[l], N.b[l], w8,
                                        reinterpret_cast<float*>(w8 + kbs_sb_bytes_kind(kind, 4 * H, 2 * H)), H, H, H)));
    }
    if (!persist_shape_ok(h)) continue;
    if (kind == KBS_KIND_TF32)
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_lstm_weights_kernel<KBS_KIND_TF32, kTileColsP><<<gb, 256, 0, st>>>(
                                        N.w_ih[l], N.w_hh[l], N.b[l], layer_w_p(h, net, l), layer_bias_p(h, net, l), H, H, H)));
    else
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_lstm_weights_kernel<KBS_KIND_F16, kTileColsP><<<gb, 256, 0, st>>>(
                                        N.w_ih[l], N.w_hh[l], N.b[l], layer_w_p(h, net, l), layer_bias_p(h, net, l), H, H, H)));
  }
  {
    const int Kp = proj_kp(h, net);
    const int cols = proj_cols(h);
    const int64_t total = int64_t(cols) * (Kp / 4);
    const unsigned gb = unsigned((total + 255) / 256);
    if (kind == KBS_KIND_TF32)
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_proj_weights_kernel<KBS_KIND_TF32><<<gb, 256, 0, st>>>(
                                        N.w_in, N.kin_pad, N.b_in, proj_w(h, net), proj_bias(h, net), H, Kp, cols)));
    else
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_proj_weights_kernel<KBS_KIND_F16><<<gb, 256, 0, st>>>(
                                        N.w_in, N.kin_pad, N.b_in, proj_w(h, net), proj_bias(h, net), H, Kp, cols)));
  }
  if (projq_shape(h)) {   // W_in as one 256-column tile in input_proj_fused_kernel's K order (plain and, for the critic, dump layout)
    for (int which = 0; which < (projq_has_dump_layout(h, net) ? 2 : 1); ++which) {
      const FLayout L = projq_layout(h, net, which);
      const int Kq = projq_kq(h, net, which);
      FPackLayout P{};
      P.kb = L.kb;
      for (int b = 0; b < L.kb; ++b) { P.fbase[b] = L.fbase[b]; P.nvalid[b] = L.nvalid[b]; }
      const int64_t total = int64_t(256) * (Kq / 4);
      const unsigned gb = unsigned((total + 255) / 256);
      if (kind == KBS_KIND_TF32)
        KBS_LAUNCH(h, KBS_K_PACK, st, (pack_proj_weights_kmap_kernel<KBS_KIND_TF32><<<gb, 256, 0, st>>>(
                                          N.w_in, N.kin_pad, N.b_in, P, projq_w(h, net, which), projq_bias(h, net, which), H, Kq)));
      else
        KBS_LAUNCH(h, KBS_K_PACK, st, (pack_proj_weights_kmap_kernel<KBS_KIND_F16><<<gb, 256, 0, st>>>(
                                          N.w_in, N.kin_pad, N.b_in, P, projq_w(h, net, which), projq_bias(h, net, which), H, Kq)));
    }
  }
  if (persist_shape_ok(h) && fused_shape(h, net)) {   // layer 0 with the input projection folded in
    const int Kf = fused_kp(h, net);
    const int64_t tot_f = int64_t(4 * H) * (Kf + 1);
    KBS_LAUNCH(h, KBS_K_PACK, st, (fuse_input_weights_kernel<<<unsigned((tot_f + 255) / 256), 256, 0, st>>>(
                                      N.w_ih[0], N.w_in, N.kin_pad, N.num_in, N.b_in, N.b[0], fused_wf(h, net), fused_bf(h, net), H, Kf)));
    const int64_t total = int64_t(4 * H) * ((Kf + H) / 4);
    const unsigned gb = unsigned((total + 255) / 256);
    if (kind == KBS_KIND_TF32)
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_lstm_weights_kernel<KBS_KIND_TF32, kTileColsP><<<gb, 256, 0, st>>>(
                                        fused_wf(h, net), N.w_hh[0], fused_bf(h, net), fused_w(h, net), fused_bias(h, net), H, Kf, Kf)));
    else
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_lstm_weights_kernel<KBS_KIND_F16, kTileColsP><<<gb, 256, 0, st>>>(
                                        fused_wf(h, net), N.w_hh[0], fused_bf(h, net), fused_w(h, net), fused_bias(h, net), H, Kf, Kf)));
  }
  if (persist_shape_ok(h)) {   // output head tile (persistent rollout kernel)
    const int64_t total = int64_t(kTileColsP) * (H / 4);
    const unsigned gb = unsigned((total + 255) / 256);
    if (kind == KBS_KIND_TF32)
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_head_weights_kernel<KBS_KIND_TF32><<<gb, 256, 0, st>>>(
                                        N.w_out, N.b_out, head_w(h, net), head_bias(h, net), H, N.num_out)));
    else
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_head_weights_kernel<KBS_KIND_F16><<<gb, 256, 0, st>>>(
                                        N.w_out, N.b_out, head_w(h, net), head_bias(h, net), H, N.num_out)));
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

static int pack_rows(kbs_handle* h, const float* src, int64_t ld, char* sb, int64_t n, int64_t np, int K, cudaStream_t st) {
  const int64_t chunks = np * (K / 4);
  const unsigned gb = unsigned((chunks + 255) / 256);
  if (tc_kind(h) == KBS_KIND_TF32)
    KBS_LAUNCH(h, KBS_K_PACK, st, (pack_rows_sb_kernel<KBS_KIND_TF32><<<gb, 256, 0, st>>>(src, ld, sb, n, np, K)));
  else
    KBS_LAUNCH(h, KBS_K_PACK, st, (pack_rows_sb_kernel<KBS_KIND_F16><<<gb, 256, 0, st>>>(src, ld, sb, n, np, K)));
  return KBS_OK;
}

// bytes of one [n][H] SB activation buffer
static size_t act_sb_bytes(const kbs_handle* h, int64_t n) { return kbs_sb_bytes_kind(tc_kind(h), pad_rows(n), h->p.hidden_size); }

KbsTcStackWs kbs_tc_stack_ws(KbsScratch& s, const kbs_handle* h, int64_t n) {
  const size_t sbb = act_sb_bytes(h, n), depth = size_t(h->p.depth);
  return {s.take<char>(2 * sbb), s.take<char>(2 * depth * sbb), s.take<float>(2 * depth * size_t(pad_rows(n)) * h->p.hidden_size)};
}

static int fb_convert(kbs_handle* h, float* rm, float* fb, int64_t n, int64_t np, int H, int to_fb, cudaStream_t st) {
  const int64_t tot = np * (H / 4);
  KBS_LAUNCH(h, KBS_K_PACK, st, (fb_convert_kernel<<<unsigned((tot + 255) / 256), 256, 0, st>>>(rm, fb, n, np, H, to_fb)));
  return KBS_OK;
}

static int carry_convert(kbs_handle* h, const CarryJobs& J, int jobs, int64_t n, int64_t np, int H, cudaStream_t st) {
  const int kt = (H / 8 + 31) / 32;
  const dim3 grid(unsigned((np / 32) * kt), unsigned(jobs));
  if (tc_kind(h) == KBS_KIND_TF32)
    KBS_LAUNCH(h, KBS_K_PACK, st, (carry_convert_kernel<KBS_KIND_TF32><<<grid, 256, 0, st>>>(J, n, np, H)));
  else
    KBS_LAUNCH(h, KBS_K_PACK, st, (carry_convert_kernel<KBS_KIND_F16><<<grid, 256, 0, st>>>(J, n, np, H)));
  return KBS_OK;
}

static int epi_debug() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("KBS_TC_EPI_DEBUG"); v = e ? atoi(e) : 0; }
  return v;
}
static void fill_lstm_args(const kbs_handle* h, int net, int l, LayerArgs& a) {
  a.dbg = epi_debug();
  const int H = h->p.hidden_size, kb = H / kbs_block_k(tc_kind(h));
  a.w_sb = layer_w(h, net, l);
  a.bias_t = layer_bias(h, net, l);
  a.H = H; a.kb_x = kb; a.kb_h = kb; a.mode = MODE_LSTM;
  a.tiles = H / kUnitsPerTile;
}

// Runs depth LSTM layers on the tensor cores.  x_rm: [n][H] row-major layer-0 input (input_proj output);
// carry: ABI layout [depth][2][n][H]; out_h_rm: [n][H] row-major un-reset top-layer output.
int kbs_tc_lstm_stack(kbs_handle* h, int net, const float* x_rm, float* carry, const uint8_t* done, float* out_h_rm,
                      const KbsTcStackWs& ws, int64_t n, bool carry_sb_valid, cudaStream_t st) {
  const KbsNet& N = h->net[net];
  if (!N.packed || !N.tc_image) return KBS_E_STATE;
  const int H = h->p.hidden_size, depth = h->p.depth;
  const int64_t np = pad_rows(n);
  const size_t sbb = act_sb_bytes(h, n);
  char* x_sb[2] = {ws.x_sb, ws.x_sb + sbb};
  char* h_sb = ws.h_sb;         // [depth][2 (in, out)]: the column-tile CTAs of a panel all read h_{t-1} while their
                                // epilogues write h_t, so in and out must be distinct buffers
  float* fb = ws.fb;            // [depth][c, h] x np*H: state in the kernel's FB layout
  const size_t fbf = size_t(np) * H;
  pack_rows(h, x_rm, H, x_sb[0], n, np, H, st);
  for (int l = 0; l < depth; ++l)
    fb_convert(h, carry + (size_t(l) * 2 + 1) * size_t(n) * H, fb + fbf * (2 * l), n, np, H, 1, st);
  if (!carry_sb_valid) {
    for (int l = 0; l < depth; ++l)
      pack_rows(h, carry + (size_t(l) * 2 + 0) * size_t(n) * H, H, h_sb + sbb * (2 * l), n, np, H, st);
  }
  for (int l = 0; l < depth; ++l) {
    LayerArgs2 a2{};
    LayerArgs& a = a2.net[0];
    fill_lstm_args(h, net, l, a);
    a.x_sb = x_sb[l & 1];
    a.h_sb_in = h_sb + sbb * (2 * l);
    a.h_sb_out = h_sb + sbb * (2 * l + 1);
    a.c = fb + fbf * (2 * l);
    a.h_carry = fb + fbf * (2 * l + 1);
    a.x_next_sb = (l + 1 < depth) ? x_sb[(l + 1) & 1] : nullptr;
    a.h_next_rm = (l + 1 < depth) ? nullptr : out_h_rm;
    a.done = done;
    a.n = n;
    a.panels = int(np / kPanelRows);
    KBS_LAUNCH(h, KBS_K_LSTM_TC, st, (launch_layer(h, tc_kind(h), a2, st)));
  }
  for (int l = 0; l < depth; ++l) {   // FB state -> ABI carry
    fb_convert(h, carry + (size_t(l) * 2 + 1) * size_t(n) * H, fb + fbf * (2 * l), n, np, H, 0, st);
    fb_convert(h, carry + (size_t(l) * 2 + 0) * size_t(n) * H, fb + fbf * (2 * l + 1), n, np, H, 0, st);
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// Debug / test entry: raw pre-activation gates (eqx order i,f,g,o; bias added) of one layer from row-major inputs.
int kbs_tc_debug_gates(kbs_handle* h, int net, int layer, const float* x_rm, const float* h_rm, float* gates_out,
                       float* ws, int64_t n, cudaStream_t st) {
  const KbsNet& N = h->net[net];
  if (!N.packed || !N.tc_image) return KBS_E_STATE;
  const int H = h->p.hidden_size;
  const int64_t np = pad_rows(n);
  const size_t sbb = act_sb_bytes(h, n);
  char* wsb = reinterpret_cast<char*>(ws);
  pack_rows(h, x_rm, H, wsb, n, np, H, st);
  pack_rows(h, h_rm, H, wsb + sbb, n, np, H, st);
  LayerArgs2 a2{};
  LayerArgs& a = a2.net[0];
  fill_lstm_args(h, net, layer, a);
  a.x_sb = wsb;
  a.h_sb_in = wsb + sbb;
  a.raw = gates_out;
  a.mode = MODE_RAW;
  a.n = n;
  a.panels = int(np / kPanelRows);
  KBS_LAUNCH(h, KBS_K_LSTM_TC, st, (launch_layer(h, tc_kind(h), a2, st)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// ---- tensor-core GEMMs of the PPO update (kbs_ppo_update.cu): split-precision, fp32-accurate ---------------------------
// gates_out [n][4H] (eqx order, bias added) = [x | h] . Wcat^T from SB operands the caller already holds
int kbs_tc_gates_fwd(kbs_handle* h, int net, int layer, const void* x_sb, const void* h_sb, float* gates_out, int64_t n,
                     cudaStream_t st) {
  const KbsNet& N = h->net[net];
  if (!N.packed || !N.tc_image) return KBS_E_STATE;
  LayerArgs2 a2{};
  LayerArgs& a = a2.net[0];
  fill_lstm_args(h, net, layer, a);
  a.x_sb = reinterpret_cast<const char*>(x_sb);
  a.h_sb_in = reinterpret_cast<const char*>(h_sb);
  a.raw = gates_out;
  a.mode = MODE_RAW;
  a.n = n;
  a.panels = int(pad_rows(n) / kPanelRows);
  KBS_LAUNCH(h, KBS_K_LSTM_TC, st, (launch_layer(h, tc_kind(h), a2, st)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// backward weights of one layer: Wb [2H][4H], Wb[c][k] = W_ih[k][c] (c < H) | W_hh[k][c - H]: [dx | dh] = dG . Wb^T
template <int KIND, int TILE>
__global__ void __launch_bounds__(256)
pack_bwd_weights_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh, char* __restrict__ w_sb,
                        float* __restrict__ bias_t, int H) {
  const int kq = 4 * H / 4;
  const int64_t idx = int64_t(blockIdx.x) * 256 + threadIdx.x;
  if (idx >= int64_t(2 * H) * kq) return;
  const int col = int(idx / kq), k = int(idx % kq) * 4;
  const float* w = col < H ? w_ih : w_hh;
  const int c = col < H ? col : col - H;
  const float x[4] = {w[size_t(k) * H + c], w[size_t(k + 1) * H + c], w[size_t(k + 2) * H + c], w[size_t(k + 3) * H + c]};
  sb_store4<TILE, KIND, true>(w_sb, col, k, 4 * H / kbs_block_k(KIND), x);
  if (k == 0) bias_t[col] = 0.0f;
}

static size_t bwd_layer_bytes(const kbs_handle* h) {
  const int H = h->p.hidden_size;
  return kbs_sb_bytes_kind(tc_kind(h), 2 * H, 4 * H) + size_t(2 * H) * 4;
}

// (re)builds the backward operand image of `net` from its current fp32 weights (call after every weight update)
int kbs_tc_pack_bwd(kbs_handle* h, int net, cudaStream_t st, int tile) {
  KbsNet& N = h->net[net];
  if (!N.packed) return KBS_E_STATE;
  const int H = h->p.hidden_size, kind = tc_kind(h);
  if ((2 * H) % kTileCols || (4 * H) % kbs_block_k(kind) || (tile != kTileCols && (tile != kBT || kind != KBS_KIND_F16))) return KBS_E_SHAPE;
  const size_t bytes = bwd_layer_bytes(h) * h->p.depth;
  float*& image = tile == kBT ? N.tc_bwd_image64 : N.tc_bwd_image;     // same bytes per layer for either tile width
  if (!image) KBS_CUDA_TRY(cudaMalloc(&image, bytes));
  for (int l = 0; l < h->p.depth; ++l) {
    char* w = reinterpret_cast<char*>(image) + bwd_layer_bytes(h) * l;
    float* bias = reinterpret_cast<float*>(w + kbs_sb_bytes_kind(kind, 2 * H, 4 * H));
    const int64_t total = int64_t(2 * H) * (4 * H / 4);
    const unsigned gb = unsigned((total + 255) / 256);
    if (tile == kBT)
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_bwd_weights_kernel<KBS_KIND_F16, kBT><<<gb, 256, 0, st>>>(N.w_ih[l], N.w_hh[l], w, bias, H)));
    else if (kind == KBS_KIND_TF32)
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_bwd_weights_kernel<KBS_KIND_TF32, kTileCols><<<gb, 256, 0, st>>>(N.w_ih[l], N.w_hh[l], w, bias, H)));
    else
      KBS_LAUNCH(h, KBS_K_PACK, st, (pack_bwd_weights_kernel<KBS_KIND_F16, kTileCols><<<gb, 256, 0, st>>>(N.w_ih[l], N.w_hh[l], w, bias, H)));
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// out [n][2H] row-major = out_scale * dG [n][4H] (SB) . [W_ih | W_hh]: columns 0..H-1 = gradient wrt the layer input,
// H..2H-1 wrt h_in.  Gradients are ~1 / (T n) small: the caller scales dG by a power of two before splitting it into FP16
// planes (whose range ends at 6e-5 / 6e-8) and passes the inverse here.
int kbs_tc_bwd_gemm(kbs_handle* h, int net, int layer, const void* dG_sb, float* out, int64_t n, float out_scale, cudaStream_t st) {
  const KbsNet& N = h->net[net];
  if (!N.packed || !N.tc_bwd_image) return KBS_E_STATE;
  const int H = h->p.hidden_size, kind = tc_kind(h);
  char* w = reinterpret_cast<char*>(N.tc_bwd_image) + bwd_layer_bytes(h) * layer;
  LayerArgs2 a2{};
  LayerArgs& a = a2.net[0];
  a.dbg = 0;
  a.x_sb = reinterpret_cast<const char*>(dG_sb);
  a.h_sb_in = a.x_sb;
  a.w_sb = w;
  a.bias_t = reinterpret_cast<const float*>(w + kbs_sb_bytes_kind(kind, 2 * H, 4 * H));
  a.raw = out; a.ldo = 2 * H; a.oscale = out_scale;
  a.mode = MODE_PLAIN;
  a.n = n;
  a.H = H; a.kb_x = 4 * H / kbs_block_k(kind); a.kb_h = 0;
  a.panels = int(pad_rows(n) / kPanelRows); a.tiles = 2 * H / kTileCols;
  KBS_LAUNCH(h, KBS_K_LSTM_TC, st, (launch_layer(h, kind, a2, st)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// ---- weight-gradient GEMMs: C = out_scale * A^T B over K = `rows` stored rows, on the tensor cores, split-K ----------------
KbsTnPlan kbs_tc_tn_plan(const kbs_handle* h, int64_t rows) {
  KbsTnPlan p{};
  const int bk = kbs_block_k(tc_kind(h));
  const int64_t kb_raw = (rows + bk - 1) / bk;
  // <= 3200 rows (FP16: 100 blocks) per accumulation run, at least 16 runs when there is enough work to split
  int64_t per = (kb_raw + 15) / 16;
  const int64_t cap = 3200 / bk;
  if (per > cap) per = cap;
  if (per < 1) per = 1;
  p.kb_split = int(per);
  p.ksplit = int((kb_raw + per - 1) / per);
  p.kb_total = p.kb_split * p.ksplit;
  p.col_bytes = size_t(p.kb_total) * kABlockBytes;          // bytes of one 128-column panel / tile of a transposed operand
  return p;
}

int kbs_tc_pack_tn(kbs_handle* h, const KbsTnPlan& plan, bool b_operand, const float* src, int64_t ld, int col0, int ncols,
                   int ncols_pad, int64_t rows, char* dst, float scale, int ones_col, cudaStream_t st, int64_t n_step,
                   int64_t np_step) {
  if (ncols_pad % kTileCols) return KBS_E_SHAPE;
  { const int rc0 = kbs_status_init(h); if (rc0) return rc0; }
  const int kind = tc_kind(h);
  // one launch per 128-column panel / tile: each has its own [kb_total] block run
  for (int c = 0; c < ncols_pad; c += kTileCols) {
    const int nc = ncols - c < kTileCols ? (ncols - c > 0 ? ncols - c : 0) : kTileCols;
    const int oc = (ones_col >= c && ones_col < c + kTileCols) ? ones_col - c : -1;
    const int64_t total = int64_t(plan.kb_total) * 4 * kTileCols;
    const unsigned gb = unsigned((total + 255) / 256);
    char* d = dst + size_t(c / kTileCols) * plan.col_bytes;
#define KBS_PACK_TN(K_, WB_) KBS_LAUNCH(h, KBS_K_PACK, st, (pack_tn_kernel<K_, WB_><<<gb, 256, 0, st>>>( \
        src, ld, col0 + c, nc, kTileCols, rows, plan.kb_total, d, scale, oc, h->persist_status, n_step, np_step)))
    if (kind == KBS_KIND_TF32) { if (b_operand) KBS_PACK_TN(KBS_KIND_TF32, true); else KBS_PACK_TN(KBS_KIND_TF32, false); }
    else { if (b_operand) KBS_PACK_TN(KBS_KIND_F16, true); else KBS_PACK_TN(KBS_KIND_F16, false); }
#undef KBS_PACK_TN
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// partial [ksplit][m_panels * 128][ldc] with ldc = (n_tiles + ones) * 128; zero_bias: >= ldc zero floats; ones_blk: the ones block
int kbs_tc_gemm_tn(kbs_handle* h, const KbsTnPlan& plan, const char* a_t, int m_panels, int m_valid, const char* b_t, int n_tiles,
                   const char* ones_blk, const float* zero_bias, float* partial, float out_scale, cudaStream_t st) {
  const int kind = tc_kind(h);
  const int tiles = n_tiles + (ones_blk ? 1 : 0);
  if (tiles * kTileCols > kMaxBias || m_panels < 1) return KBS_E_SHAPE;
  LayerArgs2 a2{};
  LayerArgs& a = a2.net[0];
  a.x_sb = a_t; a.h_sb_in = a_t;
  a.w_sb = b_t;
  a.bias_t = zero_bias;
  a.raw = partial; a.ldo = tiles * kTileCols; a.oscale = out_scale;
  a.mode = MODE_PLAIN;
  a.n = m_valid;
  a.H = 0; a.kb_x = plan.kb_split; a.kb_h = 0;
  a.panels = m_panels; a.tiles = tiles;
  a.ksplit = plan.ksplit; a.kb_stride = plan.kb_total;
  a.raw_split_stride = size_t(m_panels) * kPanelRows * size_t(a.ldo);
  a.ones_tile = ones_blk ? n_tiles : -1; a.ones_block = ones_blk;
  KBS_LAUNCH(h, KBS_K_GEMM_TN, st, (launch_layer(h, kind, a2, st)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_tc_ones_block(kbs_handle* h, char* blk, cudaStream_t st) {
  if (tc_kind(h) == KBS_KIND_TF32) KBS_LAUNCH(h, KBS_K_PACK, st, (ones_block_kernel<KBS_KIND_TF32><<<4, 256, 0, st>>>(blk)));
  else KBS_LAUNCH(h, KBS_K_PACK, st, (ones_block_kernel<KBS_KIND_F16><<<4, 256, 0, st>>>(blk)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_tc_sb_to_tn(kbs_handle* h, const KbsTnPlan& plan, bool b_operand, const char* src, size_t step_bytes, int kb_src, int blk0,
                    int nblk, int64_t n, int64_t T, char* dst, cudaStream_t st) {
  if (tc_kind(h) != KBS_KIND_F16 || nblk % 4) return KBS_E_STATE;
  const int panels = int(pad_rows(n) / kPanelRows);
  const int64_t kb_used = (T * panels * kPanelRows + 31) / 32;
  if (kb_used > plan.kb_total) return KBS_E_SHAPE;
  if (kb_used < plan.kb_total)                   // K padding behind the last stored row: zero in every panel / tile
    for (int c = 0; c < nblk / 4; ++c)
      KBS_CUDA_TRY(cudaMemsetAsync(dst + size_t(c) * plan.col_bytes + size_t(kb_used) * kABlockBytes, 0,
                                   size_t(plan.kb_total - kb_used) * kABlockBytes, st));
  const int64_t nblocks = T * panels * int64_t(nblk) * 2;
  if (nblocks > 0x7fffffffLL) return KBS_E_SHAPE;
  const unsigned gb = unsigned(nblocks);
  if (b_operand)
    KBS_LAUNCH(h, KBS_K_PACK_TN, st, (sb_to_tn_kernel<true><<<gb, 256, 0, st>>>(src, step_bytes, kb_src, blk0, nblk, n, panels, T, dst,
                                                                           plan.kb_total, plan.col_bytes)));
  else
    KBS_LAUNCH(h, KBS_K_PACK_TN, st, (sb_to_tn_kernel<false><<<gb, 256, 0, st>>>(src, step_bytes, kb_src, blk0, nblk, n, panels, T, dst,
                                                                            plan.kb_total, plan.col_bytes)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_tc_soa_to_tn(kbs_handle* h, const KbsTnPlan& plan, const float* soa, int F, int64_t ld, int64_t n, int64_t T, int ncols_pad,
                     bool ones, char* dst, cudaStream_t st) {
  if (tc_kind(h) != KBS_KIND_F16 || ncols_pad % kTileCols || F + (ones ? 1 : 0) > ncols_pad) return KBS_E_STATE;
  { const int rc0 = kbs_status_init(h); if (rc0) return rc0; }
  const int64_t np = pad_rows(n);
  const int64_t kb_used = (T * np + 31) / 32;
  if (kb_used > plan.kb_total) return KBS_E_SHAPE;
  if (kb_used < plan.kb_total)
    for (int c = 0; c < ncols_pad / kTileCols; ++c)
      KBS_CUDA_TRY(cudaMemsetAsync(dst + size_t(c) * plan.col_bytes + size_t(kb_used) * kABlockBytes, 0,
                                   size_t(plan.kb_total - kb_used) * kABlockBytes, st));
  if (T > 65535) return KBS_E_SHAPE;
  const dim3 grid(unsigned(np / 64), unsigned(ncols_pad / 32), unsigned(T));
  KBS_LAUNCH(h, KBS_K_PACK, st, (soa_to_tn_kernel<<<grid, 256, 0, st>>>(
                                    soa, F, ld, n, np, T, ncols_pad, ones ? 1 : 0, dst, plan.kb_total, plan.col_bytes, h->persist_status)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// ---- backward recurrence of the PPO update: one persistent launch ----
size_t kbs_tc_bptt_flag_bytes(const kbs_handle* h, int64_t n) {
  return (size_t(h->p.depth) * 2 * size_t(pad_rows(n) / kPanelRows) * 4 + 255) / 256 * 256;
}
bool kbs_tc_bptt_available(const kbs_handle* h, int64_t n, int64_t T) {
  const int H = h->p.hidden_size, depth = h->p.depth;
  if (tc_kind(h) != KBS_KIND_F16 || !persist_shape_ok(h) || H % kTileCols || H % kBT) return false;
  if (!kbs_tc_persistent_available(h, n, T, 2)) return false;
  const int64_t panels = pad_rows(n) / kPanelRows;
  return (T + 2 * depth) * 2 * panels * depth * 2 * (H / kBT) < (int64_t(1) << 31);
}
// tile width of bptt_persist_kernel: 64 columns.  The 128-column instantiation (KBS_BPTT_TILE=128; the caller packs the
// weights for whichever this returns) was meant for large minibatches, where every SM has several items per slot and tcgen05
// issue -- 2 instructions per k-step whatever the width -- could bound an item; MEASURED at 8 192 x 100: 20.1 ms against 19.9 ms
// with 64 columns (the cell's backward in the epilogue, 32 units per thread, takes as long as the item's MMAs), so it stays
// an A/B option.
int kbs_tc_bptt_tile(const kbs_handle* h, int64_t n) {
  (void)h; (void)n;
  const char* e = getenv("KBS_BPTT_TILE");
  return (e && atoi(e) == kTileCols) ? kTileCols : kBT;
}
int kbs_tc_bptt(kbs_handle* h, const KbsBpttArgs& b, cudaStream_t st) {
  const int H = h->p.hidden_size, depth = h->p.depth;
  if (!kbs_tc_bptt_available(h, b.n, b.T)) return KBS_E_STATE;
  { const int rc0 = kbs_status_init(h); if (rc0) return rc0; }
  if (!h->bptt_attr_set) {
    KBS_CUDA_TRY((cudaFuncSetAttribute(bptt_persist_kernel<KBS_KIND_F16, kBT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       BTile<kBT>::kSmemBytes)));
    KBS_CUDA_TRY((cudaFuncSetAttribute(bptt_persist_kernel<KBS_KIND_F16, kTileCols>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       BTile<kTileCols>::kSmemBytes)));
    h->bptt_attr_set = true;
  }
  const int bt = kbs_tc_bptt_tile(h, b.n);
  const int64_t np = pad_rows(b.n);
  BArgs a{};
  for (int k = 0; k < b.nets; ++k) {
    const KbsNet& Nn = h->net[k];
    const float* image = bt == kBT ? Nn.tc_bwd_image64 : Nn.tc_bwd_image;
    if (!Nn.packed || !image) return KBS_E_STATE;
    BNet& N = a.net[k];
    for (int l = 0; l < depth; ++l) N.w_bwd[l] = reinterpret_cast<const char*>(image) + bwd_layer_bytes(h) * l;
    N.dG = b.net[k].dG; N.save_g = b.net[k].save_g; N.c_hist = b.net[k].c_hist; N.dh_top = b.net[k].dh_top;
    N.dv = b.net[k].dv; N.w_out = b.net[k].w_out;
    if (!N.dh_top && !(N.dv && N.w_out)) return KBS_E_NULL;
    N.dx = b.net[k].dx; N.dx0 = b.net[k].dx0; N.dc = b.net[k].dc; N.flags = b.net[k].flags;
    for (int l = 0; l < depth; ++l) N.tn_dG[l] = b.net[k].tn_dG[l];
  }
  a.nets = b.nets; a.depth = depth; a.H = H; a.panels = int(np / kPanelRows);
  a.n = b.n; a.ld = b.ld; a.T = b.T;
  a.sbb = kbs_sb_bytes_kind(KBS_KIND_F16, np, H); a.sb4 = kbs_sb_bytes_kind(KBS_KIND_F16, np, 4 * H);
  a.done = b.done; a.gscale = b.gscale; a.inv_gscale = 1.0f / b.gscale;
  a.status = h->persist_status;
  { const char* e = getenv("KBS_PERSIST_DBG"); a.dbg = e ? atoi(e) : 0; }
  a.trace = h->trace_buf ? h->trace_buf + 2 * 148 * 16 : nullptr;  // third region of the debug buffer (forward kernel, input projection, this)
  const int64_t per_slot = int64_t(b.nets) * a.panels * depth * 2 * (H / bt);
  const int n_cc = int(per_slot < h->num_sms ? per_slot : h->num_sms);
  // The X tiles re-pack dG for the weight-gradient GEMMs on the fly when a CTA has (about) one item per slot: its epilogue
  // warps are idle during the MMAs then.  With many items per CTA and slot the epilogue of item j overlaps the MMAs of item
  // j + 1 and must not be held up: the caller runs kbs_tc_sb_to_tn after the kernel instead (*transposed_out says which).
  int tn = (b.tn_plan && b.net[0].tn_dG[0] && per_slot <= 2 * int64_t(h->num_sms)) ? 1 : 0;
  { const char* e = getenv("KBS_BPTT_TN"); if (e && b.tn_plan && b.net[0].tn_dG[0]) tn = atoi(e) ? 1 : 0; }
  a.tn = tn;
  if (tn) { a.tn_kb_total = b.tn_plan->kb_total; a.tn_col_bytes = b.tn_plan->col_bytes; }
  if (b.transposed_out) *b.transposed_out = tn != 0;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(unsigned(n_cc));
  cfg.blockDim = dim3(kBThreads);
  cfg.dynamicSmemBytes = bt == kBT ? BTile<kBT>::kSmemBytes : BTile<kTileCols>::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative;      // every CTA must be resident: they wait on each other's counters
  at[0].val.cooperative = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaError_t le = cudaSuccess;
  if (bt == kBT) KBS_LAUNCH(h, KBS_K_BPTT_TC, st, (le = cudaLaunchKernelEx(&cfg, bptt_persist_kernel<KBS_KIND_F16, kBT>, a)));
  else KBS_LAUNCH(h, KBS_K_BPTT_TC, st, (le = cudaLaunchKernelEx(&cfg, bptt_persist_kernel<KBS_KIND_F16, kTileCols>, a)));
  KBS_CUDA_TRY(le);
  { const int rc0 = kbs_status_publish(h, st); if (rc0) return rc0; }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// ---- forward recurrence of the PPO update: lstm_fwd_save_kernel ----
size_t kbs_tc_fwd_save_flag_bytes(const kbs_handle* h, int64_t n) {
  return (size_t(h->p.depth) * size_t(pad_rows(n) / kPanelRows) * 4 + 255) / 256 * 256;
}
bool kbs_tc_fwd_save_available(const kbs_handle* h, int64_t n, int64_t T) {
  const int H = h->p.hidden_size, depth = h->p.depth;
  if (tc_kind(h) != KBS_KIND_F16 || H % 32 || H > kMaxBias / 4 || depth > kPMaxDepth) return false;
  const int64_t panels = pad_rows(n) / kPanelRows;
  return (T + depth) * 2 * panels * depth * (H / 32) < (int64_t(1) << 31);
}
int kbs_tc_fwd_save(kbs_handle* h, const KbsFwdSaveArgs& f, cudaStream_t st) {
  const int H = h->p.hidden_size, depth = h->p.depth;
  if (!kbs_tc_fwd_save_available(h, f.n, f.T)) return KBS_E_STATE;
  { const int rc0 = kbs_status_init(h); if (rc0) return rc0; }
  if (!h->fwd_save_attr_set) {
    KBS_CUDA_TRY(cudaFuncSetAttribute(lstm_fwd_save_kernel<KBS_KIND_F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSSmemBytes));
    h->fwd_save_attr_set = true;
  }
  const int64_t n = f.n, np = pad_rows(n);
  const size_t sbb = act_sb_bytes(h, n), fbf = size_t(np) * H;
  SArgs a{};
  CarryJobs J{};
  J.ld_rm = H; J.status = h->persist_status;
  int jobs = 0;
  for (int k = 0; k < f.nets; ++k) {
    const KbsNet& Nn = h->net[k];
    if (!Nn.packed || !Nn.tc_fwd8_image) return KBS_E_STATE;
    SNet& N = a.net[k];
    N.x0 = f.net[k].x0; N.x0_stride = sbb; N.xmid = f.net[k].xmid; N.hsb = f.net[k].hsb; N.c_hist = f.net[k].c_hist;
    N.save_g = f.net[k].save_g; N.h_top_rm = f.net[k].h_top_rm; N.flags = f.net[k].flags;
    for (int l = 0; l < depth; ++l) {
      const char* w8 = reinterpret_cast<const char*>(Nn.tc_fwd8_image) + layer_image_bytes(h) * l;
      N.w[l] = w8;
      N.bias[l] = reinterpret_cast<const float*>(w8 + kbs_sb_bytes_kind(KBS_KIND_F16, 4 * H, 2 * H));
      N.tn_xh[l] = f.net[k].tn_xh[l];
      // the carries the first step reads: ABI layout [depth][2][n][H], or zeros (get_initial_model_carry)
      char* h_dst = f.net[k].hsb + sbb * (size_t(l) * (f.T + 1));
      float* c_dst = f.net[k].c_hist + fbf * (size_t(l) * (f.T + 1));
      if (!f.net[k].carry0) {
        KBS_CUDA_TRY(cudaMemsetAsync(h_dst, 0, sbb, st));
        KBS_CUDA_TRY(cudaMemsetAsync(c_dst, 0, fbf * sizeof(float), st));
      } else {
        float* c0 = const_cast<float*>(f.net[k].carry0);
        J.rm[jobs] = c0 + (size_t(l) * 2 + 0) * size_t(n) * H; J.blk[jobs] = h_dst; J.mode[jobs++] = 0;
        J.rm[jobs] = c0 + (size_t(l) * 2 + 1) * size_t(n) * H; J.blk[jobs] = c_dst; J.mode[jobs++] = 1;
      }
    }
    KBS_CUDA_TRY(cudaMemsetAsync(f.net[k].flags, 0, kbs_tc_fwd_save_flag_bytes(h, n), st));
  }
  if (jobs) carry_convert(h, J, jobs, n, np, H, st);
  a.nets = f.nets; a.depth = depth; a.H = H; a.panels = int(np / kPanelRows);
  a.n = n; a.ld = f.ld; a.T = f.T; a.sbb = sbb; a.done = f.done; a.status = h->persist_status;
  { const char* e = getenv("KBS_PERSIST_DBG"); a.dbg = e ? atoi(e) : 0; }
  const int64_t per_slot = int64_t(f.nets) * a.panels * depth * (H / 32);
  int tn = (f.tn_plan && f.net[0].tn_xh[0] && per_slot <= 2 * int64_t(h->num_sms)) ? 1 : 0;
  { const char* e = getenv("KBS_FWD_TN"); if (e && f.tn_plan && f.net[0].tn_xh[0]) tn = atoi(e) ? 1 : 0; }
  a.tn = tn;
  if (tn) { a.tn_kb_total = f.tn_plan->kb_total; a.tn_col_bytes = f.tn_plan->col_bytes; }
  if (f.transposed_out) *f.transposed_out = tn != 0;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(unsigned(per_slot < h->num_sms ? per_slot : h->num_sms));
  cfg.blockDim = dim3(kSThreads);
  cfg.dynamicSmemBytes = kSSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative;
  at[0].val.cooperative = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaError_t le = cudaSuccess;
  KBS_LAUNCH(h, KBS_K_ROLLOUT_TC, st, (le = cudaLaunchKernelEx(&cfg, lstm_fwd_save_kernel<KBS_KIND_F16>, a)));
  KBS_CUDA_TRY(le);
  { const int rc0 = kbs_status_publish(h, st); if (rc0) return rc0; }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// ---- weight-gradient GEMMs straight from the kept history: dw_gemm_kernel ------------------------------------------------
// dW_l = dG_l^T [x_l | h_in_l] contracts over ROWS (K' = step x env), and the recurrence kernels keep dG / x / h as per-step
// split-blocked operands that are K-major over FEATURES: [panel][32-feature block][hi|lo][8-feature chunk][128 rows][16 B].
// Read the other way round that is already a canonical UMMA operand -- MN-major, no swizzle: a 16-byte unit = 8 consecutive
// features (MN) of one row, the 8 rows (K') of a core matrix 16 bytes apart, the next chunk of features one chunk stride
// further -- so the GEMM takes the history IN PLACE (instruction-descriptor bits a_major = b_major = MN) and the K = row
// re-pack (sb_to_tn_kernel: 44 GB of traffic and 10 ms of a 64 ms update at 8 192 trajectories; the in-kernel transposes of
// the recurrence kernels at 512) is not needed for the four big GEMMs of an update.
// Work item = (128 gate rows of dG, 256 columns of x or of h_in | the bias column, one accumulation run of <= 3 200 rows),
// ordered run-major so that the items in flight share their operands in L2.
// Stage = 32 rows: 4-D TMA boxes {32 rows x 16 B, 4 chunks, 4 | 8 blocks, 1 (step, panel)} land as [block][chunk][row][16 B]
// per plane = 16 core matrices (A) / 32 (B) along MN at a uniform 512 B, 8-row groups 128 B apart.  Per 16-row k-step three
// N = 256 MMAs: hi.hi -> main, hi.lo + lo.hi -> correction columns (the truncating accumulator, profiles/r01_tc_accumulation.md).
// The bias gradient (column sums of dG) is a third kind of item: B = a constant block with a one in feature 0, N = 16.
// Partial sums go to the same [run][4H][2H + 128] slabs the K-major GEMM writes: tn_reduce_kernel adds them in fixed order.
constexpr int kDwRows = 32;                                                          // K' rows per stage
constexpr int kDwParts = kPanelRows / kDwRows;                                       // stages per (step, panel) unit
constexpr int kDwAPlane = 128 * kDwRows * 2, kDwBPlane = 256 * kDwRows * 2;          // 8 KB, 16 KB
constexpr int kDwStageBytes = 2 * kDwAPlane + 2 * kDwBPlane;                         // 48 KB
constexpr int kDwStages = 4;          // (2 stages of 64 rows: a stage's load could only start behind the MMAs of the stage before the last)
constexpr int kDwOnesBytes = 2 * kDwRows * 16;                                       // 2 chunks x kDwRows rows x 16 B
constexpr int kDwSmemBytes = kDwStages * kDwStageBytes + kDwOnesBytes + 256 + 1024;
constexpr int kDwThreads = 32 * 6;                                                   // issuer, producer, 4 epilogue warps
struct alignas(64) DwArgs {
  CUtensorMap a_map[2];         // dG of the layer, hi / lo plane
  CUtensorMap b_map[2][2];      // [x | h_in][hi | lo]
  int units, units_per_run, ksplit, m_tiles;     // unit = one (step, panel) pair = 128 rows
  float* partial; int ldc; size_t split_stride;
  float oscale;
};
// c0 = first row of the box x 4 (32-bit elements: the 128 rows x 16 B of a chunk are one contiguous 2 KB line of the tensor)
__device__ __forceinline__ void tma_load_sb(void* dst, const CUtensorMap* map, int row0, int kb0, int unit, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
          smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(row0 * 4), "r"(0), "r"(kb0), "r"(unit), "r"(smem_u32(bar))
      : "memory");
}
template <int N>
__device__ __forceinline__ void umma_f16_mn(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  constexpr uint32_t idesc = idesc_f16<N>() | (1u << 15) | (1u << 16);               // a_major = b_major = MN
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__global__ void __launch_bounds__(kDwThreads, 1) dw_gemm_kernel(const __grid_constant__ DwArgs args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ones = smem + kDwStages * kDwStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ones + kDwOnesBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + kDwStages;
  uint64_t* acc_full = bars + 2 * kDwStages;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kDwStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // the bias item's B operand: [2 chunks][kDwRows rows][16 B], feature 0 of every row = 1.0 (fp16), everything else 0
  for (int i = threadIdx.x; i < kDwOnesBytes / 16; i += kDwThreads)
    reinterpret_cast<uint4*>(ones)[i] = i < kDwRows ? make_uint4(0x3C00u, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Item order: all 256-column items first, run-major (the 2 m_tiles of a run are taken by neighbouring CTAs at the same time, so
  // each dG tile is fetched from HBM once for its readers and each [x | h] tile once for its m_tiles readers: gate-tile-major
  // order streamed every operand from HBM per item, 1.4 GB instead of 0.3 GB per GEMM), then the bias items (about half the
  // cost of a big one), run-major as well.  With round-robin over the CTAs the cheap items land on the CTAs that got one big
  // item less: at 16 runs 148 CTAs carry at most 2 big + 1 bias item instead of 3 big ones.
  const int per_run = args.m_tiles * 2, n_big = per_run * args.ksplit, n_items = n_big + args.m_tiles * args.ksplit;
  auto decode = [&](int it, int& m, int& nt, int& run) {
    if (it < n_big) { run = it / per_run; const int q = it - run * per_run; m = q >> 1; nt = q & 1; }
    else { const int j = it - n_big; run = j / args.m_tiles; m = j - run * args.m_tiles; nt = 2; }
  };
  if (warp == 1) {
    if (lane == 0) {
      // ===== producer =====
      uint32_t g = 0;
      for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
        int m, nt, run; decode(it, m, nt, run);
        const int u0 = run * args.units_per_run, u1 = min(u0 + args.units_per_run, args.units);
        for (int u = u0; u < u1; ++u)
          for (int half = 0; half < kDwParts; ++half, ++g) {
            const int s = g % kDwStages;
            mbar_wait(&empty[s], ((g / kDwStages) & 1) ^ 1);
            uint8_t* st = smem + size_t(s) * kDwStageBytes;
            mbar_expect_tx(&full[s], uint32_t(2 * kDwAPlane + (nt < 2 ? 2 * kDwBPlane : 0)));
            tma_load_sb(st, &args.a_map[0], half * kDwRows, 4 * m, u, &full[s]);
            tma_load_sb(st + kDwAPlane, &args.a_map[1], half * kDwRows, 4 * m, u, &full[s]);
            if (nt < 2) {
              tma_load_sb(st + 2 * kDwAPlane, &args.b_map[nt][0], half * kDwRows, 0, u, &full[s]);
              tma_load_sb(st + 2 * kDwAPlane + kDwBPlane, &args.b_map[nt][1], half * kDwRows, 0, u, &full[s]);
            }
          }
      }
    }
    __syncwarp();
  } else if (warp == 0) {
    // ===== MMA issuer =====
    uint32_t g = 0;
    int j = 0;
    const uint32_t d_main = tmem_base, d_corr = tmem_base + 256;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
      int m, nt, run; decode(it, m, nt, run);
      const int u0 = run * args.units_per_run, u1 = min(u0 + args.units_per_run, args.units);
      if (u1 <= u0) continue;                                   // a run behind the last unit: the epilogue writes zeros
      mbar_wait(acc_empty, (j & 1) ^ 1);
      tc_fence_after();
      uint32_t first = 0;
      for (int q = 0; q < kDwParts * (u1 - u0); ++q, ++g) {
        const int s = g % kDwStages;
        mbar_wait(&full[s], (g / kDwStages) & 1);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + size_t(s) * kDwStageBytes);
        // MN-major, no swizzle: LBO = distance of the 8-row groups (128 B), SBO = distance of the 8-feature chunks (kDwRows x 16 B)
        const uint64_t a_hi = umma_desc(sa, 128, kDwRows * 16), a_lo = umma_desc(sa + kDwAPlane, 128, kDwRows * 16);
        const uint64_t b_hi = nt < 2 ? umma_desc(sa + 2 * kDwAPlane, 128, kDwRows * 16) : umma_desc(smem_u32(ones), 128, kDwRows * 16);
        const uint64_t b_lo = umma_desc(sa + 2 * kDwAPlane + kDwBPlane, 128, kDwRows * 16);
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < kDwRows / 16; ++ks) {
            const uint64_t o = uint64_t(ks * 256) >> 4;                 // 16 rows further
            if (nt < 2) {
              umma_f16_mn<256>(d_main, a_hi + o, b_hi + o, first | uint32_t(ks));
              umma_f16_mn<256>(d_corr, a_hi + o, b_lo + o, first | uint32_t(ks));
              umma_f16_mn<256>(d_corr, a_lo + o, b_hi + o, 1);
            } else {
              umma_f16_mn<16>(d_main, a_hi + o, b_hi + o, first | uint32_t(ks));
              umma_f16_mn<16>(d_corr, a_lo + o, b_hi + o, first | uint32_t(ks));
            }
          }
          umma_commit(&empty[s]);
        }
        __syncwarp();
        first = 1;
      }
      if (elect_one()) umma_commit(acc_full);
      __syncwarp();
      ++j;
    }
  } else {
    // ===== epilogue: 4 warps, warp % 4 = TMEM lane quarter; thread = one gate row of the tile =====
    const int q4 = warp & 3, r = q4 * 32 + lane;
    constexpr float kCorr = 1.0f / kKbsF16LoScale;
    int j = 0;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
      int m, nt, run; decode(it, m, nt, run);
      float* dst = args.partial + size_t(run) * args.split_stride + size_t(m * 128 + r) * args.ldc + nt * 256;
      if (run * args.units_per_run >= args.units) {
        if (nt < 2) for (int c = 0; c < 256; c += 4) *reinterpret_cast<float4*>(dst + c) = make_float4(0.f, 0.f, 0.f, 0.f);
        else dst[0] = 0.0f;
        continue;
      }
      mbar_wait(acc_full, j & 1);
      tc_fence_after();
      const uint32_t tq = tmem_base + (uint32_t(q4 * 32) << 16);
      if (nt < 2) {
#pragma unroll 1
        for (int c = 0; c < 256; c += 16) {
          float v[16], cr[16];
          tmem_ld16(tq + c, v);
          tmem_ld16(tq + 256 + c, cr);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; i += 4)
            *reinterpret_cast<float4*>(dst + c + i) =
                make_float4(args.oscale * (v[i] + kCorr * cr[i]), args.oscale * (v[i + 1] + kCorr * cr[i + 1]),
                            args.oscale * (v[i + 2] + kCorr * cr[i + 2]), args.oscale * (v[i + 3] + kCorr * cr[i + 3]));
        }
      } else {
        float v[8], cr[8];
        tmem_ld8(tq, v);
        tmem_ld8(tq + 256, cr);
        tmem_ld_wait();
        dst[0] = args.oscale * (v[0] + kCorr * cr[0]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
      ++j;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}

// 4-D map over per-step split-blocked buffers (one plane), 32-bit elements: {128 rows x 4 words (one chunk: contiguous), 4 chunks,
// kb blocks, slots * panels}; box = {kDwRows rows x 4 words, 4, box_kb, 1}.  (With the 16 bytes of a row as the innermost dimension
// the copy engine moved 16-byte lines: the GEMM ran at a quarter of the speed.)
static bool encode_sb_plane_map(CUtensorMap* m, const char* base, int kb, int64_t units, int box_kb) {
  KbsTensorMapEncodeFn fn = tensor_map_encode_fn();
  if (!fn || !base) return false;
  const cuuint64_t gdim[4] = {cuuint64_t(kPanelRows) * 4, 4, cuuint64_t(kb), cuuint64_t(units)};
  const cuuint64_t gstride[3] = {cuuint64_t(kPanelRows) * 16, cuuint64_t(kABlockBytes), cuuint64_t(kb) * kABlockBytes};
  const cuuint32_t box[4] = {cuuint32_t(kDwRows) * 4, 4, cuuint32_t(box_kb), 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, const_cast<char*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool kbs_tc_dw_direct_available(const kbs_handle* h, int64_t n) {
  const char* e = getenv("KBS_DW_DIRECT");
  if (e && !atoi(e)) return false;
  // rows beyond n of the last panel are never written by the recurrence kernels: the in-place operands need whole panels
  return tc_kind(h) == KBS_KIND_F16 && h->p.hidden_size == 256 && (n % kPanelRows) == 0 && tensor_map_encode_fn() != nullptr;
}

// partial [ksplit][4H][ldc] (ldc = 2H + 128) <- dG^T [x | h_in | 1] over units = slots-in-use x panels; dG / x / h_in: bases of slot 0
int kbs_tc_dw_direct(kbs_handle* h, const KbsTnPlan& plan, const char* dG, const char* x_hist, const char* h_hist, int64_t n, int64_t T,
                     float* partial, float out_scale, cudaStream_t st) {
  const int H = h->p.hidden_size;
  if (!kbs_tc_dw_direct_available(h, n)) return KBS_E_STATE;
  const int panels = int(n / kPanelRows);
  const int64_t units = T * panels;
  if (units > 0x7fffffffLL) return KBS_E_SHAPE;
  if (!h->dw_attr_set) {
    KBS_CUDA_TRY(cudaFuncSetAttribute(dw_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDwSmemBytes));
    h->dw_attr_set = true;
  }
  DwArgs a{};
  for (int pl = 0; pl < 2; ++pl) {
    if (!encode_sb_plane_map(&a.a_map[pl], dG + pl * (kABlockBytes / 2), 4 * H / 32, units, 4)) return KBS_E_STATE;
    if (!encode_sb_plane_map(&a.b_map[0][pl], x_hist + pl * (kABlockBytes / 2), H / 32, units, 8)) return KBS_E_STATE;
    if (!encode_sb_plane_map(&a.b_map[1][pl], h_hist + pl * (kABlockBytes / 2), H / 32, units, 8)) return KBS_E_STATE;
  }
  // the runs of the K-major plan (<= 3 200 rows each) in whole units, so that the slabs line up with tn_reduce_kernel's
  a.units = int(units);
  a.ksplit = plan.ksplit;
  a.units_per_run = int((units + plan.ksplit - 1) / plan.ksplit);
  if (int64_t(a.units_per_run) * kPanelRows > 3200 + kPanelRows) return KBS_E_SHAPE;
  a.m_tiles = 4 * H / 128;
  a.partial = partial; a.ldc = 2 * H + 128; a.split_stride = size_t(4 * H) * size_t(a.ldc);
  a.oscale = out_scale;
  const int items = a.m_tiles * 3 * a.ksplit;
  const int grid = items < h->num_sms ? items : h->num_sms;
  KBS_LAUNCH(h, KBS_K_GEMM_TN, st, (dw_gemm_kernel<<<grid, kDwThreads, kDwSmemBytes, st>>>(a)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

int kbs_tc_tn_reduce(kbs_handle* h, const KbsTnPlan& plan, const float* partial, int m_panels, int ldc, int col0, int nrows,
                     int ncols, float* dst, int ld_dst, cudaStream_t st) {
  const int64_t total = int64_t(nrows) * ncols;
  KBS_LAUNCH(h, KBS_K_TN_REDUCE, st, (tn_reduce_kernel<<<unsigned((total + 255) / 256), 256, 0, st>>>(
                                         partial, plan.ksplit, size_t(m_panels) * kPanelRows * size_t(ldc), ldc, col0, nrows, ncols, dst, ld_dst)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// several column ranges of the same slabs in one launch: seg = {col0, ncols, ld_dst} x nseg, dst[nseg]
int kbs_tc_tn_reduce_multi(kbs_handle* h, const KbsTnPlan& plan, const float* partial, int m_panels, int ldc, int nrows, int nseg,
                           const int (*seg)[3], float* const* dst, cudaStream_t st) {
  if (nseg < 1 || nseg > 3) return KBS_E_SHAPE;
  TnSegs sg{};
  sg.nseg = nseg;
  for (int k = 0; k < nseg; ++k) {
    sg.col0[k] = seg[k][0]; sg.ncols[k] = seg[k][1]; sg.ld_dst[k] = seg[k][2]; sg.dst[k] = dst[k];
    sg.total_cols += seg[k][1];
  }
  const int64_t total = int64_t(nrows) * sg.total_cols;
  KBS_LAUNCH(h, KBS_K_TN_REDUCE, st, (tn_reduce_multi_kernel<<<unsigned((total + 255) / 256), 256, 0, st>>>(
                                         partial, plan.ksplit, size_t(m_panels) * kPanelRows * size_t(ldc), ldc, nrows, sg)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

size_t kbs_tc_rows_sb_bytes(const kbs_handle* h, int64_t n, int K) { return kbs_sb_bytes_kind(tc_kind(h), pad_rows(n), K); }
int kbs_tc_kind_of(const kbs_handle* h) { return tc_kind(h); }

// ---- fused rollout: tensor-core input projection of all T steps + the recurrent phase --------------------------------
KbsTcRolloutWs kbs_tc_rollout_ws(KbsScratch& s, const kbs_handle* h, int64_t n, int nets) {
  const size_t sbb = act_sb_bytes(h, n), depth = size_t(h->p.depth), H = size_t(h->p.hidden_size), np = size_t(pad_rows(n));
  KbsTcRolloutWs w{};
  for (int k = 0; k < nets; ++k) {
    w.hsb[k] = s.take<char>(2 * depth * sbb);
    w.xmid[k] = s.take<char>(2 * depth * sbb);    // the per-step launch path uses the first two
    w.h2rm[k] = s.take<float>(2 * size_t(n) * H);  // top-layer output (per-step path)
    w.fb[k] = s.take<float>(2 * depth * np * H);
    w.flags[k] = s.take<unsigned int>((depth + 1) * (np / kPanelRows));
  }
  return w;
}
int64_t kbs_tc_sb_floats(const kbs_handle* h, int64_t n) { return int64_t(act_sb_bytes(h, n) / 4); }
// floats of the SB observation staging buffer of `net` for T steps
int64_t kbs_tc_obs_sb_floats(const kbs_handle* h, int net, int64_t n, int64_t T) {
  const int kp = proj_kp(h, net), kf = fused_shape(h, net) ? fused_kp(h, net) : 0;
  return int64_t(kbs_sb_bytes_kind(tc_kind(h), T * pad_rows(n), kp > kf ? kp : kf) / 4);
}

// true: kbs_tc_input_proj_all(.., r_out) will fold net's input projection into layer 0 of the persistent kernel
bool kbs_tc_fused_input(const kbs_handle* h, int net, int64_t n, int64_t T, int nets) {
  const char* off_env = getenv("KBS_NO_FUSED_INPUT");          // A/B + cross-check (tests): keep the projection launch
  const char* legacy_env = getenv("KBS_TC_PER_STEP");
  if ((off_env && atoi(off_env)) || (legacy_env && atoi(legacy_env))) return false;
  return fused_shape(h, net) && kbs_tc_persistent_available(h, n, T, nets);
}

// obs_soa[k]: [T][num_in][ld] observations of net k; obs_sb[k]: staging (kbs_tc_obs_sb_floats); x_sb_all[k]: [T] x act SB.
int kbs_tc_input_proj_all(kbs_handle* h, int nets, const float* const* obs_soa, float* const* obs_sb, float* const* x_sb_all,
                          int64_t ld, int64_t n, int64_t T, cudaStream_t st, const float* cinert, const float* cvel,
                          KbsTcRolloutArgs* r_out) {
  const int H = h->p.hidden_size, kind = tc_kind(h);
  { const int rc0 = kbs_status_init(h); if (rc0) return rc0; }
  int proj_nets = 0;
  const int64_t np = pad_rows(n);
  // Default: input_proj_fused_kernel (FP16-split datapath, H = 256) straight from the SoA observations.  Otherwise the staged
  // form: pack kernel -> SB staging buffer -> MODE_PROJ launch.  KBS_PROJ_FUSED=1 (historical): the MODE_PROJ kernel's own
  // producer warps read the SoA observations into registers (MODE_PROJ_SOA) -- MEASURED 3.87 ms instead of 0.45 + 0.49 ms per
  // 100-step rollout: 128 threads x 32 register-staged loads are ~16 KB in flight per SM where HBM latency needs ~90 KB.
  static int staged = -1;
  if (staged < 0) { const char* e = getenv("KBS_PROJ_FUSED"); staged = (e && atoi(e)) ? 0 : 1; }
  LayerArgs2 a2{};
  for (int k = 0; k < nets; ++k) {
    const KbsNet& N = h->net[k];
    if (!N.packed || !N.tc_image) return KBS_E_STATE;
    const bool fuse = r_out && kbs_tc_fused_input(h, k, n, T, nets);
    const int Kp = fuse ? fused_kp(h, k) : proj_kp(h, k);
    const float* ci = (k == KBS_NET_CRITIC) ? cinert : nullptr;
    const float* cv = (k == KBS_NET_CRITIC) ? cvel : nullptr;
    char* osb = reinterpret_cast<char*>(obs_sb[k]);
    LayerArgs& a = a2.net[k];
    if (r_out) { r_out->x_sb_all[k] = fuse ? obs_sb[k] : x_sb_all[k]; r_out->x_is_obs[k] = fuse; }
    const char* staged_env = getenv("KBS_PROJ_STAGED");            // A/B + cross-check: pack kernel + MODE_PROJ launch
    if (!fuse && staged && projq_shape(h) && !(staged_env && atoi(staged_env)) && tensor_map_encode_fn()) {
      // straight from the SoA observations (input_proj_fused_kernel): no staging buffer, one launch per net
      const int which = (ci && cv && projq_has_dump_layout(h, k)) ? 1 : 0;
      const FLayout Lq = projq_layout(h, k, which);
      FProjArgs fa{};
      const int kf = kbs_block_k(kind);
      bool ok = encode_rows_map(&fa.tmap[0], obs_soa[k], ld, T * int64_t(N.num_in), kf);
      fa.rows_per_step[0] = N.num_in;
      if (which == 1) {
        ok = ok && encode_rows_map(&fa.tmap[1], ci, ld, T * int64_t(10 * KBS_NBODY), kf) &&
             encode_rows_map(&fa.tmap[2], cv, ld, T * int64_t(6 * KBS_NBODY), kf);
        fa.rows_per_step[1] = 10 * KBS_NBODY; fa.rows_per_step[2] = 6 * KBS_NBODY;
      }
      if (ok) {
        fa.kb = Lq.kb; fa.H = H;
        for (int b = 0; b < Lq.kb; ++b) { fa.blk_src[b] = Lq.src[b]; fa.blk_row0[b] = Lq.row0[b]; fa.blk_nvalid[b] = Lq.nvalid[b]; }
        fa.n = n; fa.n_pad = np;
        fa.w_sb = projq_w(h, k, which); fa.bias = projq_bias(h, k, which);
        fa.x_sb = reinterpret_cast<char*>(x_sb_all[k]); fa.sbb = act_sb_bytes(h, n);
        fa.items = int(T * np / kPanelRows);
        fa.status = h->persist_status;
        { const char* e = getenv("KBS_FPROJ_DBG"); fa.dbg = e ? atoi(e) : 0; }
        fa.trace = h->trace_buf;
        const unsigned grid = unsigned(fa.items < h->num_sms ? fa.items : h->num_sms);
        if (kind == KBS_KIND_TF32)
          KBS_LAUNCH(h, KBS_K_PROJ_TC, st, (input_proj_fused_kernel<KBS_KIND_TF32><<<grid, kFThreads, kFSmemBytes, st>>>(fa)));
        else
          KBS_LAUNCH(h, KBS_K_PROJ_TC, st, (input_proj_fused_kernel<KBS_KIND_F16><<<grid, kFThreads, kFSmemBytes, st>>>(fa)));
        continue;                     // no MODE_PROJ items for this net (panels = 0)
      }
    }
    if (staged || fuse) {
      const int64_t total = T * np * (Kp / 8);
      const unsigned gb = unsigned((total + 255) / 256);
      if (kind == KBS_KIND_TF32)
        KBS_LAUNCH(h, KBS_K_PACK, st, (pack_soa_sb_kernel<KBS_KIND_TF32><<<gb, 256, 0, st>>>(obs_soa[k], N.num_in, ld, osb, n, np, Kp, T, ci, cv, h->persist_status)));
      else
        KBS_LAUNCH(h, KBS_K_PACK, st, (pack_soa_sb_kernel<KBS_KIND_F16><<<gb, 256, 0, st>>>(obs_soa[k], N.num_in, ld, osb, n, np, Kp, T, ci, cv, h->persist_status)));
      a.mode = MODE_PROJ;
      if (fuse) continue;            // the packed observations ARE layer 0's input operand: no projection items (panels = 0)
    } else {
      // fused: the projection kernel's producer warps read the SoA observations (and the critic's cinert / cvel dump from the
      // recorded state) themselves and build the MMA operand in shared memory
      a.mode = MODE_PROJ_SOA;
      a.soa = obs_soa[k]; a.cinert = ci; a.cvel = cv; a.F = N.num_in; a.soa_ld = ld; a.n_env = n; a.n_pad = np;
    }
    a.x_sb = osb;
    a.h_sb_in = osb;
    a.w_sb = proj_w(h, k);
    a.bias_t = proj_bias(h, k);
    a.x_next_sb = reinterpret_cast<char*>(x_sb_all[k]);
    a.status = h->persist_status;
    a.n = T * np;                    // every staged row is written (pad rows carry the bias: harmless, never read back)
    a.H = H; a.kb_x = Kp / kbs_block_k(kind); a.kb_h = 0;
    a.panels = int(T * np / kPanelRows); a.tiles = proj_cols(h) / kTileCols;
    ++proj_nets;
  }
  if (!proj_nets) { KBS_LAUNCH_CHECK(); return KBS_OK; }
  for (int k = 0; k < 2; ++k)
    if (!a2.net[k].panels) a2.net[k].mode = a2.net[k ^ 1].mode;
  KBS_LAUNCH(h, KBS_K_PROJ_TC, st, (launch_layer(h, kind, a2, st)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

bool kbs_tc_persistent_available(const kbs_handle* h, int64_t n, int64_t T, int nets) {
  const int H = h->p.hidden_size, depth = h->p.depth;
  if (!persist_shape_ok(h)) return false;
  const int64_t panels = pad_rows(n) / kPanelRows, tiles = H / kUnitsPerTileP;
  return (T + depth) * int64_t(nets) * panels * (depth * tiles + 1) < (int64_t(1) << 31);
}

int kbs_tc_rollout_recurrent(kbs_handle* h, const KbsTcRolloutArgs& r, cudaStream_t st) {
  const int H = h->p.hidden_size, depth = h->p.depth, kind = tc_kind(h);
  const int nets = r.with_critic ? 2 : 1;
  for (int k = 0; k < nets; ++k)
    if (!h->net[k].packed || !h->net[k].tc_image) return KBS_E_STATE;
  { const int rc0 = kbs_status_init(h); if (rc0) return rc0; }
  const int head_smem = (kHeadEnvs * (H + 4) + KBS_ACTOR_OUT * H + kHeadEnvs * 41 + 4 * 32 * 2) * 4;
  if (!h->head_attr_set) {
    KBS_CUDA_TRY(cudaFuncSetAttribute(rollout_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    h->head_attr_set = true;
  }
  const int64_t n = r.n, ld = r.ld, np = pad_rows(n);
  const size_t sbb = act_sb_bytes(h, n);
  char* hsb[2] = {r.ws.hsb[0], r.ws.hsb[1]}; char* xmid[2] = {r.ws.xmid[0], r.ws.xmid[1]};
  float* const* h2rm = r.ws.h2rm; float* fb[2] = {r.ws.fb[0], r.ws.fb[1]}; unsigned int* const* flags = r.ws.flags;
  const size_t fbf = size_t(np) * H;
  const bool resident = r.res_hsb_slot != nullptr;
  const char* legacy_env = getenv("KBS_TC_PER_STEP");          // A/B and cross-check against the per-step launches
  const int legacy = (legacy_env && !r.save && !resident) ? atoi(legacy_env) : 0;
  const bool persistent = !legacy && kbs_tc_persistent_available(h, n, r.T, nets);
  if (resident) {                                              // the step state's own operands: nothing to convert
    if (!persistent || r.save || r.carry_ld) return KBS_E_SHAPE;
    for (int k = 0; k < nets; ++k) { hsb[k] = r.res_hsb[k]; fb[k] = r.res_fb[k]; }
  }
  if (r.save) {                                                // forward pass of the PPO update: per-step history buffers
    if (!persistent || kind != KBS_KIND_F16 || r.carry_ld) return KBS_E_STATE;
    for (int k = 0; k < nets; ++k) { hsb[k] = r.hsb_hist[k]; xmid[k] = r.xmid_hist[k]; }
  }
  const size_t hstep = r.save ? size_t(r.T + 1) : 2;           // slots per layer of hsb / c_hist
  if ((r.x_is_obs[0] || r.x_is_obs[1]) && !persistent) return KBS_E_STATE;         // folded input projection: persistent only
  if (r.mean && !persistent) return KBS_E_STATE;                                   // dist.mean() output: persistent kernel only
  if (r.carry_ld && (!persistent || nets * depth * 2 > 8 || H % 8)) return KBS_E_STATE;   // flat carries: persistent kernel only
  const size_t slot_f = r.carry_ld ? size_t(H) : size_t(n) * H;                  // floats between carry slots
  if (resident) {
    // read in place: the h slot the last step wrote, the fp32 c it left
  } else if (nets * depth * 2 <= 8 && H % 8 == 0) {                // ABI carry: h -> SB (parity 0), c -> FB; one launch
    CarryJobs J{};
    J.ld_rm = r.carry_ld ? r.carry_ld : H;
    J.status = h->persist_status;
    int j = 0;
    for (int k = 0; k < nets; ++k)
      for (int l = 0; l < depth; ++l) {
        char* h_dst = hsb[k] + sbb * (hstep * l);
        float* c_dst = r.save ? r.c_hist[k] + fbf * (hstep * l) : fb[k] + fbf * (2 * l);
        if (!r.carry[k]) {                                     // get_initial_model_carry: zeros
          KBS_CUDA_TRY(cudaMemsetAsync(h_dst, 0, sbb, st));
          KBS_CUDA_TRY(cudaMemsetAsync(c_dst, 0, fbf * sizeof(float), st));
          continue;
        }
        J.rm[j] = r.carry[k] + (size_t(l) * 2 + 0) * slot_f; J.blk[j] = h_dst; J.mode[j++] = 0;
        J.rm[j] = r.carry[k] + (size_t(l) * 2 + 1) * slot_f; J.blk[j] = c_dst; J.mode[j++] = 1;
      }
    if (j) carry_convert(h, J, j, n, np, H, st);
  } else {
    for (int k = 0; k < nets; ++k)
      for (int l = 0; l < depth; ++l) {
        pack_rows(h, r.carry[k] + (size_t(l) * 2 + 0) * size_t(n) * H, H, hsb[k] + sbb * (2 * l), n, np, H, st);
        fb_convert(h, r.carry[k] + (size_t(l) * 2 + 1) * size_t(n) * H, fb[k] + fbf * (2 * l), n, np, H, 1, st);
      }
  }
  const int panels = int(np / kPanelRows), tiles = H / kUnitsPerTileP;
  if (persistent) {
    // ---- persistent recurrence: one cooperative launch for all T steps (rollout_persist_kernel) ----
    // Phase A produced on the aux stream in chunks (KBS_ROLLOUT_CHUNKS > 1): this kernel reads the operands of ALL T
    // steps, so every chunk must have landed before it starts (the per-step loop below waits chunk by chunk instead).
    if (r.chunk_len > 0)
      for (int64_t c = 0; c * r.chunk_len < r.T; ++c) KBS_CUDA_TRY(cudaStreamWaitEvent(st, r.chunk_events[c], 0));
    PArgs a{};
    for (int k = 0; k < nets; ++k) {
      PNet& N = a.net[k];
      N.x_sb_all = reinterpret_cast<const char*>(r.x_sb_all[k]);
      N.kb_x0 = r.x_is_obs[k] ? fused_kp(h, k) / kbs_block_k(kind) : H / kbs_block_k(kind);
      N.x0_stride = r.x_is_obs[k] ? kbs_sb_bytes_kind(kind, np, fused_kp(h, k)) : sbb;
      N.hsb = hsb[k]; N.xmid = xmid[k]; N.fb = fb[k]; N.flags = flags[k];
      N.c_hist = r.save ? r.c_hist[k] : nullptr; N.save_g = r.save ? r.save_g[k] : nullptr;
      for (int l = 0; l < depth; ++l) { N.w_sb[l] = layer_w_p(h, k, l); N.bias_t[l] = layer_bias_p(h, k, l); }
      if (r.x_is_obs[k]) { N.w_sb[0] = fused_w(h, k); N.bias_t[0] = fused_bias(h, k); }
      N.w_head = head_w(h, k); N.bias_head = head_bias(h, k);
      KBS_CUDA_TRY(cudaMemsetAsync(flags[k], 0, size_t(depth + 1) * panels * sizeof(unsigned int), st));
    }
    a.nets = nets; a.depth = depth; a.H = H; a.panels = panels; a.tiles = tiles;
    a.n = n; a.ld = ld; a.T = r.T; a.sbb = sbb;
    {
      // panel groups (p_decode).  MEASURED (4 096 envs x 100 steps, profiles/r02_persist_groups.md): grouping trades L2
      // residency for items in flight, and the kernel needs the items: 8 / 11 / 16 / 17 panels per group = 6.82 / 5.90 / 5.25 /
      // 4.74 ms against 4.69 ms ungrouped (with ~2 items per CTA and slot the wavefront becomes dependency-latency-bound).
      // The DRAM traffic of the ungrouped order (9 GB per launch) is not what bounds the kernel.  Default: one group;
      // KBS_PERSIST_GROUP = panels per group for experiments.
      int gp = panels;
      const char* e = getenv("KBS_PERSIST_GROUP");
      if (e) { const int v = atoi(e); gp = (v <= 0 || v > panels) ? panels : v; }
      a.gpanels = gp;
    }
    a.done = r.done;
    a.arm_cmd = r.actor_obs + size_t(55) * ld;
    a.lpf = r.lpf; a.eps = r.eps_action;
    a.q = r.qpos ? r.qpos + size_t(7) * ld : nullptr;
    a.qd = r.qvel ? r.qvel + size_t(6) * ld : nullptr;
    a.ep = r.ep;
    a.action = r.action; a.log_prob = r.log_prob; a.ctrl = (r.ctrl && r.qpos && r.qvel) ? r.ctrl : nullptr; a.value = r.value;
    a.action_in = r.action_in; a.entropy = r.entropy; a.std = r.action_std; a.mean = r.mean;
    a.sraw = r.save ? r.sraw : nullptr; a.hist = r.save ? 1 : 0;
    a.status = h->persist_status;
    a.hsb_slot = r.res_hsb_slot;
    { const char* e = getenv("KBS_PERSIST_DBG"); a.dbg = e ? atoi(e) : 0; }
    a.trace = h->trace_buf;
    cudaLaunchConfig_t cfg{};
    const int64_t per_slot = int64_t(nets) * a.gpanels * (depth * tiles + 1);
    cfg.gridDim = dim3(unsigned(per_slot < h->num_sms ? per_slot : h->num_sms));
    { const char* e = getenv("KBS_PERSIST_GRID"); if (e && atoi(e) > 0 && atoi(e) < int(cfg.gridDim.x)) cfg.gridDim.x = unsigned(atoi(e)); }   // profiling only
    cfg.blockDim = dim3(kThreadsP);
    cfg.dynamicSmemBytes = kPSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;      // every CTA must be resident: they wait on each other's counters
    at[0].val.cooperative = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaError_t le = cudaSuccess;
    if (r.save)
      KBS_LAUNCH(h, KBS_K_ROLLOUT_TC, st, (le = cudaLaunchKernelEx(&cfg, rollout_persist_kernel<KBS_KIND_F16, true>, h->p, a)));
    else if (kind == KBS_KIND_TF32)
      KBS_LAUNCH(h, KBS_K_ROLLOUT_TC, st, (le = cudaLaunchKernelEx(&cfg, rollout_persist_kernel<KBS_KIND_TF32, false>, h->p, a)));
    else
      KBS_LAUNCH(h, KBS_K_ROLLOUT_TC, st, (le = cudaLaunchKernelEx(&cfg, rollout_persist_kernel<KBS_KIND_F16, false>, h->p, a)));
    KBS_CUDA_TRY(le);
    { const int rc0 = kbs_status_publish(h, st); if (rc0) return rc0; }
    if (r.save || resident) { KBS_LAUNCH_CHECK(); return KBS_OK; }   // the update does not need the final carries; the
                                                                      // online step leaves them in its state
    if (nets * depth * 2 <= 8 && H % 8 == 0) {                       // FB state -> ABI carry; one launch
      CarryJobs J{};
      J.ld_rm = r.carry_ld ? r.carry_ld : H;
      J.status = nullptr;
      int j = 0;
      for (int k = 0; k < nets; ++k) {
        float* dst = (r.carry_ld && r.carry_out[k]) ? r.carry_out[k] : r.carry[k];
        for (int l = 0; l < depth; ++l) {
          J.rm[j] = dst + (size_t(l) * 2 + 1) * slot_f; J.blk[j] = fb[k] + fbf * (2 * l); J.mode[j++] = 2;
          J.rm[j] = dst + (size_t(l) * 2 + 0) * slot_f; J.blk[j] = fb[k] + fbf * (2 * l + 1); J.mode[j++] = 2;
        }
      }
      carry_convert(h, J, j, n, np, H, st);
    } else {
      for (int k = 0; k < nets; ++k)
        for (int l = 0; l < depth; ++l) {
          fb_convert(h, r.carry[k] + (size_t(l) * 2 + 1) * size_t(n) * H, fb[k] + fbf * (2 * l), n, np, H, 0, st);
          fb_convert(h, r.carry[k] + (size_t(l) * 2 + 0) * size_t(n) * H, fb[k] + fbf * (2 * l + 1), n, np, H, 0, st);
        }
    }
    KBS_LAUNCH_CHECK();
    return KBS_OK;
  }
  // The head of step t (out-projection, sampling, log-prob, torque, value) feeds nothing back into the recurrence, so
  // it runs on the handle's side stream, forked from and joined back into the caller's stream with events, while the
  // LSTM launches of step t+1 proceed: it lands on the SMs the 256-CTA LSTM grid leaves idle in its second wave.
  { const int rc0 = kbs_side_stream_init(h); if (rc0) return rc0; }
  cudaStream_t side = h->side_stream;
  for (int64_t t = 0; t < r.T; ++t) {
    const int pin = int(t & 1), pout = pin ^ 1;
    const uint8_t* done_t = r.done ? r.done + t * ld : nullptr;
    if (r.chunk_len > 0 && t % r.chunk_len == 0) KBS_CUDA_TRY(cudaStreamWaitEvent(st, r.chunk_events[t / r.chunk_len], 0));
    // top layer of step t overwrites h2rm[pin], last read by the head of step t-2
    if (t >= 2) KBS_CUDA_TRY(cudaStreamWaitEvent(st, h->ev_head[pin], 0));
    for (int l = 0; l < depth; ++l) {
      LayerArgs2 a2{};
      for (int k = 0; k < nets; ++k) {
        LayerArgs& a = a2.net[k];
        fill_lstm_args(h, k, l, a);
        a.x_sb = (l == 0) ? reinterpret_cast<const char*>(r.x_sb_all[k]) + size_t(t) * sbb : xmid[k] + sbb * ((l - 1) & 1);
        a.h_sb_in = hsb[k] + sbb * (2 * l + pin);
        a.h_sb_out = hsb[k] + sbb * (2 * l + pout);
        a.c = fb[k] + fbf * (2 * l);
        a.h_carry = fb[k] + fbf * (2 * l + 1);
        a.x_next_sb = (l + 1 < depth) ? xmid[k] + sbb * (l & 1) : nullptr;
        a.h_next_rm = (l + 1 < depth) ? nullptr : h2rm[k] + size_t(pin) * n * H;
        a.done = done_t;
        a.n = n;
        a.panels = int(np / kPanelRows);
        if (h->trace_buf && t == h->trace_step && l == h->trace_layer) a.trace = h->trace_buf;
      }
      KBS_LAUNCH(h, KBS_K_LSTM_TC, st, (launch_layer(h, kind, a2, st)));
    }
    KBS_CUDA_TRY(cudaEventRecord(h->ev_lstm[pin], st));
    KBS_CUDA_TRY(cudaStreamWaitEvent(side, h->ev_lstm[pin], 0));
    HeadArgs ha{};
    for (int k = 0; k < nets; ++k) {
      ha.h2[k] = h2rm[k] + size_t(pin) * n * H; ha.w_out[k] = h->net[k].w_out; ha.b_out[k] = h->net[k].b_out;
    }
    ha.arm_cmd = r.actor_obs + (size_t(t) * KBS_ACTOR_OBS + 55) * ld;
    ha.lpf = r.lpf;
    ha.eps = r.eps_action ? r.eps_action + size_t(t) * KBS_NUM_JOINTS * ld : nullptr;
    ha.done = done_t;
    ha.q = r.qpos ? r.qpos + (size_t(t) * KBS_NQ + 7) * ld : nullptr;
    ha.qd = r.qvel ? r.qvel + (size_t(t) * KBS_NV + 6) * ld : nullptr;
    ha.ep = r.ep;
    ha.action = r.action ? r.action + size_t(t) * KBS_NUM_JOINTS * ld : nullptr;
    ha.log_prob = r.log_prob ? r.log_prob + size_t(t) * ld : nullptr;
    ha.ctrl = r.ctrl ? r.ctrl + size_t(t) * KBS_NUM_JOINTS * ld : nullptr;
    ha.value = r.value ? r.value + size_t(t) * ld : nullptr;
    ha.action_in = r.action_in ? r.action_in + size_t(t) * KBS_NUM_JOINTS * ld : nullptr;
    ha.entropy = r.entropy ? r.entropy + size_t(t) * ld : nullptr;
    ha.std = r.action_std ? r.action_std + size_t(t) * KBS_NUM_JOINTS * ld : nullptr;
    ha.n = n; ha.ld = ld; ha.H = H;
    static int skip_head = -1;
    if (skip_head < 0) { const char* e = getenv("KBS_SKIP_HEAD"); skip_head = e ? atoi(e) : 0; }   // profiling only
    if (!skip_head)
    KBS_LAUNCH(h, KBS_K_ACTOR_HEAD, side,
               (rollout_head_kernel<<<dim3(unsigned((n + kHeadEnvs - 1) / kHeadEnvs), unsigned(nets)), 128, head_smem, side>>>(
                   h->p, ha)));
    KBS_CUDA_TRY(cudaEventRecord(h->ev_head[pin], side));
  }
  // join: everything the heads wrote (and the lpf state) is visible to the caller's stream
  KBS_CUDA_TRY(cudaStreamWaitEvent(st, h->ev_head[0], 0));
  if (r.T > 1) KBS_CUDA_TRY(cudaStreamWaitEvent(st, h->ev_head[1], 0));
  for (int k = 0; k < nets; ++k)
    for (int l = 0; l < depth; ++l) {                // FB state -> ABI carry
      fb_convert(h, r.carry[k] + (size_t(l) * 2 + 1) * size_t(n) * H, fb[k] + fbf * (2 * l), n, np, H, 0, st);
      fb_convert(h, r.carry[k] + (size_t(l) * 2 + 0) * size_t(n) * H, fb[k] + fbf * (2 * l + 1), n, np, H, 0, st);
    }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// Debug: one LSTM-mode layer launch for both nets on scratch data with per-CTA clock64 stamps.
// trace_out (device) [2 * tiles * panels][8]: start, setup done, first stage landed, MMAs issued, accumulators ready,
// epilogue done, smid, unused.
// Both nets run on zeroed layer-0 buffers of the rollout workspace of net 0.
int kbs_tc_debug_trace(kbs_handle* h, long long* trace_out, const KbsTcRolloutWs& ws, int64_t n, cudaStream_t st) {
  const int H = h->p.hidden_size;
  for (int k = 0; k < 2; ++k)
    if (!h->net[k].packed || !h->net[k].tc_image) return KBS_E_STATE;
  const int64_t np = pad_rows(n);
  const size_t sbb = act_sb_bytes(h, n);
  KBS_CUDA_TRY(cudaMemsetAsync(ws.hsb[0], 0, sbb * 2, st));
  KBS_CUDA_TRY(cudaMemsetAsync(ws.xmid[0], 0, sbb * 2, st));
  KBS_CUDA_TRY(cudaMemsetAsync(ws.fb[0], 0, size_t(np) * H * 4 * 2, st));
  LayerArgs2 a2{};
  for (int k = 0; k < 2; ++k) {
    LayerArgs& a = a2.net[k];
    fill_lstm_args(h, k, 0, a);
    a.x_sb = ws.xmid[0]; a.h_sb_in = ws.hsb[0]; a.h_sb_out = ws.hsb[0] + sbb; a.x_next_sb = ws.xmid[0] + sbb;
    a.c = ws.fb[0]; a.h_carry = ws.fb[0] + size_t(np) * H; a.h_next_rm = nullptr; a.done = nullptr; a.n = n;
    a.trace = trace_out;
    a.panels = int(np / kPanelRows);
  }
  KBS_LAUNCH(h, KBS_K_LSTM_TC, st, (launch_layer(h, tc_kind(h), a2, st)));
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}

// ---- the online step's resident carries (kbs_step_state_*, kbs_rollout_step) -----------------------------------------------
// One net's piece of a step state: hsb [depth][2] x act SB (the h operand; the state's slot word names the one the next step
// reads) and fb [depth][c, h] x np*H (the fp32 cell state, and the fp32 h the last step wrote).
KbsTcStepNet kbs_tc_step_net(KbsScratch& s, const kbs_handle* h, int64_t n) {
  const size_t depth = size_t(h->p.depth), H = size_t(h->p.hidden_size), np = size_t(pad_rows(n));
  KbsTcStepNet w;
  w.hsb = s.take<char>(2 * depth * act_sb_bytes(h, n));
  w.fb = s.take<float>(2 * depth * np * H);
  return w;
}

// ABI carry [depth][2][n][H] <-> one net's resident operands.  to_state: h -> hsb slot 0 (split) and fb h, c -> fb c
// (carry == nullptr: zeros); else fb c / fb h -> the ABI c / h (what kbs_tc_rollout_recurrent writes back after a call).
int kbs_tc_step_carry(kbs_handle* h, float* carry, const KbsTcStepNet& w, int64_t n, bool to_state, cudaStream_t st) {
  const int H = h->p.hidden_size, depth = h->p.depth;
  const int64_t np = pad_rows(n);
  const size_t sbb = act_sb_bytes(h, n), fbf = size_t(np) * H;
  { const int rc0 = kbs_status_init(h); if (rc0) return rc0; }
  if (to_state) {
    KBS_CUDA_TRY(cudaMemsetAsync(w.hsb, 0, 2 * size_t(depth) * sbb, st));
    if (!carry) { KBS_CUDA_TRY(cudaMemsetAsync(w.fb, 0, 2 * size_t(depth) * fbf * sizeof(float), st)); return KBS_OK; }
  }
  CarryJobs J{};
  J.ld_rm = H;
  J.status = to_state ? h->persist_status : nullptr;
  int j = 0;
  for (int l = 0; l < depth; ++l) {
    float* hrm = carry + (size_t(l) * 2 + 0) * size_t(n) * H;
    float* crm = carry + (size_t(l) * 2 + 1) * size_t(n) * H;
    if (to_state) {
      J.rm[j] = hrm; J.blk[j] = w.hsb + sbb * (2 * l); J.mode[j++] = 0;
      J.rm[j] = hrm; J.blk[j] = w.fb + fbf * (2 * l + 1); J.mode[j++] = 1;
      J.rm[j] = crm; J.blk[j] = w.fb + fbf * (2 * l); J.mode[j++] = 1;
    } else {
      J.rm[j] = crm; J.blk[j] = w.fb + fbf * (2 * l); J.mode[j++] = 2;
      J.rm[j] = hrm; J.blk[j] = w.fb + fbf * (2 * l + 1); J.mode[j++] = 2;
    }
    if (j > 5 || l + 1 == depth) {         // at most 8 jobs per launch
      if (const int rc = carry_convert(h, J, j, n, np, H, st)) return rc;
      j = 0;
    }
  }
  KBS_LAUNCH_CHECK();
  return KBS_OK;
}
