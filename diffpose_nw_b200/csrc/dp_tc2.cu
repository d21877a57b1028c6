// Tensor-core engine, second generation ("tcg"): persistent sm_100a kernel, one 128-row tile (7 poses x 17 joints) per
// CTA, all DDIM steps and layers executed without leaving the SM.  Every contraction of the denoiser runs on tcgen05:
//
//   * dense projections (QKV, out-proj, GraphNet fc1/fc2, Chebyshev convolutions) as M=128, N=96, K=16 fp16 MMAs with
//     fp32 accumulators in TMEM; biases ride along as one extra K step against a constant-one slab.  An activation
//     that is only ever the A side of a GEMM never touches shared memory: the epilogue writes it as packed fp16 pairs
//     into tensor memory (TS-form MMA); only B operands (K, V, LN1(x), z, x, h) and Q live in shared memory;
//   * LayerNorm writes the plain normalised row: the gains are folded into the consumer's weights and bias at pack
//     time (for LN1, whose output first goes through L^, the shift enters through a per-joint K slab); the sampler's
//     time embedding enters GC2 as one more bias K step (Chebyshev slab x per-(step, layer) block);
//   * the residual stream X lives in TMEM (96 fp32 columns).  Residual additions are free: the out-projection, the
//     second GraphNet aggregation and the b2 bias accumulate straight into those columns (D += A*B);
//   * the 17x17 graph operators (Chebyshev T1/T2, learnable-adjacency L^).  Joints 0..15: a graph matrix G is stored
//     once as a "tall" K-major operand [256 rows x 16] whose rows 128..144 hold G[:, 0:16] and every other row is zero;
//     the window starting at row 128-18p is the 128x16 matrix that applies G to pose p and nothing to the other poses,
//     and the activations are consumed in place as an MN-major B operand starting at row 18p: one K=16 MMA per pose.
//     Joint 16: the epilogues also drop the joint-16 row of every pose into a compact 16-row side buffer, and one more
//     MMA applies [G[i][16] at (18p+i, p)] to it.  OUT[128 x 96] = G per pose in 8 MMAs and no data movement;
//   * attention: S_h = Q_h K_h^T for the whole tile (N = 128 key rows), softmax on the compute warps straight out of
//     TMEM (each row keeps the 17 columns of its own pose), probabilities written back to TMEM as packed fp16 and used
//     as the A operand of O_h = P_h V_h (V consumed in place as an MN-major operand);
//   * the input (K = 15) and output (N = 15) Chebyshev convolutions with hi/lo fp16 splits of both operands (three
//     MMAs per product), i.e. at fp32-level accuracy.
//
// Warp roles: 8 compute warps (epilogues TMEM -> registers -> fp16 operand in tensor or shared memory, LayerNorm,
// softmax, DDIM update), one producer warp (weights and per-layer parameters L2 -> shared memory with cp.async.bulk + mbarrier
// complete_tx, 4-stage ring of 21.5 KB blocks), one issuer warp (every tcgen05.mma, following a static per-layer
// program).  Compute warps and issuer hand over through two 4-deep event rings, both sides walking the same static
// sequence: "operands ready" = hardware named barriers (bar.arrive by the 256 compute threads, bar.sync by the issuer warp:
// measurably faster to wake than an mbarrier), "accumulator ready" = mbarriers armed by tcgen05.commit.
//
// Reference semantics: see the list at the top of dp_simt.cu (same functions, same file:line).
#include <cuda_fp16.h>
#include <cmath>
#include "dp_internal.h"
#include "dp_sm100.cuh"
#include "dp_metrics_dev.cuh"
#include "dp_tc_layout.cuh"

namespace dp {

namespace {

using namespace sm100;
using namespace tc;

constexpr int PS = 18;               // tile rows per pose: 17 joints + 1 pad row, so every pose starts on an even row and the
                                     // rows of a warp (32) always begin 0, 14, 10 or 6 rows into a pose -> one softmax code path
constexpr int TR = TP * PS;          // 126 rows carry poses
constexpr int NSTAGE = 4;
constexpr int T_ROWS = 256;                         // tall graph operand: rows 128..144 hold the matrix
constexpr int T_LBO = T_ROWS * 16 + 16;             // 4112
constexpr int TALL_BYTES = 2 * T_LBO;               // 8224: K = joints 0..15 (joint 16 goes through the side operands below)
constexpr int SIDE_LBO = 256;                       // side buffer [16 rows x 96 ch]: 8-channel groups 256 B apart
constexpr int SIDE_BYTES = 12 * SIDE_LBO;           // 3072
constexpr int A16_BYTES = A_LBO;                    // joint-16 operand of a graph matrix: one chunk column [128 rows x 8]
constexpr int OUT_LBO = 256;                        // output-convolution block: N = 16 rows, K-adjacent core matrices 256 B apart
constexpr int LP_LHAT_BYTES = 4 * NP * 16;          // per-layer parameters: L^ as fp16 [4 chunk columns][17 rows][8]
constexpr int LP_JS_BYTES = PS * 16;                //   + the joint slab rows (1, 1, r_hi, r_hi, r_lo, 0, 0, 0), r = row sums of L^
constexpr int LP_BYTES = LP_LHAT_BYTES + LP_JS_BYTES;   // 1376, copied from the packed parameter array
constexpr int LP_TAU_BYTES = H * 16;                // time-embedding block of one (step, layer): [96 outputs][8] fp16 (tc2_tau_kernel)
constexpr int PAR_BYTES = LP_BYTES + LP_TAU_BYTES;  // 2912 per stage
constexpr int JS_BYTES = TM * 16;                   // joint slab: one chunk column [128 rows x 8]
constexpr int kComputeThreads = 256;
constexpr int kProducerWarp = 8, kIssuerWarp = 9;
constexpr int kThreads = kComputeThreads + 64;
constexpr int NEV = 4;               // depth of the two hand-over rings ("operands ready", "accumulator ready")
constexpr uint32_t COL_X = 0;        // residual stream
constexpr uint32_t COL_ACC = 96;     // GEMM accumulators (up to 288 columns)
constexpr uint32_t COL_S0 = 96;      // attention: scores of the even head of a pair [128 x 128]; its probabilities
constexpr uint32_t COL_S1 = 224;     //   overwrite the first 64 columns as packed fp16 (A operand of P V); odd head
constexpr uint32_t COL_O = 352;      // attention output [128 x 96] (+8 scratch columns); before that the V accumulator
constexpr uint32_t COL_ACC2 = 288;   // third accumulator group: GEMMs that start while groups 0/1 are still being read
constexpr uint32_t COL_TA0 = 448;    // fp16 A operands kept in tensor memory (48 columns = 96 channels each): operands that
constexpr uint32_t COL_TA1 = 384;    //   only ever feed a GEMM as A skip shared memory (its bandwidth bounds the epilogues)

// shared memory map (bytes)
constexpr int OFF_A = 0;                                   // three fp16 operand blocks; fp32 scratch [128][17] aliases block 0
constexpr int OFF_SIDE = OFF_A + 3 * ABLK_BYTES;           // per operand block: the joint-16 rows of the 7 poses, compacted (rows 7..15 zero)
constexpr int OFF_A16 = OFF_SIDE + 3 * SIDE_BYTES;         // per graph matrix (T1, T2, L^): element (18p+i, p) = G[i][16]
constexpr int OFF_MK = OFF_A16 + 3 * A16_BYTES;            // key-mask chunk column: element (key row, 0) = -65504 for a masked joint, else 0
constexpr int OFF_CS = OFF_MK + JS_BYTES;                  // Chebyshev slab: rows (1, 1, p1_hi, p1_hi, p1_lo, p2_hi, p2_hi, p2_lo), p_k = row sums of T_k
constexpr int OFF_JS = OFF_CS + JS_BYTES;                  // joint slab of the current layer (fc1 bias + the LayerNorm shift seen through L^)
constexpr int OFF_ONES = OFF_JS + JS_BYTES;                // constant-one K slab (bias rides in the MMA) + a zero chunk column
constexpr int OFF_TALL = OFF_ONES + ONES_BYTES;            // tall T1, T2, L^
constexpr int OFF_W = (OFF_TALL + 3 * TALL_BYTES + 127) / 128 * 128;
constexpr int OFF_XT = OFF_W + NSTAGE * WBLK_BYTES;        // x_t [128][XS] fp32
constexpr int XS = 9;                                      // x_t row stride in floats: odd, so row-per-lane access is conflict free
constexpr int OFF_PAR = al16(OFF_XT + TM * XS * 4);        // per-layer parameters, 2 stages
constexpr int OFF_TEP = OFF_PAR + 2 * PAR_BYTES;           // per-pose temb [7][96] fp32 (forward mode: per-sample timesteps)
constexpr int OFF_T12 = OFF_TEP + TP * H * 4;              // (T1, T2)[17][17] as float2, fp32: the 5-wide input / output convolutions
constexpr int OFF_STAT = al16(OFF_T12 + NP * NP * 8);      // LayerNorm partial statistics [2][128] float2
constexpr int OFF_MASK = OFF_STAT + 2 * TM * 8;            // key mask [32]
constexpr int OFF_BAR = OFF_MASK + 128;                    // mbarriers: full[4], empty[4], pfull[2], pempty[2], (unused)[4], acc[4]
constexpr int OFF_TMEM = OFF_BAR + 192;
constexpr int OFF_EV = OFF_TMEM + 16;                      // fused evaluation: xyz of the tile's finished poses [7][17][3] fp32, then their targets
constexpr int EV_FLOATS = TP * NP * 3;
constexpr int SMEM_BYTES = OFF_EV + 2 * EV_FLOATS * 4;
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
static_assert(OFF_W % 128 == 0 && OFF_ONES % 16 == 0 && OFF_JS % 16 == 0 && OFF_CS % 16 == 0 && OFF_MK % 16 == 0 && OFF_TALL % 16 == 0 && OFF_SIDE % 16 == 0 && OFF_A16 % 16 == 0 && OFF_BAR % 16 == 0 && OFF_T12 % 16 == 0 && OFF_XT % 16 == 0 &&
              OFF_STAT % 16 == 0 && OFF_PAR % 16 == 0 && OFF_TEP % 16 == 0 && PAR_BYTES % 16 == 0 && LP_BYTES % 16 == 0, "alignment");

__device__ __forceinline__ void bar_compute() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// byte offset of the 16-byte chunk holding elements (row, 8*kc .. 8*kc+7) inside an fp16 operand block
__device__ __forceinline__ uint32_t a_chunk(int row, int kc) { return kc * A_LBO + row * 16; }

#define DP_PHASE_FN __forceinline__

struct Tc2Args {
  const Weights* w;          // fp32 blob (T1/T2 for the gathers, output bias)
  const uint8_t* wpack;      // fp16 weight blocks [n_layer][14][21504 B]
  const uint8_t* ioblocks;   // [2][21504 B]: input-convolution block, output-convolution block
  const uint8_t* lparams;    // [n_layer][LP_BYTES]
  int n_layer;
  int c_in, c_out;           // coordinate widths (<= 5): uvxyz -> uvxyz for GCNdiff, uv -> xyz for GCNpose
  int forward_only;          // 1: a single denoiser/lifter forward, the output is eps (dp_forward); 0: the DDIM loop
  int has_temb;              // GCNpose has no time embedding
  const float* x_in;
  int x_is_repeated;
  float* out;
  long n_rows, n_pose;
  int n_hyp;
  int mean_over_hyp;         // sampler: out = mean over the hypotheses of a pose, [n_pose][17][c] (runners/diffpose_frame.py:382).
                             // Rows are then walked pose-major (row g = pose g / n_hyp, hypothesis g % n_hyp) and every CTA owns a
                             // contiguous range of POSES, so all hypotheses of a pose pass through the same CTA in order
  int n_steps;
  const float* temb;         // [n_rows][n_layer][96]: per-sample time embeddings of a forward call (forward_only)
  const uint8_t* tau;        // [n_steps][n_layer][LP_TAU_BYTES]: the sampler's time embedding as a bias block of GC2 (tc2_tau)
  const float* noise;
  const unsigned char* mask;
  const dp_step* steps_dev;
  const float* gt;           // fused evaluation (dp_sample with targets_xyz): targets [n_pose][17][3]; every finished pose (after the hypothesis
  double* sums;              //   mean, if any) adds its MPJPE / P-MPJPE to sums[0..1] and 1 to sums[2] (common/loss.py, dp_metrics)
  long long* trace;          // optional diagnostic: CTA 0 records clock64() at every hand-over (see dp_set_trace)
  int trace_cap;
  NoiseKey key;              // key.on: z from the keyed stream instead of noise (NULL); runs the KEYED instantiation
};

// ------------------------------------------------------------------------------------------------ compute-warp pieces
struct Ctx {
  long long* trace;     // non-null on one thread of CTA 0 only
  int trace_n, trace_cap;
  uint8_t* smem;
  uint32_t tmem_lane;   // tmem base + (lane quarter << 16)
  uint32_t rdy, acc;    // first mbarrier of each ring
  uint32_t rdy_i, acc_i, acc_phase;   // ring positions (events are produced and consumed in one global program order)
  int row, hh, lane;
};

// stamps are (clock64() << 1) | kind, kind 0 = about to signal "operands ready", 1 = "accumulator ready" observed
template <bool TRACE>
__device__ __forceinline__ void trace_mark(Ctx& c, int kind) {
  if (TRACE && c.trace != nullptr && c.trace_n < c.trace_cap) c.trace[c.trace_n++] = (clock64() << 1) | kind;
}
// "my operands are in shared memory / my TMEM accesses are done": one arrival per compute warp
// SMEM = false: the phase wrote tensor memory only (softmax), no shared-memory operand needs publishing to the async proxy
template <bool TRACE, bool SMEM = true>
__device__ __forceinline__ void signal_ready_t(Ctx& c) {
  trace_mark<TRACE>(c, 0);
  if (SMEM) fence_async_smem();
  tc_fence_before();
  // hardware named barrier 2 + ring slot: 256 compute threads arrive, the issuer warp (32 threads) waits
  asm volatile("bar.arrive %0, 288;" ::"r"(2 + c.rdy_i) : "memory");
  c.rdy_i = (c.rdy_i + 1) & (NEV - 1);
}
template <bool TRACE>
__device__ __forceinline__ void wait_acc_t(Ctx& c) {
  mbar_wait(c.acc + 8 * c.acc_i, c.acc_phase);
  c.acc_i = (c.acc_i + 1) & (NEV - 1);
  if (c.acc_i == 0) c.acc_phase ^= 1;
  tc_fence_after();
  trace_mark<TRACE>(c, 1);
}

// One epilogue group: 48 accumulator columns of this thread's lane: TMEM -> registers -> (row scale) -> clamp (lo = 0: relu,
// -inf: none) -> (+ temb) -> fp16 -> six 16-byte chunks of an operand block.  Inlined on purpose: measured on this part, a
// call or a taken branch to code that is not next in line costs an instruction-cache miss (100-250 cycles), and a stack
// lives in L2 because the shared-memory carve-out leaves next to no L1.
// side: for the joint-16 row of a pose, where its chunks go in the block's side buffer (nullptr for every other row and
// for blocks that are never aggregated)
__device__ DP_PHASE_FN void epi_run(uint8_t* dst, uint32_t col, float lo, const float* temb, float scale = 1.0f, bool scaled = false,
                                    uint8_t* side = nullptr, bool relu_in_cvt = false, bool b_only = false, uint32_t tdst = 0) {
  float v[48];
  tmem_ld48(col, v);
  if (scaled) {              // row scale of an integerised graph matrix
#pragma unroll
    for (int i = 0; i < 48; i += 2) mul2(v[i], v[i + 1], v[i], v[i + 1], scale, scale);
  }
  if (lo == 0.f && !relu_in_cvt) {
#pragma unroll
    for (int i = 0; i < 48; ++i) v[i] = fmaxf(v[i], 0.f);
  }
  if (temb != nullptr) {
#pragma unroll
    for (int i = 0; i < 48; i += 4) {
      const float4 t = *reinterpret_cast<const float4*>(temb + i);
      add2(v[i], v[i + 1], v[i], v[i + 1], t.x, t.y);
      add2(v[i + 2], v[i + 3], v[i + 2], v[i + 3], t.z, t.w);
    }
  }
  if (b_only) {
    // the shared-memory copy is only ever read as a B operand (per-pose windows over joints 0..15 + the side buffer): a
    // joint-16 row goes to the side buffer alone -- one store per chunk instead of two (the phase is bound by shared-memory
    // store issue).  tdst: the same operand is also the A side of a GEMM -> second copy in tensor memory.
    uint8_t* const d = side != nullptr ? side : dst;
    const int stride = side != nullptr ? SIDE_LBO : A_LBO;
    uint32_t pk[24];
#pragma unroll
    for (int i = 0; i < 24; ++i) pk[i] = relu_in_cvt ? pack2_relu(v[2 * i], v[2 * i + 1]) : pack2(v[2 * i], v[2 * i + 1]);
#pragma unroll
    for (int q = 0; q < 6; ++q) *reinterpret_cast<uint4*>(d + q * stride) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
    if (tdst != 0) tmem_st24_u32(tdst, pk);
    return;
  }
#pragma unroll
  for (int q = 0; q < 6; ++q) {
    const uint4 u = relu_in_cvt ? pack8_relu(v + 8 * q) : pack8(v + 8 * q);
    *reinterpret_cast<uint4*>(dst + q * A_LBO) = u;
    if (side != nullptr) *reinterpret_cast<uint4*>(side + q * SIDE_LBO) = u;
  }
}

// The same for an operand that is only ever the A side of a GEMM: fp16 pairs into 24 tensor-memory columns (TS-form MMA).
// No shared-memory store, no generic->async proxy fence.
__device__ DP_PHASE_FN void epi_tmem(uint32_t dcol, uint32_t col, float scale, bool scaled, bool relu) {
  float v[48];
  tmem_ld48(col, v);
  if (scaled) {
#pragma unroll
    for (int i = 0; i < 48; i += 2) mul2(v[i], v[i + 1], v[i], v[i + 1], scale, scale);
  }
  uint32_t pk[24];
#pragma unroll
  for (int i = 0; i < 24; ++i) pk[i] = relu ? pack2_relu(v[2 * i], v[2 * i + 1]) : pack2(v[2 * i], v[2 * i + 1]);
  tmem_st24_u32(dcol, pk);
}

// LayerNorm phase: residual row (48 of its 96 channels per thread) from TMEM -> LayerNorm -> fp16 operand block
// With acol != 0 the closing residual of the previous layer's Chebyshev block is applied first: x += relu(acc), written
// back to TMEM (later MMAs accumulate onto it).
__device__ DP_PHASE_FN void ln_run(uint8_t* smem, uint32_t xcol, uint32_t acol, int row, int hh, uint32_t dst_off, uint8_t* side = nullptr,
                                   uint32_t tdst = 0) {
  float v[48];
  if (acol != 0) {
    float u[48];
    tmem_ld16_async(acol, u);
    tmem_ld16_async(acol + 16, u + 16);
    tmem_ld16_async(acol + 32, u + 32);
    tmem_ld48(xcol, v);
    launder<48>(u);
#pragma unroll
    for (int i = 0; i < 48; i += 2) add2(v[i], v[i + 1], v[i], v[i + 1], fmaxf(u[i], 0.f), fmaxf(u[i + 1], 0.f));
    tmem_st16(xcol, v);            // completion is awaited at the end of the phase, behind the LayerNorm arithmetic
    tmem_st16(xcol + 16, v + 16);
    tmem_st16(xcol + 32, v + 32);
  } else {
    tmem_ld48(xcol, v);
  }
  // one pass: sum and sum of squares of this thread's 48 channels (fp32; the row has 96 values of comparable size, so the
  // cancellation in sum(x^2) - n mean^2 costs a few ulp of the variance -- far below the fp16 rounding of the output)
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
#pragma unroll
  for (int i = 0; i < 48; i += 4) {
    add2(s0, s1, s0, s1, v[i], v[i + 1]);
    add2(s2, s3, s2, s3, v[i + 2], v[i + 3]);
    fma2(q0, q1, v[i], v[i + 1], v[i], v[i + 1], q0, q1);
    fma2(q2, q3, v[i + 2], v[i + 3], v[i + 2], v[i + 3], q2, q3);
  }
  const float sh = (s0 + s1) + (s2 + s3), qh = (q0 + q1) + (q2 + q3);
  float2* stat = reinterpret_cast<float2*>(smem + OFF_STAT);
  stat[hh * TM + row] = make_float2(sh, qh);
  bar_compute();
  const float2 o = stat[(hh ^ 1) * TM + row];
  const float mean = (sh + o.x) * (1.0f / (float)H);
  const float m2 = fmaxf(fmaf(-(sh + o.x), mean, qh + o.y), 0.f);          // sum (x - mean)^2
  float sd;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sd) : "f"(m2 * (1.0f / (float)(H - 1))));
  const float inv = rcp_fast(sd + 1e-6f);
  // (x - mean) / (std + eps): the gains a_2, b_2 are folded into the weights and biases of the GEMMs that consume this
  // operand (tc2_pack), so nothing is read from shared memory here -- the phase is bound by shared-memory bandwidth
  const float shift = -mean * inv;
#pragma unroll
  for (int i = 0; i < 48; i += 2) fma2(v[i], v[i + 1], v[i], v[i + 1], inv, inv, shift, shift);
  if (tdst != 0) {     // the operand only feeds GEMMs as A: keep it in tensor memory (the wait inside covers the residual store too)
    uint32_t pk[24];
#pragma unroll
    for (int i = 0; i < 24; ++i) pk[i] = pack2(v[2 * i], v[2 * i + 1]);
    tmem_st24_u32(tdst, pk);
    return;
  }
  // shared-memory destination: a B operand (LN1 -> L^ aggregation); joint-16 rows go to the side buffer only (see epi_run)
  uint8_t* const d = side != nullptr ? side : smem + dst_off;
  const int stride = side != nullptr ? SIDE_LBO : A_LBO;
#pragma unroll
  for (int q = 0; q < 6; ++q) *reinterpret_cast<uint4*>(d + q * stride) = pack8(v + 8 * q);
  if (acol != 0) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// Softmax of one head's scores for this thread's row (GraFormer.py:104-111).  The scores of the whole tile sit in
// TMEM as S[128 x 128] (row = query, column = key row of the tile); a row only needs the 17 columns of its own pose.
// Poses start every PS = 18 rows, so the 32 rows of a warp span at most three poses beginning at pose p0 = 32*wq/18:
// the warp loads the 64 columns from 18*p0 and every lane picks its pose's 17 with selects at compile-time offsets.
// The probabilities go back to TMEM as fp16 pairs, zero outside the pose (block-diagonal P[128 x 128]), and feed the
// P V product as its A operand.  One code path for all warps.
// The key mask (GraFormer.py:107-108, masked_fill(mask == 0, -1e9)) is not applied here: the second K step of the score
// MMA multiplies a column of ones on the Q side with the mask chunk column on the K side, so a masked key arrives with
// -65504 added to its score and its probability flushes to exactly 0 like the reference's.  k2 = log2(e)/sqrt(d_k), or 0
// when every key is masked (the reference's softmax over seventeen equal -1e9 is uniform).
__device__ DP_PHASE_FN void softmax_run(uint32_t region, int row, float k2) {
  const int p0 = ((row & ~31) * 57) >> 10;          // (32*wq) / 18 for wq = 0..3  ->  0, 1, 3, 5
  const int p = min(row / PS, TP - 1);              // pad rows 126, 127 ride along as pose 6
  const int q = p - p0;
  float v[64];
#pragma unroll
  for (int i = 0; i < 64; i += 16) tmem_ld16_async(region + PS * p0 + i, v + i);
  tmem_ld_wait();
  launder<64>(v);
  float sc[NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const float t = q == 0 ? v[j] : v[PS + j];
    sc[j] = q == 2 ? v[2 * PS + j] : t;
  }
  float m0 = fmaxf(sc[0], sc[1]), m1 = fmaxf(sc[2], sc[3]), m2 = fmaxf(sc[4], sc[5]), m3 = fmaxf(sc[6], sc[7]);
  m0 = fmaxf(m0, fmaxf(sc[8], sc[9])); m1 = fmaxf(m1, fmaxf(sc[10], sc[11])); m2 = fmaxf(m2, fmaxf(sc[12], sc[13])); m3 = fmaxf(m3, fmaxf(sc[14], sc[15]));
  const float mk = fmaxf(fmaxf(m0, m1), fmaxf(fmaxf(m2, m3), sc[16])) * k2;
  const float nmk = -mk;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
  for (int j = 0; j < 16; j += 4) {
    fma2(sc[j], sc[j + 1], sc[j], sc[j + 1], k2, k2, nmk, nmk);
    fma2(sc[j + 2], sc[j + 3], sc[j + 2], sc[j + 3], k2, k2, nmk, nmk);
    sc[j] = ex2(sc[j]); sc[j + 1] = ex2(sc[j + 1]); sc[j + 2] = ex2(sc[j + 2]); sc[j + 3] = ex2(sc[j + 3]);
    add2(s0, s1, s0, s1, sc[j], sc[j + 1]);
    add2(s2, s3, s2, s3, sc[j + 2], sc[j + 3]);
  }
  sc[16] = ex2(fmaf(sc[16], k2, nmk));
  const float inv = rcp_fast((s0 + s1) + (s2 + s3) + sc[16]);
#pragma unroll
  for (int j = 0; j < 16; j += 2) mul2(sc[j], sc[j + 1], sc[j], sc[j + 1], inv, inv);
  sc[16] *= inv;
  // P[128 x 128] as the A operand of P V, 64 packed columns: slot s < 7 (columns 8s..8s+7) = joints 0..15 of pose s,
  // slot 7 = joint 16 of poses 0..6 (K position = pose).  A row is non-zero only in its own pose's slot and position, so
  // every pose sees the same summation order in P V, whatever its place in the tile.
  uint32_t w[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) w[i] = pack2(sc[2 * i], sc[2 * i + 1]);
  const uint32_t w16 = (p & 1) ? (pack2(0.f, sc[16])) : (pack2(sc[16], 0.f));
#pragma unroll
  for (int piece = 0; piece < 4; ++piece) {
    uint32_t pk[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int col = 16 * piece + i, slot = col >> 3;
      if (slot < TP) pk[i] = (p == slot) ? w[col & 7] : 0u;
      else pk[i] = ((col & 7) < 4 && (p >> 1) == (col & 7)) ? w16 : 0u;
    }
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(region + 16 * piece),
        "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]), "r"(pk[4]), "r"(pk[5]), "r"(pk[6]), "r"(pk[7]), "r"(pk[8]), "r"(pk[9]),
        "r"(pk[10]), "r"(pk[11]), "r"(pk[12]), "r"(pk[13]), "r"(pk[14]), "r"(pk[15]) : "memory");
  }
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// element (tall row, k) of tall graph operand `which`
__device__ __forceinline__ __half* tall_elem(uint8_t* smem, int which, int trow, int k) {
  return reinterpret_cast<__half*>(smem + OFF_TALL + which * TALL_BYTES + (k >> 3) * T_LBO + trow * 16 + (k & 7) * 2);
}

// ------------------------------------------------------------------------------------------------ the kernel
// TRACE = true compiles the clock64() stamps of dp_set_trace in; the production instantiation carries none of it.
// EVAL = true compiles the fused evaluation tail (dp_sample with targets_xyz) in: ~3 000 instructions that the plain sampler instantiation
// does not carry either.
// KEYED = true draws z from the keyed stream (a.key, dp_philox.cuh) instead of reading a.noise; the unkeyed instantiations
// carry none of the Philox code, so their schedule is the one they had before keyed noise existed.
template <bool TRACE, bool EVAL, bool KEYED>
__global__ void __launch_bounds__(kThreads, 1) tc2_kernel(Tc2Args a, StepsArg inl) {
  auto signal_ready = [](Ctx& c) { signal_ready_t<TRACE>(c); };
  auto signal_ready_tmem = [](Ctx& c) { signal_ready_t<TRACE, false>(c); };
  auto wait_acc = [](Ctx& c) { wait_acc_t<TRACE>(c); };
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  float* xt = reinterpret_cast<float*>(smem + OFF_XT);
  float* maskf = reinterpret_cast<float*>(smem + OFF_MASK);
  float2* t12 = reinterpret_cast<float2*>(smem + OFF_T12);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_TMEM);
  // diagnostic stamps of CTA 0 (last four slots of the trace buffer): kernel entry, setup done, tiles done
  long long* const ktrace = (TRACE && blockIdx.x == 0 && tid == 0 && a.trace != nullptr && a.trace_cap >= 8) ? a.trace + a.trace_cap - 4 : nullptr;
  if (ktrace) ktrace[0] = clock64();

  const uint32_t full0 = sbase + OFF_BAR, empty0 = sbase + OFF_BAR + 32, pfull0 = sbase + OFF_BAR + 64, pempty0 = sbase + OFF_BAR + 80,
                 rdy = sbase + OFF_BAR + 96, accb = sbase + OFF_BAR + 128;

  // ---------------------------------------------------------------- one-time setup
  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(pfull0 + 8 * s, 1); mbar_init(pempty0 + 8 * s, kComputeThreads / 32); }
    for (int s = 0; s < NEV; ++s) { mbar_init(rdy + 8 * s, kComputeThreads / 32); mbar_init(accb + 8 * s, 1); }
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(sbase + OFF_TMEM, TMEM_COLS);
  // operand blocks, ones slab and tall operands start as zeros (every byte an MMA can touch must be a finite fp16)
  for (int i = tid; i < (OFF_W - OFF_A) / 16; i += kThreads) reinterpret_cast<uint4*>(smem + OFF_A)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  // constant-one K slab: element (row, 0) = (row, 1) = 1
  for (int i = tid; i < TM; i += kThreads) *reinterpret_cast<uint32_t*>(smem + OFF_ONES + a_chunk(i, 0)) = pack2(1.0f, 1.0f);
  // Programmatic dependent launch: this grid may have started while the previous kernel of the stream was still
  // draining.  Nothing above touches global memory; wait here for the previous kernel's results (x_in may be its
  // output, the temb table and the packed weights are written by earlier kernels of the same stream).
  asm volatile("griddepcontrol.wait;" ::: "memory");
  // Tile schedule of this CTA.  Default: tiles blockIdx.x, blockIdx.x + gridDim.x, ... of the hypothesis-major row list.
  // mean_over_hyp: a contiguous, balanced range of poses; its n_hyp rows per pose form this CTA's own tile list.
  long row_lo = 0, row_hi = 0;
  int my_tiles;
  if (a.mean_over_hyp) {
    const long base = a.n_pose / gridDim.x, rem = a.n_pose % gridDim.x;
    const long p_lo = blockIdx.x * base + min((long)blockIdx.x, rem);
    row_lo = p_lo * a.n_hyp;
    row_hi = row_lo + (base + ((long)blockIdx.x < rem ? 1 : 0)) * a.n_hyp;
    my_tiles = (int)((row_hi - row_lo + TP - 1) / TP);
  } else {
    const int n_tiles = (int)((a.n_rows + TP - 1) / TP);   // the host refuses more than INT_MAX tiles
    my_tiles = (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  }
  // The poses of this CTA's first tile are requested from global memory right here, before the one-time set-up loads below
  // and its barrier: their DRAM / L2 latency (the bench rotates inputs through a pool larger than L2) then overlaps the
  // set-up instead of sitting between it and the first panel.  One compute thread holds up to three values.
  constexpr int kPre = (TP * NP * 5 + kComputeThreads - 1) / kComputeThreads;
  float xpre[kPre];
  if (warp < kProducerWarp && my_tiles > 0) {
    const long g0 = a.mean_over_hyp ? row_lo : (long)blockIdx.x * TP;
    const int npose0 = (int)min((long)TP, (a.mean_over_hyp ? row_hi : a.n_rows) - g0);
    const int per = NP * a.c_in, nin0 = npose0 * per;
#pragma unroll
    for (int k = 0; k < kPre; ++k) {
      const int idx = tid + k * kComputeThreads;
      xpre[k] = 0.f;
      if (idx < nin0) {
        const int p = idx / per, rem = idx - p * per;
        const long g = g0 + p;
        long src;
        if (a.mean_over_hyp) { const long b = g / a.n_hyp; src = a.x_is_repeated ? (g - b * a.n_hyp) * a.n_pose + b : b; }
        else src = a.x_is_repeated ? g : (g % a.n_pose);
        xpre[k] = __ldg(a.x_in + src * per + rem);
      }
    }
  }

  const Weights& w = *a.w;
  for (int i = tid; i < NP * NP; i += kThreads) {
    const int r = i / NP, k = i - r * NP;
    const __half g1 = __float2half_rn(__ldg(w.t1m + i)), g2 = __float2half_rn(__ldg(w.t2m + i));   // integer rows, exact in fp16;
    if (k < 16) {                                                                                    // the epilogue applies the row scale
      *tall_elem(smem, 0, 128 + r, k) = g1;
      *tall_elem(smem, 1, 128 + r, k) = g2;
    } else {
      for (int p = 0; p < TP; ++p) {
        *reinterpret_cast<__half*>(smem + OFF_A16 + (p * PS + r) * 16 + p * 2) = g1;
        *reinterpret_cast<__half*>(smem + OFF_A16 + A16_BYTES + (p * PS + r) * 16 + p * 2) = g2;
      }
    }
  }
  if (tid < TR && tid % PS < NP) {
    // Chebyshev slab (static): GC2 sees h + 1 temb^T, and T_k (1 temb^T) = p_k temb^T with p_k the row sums of T_k
    // (p_0 = 1; for a row-normalised adjacency p_1 = 0, p_2 = -1, but nothing here relies on it)
    const int i = tid % PS;
    float p1 = 0.f, p2 = 0.f;
    for (int j = 0; j < NP; ++j) { p1 += __ldg(w.t1 + i * NP + j); p2 += __ldg(w.t2 + i * NP + j); }
    const float p1h = __half2float(__float2half_rn(p1)), p2h = __half2float(__float2half_rn(p2));
    *reinterpret_cast<uint4*>(smem + OFF_CS + tid * 16) = make_uint4(pack2(1.f, 1.f), pack2(p1h, p1h), pack2(p1 - p1h, p2h), pack2(p2h, p2 - p2h));
  }
  if (tid < 32) {
    int n_masked = 0;
    if (a.mask) for (int j = 0; j < NP; ++j) n_masked += a.mask[j] == 0;
    // [20] the softmax scale, [24,29) output bias
    maskf[tid] = (tid >= 24 && tid < 24 + a.c_out) ? __ldg(w.bout + tid - 24)
                 : (tid == 20 ? (n_masked == NP ? 0.f : 0.20412414523193151f * 1.4426950408889634f) : 0.f);   // log2(e) / sqrt(24)
  }
  if (a.mask != nullptr && tid >= 32 && tid < 32 + TR) {
    int n_masked = 0;
    for (int j = 0; j < NP; ++j) n_masked += a.mask[j] == 0;
    const int r = tid - 32, j = r % PS;
    if (j < NP && a.mask[j] == 0 && n_masked < NP) *reinterpret_cast<__half*>(smem + OFF_MK + r * 16) = __float2half_rn(-65504.f);
  }
  if (tid < NP * NP) t12[tid] = make_float2(__ldg(w.t1 + tid), __ldg(w.t2 + tid));
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (ktrace) ktrace[1] = clock64();
  // let the next kernel of the stream begin its launch: its CTAs take over each SM as ours retire
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  const int L = a.n_layer;
  if (warp == kProducerWarp) {
    // ---------------------------------------------------------------- producer (TMA bulk copies): per step the input-convolution
    // block, per layer its parameters (double buffered) + 14 weight blocks, then the output-convolution block
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, ps = 0, pphase = 0;
      auto put_block = [&](const uint8_t* src) {
        mbar_wait_sleep(empty0 + 8 * stage, phase ^ 1);
        mbar_expect_tx(full0 + 8 * stage, WBLK_BYTES);
        bulk_g2s(sbase + OFF_W + stage * WBLK_BYTES, src, WBLK_BYTES, full0 + 8 * stage);
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
      };
      for (int it = 0; it < my_tiles; ++it)
        for (int step = 0; step < a.n_steps; ++step) {
          put_block(a.ioblocks);
          for (int l = 0; l < L; ++l) {
            mbar_wait_sleep(pempty0 + 8 * ps, pphase ^ 1);
            const bool step_temb = !a.forward_only && a.has_temb;     // one temb row per (step, layer), shared by the batch
            mbar_expect_tx(pfull0 + 8 * ps, step_temb ? PAR_BYTES : LP_BYTES);
            bulk_g2s(sbase + OFF_PAR + ps * PAR_BYTES, a.lparams + (size_t)l * LP_BYTES, LP_BYTES, pfull0 + 8 * ps);
            if (step_temb) bulk_g2s(sbase + OFF_PAR + ps * PAR_BYTES + LP_BYTES, a.tau + ((size_t)step * L + l) * LP_TAU_BYTES, LP_TAU_BYTES, pfull0 + 8 * ps);
            if (++ps == 2) { ps = 0; pphase ^= 1; }
            for (int blk = 0; blk < BLOCKS_PER_LAYER; ++blk) put_block(a.wpack + ((size_t)l * BLOCKS_PER_LAYER + blk) * WBLK_BYTES);
          }
          put_block(a.ioblocks + WBLK_BYTES);
        }
    }
    __syncwarp();
  } else if (warp == kIssuerWarp) {
    // ---------------------------------------------------------------- MMA issuer: the whole warp runs the static program
    // (every value is warp-uniform), one elected lane issues
    const uint32_t leader = elect_one() ? 1u : 0u;
    uint32_t stage = 0, phase = 0, rdy_i = 0, acc_i = 0;
    long long* itrace = (TRACE && blockIdx.x == 0 && a.trace != nullptr && leader) ? a.trace + a.trace_cap / 2 : nullptr;   // issuer stamps: second half
    int itrace_n = 0;
    auto imark = [&]() { if (TRACE && itrace != nullptr && itrace_n < a.trace_cap / 2) itrace[itrace_n++] = clock64(); };
    auto wait_rdy = [&]() {
      imark();
      asm volatile("bar.sync %0, 288;" ::"r"(2 + rdy_i) : "memory");
      rdy_i = (rdy_i + 1) & (NEV - 1);
      tc_fence_after();
      imark();
    };
    auto commit_acc = [&]() { umma_commit(accb + 8 * acc_i, leader); acc_i = (acc_i + 1) & (NEV - 1); };
    auto w_acquire = [&]() -> uint32_t { mbar_wait(full0 + 8 * stage, phase); tc_fence_after(); return sbase + OFF_W + stage * WBLK_BYTES; };
    auto w_release = [&]() { umma_commit(empty0 + 8 * stage, leader); if (++stage == NSTAGE) { stage = 0; phase ^= 1; } };
    const uint32_t tb = tmem_base;
    const uint32_t ones_lo = desc_lo(sbase + OFF_ONES, A_LBO);
    constexpr uint32_t kHiK = desc_hi(128);          // K-major operands of every kind: 8-row groups 128 B apart
    constexpr uint32_t kHiActMn = desc_hi(A_LBO);    // activations as MN-major B: 8-channel groups one chunk column apart
    constexpr uint32_t kN96 = idesc_f16(96, false), kN96Mn = idesc_f16(96, true), kN128 = idesc_f16(128, false), kN32Mn = idesc_f16(32, true),
                       kN16 = idesc_f16(16, false);
    // D[:, dcol..dcol+96) (+)= A [128 x 96] * W^T with A in tensor memory (48 columns of fp16 pairs from acol)
    auto gemm_ts = [&](uint32_t wa, uint32_t acol, uint32_t dcol, uint32_t accumulate) {
      uint32_t b_lo = desc_lo(wa, W_LBO), acc = accumulate;
#pragma unroll
      for (int ks = 0; ks < 6; ++ks) {
        umma_ts(tb + dcol, tb + acol + 8 * ks, b_lo, kHiK, kN96, acc, leader);
        b_lo += 2 * W_LBO >> 4; acc = 1u;
      }
    };
    // A converted in place inside its own fp32 accumulator [abase, abase+96): each half of the columns holds the 24 fp16
    // pairs of its own 48 channels (the two threads of a row convert their halves independently)
    auto gemm_ts_inplace = [&](uint32_t wa, uint32_t abase, uint32_t dcol, uint32_t accumulate) {
      uint32_t b_lo = desc_lo(wa, W_LBO), acc = accumulate;
#pragma unroll
      for (int ks = 0; ks < 6; ++ks) {
        umma_ts(tb + dcol, tb + abase + 8 * ks + (ks >= 3 ? 24 : 0), b_lo, kHiK, kN96, acc, leader);
        b_lo += 2 * W_LBO >> 4; acc = 1u;
      }
    };
    auto bias = [&](uint32_t wa, uint32_t dcol) {
      umma_ss(tb + dcol, ones_lo, kHiK, desc_lo(wa + 12 * W_LBO, W_LBO), kHiK, kN96, 1u, leader);
    };
    // the same with the joint slab as A: bias + r_i * beta (k = 98..100 of the block), second chunk column = the zero one
    const uint32_t js_lo = desc_lo(sbase + OFF_JS, OFF_ONES + A_LBO - OFF_JS);
    // sampler: the time embedding enters GC2 as one more K step, A = Chebyshev slab, B = this (step, layer)'s block in the
    // parameter stage (its second chunk column repeats the first: LBO = 0; the slab's second one is the zero column)
    const uint32_t cs_lo = desc_lo(sbase + OFF_CS, OFF_ONES + A_LBO - OFF_CS);
    const bool tau_step = a.has_temb && !a.forward_only;
    uint32_t ips = 0, ipphase = 0;
    auto bias_joint = [&](uint32_t wa, uint32_t dcol) {
      umma_ss(tb + dcol, js_lo, kHiK, desc_lo(wa + 12 * W_LBO, W_LBO), kHiK, kN96, 1u, leader);
    };
    // D[:, dcol..dcol+96) (+)= blockdiag_p(G) * block b_blk, G = graph operand `which`: one K=16 MMA per pose over joints
    // 0..15 (window into the tall operand x the pose's rows in place), one over the joint-16 rows in the side buffer
    auto aggregate = [&](int which, int b_blk, uint32_t dcol, uint32_t accumulate) {
      uint32_t a_lo = desc_lo(sbase + OFF_TALL + which * TALL_BYTES + 128 * 16, T_LBO);
      uint32_t b_lo = desc_lo(sbase + OFF_A + b_blk * ABLK_BYTES, 128);
      uint32_t acc = accumulate;
#pragma unroll 1
      for (int p = 0; p < TP; ++p) {
        umma_ss(tb + dcol, a_lo, kHiK, b_lo, kHiActMn, kN96Mn, acc, leader);
        acc = 1u;
        a_lo -= PS;      // window start moves up one pose (PS rows of 16 B, >> 4)
        b_lo += PS;      // activations of the next pose
      }
      const uint32_t a16 = sbase + OFF_A16 + which * A16_BYTES;
      umma_ss(tb + dcol, desc_lo(a16, (sbase + OFF_ONES + A_LBO) - a16), kHiK, desc_lo(sbase + OFF_SIDE + b_blk * SIDE_BYTES, 128), desc_hi(SIDE_LBO),
              kN96Mn, 1u, leader);
    };
    // S_h[:, 0..128) = Q_h K_h^T (+ key mask); Q = block 0, K = block 1, chunk columns 3h..3h+2.  The 4th chunk column of
    // the second K step is reached through the descriptor's leading-dimension offset: the ones slab (1, 1, 0, ...) for Q
    // and the key-mask chunk column (m_j, 0, 0, ...) for K, so that every score gets + m_j of its key
    auto scores_head = [&](int h, uint32_t dcol) {
      const uint32_t qa = sbase + OFF_A + 3 * h * A_LBO, ka = qa + ABLK_BYTES;
      umma_ss(tb + dcol, desc_lo(qa, A_LBO), kHiK, desc_lo(ka, A_LBO), kHiK, kN128, 0u, leader);
      umma_ss(tb + dcol, desc_lo(qa + 2 * A_LBO, (sbase + OFF_ONES) - (qa + 2 * A_LBO)), kHiK,
              desc_lo(ka + 2 * A_LBO, (sbase + OFF_MK) - (ka + 2 * A_LBO)), kHiK, kN128, 1u, leader);
    };
    // O[:, 24h..24h+32) = P_h V[:, 24h..24h+32): P_h in TMEM at pcol (slot layout, see softmax_run), V = block 2 in place as an
    // MN-major operand: one K=16 MMA per pose (joints 0..15), one for the joint-16 rows in the side buffer of block 2
    auto pv_head = [&](int h, uint32_t pcol) {
      uint32_t b_lo = desc_lo(sbase + OFF_A + 2 * ABLK_BYTES + 3 * h * A_LBO, 128);
#pragma unroll
      for (int p = 0; p < TP; ++p) {
        umma_ts(tb + COL_O + 24 * h, tb + pcol + 8 * p, b_lo, kHiActMn, kN32Mn, p > 0 ? 1u : 0u, leader);
        b_lo += PS;
      }
      umma_ts(tb + COL_O + 24 * h, tb + pcol + 8 * TP, desc_lo(sbase + OFF_SIDE + 2 * SIDE_BYTES + 3 * h * SIDE_LBO, 128), desc_hi(SIDE_LBO), kN32Mn, 1u,
              leader);
    };
    for (int it = 0; it < my_tiles; ++it)
      for (int step = 0; step < a.n_steps; ++step) {
        uint32_t wa;
        // 0. x = [x_t | T1 x_t | T2 x_t] Win + b at hi/lo precision: A = block 0 chunk columns 0..5 (hi, lo, hi),
        //    B = [Win_hi ; Win_hi ; Win_lo] (row 15 of each slab carries the bias)
        wa = w_acquire();     // (before the wait: the weights are there long before the operands)
        wait_rdy();
        {
          const uint32_t a_lo = desc_lo(sbase + OFF_A, A_LBO), b_lo = desc_lo(wa, W_LBO);
#pragma unroll
          for (int ks = 0; ks < 3; ++ks)
            umma_ss(tb + COL_X, a_lo + ks * (2 * A_LBO >> 4), kHiK, b_lo + ks * (2 * W_LBO >> 4), kHiK, kN96, ks > 0 ? 1u : 0u, leader);
        }
        w_release();
        commit_acc();
        for (int l = 0; l < L; ++l) {
          // Every "wait_rdy" consumes the next "operands ready" event of the compute warps, every "commit_acc" produces
          // the next "accumulator ready" event; both sides walk the same static sequence.  Accumulator groups: ACC+0,
          // ACC+96 (also the two score regions), ACC2 and the O region, arranged so that a GEMM may start while the
          // compute warps are still reading the groups of the previous one.
          // 1. q, k, v = LN0(x) W + b                         A = TA0 (tensor memory); one event per output block
          wa = w_acquire();     // (before the wait: the weights are there long before the operands)
          //    (k's bias only shifts every score of a query row by the same constant and v's could be folded into the
          //    out-projection: tried in round 2, 2 MMAs fewer per layer, no measurable gain -- 96.8 vs 96.6 us per batch -- while
          //    every rounding point downstream moves; not taken)
          wait_rdy(); gemm_ts(wa, COL_TA0, COL_ACC, 0u); bias(wa, COL_ACC); w_release(); commit_acc();
          wa = w_acquire(); gemm_ts(wa, COL_TA0, COL_ACC + 96, 0u); bias(wa, COL_ACC + 96); w_release(); commit_acc();
          wa = w_acquire(); gemm_ts(wa, COL_TA0, COL_O, 0u); bias(wa, COL_O); w_release(); commit_acc();
          // 1b. attention, two heads at a time: S = Q_h K_h^T (d_k = 24 = K step of 16 + 8 real | 8 zero columns),
          //     softmax on the compute warps (P back into TMEM), O_h = P V_h with V as an MN-major operand
          wait_rdy();                                             // q, k in blocks 0, 1
          scores_head(0, COL_S0); scores_head(1, COL_S1);
          commit_acc();
          wait_rdy();                                             // v in block 2 (its accumulator, the O region, is free)
          wait_rdy();                                             // P of heads 0, 1
          pv_head(0, COL_S0); pv_head(1, COL_S1);
          scores_head(2, COL_S0); scores_head(3, COL_S1);
          commit_acc();
          wait_rdy();                                             // P of heads 2, 3
          pv_head(2, COL_S0); pv_head(3, COL_S1);
          commit_acc();
          // 2. x += attn Wo + bo                              A = TA0
          wa = w_acquire();     // (before the wait: the weights are there long before the operands)
          wait_rdy(); gemm_ts(wa, COL_TA0, COL_X, 1u); bias(wa, COL_X); w_release();
          commit_acc();
          // 3. g1 = L^ LN1(x)                                 B = block 0
          wait_rdy();
          aggregate(2, 0, COL_ACC, 0u);
          commit_acc();
          // 4. h = g1 W1 + b1 (192 outputs)                   A = TA0; one event per half
          wa = w_acquire();     // (before the wait: the weights are there long before the operands)
          wait_rdy(); gemm_ts(wa, COL_TA0, COL_ACC, 0u); bias_joint(wa, COL_ACC); w_release(); commit_acc();
          wa = w_acquire(); gemm_ts(wa, COL_TA0, COL_ACC + 96, 0u); bias_joint(wa, COL_ACC + 96); w_release(); commit_acc();
          // 5. z = relu(h) W2 ; x += b2                       A = TA1, TA0, each as soon as its half of h is there
          wa = w_acquire();     // (before the wait: the weights are there long before the operands)
          wait_rdy(); gemm_ts(wa, COL_TA1, COL_ACC2, 0u); bias(wa, COL_X); w_release();
          wa = w_acquire();     // (before the wait: the weights are there long before the operands)
          wait_rdy(); gemm_ts(wa, COL_TA0, COL_ACC2, 1u); w_release();
          commit_acc();
          // 6. x += L^ z                                      B = block 1
          wait_rdy();
          aggregate(2, 1, COL_X, 1u);
          commit_acc();
          // 7/8, 9/10. the two Chebyshev convolutions: [T1 v | T2 v] (B = block 0, one event each), and
          //     [v | T1 v | T2 v] Wc + b into ACC2 -- the v part right away, the others as their operands arrive
          if (tau_step) { mbar_wait(pfull0 + 8 * ips, ipphase); tc_fence_after(); }   // complete long ago: the compute warps waited on it
          for (int conv = 0; conv < 2; ++conv) {
            wait_rdy();
            aggregate(0, 0, COL_ACC, 0u); commit_acc();
            aggregate(1, 0, COL_ACC + 96, 0u); commit_acc();
            wa = w_acquire(); gemm_ts(wa, conv == 0 ? COL_TA0 : COL_TA1, COL_ACC2, 0u); bias(wa, COL_ACC2);
            if (conv == 1 && tau_step) umma_ss(tb + COL_ACC2, cs_lo, kHiK, desc_lo(sbase + OFF_PAR + ips * PAR_BYTES + LP_BYTES, 0), kHiK, kN96, 1u, leader);
            w_release();
            wa = w_acquire();     // (before the wait: the weights are there long before the operands)
            wait_rdy(); gemm_ts_inplace(wa, COL_ACC, COL_ACC2, 1u); w_release();
            wa = w_acquire();     // (before the wait: the weights are there long before the operands)
            wait_rdy(); gemm_ts_inplace(wa, COL_ACC + 96, COL_ACC2, 1u); w_release();
            commit_acc();
          }
          if (++ips == 2) { ips = 0; ipphase ^= 1; }
        }
        // 11. U = [X_hi | X_lo | X_hi] [Wout_hi ; Wout_hi ; Wout_lo]   (N = 16: 3 Chebyshev orders x 5 outputs)
        wa = w_acquire();     // (before the wait: the weights are there long before the operands)
        wait_rdy();
        {
          const uint32_t b_lo = desc_lo(wa, OUT_LBO);
#pragma unroll
          for (int part = 0; part < 3; ++part) {
            const uint32_t acol = part == 1 ? COL_TA1 : COL_TA0;     // X_hi, X_lo, X_hi as TMEM-resident A operands
#pragma unroll
            for (int ks = 0; ks < 6; ++ks)
              umma_ts(tb + COL_ACC, tb + acol + 8 * ks, b_lo + (part * 6 + ks) * (2 * OUT_LBO >> 4), kHiK, kN16, (part | ks) ? 1u : 0u, leader);
          }
        }
        w_release();
        commit_acc();
      }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- compute warps
    Ctx c;
    c.smem = smem;
    c.lane = lane;
    c.row = (warp & 3) * 32 + lane;
    c.hh = warp >> 2;
    c.tmem_lane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
    c.rdy = rdy; c.acc = accb; c.acc_phase = 0; c.rdy_i = 0; c.acc_i = 0;
    c.trace = (blockIdx.x == 0 && tid == 0) ? a.trace : nullptr;
    c.trace_n = 0; c.trace_cap = a.trace_cap / 2;
    const int row = c.row, hh = c.hh;
    float* scratch = reinterpret_cast<float*>(smem + OFF_A);   // [128][SCR] fp32, aliases the head of operand block 0
    constexpr int SCR = 17;                                    // odd row stride: one thread per row reads without bank conflicts
    const float k2 = maskf[20];
    uint32_t ps = 0, pphase = 0;                               // parameter stage of the current layer
    const uint32_t xcol = c.tmem_lane + COL_X + hh * 48;       // this thread's half of its residual row
    const uint32_t my_chunk = (uint32_t)(OFF_A + a_chunk(row, hh * 6));   // its first chunk inside operand block 0
    // row scales of the integerised Chebyshev matrices for this thread's joint (pad rows: anything finite)
    const float t1scale = __ldg(w.t1s + min(row % PS, NP - 1)), t2scale = __ldg(w.t2s + min(row % PS, NP - 1));
    // the joint-16 row of a pose also goes to the side buffer of the block it is written to (row = pose, same chunk columns)
    uint8_t* const side0 = (row % PS == NP - 1 && row / PS < TP) ? smem + OFF_SIDE + (hh * 6) * SIDE_LBO + (row / PS) * 16 : nullptr;
    uint8_t* const side1 = side0 ? side0 + SIDE_BYTES : nullptr;
    uint8_t* const side2 = side0 ? side0 + 2 * SIDE_BYTES : nullptr;

    float macc = 0.f;     // mean_over_hyp: running hypothesis sum of output element `tid` of the pose being completed
    double ev1 = 0.0, ev2 = 0.0, evn = 0.0;   // fused evaluation: this warp's partial sums (the same on every lane)
    for (int it = 0; it < my_tiles; ++it) {
      const long g0 = a.mean_over_hyp ? row_lo + (long)it * TP : ((long)blockIdx.x + (long)it * gridDim.x) * TP;
      const int npose = (int)min((long)TP, (a.mean_over_hyp ? row_hi : a.n_rows) - g0);
      const int ci = a.c_in, co = a.c_out;
      const int nin = npose * NP * ci, nval = npose * NP * co;  // valid (pose, joint, coordinate) triples: input, output
      for (int idx = tid; idx < TM * XS; idx += kComputeThreads) xt[idx] = 0.f;
      bar_compute();
      if (it == 0) {          // requested before the set-up barrier (xpre)
#pragma unroll
        for (int k = 0; k < kPre; ++k) {
          const int idx = tid + k * kComputeThreads;
          if (idx < nin) {
            const int p = idx / (NP * ci), rem = idx - p * (NP * ci);
            xt[(p * PS + rem / ci) * XS + rem % ci] = xpre[k];
          }
        }
      } else {
        for (int idx = tid; idx < nin; idx += kComputeThreads) {
          const int p = idx / (NP * ci), rem = idx - p * (NP * ci);
          const long g = g0 + p;
          long src;
          if (a.mean_over_hyp) { const long b = g / a.n_hyp; src = a.x_is_repeated ? (g - b * a.n_hyp) * a.n_pose + b : b; }
          else src = a.x_is_repeated ? g : (g % a.n_pose);
          xt[(p * PS + rem / ci) * XS + rem % ci] = a.x_in[src * (NP * ci) + rem];
        }
      }
      if ((EVAL && a.gt != nullptr)) {        // targets of the poses this tile finishes: requested now, read in the tile's tail
        float* evg = reinterpret_cast<float*>(smem + OFF_EV) + EV_FLOATS;
        for (int idx = tid; idx < npose * NP * 3; idx += kComputeThreads) {
          const int p = idx / (NP * 3);
          const long g = g0 + p;
          const long b = a.mean_over_hyp ? g / a.n_hyp : g % a.n_pose;
          if (!a.mean_over_hyp || g - b * a.n_hyp == a.n_hyp - 1) evg[idx] = __ldg(a.gt + b * (NP * 3) + (idx - p * (NP * 3)));
        }
      }
      bar_compute();

      // ---- input ChebConv (ChebConv.py:74-88, K = 15): the panel [x | T1 x | T2 x | 1] of every row, split into
      //      fp16 hi and lo parts, becomes chunk columns 0..5 of operand block 0 (hi, lo, hi)
      auto build_panel = [&]() {
        if (tid < TM) {
          const int r = tid;
          float pv[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) pv[i] = 0.f;
          const int p = r / PS, i = r - p * PS;
          if (p < TP && i < NP) {
#pragma unroll
            for (int cc = 0; cc < 5; ++cc) pv[cc] = xt[r * XS + cc];
            // dense over the 17 joints of the pose: no index indirection, every load is independent of the others (a
            // neighbour list would save multiplications by zero but chain two shared-memory latencies per entry)
#pragma unroll
            for (int n = 0; n < NP; ++n) {
              const float* u = xt + (p * PS + n) * XS;
              const float2 cf = t12[i * NP + n];
#pragma unroll
              for (int cc = 0; cc < 5; ++cc) { pv[5 + cc] = fmaf(cf.x, u[cc], pv[5 + cc]); pv[10 + cc] = fmaf(cf.y, u[cc], pv[10 + cc]); }
            }
          }
          pv[15] = 1.0f;      // multiplies the bias row of the weight slabs
          uint4 h0, l0, h1, l1;
          split8(pv, h0, l0);
          split8(pv + 8, h1, l1);
          uint8_t* dst = smem + OFF_A;
          *reinterpret_cast<uint4*>(dst + a_chunk(r, 0)) = h0; *reinterpret_cast<uint4*>(dst + a_chunk(r, 1)) = h1;
          *reinterpret_cast<uint4*>(dst + a_chunk(r, 2)) = l0; *reinterpret_cast<uint4*>(dst + a_chunk(r, 3)) = l1;
          *reinterpret_cast<uint4*>(dst + a_chunk(r, 4)) = h0; *reinterpret_cast<uint4*>(dst + a_chunk(r, 5)) = h1;
        }
      };
      build_panel();
      signal_ready(c);                                             // -> 0 (in-conv operands of step 0)
      for (int step = 0; step < a.n_steps; ++step) {
        mbar_wait(pfull0 + 8 * ps, pphase);                        // layer 0's parameters (checked here, off the critical path)
        wait_acc(c);
        const uint32_t acol = c.tmem_lane + COL_ACC + hh * 48;      // this thread's half of accumulator group 0
        const uint32_t acol2 = c.tmem_lane + COL_ACC2 + hh * 48, ocol = c.tmem_lane + COL_O + hh * 48;
        const uint32_t ta0 = c.tmem_lane + COL_TA0 + hh * 24, ta1 = c.tmem_lane + COL_TA1 + hh * 24;   // this thread's half of a TMEM operand
        // The loop is rotated: LN0 of a layer runs at the end of the previous iteration (here for layer 0), so that the
        // backward branch -- an instruction-cache miss on this part -- and the parameter copies below fall into the wait
        // for the q GEMM instead of sitting in front of LN0 on the critical path.
        ln_run(smem, xcol, 0u, row, hh, 0u, nullptr, ta0);
        signal_ready_tmem(c);                                        // LN0(x) in TA0

        for (int l = 0; l < L; ++l) {
          // this layer's parameters (L^, joint slab, time-embedding block) have been staged by the producer
          const uint8_t* par = smem + OFF_PAR + ps * PAR_BYTES;
          if (a.forward_only && a.has_temb && tid < TP * (H / 4)) {   // per-sample timesteps: this layer's temb row of every pose
            const int p = tid / (H / 4), c4 = tid - p * (H / 4);
            float4 tv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p < npose) tv = __ldg(reinterpret_cast<const float4*>(a.temb + ((size_t)(g0 + p) * L + l) * H) + c4);
            reinterpret_cast<float4*>(smem + OFF_TEP)[tid] = tv;
          }
          if (tid < 2 * NP) {   // L^[:, 0:16] into rows 128..144 of its tall operand
            const int kc = tid / NP, r = tid - kc * NP;
            *reinterpret_cast<uint4*>(smem + OFF_TALL + 2 * TALL_BYTES + kc * T_LBO + (128 + r) * 16) = *reinterpret_cast<const uint4*>(par + tid * 16);
          } else if (tid >= 64 && tid < 64 + TP * NP) {   // L^[:, 16] into its joint-16 operand: element (18p+i, p)
            const int p = (tid - 64) / NP, i = (tid - 64) - p * NP;
            *reinterpret_cast<__half*>(smem + OFF_A16 + 2 * A16_BYTES + (p * PS + i) * 16 + p * 2) =
                *reinterpret_cast<const __half*>(par + (2 * NP + i) * 16);
          }
          if (tid < TR)     // joint slab of this layer (the previous layer's fc1 finished reading it long ago)
            *reinterpret_cast<uint4*>(smem + OFF_JS + tid * 16) = *reinterpret_cast<const uint4*>(par + LP_LHAT_BYTES + (tid % PS) * 16);
          // The layer is a fixed sequence of compute phases, each followed by "operands ready" and a wait for the
          // accumulators of the MMA group it feeds (the issuer runs the matching program).  Straight-line code on
          // purpose: on this part every taken branch to code that is not next in line costs an instruction-cache miss.
          uint8_t* const blk0 = smem + my_chunk;                     // its chunks in operand blocks 0, 1, 2
          uint8_t* const blk1 = blk0 + ABLK_BYTES;
          uint8_t* const blk2 = blk0 + 2 * ABLK_BYTES;
          const float ninf = -INFINITY;
          // temb added after GC1 (gcndiff.py:51).  Sampler: the issuer adds it to GC2 as a bias block, nothing to do here.
          // Forward call: one row per pose, added in the epilogue.  GCNpose: none.
          const bool pose_temb = a.forward_only && a.has_temb;
          const float* temb_row = reinterpret_cast<const float*>(smem + OFF_TEP) + min(row / PS, TP - 1) * H + hh * 48;
          // ======== x = x + attn(LN0(x))   (LN0 has been signalled already)
          wait_acc(c); epi_run(blk0, acol, ninf, nullptr);           // q
          wait_acc(c); epi_run(blk1, acol + 96, ninf, nullptr);      // k
          signal_ready(c);                                           // q, k ready -> scores of heads 0, 1
          wait_acc(c); epi_run(blk2, ocol, ninf, nullptr, 1.0f, false, side2, false, true);   // v
          signal_ready(c);                                           // v ready
          wait_acc(c);
          softmax_run(c.tmem_lane + (hh ? COL_S1 : COL_S0), row, k2);
          signal_ready_tmem(c);                                      // -> P V of heads 0, 1; scores of heads 2, 3
          wait_acc(c);
          softmax_run(c.tmem_lane + (hh ? COL_S1 : COL_S0), row, k2);
          signal_ready_tmem(c);                                      // -> P V of heads 2, 3
          wait_acc(c);
          epi_tmem(ta0, ocol, 1.0f, false, false);
          signal_ready_tmem(c);                                      // -> out projection (accumulates into x)
          wait_acc(c);
          // ======== x = x + GraphNet(LN1(x))
          ln_run(smem, xcol, 0u, row, hh, my_chunk, side0);
          signal_ready(c);                                           // -> L^ y
          wait_acc(c);
          epi_tmem(ta0, acol, 1.0f, false, false);
          signal_ready_tmem(c);                                      // -> fc1
          wait_acc(c); epi_tmem(ta1, acol, 1.0f, false, true);
          signal_ready_tmem(c);                                      // first half of relu(h) -> fc2, first K block
          wait_acc(c); epi_tmem(ta0, acol + 96, 1.0f, false, true);  // (fc1 has finished reading TA0)
          signal_ready_tmem(c);                                      // second half
          wait_acc(c);
          epi_run(blk1, acol2, ninf, nullptr, 1.0f, false, side1, false, true);
          signal_ready(c);                                           // -> L^ z (accumulates into x)
          wait_acc(c);
          // ======== x = x + GC2(GC1(x) + temb)
          epi_run(blk0, xcol, ninf, nullptr, 1.0f, false, side0, false, true, ta0);
          signal_ready(c);                                           // x as an operand: B (block 0) -> [T1 x | T2 x], A (TA0) -> x Wc1_0
          wait_acc(c); epi_tmem(acol, acol, t1scale, true, false);   // T1 x, converted in place
          signal_ready_tmem(c);
          wait_acc(c); epi_tmem(acol + 96, acol + 96, t2scale, true, false);   // T2 x
          signal_ready_tmem(c);
          wait_acc(c);
          if (pose_temb) epi_run(blk0, acol2, 0.f, temb_row, 1.0f, false, side0, false, true, ta1);
          else epi_run(blk0, acol2, 0.f, nullptr, 1.0f, false, side0, true, true, ta1);
          signal_ready(c);                                           // h = relu(GC1) (+ temb) -> [T1 h | T2 h] and h Wc2_0
          wait_acc(c); epi_tmem(acol, acol, t1scale, true, false);
          signal_ready_tmem(c);
          wait_acc(c); epi_tmem(acol + 96, acol + 96, t2scale, true, false);
          signal_ready_tmem(c);
          const uint32_t ps_done = ps;
          if (++ps == 2) { ps = 0; pphase ^= 1; }
          if (l + 1 < L) mbar_wait(pfull0 + 8 * ps, pphase);        // the next layer's parameters, while the last GEMM runs
          wait_acc(c);                                               // GC2 in ACC2: the residual is applied by the next phase
          __syncwarp();
          if (lane == 0) mbar_arrive(pempty0 + 8 * ps_done);         // GC2 was the last reader of this layer's parameter stage
          if (l + 1 < L) {
            // closing residual of this layer's Chebyshev block, then LN0 of the next layer
            ln_run(smem, xcol, acol2, row, hh, 0u, nullptr, ta0);
            signal_ready_tmem(c);                                    // LN0(x) in TA0
          }
        }

        // ---- output ChebConv (N = 5): U_k = X Wout_k on the tensor cores with X = hi + lo, then
        //      eps = b + U0 + T1 U1 + T2 U2 and the DDIM update on the CUDA cores
        {
          float v[48], u[48];
          const uint32_t acol2 = c.tmem_lane + COL_ACC2 + hh * 48;
          tmem_ld16_async(acol2, u);
          tmem_ld16_async(acol2 + 16, u + 16);
          tmem_ld16_async(acol2 + 32, u + 32);
          tmem_ld48(xcol, v);
          launder<48>(u);
#pragma unroll
          for (int i = 0; i < 48; ++i) v[i] += fmaxf(u[i], 0.f);   // closing residual of the last layer
          // X = hi + lo, both fp16, both A operands in tensor memory (TA0, TA1)
          uint32_t ph[24], pl[24];
#pragma unroll
          for (int q = 0; q < 6; ++q) {
            uint4 hi, lo;
            split8(v + 8 * q, hi, lo);
            ph[4 * q] = hi.x; ph[4 * q + 1] = hi.y; ph[4 * q + 2] = hi.z; ph[4 * q + 3] = hi.w;
            pl[4 * q] = lo.x; pl[4 * q + 1] = lo.y; pl[4 * q + 2] = lo.z; pl[4 * q + 3] = lo.w;
          }
          tmem_st24_u32(ta0, ph);
          tmem_st24_u32(ta1, pl);
        }
        signal_ready_tmem(c);                                      // -> 11
        wait_acc(c);
        if (hh == 0) {
          float u[16];
          tmem_ld16_async(c.tmem_lane + COL_ACC, u);
          tmem_ld_wait();
          launder<16>(u);
#pragma unroll
          for (int i = 0; i < 16; ++i) scratch[row * SCR + i] = u[i];
        }
        tc_fence_before();
        bar_compute();
        // eps = b + U0 + T1 U1 + T2 U2, then either the DDIM update (common/utils_diff.py:59-65, same operation order, no FMA
        // contraction) or, for a plain forward call, the store of eps.  Two threads per tile row: coordinates 0..2 and 3..4.
        {
          const dp_step st = a.steps_dev ? a.steps_dev[step] : inl.s[step];
          const int r = tid & (TM - 1), part = tid >> 7;
          const int p = r / PS, i = r - p * PS;
          const int n0 = part ? 3 : 0, n1 = min(co, part ? 5 : 3);
          if (i < NP && p < npose && n0 < n1) {
            float et[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) et[k] = maskf[24 + n0 + k] + scratch[r * SCR + n0 + k];   // (slots past c_out are never stored)
#pragma unroll
            for (int q = 0; q < NP; ++q) {
              const float* u = scratch + (p * PS + q) * SCR + n0;
              const float2 cf = t12[i * NP + q];
#pragma unroll
              for (int k = 0; k < 3; ++k) et[k] = fmaf(cf.y, u[10 + k], fmaf(cf.x, u[5 + k], et[k]));
            }
            long grow = g0 + p;       // row of the caller's hypothesis-major arrays (noise, eps)
            if (a.mean_over_hyp) { const long b = grow / a.n_hyp; grow = (grow - b * a.n_hyp) * a.n_pose + b; }
            const size_t o = ((size_t)grow * NP + i) * co;
            // keyed noise: this thread's elements e0 .. e0 + 2 of row (b, h) lie in at most two Philox quads
            uint4 qa = make_uint4(0, 0, 0, 0), qb = qa;
            const uint32_t e0 = (uint32_t)(i * co + n0);
            if (KEYED) {
              const long h = grow / a.n_pose;
              const uint32_t s = a.key.step_offset + (uint32_t)step, b = a.key.pose_offset + (uint32_t)(grow - h * a.n_pose);
              qa = philox_quad(a.key, s, b, (uint32_t)h, e0 >> 2);
              qb = ((e0 + (uint32_t)(n1 - n0) - 1u) >> 2) != (e0 >> 2) ? philox_quad(a.key, s, b, (uint32_t)h, (e0 >> 2) + 1u) : qa;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
              const int n = n0 + k;
              if (n >= n1) break;
              if (a.forward_only) {
                a.out[o + n] = et[k];
              } else {
                const float xv = xt[r * XS + n];
                const float x0 = __fdiv_rn(__fsub_rn(xv, __fmul_rn(et[k], st.sqrt_1m_at)), st.sqrt_at);
                float nx = __fmul_rn(st.sqrt_an, x0);
                if (a.noise) nx = __fadd_rn(nx, __fmul_rn(st.c1, a.noise[(size_t)step * a.n_rows * NP * co + o + n]));
                else if (KEYED) {
                  const uint32_t e = e0 + (uint32_t)k;
                  nx = __fadd_rn(nx, __fmul_rn(st.c1, philox_box_muller((e >> 2) == (e0 >> 2) ? qa : qb, e & 3u)));
                }
                xt[r * XS + n] = __fadd_rn(nx, __fmul_rn(st.c2, et[k]));
              }
            }
          }
        }
        bar_compute();   // scratch (= the head of operand block 0) is free again: the next panel / epilogues overwrite it
        if (step + 1 < a.n_steps) {   // the next step's panel before the backward branch: that one then falls into the in-conv wait
          build_panel();
          signal_ready(c);
        }
      }
      if (a.mean_over_hyp) {
        // mean(reshape(H, -1, 17, c), 0) fused into the store: the rows of this CTA are pose-major, so thread e < 17 c walks
        // the tile's rows in order, carries the running sum of its element across tiles in a register and stores a pose
        // when its last hypothesis has passed (same summation order and division as hyp_mean_kernel: bit-identical)
        if (tid < NP * co) {
          const float* src = xt + (tid / co) * XS + tid % co;
          for (int p = 0; p < npose; ++p) {
            const long g = g0 + p, b = g / a.n_hyp;
            const int h = (int)(g - b * a.n_hyp);
            const float v = src[p * PS * XS];
            macc = h == 0 ? __fadd_rn(0.f, v) : __fadd_rn(macc, v);
            if (h == a.n_hyp - 1) {
              const float mval = __fdiv_rn(macc, (float)a.n_hyp);
              a.out[(size_t)b * NP * co + tid] = mval;
              if ((EVAL && a.gt != nullptr) && tid % co >= co - 3) reinterpret_cast<float*>(smem + OFF_EV)[p * (NP * 3) + (tid / co) * 3 + tid % co - (co - 3)] = mval;
            }
          }
        }
      } else if (!a.forward_only) {
        for (int idx = tid; idx < nval; idx += kComputeThreads) {
          const int p = idx / (NP * co), rem = idx - p * (NP * co);
          const float xv = xt[(p * PS + rem / co) * XS + rem % co];
          a.out[(size_t)g0 * NP * co + idx] = xv;
          if ((EVAL && a.gt != nullptr) && rem % co >= co - 3) reinterpret_cast<float*>(smem + OFF_EV)[p * (NP * 3) + (rem / co) * 3 + rem % co - (co - 3)] = xv;
        }
      }
      if ((EVAL && a.gt != nullptr)) {
        // Fused evaluation tail (runners/diffpose_frame.py:382-387): one warp per finished pose of this tile -- at most 7, on 8
        // compute warps -- computes MPJPE and P-MPJPE from the xyz just stored and the targets requested at the tile's start.
        bar_compute();
        const float* evp = reinterpret_cast<const float*>(smem + OFF_EV);
        int cnt = 0;
        for (int p = 0; p < npose; ++p) {
          const long g = g0 + p;
          if (a.mean_over_hyp && g % a.n_hyp != a.n_hyp - 1) continue;
          if ((cnt & 7) == warp) {
            const int j = lane < NP ? lane : 0;
            float pv[3], gv[3];
#pragma unroll
            for (int cc = 0; cc < 3; ++cc) { pv[cc] = evp[p * (NP * 3) + j * 3 + cc]; gv[cc] = evp[EV_FLOATS + p * (NP * 3) + j * 3 + cc]; }
            float e1, e2;
            metric::pose_errors(pv, gv, lane, e1, e2);
            ev1 += (double)e1; ev2 += (double)e2; evn += 1.0;
          }
          ++cnt;
        }
      }
      bar_compute();
    }
    if ((EVAL && a.gt != nullptr)) {     // one atomic per CTA and quantity
      double* red = reinterpret_cast<double*>(smem + OFF_STAT);      // [3][8], free after the last tile
      if (lane == 0) { red[warp] = ev1; red[8 + warp] = ev2; red[16 + warp] = evn; }
      bar_compute();
      if (tid < 3) {
        double sacc = 0.0;
        for (int wq = 0; wq < kComputeThreads / 32; ++wq) sacc += red[tid * 8 + wq];
        if (sacc != 0.0) atomicAdd(a.sums + tid, sacc);
      }
    }
  }
  if (ktrace) ktrace[2] = clock64();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
  if (ktrace) ktrace[3] = clock64();
}

__device__ __forceinline__ float hi16(float v) { return __half2float(__float2half_rn(v)); }

// fp32 [K][N] panels of the fp32 blob -> fp16 weight block in the canonical K-major no-swizzle UMMA layout.
// block element (n, k): n in [0,96) output feature, k in [0,112): k < 96 weight W[k0+k][n0+n]; k = 96/97 bias hi/lo.
// A LayerNorm in front of the GEMM is folded in (GraFormer.py:67-70: y = a_2 n + b_2 with n the normalised row): the weight
// rows are scaled by a_2, and the shift b_2 W goes
//   fold = 1: into the bias (the GEMM reads y directly: q, k, v);
//   fold = 2: into rows k = 98..100 as (hi, lo, hi) of beta = b_2 W, to be multiplied by the joint slab (r_hi, r_hi, r_lo):
//             the GEMM reads L^ y = (L^ n) a_2 + r b_2^T, r = row sums of L^ (fc1 of the GraphNet).
__global__ void tc2_pack_block_kernel(uint8_t* __restrict__ dst, const float* __restrict__ W, int ldw, int k0, int n0,
                                      const float* __restrict__ bias, const float* __restrict__ ln_a, const float* __restrict__ ln_b, int fold) {
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 96 * WK; idx += gridDim.x * blockDim.x) {
    const int n = idx / WK, k = idx - n * WK;
    float v = 0.f;
    if (k < 96) {
      v = W[(size_t)(k0 + k) * ldw + n0 + n];
      if (fold) v *= ln_a[k0 + k];
    } else if (k <= 100) {
      float beta = 0.f;
      if (fold) for (int j = 0; j < 96; ++j) beta = fmaf(ln_b[k0 + j], W[(size_t)(k0 + j) * ldw + n0 + n], beta);
      const float b = (bias != nullptr ? bias[n] : 0.f) + (fold == 1 ? beta : 0.f);
      if (k == 96) v = hi16(b);
      else if (k == 97) v = b - hi16(b);
      else if (fold == 2) v = (k == 99) ? beta - hi16(beta) : hi16(beta);
    }
    const size_t off = (size_t)(k >> 3) * W_LBO + (size_t)(n >> 3) * W_SBO + (n & 7) * 16 + (k & 7) * 2;
    *reinterpret_cast<__half*>(dst + off) = __float2half_rn(v);
  }
}

// Input convolution block [N=96][K=48]: K slabs [hi ; hi ; lo] of the panel weights Win [3*c_in][96]; panel position
// k = order*5 + coordinate (coordinates >= c_in are zero), the bias sits in row 15.
// Output convolution block [N=16][K=288] (K-adjacent core matrices OUT_LBO apart): slabs [hi ; hi ; lo] of Wout
// [3][96][c_out] reshaped to columns order*5 + output (outputs >= c_out and column 15 are zero).  Both blocks are zero
// padded to WBLK_BYTES.
__global__ void tc2_pack_io_kernel(uint8_t* __restrict__ dst, const float* __restrict__ win, const float* __restrict__ bin,
                                   const float* __restrict__ wout, int c_in, int c_out) {
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 96 * 48; idx += gridDim.x * blockDim.x) {
    const int n = idx / 48, k = idx - n * 48;
    const int slab = k >> 4, kk = k & 15;
    float full = 0.f;
    if (kk == 15) full = bin[n];
    else if (kk % 5 < c_in) full = win[((kk / 5) * c_in + kk % 5) * 96 + n];
    const float v = slab < 2 ? hi16(full) : full - hi16(full);
    const size_t off = (size_t)(k >> 3) * W_LBO + (size_t)(n >> 3) * W_SBO + (n & 7) * 16 + (k & 7) * 2;
    *reinterpret_cast<__half*>(dst + off) = __float2half_rn(v);
  }
  uint8_t* d2 = dst + WBLK_BYTES;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 16 * 288; idx += gridDim.x * blockDim.x) {
    const int n = idx / 288, k = idx - n * 288;
    const int slab = k / 96, ch = k - slab * 96;
    float full = 0.f;
    if (n < 15 && n % 5 < c_out) full = wout[((n / 5) * 96 + ch) * c_out + (n % 5)];
    const float v = slab < 2 ? hi16(full) : full - hi16(full);
    const size_t off = (size_t)(k >> 3) * OUT_LBO + (size_t)(n >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2;
    *reinterpret_cast<__half*>(d2 + off) = __float2half_rn(v);
  }
}

// per-layer parameter record: L^ as fp16 [4 chunk columns][17 rows][8], then the joint slab rows [18][8]:
// (1, 1, r_hi, r_hi, r_lo, 0, 0, 0) with r_i = sum_j L^[i][j] in fp32 (row 17, the pad row of a pose, is zero)
__global__ void tc2_pack_lparams_kernel(uint8_t* __restrict__ dst, const float* __restrict__ lhat) {
  __half* hp = reinterpret_cast<__half*>(dst);
  for (int i = threadIdx.x; i < 4 * NP * 8; i += blockDim.x) {
    const int kc = i / (NP * 8), r = (i / 8) % NP, e = i & 7;
    const int k = kc * 8 + e;
    hp[i] = __float2half_rn(k < NP ? lhat[r * NP + k] : 0.f);
  }
  __half* js = reinterpret_cast<__half*>(dst + LP_LHAT_BYTES);
  for (int i = threadIdx.x; i < PS; i += blockDim.x) {
    float r = 0.f;
    if (i < NP) for (int j = 0; j < NP; ++j) r += lhat[i * NP + j];
    const float one = i < NP ? 1.f : 0.f, rh = hi16(r);
    const float vals[8] = {one, one, rh, rh, r - rh, 0.f, 0.f, 0.f};
    for (int e = 0; e < 8; ++e) js[i * 8 + e] = __float2half_rn(i < NP ? vals[e] : 0.f);
  }
}

// Time embedding of the sampler as a bias block of GC2 (gcndiff.py:48-53: GC2(relu(GC1 x) + temb)):
// sum_k T_k (1 temb^T) W_k = sum_k p_k (temb^T W_k), p_k = row sums of T_k (the Chebyshev slab of the kernel).
// One block per (step, layer): [96 outputs][8] = (u0_hi, u0_lo, u1_hi, u1_lo, u1_hi, u2_hi, u2_lo, u2_hi), u_k = temb^T W_k.
__global__ void tc2_tau_kernel(uint8_t* __restrict__ dst, const float* __restrict__ temb, const Weights* __restrict__ w, int n_layer) {
  const float* t = temb + (size_t)blockIdx.x * H;          // table rows are [step][layer]
  const float* wc2 = w->layer[blockIdx.x % n_layer].wc2;
  const int n = threadIdx.x;
  float u[3];
  for (int k = 0; k < 3; ++k) {
    float acc = 0.f;
    for (int c = 0; c < H; ++c) acc = fmaf(t[c], wc2[(size_t)(k * H + c) * H + n], acc);
    u[k] = acc;
  }
  const float h0 = hi16(u[0]), h1 = hi16(u[1]), h2 = hi16(u[2]);
  *reinterpret_cast<uint4*>(dst + (size_t)blockIdx.x * LP_TAU_BYTES + n * 16) =
      make_uint4(pack2(h0, u[0] - h0), pack2(h1, u[1] - h1), pack2(h1, h2), pack2(u[2] - h2, h2));
}

}  // namespace

// m->temb holds the [n_steps][n_layer][96] table of the schedule (simt_temb): derive the GC2 bias blocks from it
int tc2_tau(dp_model* m, int n_steps, cudaStream_t s) {
  if (!m->d.has_temb) return DP_OK;
  DP_TRY(m->tc2_tau.reserve((size_t)n_steps * m->d.n_layer * LP_TAU_BYTES));
  tc2_tau_kernel<<<n_steps * m->d.n_layer, H, 0, s>>>(m->tc2_tau.get<uint8_t>(), m->temb.get<float>(), m->dw.get<Weights>(), m->d.n_layer);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

// `bias` points at the first of the 96 bias values of this block (or NULL)
static int pack_block(uint8_t* dst, const float* W, int ldw, int k0, int n0, const float* bias, cudaStream_t s, const float* ln_a = nullptr,
                      const float* ln_b = nullptr, int fold = 0) {
  tc2_pack_block_kernel<<<12, 256, 0, s>>>(dst, W, ldw, k0, n0, bias, ln_a, ln_b, fold);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

int tc2_pack(dp_model* m, cudaStream_t s) {
  const Dims& d = m->d;
  // [n_layer][14][WBLK_BYTES] weight blocks, then [2][WBLK_BYTES] io blocks, then [n_layer][LP_BYTES] per-layer parameters
  const size_t wbytes = (size_t)d.n_layer * BLOCKS_PER_LAYER * WBLK_BYTES;
  const size_t need = wbytes + 2 * WBLK_BYTES + (size_t)d.n_layer * LP_BYTES;
  DP_TRY(m->tc2_blocks.reserve(need));
  uint8_t* blocks = m->tc2_blocks.get<uint8_t>();
  DP_CUDA(cudaMemsetAsync(blocks, 0, need, s));
  for (int l = 0; l < d.n_layer; ++l) {
    const LayerW& L = m->hw.layer[l];
    uint8_t* b = blocks + (size_t)l * BLOCKS_PER_LAYER * WBLK_BYTES;
    int i = 0;
    // consumption order of the issuer: q, k, v, o, fc1 (two output halves), fc2 (two input halves; the first carries b2,
    // which the kernel adds to the residual stream), cheb1 x3, cheb2 x3
    for (int part = 0; part < 3; ++part) DP_TRY(pack_block(b + (size_t)(i++) * WBLK_BYTES, L.wqkv, 3 * H, 0, part * H, L.bqkv + part * H, s, L.ln0_a, L.ln0_b, 1));
    DP_TRY(pack_block(b + (size_t)(i++) * WBLK_BYTES, L.wo, H, 0, 0, L.bo, s));
    for (int part = 0; part < 2; ++part) DP_TRY(pack_block(b + (size_t)(i++) * WBLK_BYTES, L.w1, 2 * H, 0, part * H, L.b1 + part * H, s, L.ln1_a, L.ln1_b, 2));
    for (int part = 0; part < 2; ++part) DP_TRY(pack_block(b + (size_t)(i++) * WBLK_BYTES, L.w2, H, part * H, 0, part == 0 ? L.b2 : nullptr, s));
    for (int part = 0; part < 3; ++part) DP_TRY(pack_block(b + (size_t)(i++) * WBLK_BYTES, L.wc1, H, part * H, 0, part == 0 ? L.bc1 : nullptr, s));
    for (int part = 0; part < 3; ++part) DP_TRY(pack_block(b + (size_t)(i++) * WBLK_BYTES, L.wc2, H, part * H, 0, part == 0 ? L.bc2 : nullptr, s));
    tc2_pack_lparams_kernel<<<1, 128, 0, s>>>(blocks + wbytes + 2 * WBLK_BYTES + (size_t)l * LP_BYTES, L.lhat);
    count_launch();
    DP_CUDA(cudaGetLastError());
  }
  tc2_pack_io_kernel<<<18, 256, 0, s>>>(blocks + wbytes, m->hw.win, m->hw.bin, m->hw.wout, d.c_in, d.c_out);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

int tc2_run(dp_model* m, const EngineCall& c, cudaStream_t s) {
  const uint8_t* blocks = m->tc2_blocks.get<uint8_t>();
  if (!blocks) { set_error("tensor-core engine: weights are not packed"); return DP_ERR_STATE; }
  DP_TRY((smem_opt_in<tc2_kernel<false, false, false>>(m->device, SMEM_BYTES)));
  DP_TRY((smem_opt_in<tc2_kernel<true, false, false>>(m->device, SMEM_BYTES)));
  DP_TRY((smem_opt_in<tc2_kernel<false, true, false>>(m->device, SMEM_BYTES)));
  DP_TRY((smem_opt_in<tc2_kernel<false, false, true>>(m->device, SMEM_BYTES)));
  DP_TRY((smem_opt_in<tc2_kernel<false, true, true>>(m->device, SMEM_BYTES)));
  const size_t wbytes = (size_t)m->d.n_layer * BLOCKS_PER_LAYER * WBLK_BYTES;
  Tc2Args a{};
  a.w = m->dw.get<Weights>(); a.wpack = blocks; a.ioblocks = blocks + wbytes; a.lparams = blocks + wbytes + 2 * WBLK_BYTES;
  a.n_layer = m->d.n_layer; a.c_in = m->d.c_in; a.c_out = m->d.c_out; a.forward_only = c.forward_only; a.has_temb = m->d.has_temb;
  a.x_in = c.x_in; a.x_is_repeated = c.x_is_repeated; a.out = c.out;
  a.n_rows = c.n_pose * c.n_hyp; a.n_pose = c.n_pose; a.n_hyp = c.n_hyp; a.mean_over_hyp = c.mean_over_hyp; a.n_steps = c.n_steps;
  a.temb = m->temb.get<float>(); a.tau = m->tc2_tau.get<uint8_t>(); a.noise = c.noise; a.key = c.key; a.mask = c.mask; a.steps_dev = c.steps_dev;
  a.gt = c.gt; a.sums = c.sums; a.trace = m->trace; a.trace_cap = m->trace_cap;
  const long n_tiles = (a.n_rows + TP - 1) / TP;
  if (n_tiles > 0x7fffffffL) { set_error("tensor-core engine: more than 2^31 tiles of 7 poses in one call"); return DP_ERR_INVALID; }
  int grid = (int)(n_tiles < m->sm_count ? n_tiles : m->sm_count);
  if (a.mean_over_hyp) grid = (int)(a.n_pose < m->sm_count ? a.n_pose : m->sm_count);   // CTAs own whole poses
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  // a keyed call runs a keyed instantiation (without the hand-over trace, which only the plain sampler records)
  if (a.key.on && a.gt != nullptr) DP_CUDA(cudaLaunchKernelEx(&cfg, tc2_kernel<false, true, true>, a, *c.inl));
  else if (a.key.on) DP_CUDA(cudaLaunchKernelEx(&cfg, tc2_kernel<false, false, true>, a, *c.inl));
  else if (a.gt != nullptr) DP_CUDA(cudaLaunchKernelEx(&cfg, tc2_kernel<false, true, false>, a, *c.inl));
  else if (a.trace != nullptr) DP_CUDA(cudaLaunchKernelEx(&cfg, tc2_kernel<true, false, false>, a, *c.inl));
  else DP_CUDA(cudaLaunchKernelEx(&cfg, tc2_kernel<false, false, false>, a, *c.inl));
  count_launch();
  record_launch(m, grid, kThreads, SMEM_BYTES, TP, DP_ENGINE_TCG, n_tiles);
  return DP_OK;
}

}  // namespace dp
