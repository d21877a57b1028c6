// Split-precision tensor-core engine ("tcx"): the ACCURATE tcgen05 path.  Persistent sm_100a kernel, one 128-row tile
// (7 poses x 17 joints) per CTA, every layer (and, for the sampler, every DDIM step) executed without leaving the SM.
//
// Why it exists: the default engine (dp_tc2.cu) rounds every tensor-core operand to fp16 (11-bit significand).  Behind a
// DDIM schedule that error is damped (x_T within 1e-3 of the fp32 reference), but a plain forward call -- GCNdiff.forward
// used for a loss, and above all the GCNpose lifter whose output IS the xyz handed to the sampler -- carries it undamped:
// ~7e-4 relative, 2e-3 abs on random weights (oracle/tc_emulation.py).  Emulating the rounding points one class at a
// time shows that every class matters (activations, weights, attention probabilities, graph operands): only splitting
// all of them brings the lifter to 3e-6.  So this engine
//
//   * runs the dense projections (QKV, out-proj, GraphNet fc1/fc2, both Chebyshev convolutions: 11.0 of the 12.3 MMAC
//     per pose-forward) on tcgen05 as THREE fp16 products per K step, D += A_hi W_hi + A_lo W_hi + A_hi W_lo with
//     A = A_hi + A_lo and W = W_hi + W_lo split into fp16 pairs (~22 significand bits each, fp32 accumulation in TMEM);
//   * keeps everything else in fp32 on the CUDA cores, in shared memory: LayerNorm (unbiased std, eps on std), the
//     per-head attention with its softmax (q straight from TMEM, k and v as fp32 rows), the 17x17 graph operators
//     (Chebyshev T1/T2 over the neighbour lists, learnable-adjacency L^), the residual stream, the 5-wide input/output
//     convolutions and the DDIM update.
//
// It serves dp_forward for both model kinds (GCNdiff with per-sample timesteps, GCNpose uv -> xyz, optionally fused with
// the runner's root-centring + concat into uvxyz, runners/diffpose_frame.py:337-343) and is selectable for the sampler.
// Result: <= 2e-5 from the fp32 oracle (tests/test_gpu_tc.py) at ~6x the speed of the fp32 FMA engine.
//
// Reference semantics: see the list at the top of dp_simt.cu (same functions, same file:line).
#include <cuda_fp16.h>
#include <cmath>
#include "dp_internal.h"
#include "dp_sm100.cuh"
#include "dp_tc_layout.cuh"

namespace dp {

namespace {

using namespace sm100;
using namespace tc;

constexpr int TR = TP * NP;          // 119 valid rows (row = pose * 17 + joint)
constexpr int XLD = 100;             // fp32 row stride (floats): thread-per-row float4 access is conflict free
constexpr int NSTAGE = 3;
constexpr int A_SBO = 128;
constexpr int PAIR_BYTES = 2 * ABLK_BYTES;          // an operand = (hi block, lo block)
constexpr int NNB = NP;              // neighbour-list capacity: any graph.  The lists are padded to the longest row of the graph in
                                     // use (9 = the largest 2-hop neighbourhood of the H36M tree, support of T2 = 2L^2 - I)
constexpr int kComputeThreads = 512;   // 16 compute warps: the fp32 shared-memory phases are latency bound, so the kernel wants warps
constexpr int kThreads = kComputeThreads + 32;
constexpr int kParts = kComputeThreads / TM;          // 4 threads per tile row: 24 of the 96 channels each
constexpr int PC = H / kParts;                        // 24
constexpr int XS = 8;                // x_t / eps row stride (floats)

// shared memory map (bytes); each of the BLOCKS_PER_LAYER weight blocks is a (hi, lo) pair of ring entries
constexpr int al128(int x) { return (x + 127) / 128 * 128; }
constexpr int OFF_X = 0;                                   // fp32 residual stream [119][100]
constexpr int OFF_P0 = al128(OFF_X + TR * XLD * 4);        // operand pair 0 (hi, lo); aliased by the fp32 buffer S0 [119][100]
constexpr int OFF_P1 = OFF_P0 + al128(PAIR_BYTES);         // operand pair 1; aliased by the fp32 buffer S1
constexpr int OFF_ONES = OFF_P1 + al128(PAIR_BYTES);       // constant-one K slab (the bias rides in the MMA)
constexpr int OFF_W = al128(OFF_ONES + ONES_BYTES);        // weight ring
constexpr int OFF_XT = OFF_W + NSTAGE * WBLK_BYTES;        // x_t [128][8] fp32
constexpr int OFF_EP = OFF_XT + TM * XS * 4;               // eps [128][8] fp32
constexpr int OFF_NBI = OFF_EP + TM * XS * 4;              // neighbour index  [17][17] int, then the per-row counts [17]
constexpr int OFF_NBC = al16(OFF_NBI + (NP * NNB + NP) * 4);   // neighbour coeffs [17][17] float2 (T1, T2)
constexpr int OFF_LH = al16(OFF_NBC + NP * NNB * 8);       // L^ [17][17]
constexpr int OFF_TE = al16(OFF_LH + NP * NP * 4);         // temb rows of the current layer: [7][96] (forward) or [96] (sampler)
constexpr int OFF_MASK = OFF_TE + TP * H * 4;              // key mask [32]
constexpr int OFF_BAR = OFF_MASK + 128;                    // mbarriers: full[3], empty[3], done
constexpr int OFF_TMEM = OFF_BAR + 128;
constexpr int SMEM_BYTES = OFF_TMEM + 16;
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
static_assert(TR * XLD * 4 <= PAIR_BYTES, "an fp32 buffer must fit the operand pair it aliases");
static_assert(OFF_W % 128 == 0 && OFF_P0 % 128 == 0 && OFF_P1 % 128 == 0 && OFF_ONES % 16 == 0 && OFF_BAR % 16 == 0 && OFF_NBC % 16 == 0 &&
              OFF_XT % 16 == 0 && OFF_TE % 16 == 0, "alignment");

__device__ __forceinline__ void bar_compute() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
// Instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 (bit 4), A=B=f16 (0), K-major both, N>>3 at 17, M>>4 at 24
constexpr uint32_t kIdescN96 = (1u << 4) | ((96u >> 3) << 17) | ((128u >> 4) << 24);

// byte offset of the 16-byte chunk holding elements (row, 8*kc .. 8*kc+7) inside an fp16 operand block
__device__ __forceinline__ uint32_t a_chunk(int row, int kc) { return kc * A_LBO + (row >> 3) * A_SBO + (row & 7) * 16; }

// v[0..8) = hi + lo, both fp16 -> chunk (row, kc) of the hi and the lo block of an operand pair
__device__ __forceinline__ void store_split(uint8_t* pair, int row, int kc, const float* v) {
  uint4 hi, lo;
  split8(v, hi, lo);
  *reinterpret_cast<uint4*>(pair + a_chunk(row, kc)) = hi;
  *reinterpret_cast<uint4*>(pair + ABLK_BYTES + a_chunk(row, kc)) = lo;
}
// rows 119..127 of an operand: any finite value (their accumulator rows are never read)
__device__ __forceinline__ void store_zero(uint8_t* pair, int row, int kc) {
  *reinterpret_cast<uint4*>(pair + a_chunk(row, kc)) = make_uint4(0, 0, 0, 0);
  *reinterpret_cast<uint4*>(pair + ABLK_BYTES + a_chunk(row, kc)) = make_uint4(0, 0, 0, 0);
}

struct TcxArgs {
  const Weights* w;          // fp32 blob (LayerNorm, L^, b2, in/out convolutions)
  const uint8_t* wpack;      // fp16 weight blocks [n_layer][14][2 (hi, lo)][21504 B]
  int n_layer;
  int c_in, c_out;           // coordinate widths (<= 5): uvxyz -> uvxyz for GCNdiff, uv -> xyz for GCNpose
  int forward_only;          // 1: a single denoiser / lifter forward (dp_forward); 0: the DDIM loop
  int has_temb;
  int emit_uvxyz;            // forward_only GCNpose: write [uv | xyz - xyz_root] (5 wide) instead of xyz (dp_lift)
  const float* x_in;
  int x_is_repeated;
  float* out;
  long n_rows, n_pose;
  int n_steps;
  const float* temb;         // sampler: [n_steps][n_layer][96]; forward: [n_rows][n_layer][96]
  const float* noise;
  NoiseKey key;              // key.on: z from the keyed stream instead (noise is NULL)
  const unsigned char* mask;
  const dp_step* steps_dev;
};

struct Pipe {
  uint32_t full0, empty0, done;   // smem addresses of the barriers
  uint32_t stage, phase;          // weight ring position (thread 0 and the producer keep their own copy)
  uint32_t done_phase;            // every compute thread tracks the parity of the "GEMM finished" barrier
};

// D[:, 0..96) (+)= A W^T (+ bias) at split precision: A = operand pair (hi, lo), W = two consecutive ring entries (hi with
// the bias slab, lo).  Largest terms first.  Issued by a single thread.
__device__ __forceinline__ void issue_gemm(Pipe& p, uint32_t smem_base, uint32_t tmem_d, int pair_off, bool accumulate, bool bias) {
  const uint32_t ah = smem_base + pair_off, al = ah + ABLK_BYTES;
  mbar_wait(p.full0 + 8 * p.stage, p.phase);
  tc_fence_after();
  uint32_t wa = smem_base + OFF_W + p.stage * WBLK_BYTES;
#pragma unroll
  for (int ks = 0; ks < 6; ++ks)
    umma_f16(tmem_d, make_desc(ah + ks * 2 * A_LBO, A_LBO, A_SBO), make_desc(wa + ks * 2 * W_LBO, W_LBO, W_SBO), kIdescN96,
             (accumulate || ks > 0) ? 1u : 0u);
  if (bias)
    umma_f16(tmem_d, make_desc(smem_base + OFF_ONES, A_LBO, A_SBO), make_desc(wa + 12 * W_LBO, W_LBO, W_SBO), kIdescN96, 1u);
#pragma unroll
  for (int ks = 0; ks < 6; ++ks)
    umma_f16(tmem_d, make_desc(al + ks * 2 * A_LBO, A_LBO, A_SBO), make_desc(wa + ks * 2 * W_LBO, W_LBO, W_SBO), kIdescN96, 1u);
  umma_commit(p.empty0 + 8 * p.stage);   // the stage is free once these MMAs have read it
  if (++p.stage == NSTAGE) { p.stage = 0; p.phase ^= 1; }
  mbar_wait(p.full0 + 8 * p.stage, p.phase);
  tc_fence_after();
  wa = smem_base + OFF_W + p.stage * WBLK_BYTES;
#pragma unroll
  for (int ks = 0; ks < 6; ++ks)
    umma_f16(tmem_d, make_desc(ah + ks * 2 * A_LBO, A_LBO, A_SBO), make_desc(wa + ks * 2 * W_LBO, W_LBO, W_SBO), kIdescN96, 1u);
  umma_commit(p.empty0 + 8 * p.stage);
  if (++p.stage == NSTAGE) { p.stage = 0; p.phase ^= 1; }
}

// after an operand was written with ordinary stores: make it visible to the tensor core (async proxy), then sync
__device__ __forceinline__ void publish_operand() {
  fence_async_smem();
  tc_fence_before();
  bar_compute();
}
__device__ __forceinline__ void wait_gemm(Pipe& p) {
  mbar_wait(p.done, p.done_phase);
  p.done_phase ^= 1;
  tc_fence_after();
}

// Thread map of the 16 compute warps: warp w owns tile rows 32*(w&3).. (the TMEM lanes a warp may touch) and the 24-channel
// part (w>>2) of them.
struct Tm {
  int row, part;
  uint32_t taddr;     // TMEM address of this thread's lane, column 0
};
__device__ __forceinline__ Tm thread_map(uint32_t tmem_base) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  Tm t;
  t.row = (warp & 3) * 32 + lane;
  t.part = warp >> 2;
  t.taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
  return t;
}

// Epilogues of a 96-column accumulator: every thread handles the 24 columns of its part.
enum EpiKind { EPI_F32 = 0, EPI_XADD = 1, EPI_RELU_SPLIT = 2 };

template <int KIND>
__device__ __forceinline__ void epilogue(uint8_t* smem, const Tm& t, uint32_t acc_col, int dst_off) {
  float v[PC];
  tmem_ld24(t.taddr + acc_col + PC * t.part, v);     // (warp-collective: every lane takes part, valid row or not)
  if (KIND == EPI_RELU_SPLIT) {
    uint8_t* pair = smem + dst_off;
#pragma unroll
    for (int i = 0; i < PC; ++i) v[i] = fmaxf(v[i], 0.f);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      if (t.row < TR) store_split(pair, t.row, 3 * t.part + c, v + 8 * c);
      else store_zero(pair, t.row, 3 * t.part + c);
    }
    return;
  }
  if (t.row >= TR) return;
  float* dst = reinterpret_cast<float*>(smem + (KIND == EPI_XADD ? OFF_X : dst_off)) + t.row * XLD + PC * t.part;
#pragma unroll
  for (int i = 0; i < PC; i += 4) {
    float4 o = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
    if (KIND == EPI_XADD) {
      const float4 x = *reinterpret_cast<float4*>(dst + i);
      o.x += x.x; o.y += x.y; o.z += x.z; o.w += x.w;
    }
    *reinterpret_cast<float4*>(dst + i) = o;
  }
}

// LayerNorm of the residual stream (GraFormer.py:67-70: unbiased std, eps added to std): lanes 4r .. 4r+3 own the four
// 24-channel parts of row r.  TO_OPERAND: split into the operand pair at dst_off; else fp32 rows at dst_off.
template <bool TO_OPERAND>
__device__ __forceinline__ void layer_norm_tile(uint8_t* smem, int dst_off, const float* __restrict__ ga, const float* __restrict__ gb) {
  const int row = threadIdx.x >> 2, q4 = threadIdx.x & 3;
  const float* xr = reinterpret_cast<const float*>(smem + OFF_X) + min(row, TR - 1) * XLD + q4 * PC;
  float v[PC];
#pragma unroll
  for (int q = 0; q < PC / 4; ++q) {
    const float4 u = *reinterpret_cast<const float4*>(xr + 4 * q);
    v[4 * q] = u.x; v[4 * q + 1] = u.y; v[4 * q + 2] = u.z; v[4 * q + 3] = u.w;
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < PC; ++i) s += v[i];
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  const float mean = s * (1.0f / (float)H);
  float q2 = 0.f;
#pragma unroll
  for (int i = 0; i < PC; ++i) { v[i] -= mean; q2 = fmaf(v[i], v[i], q2); }
  q2 += __shfl_xor_sync(0xffffffffu, q2, 1);
  q2 += __shfl_xor_sync(0xffffffffu, q2, 2);
  const float inv = 1.0f / (sqrtf(q2 * (1.0f / (float)(H - 1))) + 1e-6f);
  if (row >= TR) {
    if (TO_OPERAND) {
#pragma unroll
      for (int c = 0; c < 3; ++c) store_zero(smem + dst_off, row, q4 * 3 + c);
    }
    return;
  }
#pragma unroll
  for (int q = 0; q < PC / 4; ++q) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(ga + q4 * PC) + q), b = __ldg(reinterpret_cast<const float4*>(gb + q4 * PC) + q);
    v[4 * q] = fmaf(a.x * inv, v[4 * q], b.x); v[4 * q + 1] = fmaf(a.y * inv, v[4 * q + 1], b.y);
    v[4 * q + 2] = fmaf(a.z * inv, v[4 * q + 2], b.z); v[4 * q + 3] = fmaf(a.w * inv, v[4 * q + 3], b.w);
  }
  if (TO_OPERAND) {
#pragma unroll
    for (int c = 0; c < 3; ++c) store_split(smem + dst_off, row, q4 * 3 + c, v + 8 * c);
  } else {
    float* y = reinterpret_cast<float*>(smem + dst_off) + row * XLD + q4 * PC;
#pragma unroll
    for (int q = 0; q < PC / 4; ++q) *reinterpret_cast<float4*>(y + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  }
}

// Multi-head attention over the joints of each pose (GraFormer.py:99-113) in fp32.  q: this thread's row straight from
// the accumulator columns [0, 96) in TMEM; k, v: fp32 rows in S0 / S1.  One thread per (row, head): warp w owns rows
// 32*(w&3).. and head w>>2.  The output stays in registers until every thread has finished reading v (S1 aliases the
// operand pair the result is written to).
__device__ __forceinline__ void attention_tile(uint8_t* smem, const Tm& t, int out_pair_off) {
  const int h = t.part;
  const float* maskf = reinterpret_cast<const float*>(smem + OFF_MASK);
  const float* K = reinterpret_cast<const float*>(smem + OFF_P0);
  const float* V = reinterpret_cast<const float*>(smem + OFF_P1);
  const float scale = 1.0f / sqrtf(24.0f);
  const int p = min(t.row, TR - 1) / NP;
  float q[PC];
  tmem_ld24(t.taddr + PC * h, q);
  float sc[NP];
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const float* kr = K + (p * NP + j) * XLD + PC * h;
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const float4 kv = *reinterpret_cast<const float4*>(kr + 4 * c);
      s = fmaf(q[4 * c], kv.x, s); s = fmaf(q[4 * c + 1], kv.y, s); s = fmaf(q[4 * c + 2], kv.z, s); s = fmaf(q[4 * c + 3], kv.w, s);
    }
    s = s * scale;
    if (maskf[j] == 0.f) s = -1e9f;
    sc[j] = s;
    mx = fmaxf(mx, s);
  }
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < NP; ++j) { sc[j] = expf(sc[j] - mx); sum += sc[j]; }
  const float inv = 1.0f / sum;
  float o[PC];
#pragma unroll
  for (int e = 0; e < PC; ++e) o[e] = 0.f;
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    const float* vr = V + (p * NP + j) * XLD + PC * h;
    const float pj = sc[j] * inv;
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const float4 vv = *reinterpret_cast<const float4*>(vr + 4 * c);
      o[4 * c] = fmaf(pj, vv.x, o[4 * c]); o[4 * c + 1] = fmaf(pj, vv.y, o[4 * c + 1]);
      o[4 * c + 2] = fmaf(pj, vv.z, o[4 * c + 2]); o[4 * c + 3] = fmaf(pj, vv.w, o[4 * c + 3]);
    }
  }
  tc_fence_before();
  bar_compute();               // everybody is done with k and v
  uint8_t* pair = smem + out_pair_off;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (t.row < TR) store_split(pair, t.row, 3 * h + c, o + 8 * c);
    else store_zero(pair, t.row, 3 * h + c);
  }
}

// out[i] = sum_j L^[i][j] Y[j] over the pose of row i (GraFormer.py:174-186), Y fp32 rows at src_off -> operand pair
__device__ __forceinline__ void lhat_to_operand(uint8_t* smem, int src_off, int pair_off) {
  const int row = threadIdx.x & 127;
  uint8_t* pair = smem + pair_off;
  if (row >= TR) {
    for (int kc = threadIdx.x >> 7; kc < 12; kc += kParts) store_zero(pair, row, kc);
    return;
  }
  const float* Y = reinterpret_cast<const float*>(smem + src_off);
  const float* lh = reinterpret_cast<const float*>(smem + OFF_LH);
  const int p = row / NP, i = row - p * NP;
  float co[NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) co[j] = lh[i * NP + j];
  for (int kc = threadIdx.x >> 7; kc < 12; kc += kParts) {
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const float* src = Y + (p * NP + j) * XLD + kc * 8;
      const float4 u0 = *reinterpret_cast<const float4*>(src), u1 = *reinterpret_cast<const float4*>(src + 4);
      acc[0] = fmaf(co[j], u0.x, acc[0]); acc[1] = fmaf(co[j], u0.y, acc[1]); acc[2] = fmaf(co[j], u0.z, acc[2]); acc[3] = fmaf(co[j], u0.w, acc[3]);
      acc[4] = fmaf(co[j], u1.x, acc[4]); acc[5] = fmaf(co[j], u1.y, acc[5]); acc[6] = fmaf(co[j], u1.z, acc[6]); acc[7] = fmaf(co[j], u1.w, acc[7]);
    }
    store_split(pair, row, kc, acc);
  }
}

// X[i] += sum_j L^[i][j] Z[j] + b2   (second LAM_Gconv with fc2 commuted in front of the aggregation), Z fp32 rows at src_off
__device__ __forceinline__ void lhat_residual(uint8_t* smem, int src_off, const float* __restrict__ b2) {
  const int row = threadIdx.x & 127;
  if (row >= TR) return;
  const float* Z = reinterpret_cast<const float*>(smem + src_off);
  float* X = reinterpret_cast<float*>(smem + OFF_X) + row * XLD;
  const float* lh = reinterpret_cast<const float*>(smem + OFF_LH);
  const int p = row / NP, i = row - p * NP;
  float co[NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) co[j] = lh[i * NP + j];
  for (int kc = threadIdx.x >> 7; kc < 12; kc += kParts) {
    float acc[8];
    const float4 bb0 = __ldg(reinterpret_cast<const float4*>(b2 + kc * 8)), bb1 = __ldg(reinterpret_cast<const float4*>(b2 + kc * 8 + 4));
    acc[0] = bb0.x; acc[1] = bb0.y; acc[2] = bb0.z; acc[3] = bb0.w; acc[4] = bb1.x; acc[5] = bb1.y; acc[6] = bb1.z; acc[7] = bb1.w;
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const float* src = Z + (p * NP + j) * XLD + kc * 8;
      const float4 u0 = *reinterpret_cast<const float4*>(src), u1 = *reinterpret_cast<const float4*>(src + 4);
      acc[0] = fmaf(co[j], u0.x, acc[0]); acc[1] = fmaf(co[j], u0.y, acc[1]); acc[2] = fmaf(co[j], u0.z, acc[2]); acc[3] = fmaf(co[j], u0.w, acc[3]);
      acc[4] = fmaf(co[j], u1.x, acc[4]); acc[5] = fmaf(co[j], u1.y, acc[5]); acc[6] = fmaf(co[j], u1.z, acc[6]); acc[7] = fmaf(co[j], u1.w, acc[7]);
    }
    float4 x0 = *reinterpret_cast<float4*>(X + kc * 8), x1 = *reinterpret_cast<float4*>(X + kc * 8 + 4);
    x0.x += acc[0]; x0.y += acc[1]; x0.z += acc[2]; x0.w += acc[3]; x1.x += acc[4]; x1.y += acc[5]; x1.z += acc[6]; x1.w += acc[7];
    *reinterpret_cast<float4*>(X + kc * 8) = x0;
    *reinterpret_cast<float4*>(X + kc * 8 + 4) = x1;
  }
}

// fp32 rows at src_off -> split operand pair (the A side of a Chebyshev block: [v W0 | v W1 | v W2] from one operand)
__device__ __forceinline__ void rows_to_operand(uint8_t* smem, int src_off, int pair_off) {
  const int row = threadIdx.x & 127;
  uint8_t* pair = smem + pair_off;
  const float* V = reinterpret_cast<const float*>(smem + src_off);
  for (int kc = threadIdx.x >> 7; kc < 12; kc += kParts) {
    if (row >= TR) { store_zero(pair, row, kc); continue; }
    const float* src = V + row * XLD + kc * 8;
    const float4 u0 = *reinterpret_cast<const float4*>(src), u1 = *reinterpret_cast<const float4*>(src + 4);
    const float u[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
    store_split(pair, row, kc, u);
  }
}

// Chebyshev block, aggregation AFTER the products (ChebConv.py:74-88: sum_k T_k (v W_k) = (v W0) + T1 (v W1) + T2 (v W2)):
// the three products sit in the accumulators at columns 0 (with the bias), 96 and 192.  Phase 1: Y1, Y2 -> fp32 rows S0, S1.
// Phase 2 (after a barrier): out = relu(acc0 + T1 Y1 + T2 Y2) over the neighbour list of the row's joint, 24 channels per
// thread.  One GEMM wait per block instead of three, and T1 / T2 share one pass.
__device__ __forceinline__ void cheb_stage_y(uint8_t* smem, const Tm& t) {
  epilogue<EPI_F32>(smem, t, 96, OFF_P0);
  epilogue<EPI_F32>(smem, t, 192, OFF_P1);
}
__device__ __forceinline__ void cheb_aggregate(uint8_t* smem, const Tm& t, int nnb, float* out) {
  tmem_ld24(t.taddr + PC * t.part, out);
  if (t.row >= TR) return;
  const int* nbi = reinterpret_cast<const int*>(smem + OFF_NBI);
  const float2* nbc = reinterpret_cast<const float2*>(smem + OFF_NBC);
  const float* Y1 = reinterpret_cast<const float*>(smem + OFF_P0) + PC * t.part;
  const float* Y2 = reinterpret_cast<const float*>(smem + OFF_P1) + PC * t.part;
  const int p = t.row / NP, i = t.row - p * NP;
#pragma unroll 3
  for (int n = 0; n < nnb; ++n) {
    const int rj = (p * NP + nbi[i * NNB + n]) * XLD;
    const float2 cf = nbc[i * NNB + n];
#pragma unroll
    for (int c = 0; c < PC; c += 4) {
      const float4 a = *reinterpret_cast<const float4*>(Y1 + rj + c), b = *reinterpret_cast<const float4*>(Y2 + rj + c);
      out[c] = fmaf(cf.y, b.x, fmaf(cf.x, a.x, out[c])); out[c + 1] = fmaf(cf.y, b.y, fmaf(cf.x, a.y, out[c + 1]));
      out[c + 2] = fmaf(cf.y, b.z, fmaf(cf.x, a.z, out[c + 2])); out[c + 3] = fmaf(cf.y, b.w, fmaf(cf.x, a.w, out[c + 3]));
    }
  }
#pragma unroll
  for (int c = 0; c < PC; ++c) out[c] = fmaxf(out[c], 0.f);
}

__global__ void __launch_bounds__(kThreads, 1) tcx_kernel(TcxArgs a, StepsArg inl) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  float* X = reinterpret_cast<float*>(smem + OFF_X);
  float* xt = reinterpret_cast<float*>(smem + OFF_XT);
  float* ep = reinterpret_cast<float*>(smem + OFF_EP);
  float* lh = reinterpret_cast<float*>(smem + OFF_LH);
  float* te = reinterpret_cast<float*>(smem + OFF_TE);
  float* maskf = reinterpret_cast<float*>(smem + OFF_MASK);
  int* nbi = reinterpret_cast<int*>(smem + OFF_NBI);
  float2* nbc = reinterpret_cast<float2*>(smem + OFF_NBC);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_TMEM);
  const Weights& w = *a.w;

  Pipe pp;
  pp.full0 = sbase + OFF_BAR; pp.empty0 = sbase + OFF_BAR + 32; pp.done = sbase + OFF_BAR + 64;
  pp.stage = 0; pp.phase = 0; pp.done_phase = 0;

  // ---------------------------------------------------------------- one-time setup
  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) { mbar_init(pp.full0 + 8 * s, 1); mbar_init(pp.empty0 + 8 * s, 1); }
    mbar_init(pp.done, 1);
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(sbase + OFF_TMEM, TMEM_COLS);
  // constant-one K slab: element (row, 0) = (row, 1) = 1, the other 14 of the 16 columns are 0
  for (int i = tid; i < 2 * TM; i += kThreads) {
    const int row = i & 127, kc = i >> 7;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (kc == 0) v.x = pack2(1.0f, 1.0f);
    *reinterpret_cast<uint4*>(smem + OFF_ONES + a_chunk(row, kc)) = v;
  }
  if (tid < 32) maskf[tid] = (tid < NP && a.mask && a.mask[tid] == 0) ? 0.f : 1.f;
  if (tid < NP) {
    // neighbour list of joint tid: columns where T1 or T2 is non-zero, padded with (self, 0, 0) up to the capacity
    int n = 0;
    for (int j = 0; j < NP; ++j) {
      const float c1 = __ldg(w.t1 + tid * NP + j), c2 = __ldg(w.t2 + tid * NP + j);
      if (c1 != 0.f || c2 != 0.f) { nbi[tid * NNB + n] = j; nbc[tid * NNB + n] = make_float2(c1, c2); ++n; }
    }
    nbi[NP * NNB + tid] = n;
    for (; n < NNB; ++n) { nbi[tid * NNB + n] = tid; nbc[tid * NNB + n] = make_float2(0.f, 0.f); }
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  int nnb = 1;                         // longest neighbour list of this graph (every loop over a list runs to it)
  for (int j = 0; j < NP; ++j) nnb = max(nnb, nbi[NP * NNB + j]);

  const long n_tiles = (a.n_rows + TP - 1) / TP;
  const int L = a.n_layer;
  const int ci = a.c_in, co = a.c_out;

  if (warp == kComputeThreads / 32) {
    // ---------------------------------------------------------------- weight producer (TMA bulk copies): the (hi, lo) blocks
    // of a layer in the order the kernel consumes them
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
        for (int step = 0; step < a.n_steps; ++step)
          for (int blk = 0; blk < L * BLOCKS_PER_LAYER * 2; ++blk) {
            mbar_wait_sleep(pp.empty0 + 8 * stage, phase ^ 1);
            mbar_expect_tx(pp.full0 + 8 * stage, WBLK_BYTES);
            bulk_g2s(sbase + OFF_W + stage * WBLK_BYTES, a.wpack + (size_t)blk * WBLK_BYTES, WBLK_BYTES, pp.full0 + 8 * stage);
            if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
          }
    }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- compute warps
    const Tm t = thread_map(tmem_base);
    for (long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const long g0 = tile * TP;
      const int npose = (int)min((long)TP, a.n_rows - g0);
      const int R = npose * NP;
      for (int idx = tid; idx < TM * XS; idx += kComputeThreads) {
        const int r = idx >> 3, c = idx & 7;
        float v = 0.f;
        if (r < R && c < ci) {
          const long g = g0 + r / NP;
          const long src = a.x_is_repeated ? g : (g % a.n_pose);
          v = a.x_in[(src * NP + (r % NP)) * ci + c];
        }
        xt[idx] = v;
      }
      bar_compute();

      for (int step = 0; step < a.n_steps; ++step) {
        // ---- input ChebConv (K = 3 c_in <= 15): fp32 on the CUDA cores.  B[row][order * c_in + c] = (T_order x)[row][c]
        float* Bin = reinterpret_cast<float*>(smem + OFF_P0);   // [128][16]
        for (int idx = tid; idx < TM * ci; idx += kComputeThreads) {
          const int r = idx / ci, c = idx - r * ci;
          float v0 = 0.f, v1 = 0.f, v2 = 0.f;
          if (r < TR) {
            const int p = r / NP, i = r - p * NP;
            v0 = xt[r * XS + c];
            for (int n = 0; n < nnb; ++n) {
              const float u = xt[(p * NP + nbi[i * NNB + n]) * XS + c];
              const float2 cf = nbc[i * NNB + n];
              v1 = fmaf(cf.x, u, v1);
              v2 = fmaf(cf.y, u, v2);
            }
          }
          Bin[r * 16 + c] = v0; Bin[r * 16 + ci + c] = v1; Bin[r * 16 + 2 * ci + c] = v2;
        }
        bar_compute();
        {
          const int row = tid & 127, part = tid >> 7;
          if (row < TR) {
            float acc[PC];
#pragma unroll
            for (int g = 0; g < PC / 4; ++g) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(w.bin + part * PC) + g);
              acc[4 * g] = b4.x; acc[4 * g + 1] = b4.y; acc[4 * g + 2] = b4.z; acc[4 * g + 3] = b4.w;
            }
            for (int k = 0; k < 3 * ci; ++k) {
              const float bv = Bin[row * 16 + k];
#pragma unroll
              for (int g = 0; g < PC / 4; ++g) {
                const float4 w4 = __ldg(reinterpret_cast<const float4*>(w.win + k * H + part * PC) + g);
                acc[4 * g] = fmaf(bv, w4.x, acc[4 * g]); acc[4 * g + 1] = fmaf(bv, w4.y, acc[4 * g + 1]);
                acc[4 * g + 2] = fmaf(bv, w4.z, acc[4 * g + 2]); acc[4 * g + 3] = fmaf(bv, w4.w, acc[4 * g + 3]);
              }
            }
#pragma unroll
            for (int g = 0; g < PC / 4; ++g)
              *reinterpret_cast<float4*>(X + row * XLD + part * PC + 4 * g) = make_float4(acc[4 * g], acc[4 * g + 1], acc[4 * g + 2], acc[4 * g + 3]);
          }
        }
        bar_compute();

        for (int l = 0; l < L; ++l) {
          const LayerW& Lw = w.layer[l];
          for (int i = tid; i < NP * NP; i += kComputeThreads) lh[i] = __ldg(Lw.lhat + i);
          if (a.has_temb) {
            if (a.forward_only) {      // per-sample timesteps: one projected embedding row per pose
              for (int i = tid; i < TP * H; i += kComputeThreads) {
                const int p = i / H;
                te[i] = p < npose ? __ldg(a.temb + ((size_t)(g0 + p) * L + l) * H + (i - p * H)) : 0.f;
              }
            } else if (tid < H) {
              te[tid] = __ldg(a.temb + ((size_t)step * L + l) * H + tid);
            }
          }
          // ======== x = x + attn(LN0(x))
          layer_norm_tile<true>(smem, OFF_P1, Lw.ln0_a, Lw.ln0_b);
          publish_operand();
          if (tid == 0) {
            tc_fence_after();
            issue_gemm(pp, sbase, tmem_base + 0, OFF_P1, false, true);     // Q
            issue_gemm(pp, sbase, tmem_base + 96, OFF_P1, false, true);    // K
            issue_gemm(pp, sbase, tmem_base + 192, OFF_P1, false, true);   // V
            umma_commit(pp.done);
          }
          wait_gemm(pp);
          epilogue<EPI_F32>(smem, t, 96, OFF_P0);      // k -> S0
          epilogue<EPI_F32>(smem, t, 192, OFF_P1);     // v -> S1 (the GEMMs have finished reading pair 1)
          tc_fence_before();
          bar_compute();
          attention_tile(smem, t, OFF_P0);              // (syncs inside) -> pair 0
          publish_operand();
          if (tid == 0) {
            tc_fence_after();
            issue_gemm(pp, sbase, tmem_base, OFF_P0, false, true);         // out projection
            umma_commit(pp.done);
          }
          wait_gemm(pp);
          epilogue<EPI_XADD>(smem, t, 0, 0);
          tc_fence_before();
          bar_compute();
          // ======== x = x + GraphNet(LN1(x))
          layer_norm_tile<false>(smem, OFF_P1, Lw.ln1_a, Lw.ln1_b);        // y -> S1
          bar_compute();
          lhat_to_operand(smem, OFF_P1, OFF_P0);                            // L^ y -> pair 0
          publish_operand();
          if (tid == 0) {
            tc_fence_after();
            issue_gemm(pp, sbase, tmem_base + 0, OFF_P0, false, true);     // fc1, outputs 0..95
            issue_gemm(pp, sbase, tmem_base + 96, OFF_P0, false, true);    // fc1, outputs 96..191
            umma_commit(pp.done);
          }
          wait_gemm(pp);
          epilogue<EPI_RELU_SPLIT>(smem, t, 0, OFF_P0);    // relu(h[:, 0:96]) -> pair 0
          epilogue<EPI_RELU_SPLIT>(smem, t, 96, OFF_P1);   // relu(h[:, 96:192]) -> pair 1
          publish_operand();
          if (tid == 0) {
            tc_fence_after();
            issue_gemm(pp, sbase, tmem_base + 192, OFF_P0, false, false);  // fc2, inputs 0..95
            issue_gemm(pp, sbase, tmem_base + 192, OFF_P1, true, false);   // fc2, inputs 96..191
            umma_commit(pp.done);
          }
          wait_gemm(pp);
          epilogue<EPI_F32>(smem, t, 192, OFF_P1);     // z -> S1
          tc_fence_before();
          bar_compute();
          lhat_residual(smem, OFF_P1, Lw.b2);
          bar_compute();
          // ======== x = x + GC2(GC1(x) + temb): each block = one operand, three products, aggregation in the epilogue
          rows_to_operand(smem, OFF_X, OFF_P0);
          publish_operand();
          if (tid == 0) {
            tc_fence_after();
            issue_gemm(pp, sbase, tmem_base, OFF_P0, false, true);          // x W0 + b
            issue_gemm(pp, sbase, tmem_base + 96, OFF_P0, false, false);    // x W1
            issue_gemm(pp, sbase, tmem_base + 192, OFF_P0, false, false);   // x W2
            umma_commit(pp.done);
          }
          wait_gemm(pp);
          cheb_stage_y(smem, t);
          tc_fence_before();
          bar_compute();
          {
            float h1[PC];
            cheb_aggregate(smem, t, nnb, h1);   // relu(GC1(x))
            if (a.has_temb && t.row < TR) {     // + temb (gcndiff.py:51): per pose for a forward call, per step for the sampler
              const float* tr = te + (a.forward_only ? (t.row / NP) * H : 0) + PC * t.part;
#pragma unroll
              for (int c = 0; c < PC; c += 4) {
                const float4 tv = *reinterpret_cast<const float4*>(tr + c);
                h1[c] += tv.x; h1[c + 1] += tv.y; h1[c + 2] += tv.z; h1[c + 3] += tv.w;
              }
            }
            tc_fence_before();
            bar_compute();                       // everybody is done with Y1, Y2 (they alias the operand pairs)
            uint8_t* pair = smem + OFF_P0;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              if (t.row < TR) store_split(pair, t.row, 3 * t.part + c, h1 + 8 * c);
              else store_zero(pair, t.row, 3 * t.part + c);
            }
          }
          publish_operand();
          if (tid == 0) {
            tc_fence_after();
            issue_gemm(pp, sbase, tmem_base, OFF_P0, false, true);
            issue_gemm(pp, sbase, tmem_base + 96, OFF_P0, false, false);
            issue_gemm(pp, sbase, tmem_base + 192, OFF_P0, false, false);
            umma_commit(pp.done);
          }
          wait_gemm(pp);
          cheb_stage_y(smem, t);
          tc_fence_before();
          bar_compute();
          {
            float h2[PC];
            cheb_aggregate(smem, t, nnb, h2);   // relu(GC2(h1))
            if (t.row < TR) {
              float* xr = X + t.row * XLD + PC * t.part;
#pragma unroll
              for (int c = 0; c < PC; c += 4) {
                float4 x = *reinterpret_cast<float4*>(xr + c);
                x.x += h2[c]; x.y += h2[c + 1]; x.z += h2[c + 2]; x.w += h2[c + 3];
                *reinterpret_cast<float4*>(xr + c) = x;
              }
            }
          }
          tc_fence_before();
          bar_compute();
        }

        // ---- output ChebConv (N = c_out <= 5): U_k = X Wout_k on the CUDA cores, then eps = b + U0 + T1 U1 + T2 U2.
        //      Wout [3*96][c_out] is staged in shared memory first (a warp reads one channel row at a time: broadcasts).
        float* wsm = reinterpret_cast<float*>(smem + OFF_P1);
        for (int i = tid; i < 3 * H * co; i += kComputeThreads) wsm[i] = __ldg(w.wout + i);
        bar_compute();
        {
          float* U = reinterpret_cast<float*>(smem + OFF_P0);   // [4][128][16]
          const int row = tid & 127, part = tid >> 7;
          float acc[15];
#pragma unroll
          for (int i = 0; i < 15; ++i) acc[i] = 0.f;
          if (row < TR) {
            for (int cq = 0; cq < PC / 4; ++cq) {
              const float4 xv = *reinterpret_cast<const float4*>(X + row * XLD + part * PC + cq * 4);
              const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int c = part * PC + cq * 4 + e;
#pragma unroll
                for (int k3 = 0; k3 < 3; ++k3)
#pragma unroll
                  for (int n = 0; n < 5; ++n)
                    if (n < co) acc[k3 * 5 + n] = fmaf(xs[e], wsm[(k3 * H + c) * co + n], acc[k3 * 5 + n]);
              }
            }
          }
#pragma unroll
          for (int i = 0; i < 15; ++i) U[(part * TM + row) * 16 + i] = acc[i];
        }
        bar_compute();
        {
          const float* U = reinterpret_cast<const float*>(smem + OFF_P0);
          for (int idx = tid; idx < TR * co; idx += kComputeThreads) {
            const int r = idx / co, n = idx - r * co;
            const int p = r / NP, i = r - p * NP;
            float v = __ldg(w.bout + n);
#pragma unroll
            for (int pt = 0; pt < kParts; ++pt) v += U[(pt * TM + r) * 16 + n];
            for (int q = 0; q < nnb; ++q) {
              const int rj = p * NP + nbi[i * NNB + q];
              const float2 cf = nbc[i * NNB + q];
              float u1 = 0.f, u2 = 0.f;
#pragma unroll
              for (int pt = 0; pt < kParts; ++pt) { u1 += U[(pt * TM + rj) * 16 + 5 + n]; u2 += U[(pt * TM + rj) * 16 + 10 + n]; }
              v = fmaf(cf.x, u1, v);
              v = fmaf(cf.y, u2, v);
            }
            ep[r * XS + n] = v;
          }
        }
        bar_compute();
        if (a.forward_only) {
          if (a.emit_uvxyz) {
            // the runner's glue (runners/diffpose_frame.py:337-343, with the intended out-of-place root-centring):
            // [uv | xyz - xyz[root]] as the 5-wide input of the sampler
            const int wd = ci + co;
            for (int idx = tid; idx < R * wd; idx += kComputeThreads) {
              const int r = idx / wd, n = idx - r * wd;
              const int p = r / NP;
              const float v = n < ci ? xt[r * XS + n] : __fsub_rn(ep[r * XS + (n - ci)], ep[(p * NP) * XS + (n - ci)]);
              a.out[(size_t)g0 * NP * wd + idx] = v;
            }
          } else {
            for (int idx = tid; idx < R * co; idx += kComputeThreads) a.out[(size_t)g0 * NP * co + idx] = ep[(idx / co) * XS + idx % co];
          }
        } else {
          // ---- DDIM update (common/utils_diff.py:59-65), same operation order, no FMA contraction
          const dp_step st = a.steps_dev ? a.steps_dev[step] : inl.s[step];
          for (int idx = tid; idx < R * co; idx += kComputeThreads) {
            const int r = idx / co, c = idx - r * co;
            const float et = ep[r * XS + c], xv = xt[r * XS + c];
            const float x0 = __fdiv_rn(__fsub_rn(xv, __fmul_rn(et, st.sqrt_1m_at)), st.sqrt_at);
            float nx = __fmul_rn(st.sqrt_an, x0);
            if (a.noise) {
              const float z = a.noise[((size_t)step * a.n_rows + g0) * NP * co + idx];
              nx = __fadd_rn(nx, __fmul_rn(st.c1, z));
            } else if (a.key.on) {
              // hypothesis-major row g = h * n_pose + b
              const long g = g0 + r / NP, h = g / a.n_pose;
              const float z = philox_normal(a.key, a.key.step_offset + (uint32_t)step, a.key.pose_offset + (uint32_t)(g - h * a.n_pose),
                                            (uint32_t)h, (uint32_t)((r % NP) * co + c));
              nx = __fadd_rn(nx, __fmul_rn(st.c1, z));
            }
            xt[r * XS + c] = __fadd_rn(nx, __fmul_rn(st.c2, et));
          }
        }
        bar_compute();
      }
      if (!a.forward_only)
        for (int idx = tid; idx < R * co; idx += kComputeThreads) a.out[(size_t)g0 * NP * co + idx] = xt[(idx / co) * XS + idx % co];
      bar_compute();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

// fp32 [K][N] panels of the fp32 blob -> a (hi, lo) pair of fp16 weight blocks in the canonical K-major no-swizzle UMMA
// layout.  block element (n, k): n in [0,96) output feature, k in [0,112): k < 96 weight W[k0+k][n0+n] (hi = fp16(W),
// lo = fp16(W - hi)); k = 96/97 of the hi block: bias hi/lo.
__global__ void tcx_pack_block_kernel(uint8_t* __restrict__ dst, const float* __restrict__ W, int ldw, int k0, int n0,
                                      const float* __restrict__ bias) {
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 96 * WK; idx += gridDim.x * blockDim.x) {
    const int n = idx / WK, k = idx - n * WK;
    float hi = 0.f, lo = 0.f;
    if (k < 96) {
      const float v = W[(size_t)(k0 + k) * ldw + n0 + n];
      hi = __half2float(__float2half_rn(v));
      lo = v - hi;
    } else if (bias != nullptr && k == 96) {
      hi = __half2float(__float2half_rn(bias[n0 + n]));
    } else if (bias != nullptr && k == 97) {
      const float b = bias[n0 + n];
      hi = b - __half2float(__float2half_rn(b));
    }
    const size_t off = (size_t)(k >> 3) * W_LBO + (size_t)(n >> 3) * W_SBO + (n & 7) * 16 + (k & 7) * 2;
    *reinterpret_cast<__half*>(dst + off) = __float2half_rn(hi);
    *reinterpret_cast<__half*>(dst + WBLK_BYTES + off) = __float2half_rn(lo);
  }
}

}  // namespace

static int pack_block(uint8_t* dst, const float* W, int ldw, int k0, int n0, const float* bias, cudaStream_t s) {
  tcx_pack_block_kernel<<<12, 256, 0, s>>>(dst, W, ldw, k0, n0, bias);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

// Lazy: the split weights (3 MB) are built the first time this engine runs after a dp_pack, not on every weight load.
static int tcx_ensure_packed(dp_model* m, cudaStream_t s) {
  if (m->tcx_packed) return DP_OK;
  const Dims& d = m->d;
  DP_TRY(m->tcx_blocks.reserve((size_t)d.n_layer * BLOCKS_PER_LAYER * 2 * WBLK_BYTES));
  for (int l = 0; l < d.n_layer; ++l) {
    const LayerW& L = m->hw.layer[l];
    uint8_t* b = m->tcx_blocks.get<uint8_t>() + (size_t)l * BLOCKS_PER_LAYER * 2 * WBLK_BYTES;
    int i = 0;
    // consumption order of the kernel: q, k, v, o, fc1 (two output halves), fc2 (two input halves), cheb1 x3, cheb2 x3
    for (int part = 0; part < 3; ++part) DP_TRY(pack_block(b + (size_t)(i++) * 2 * WBLK_BYTES, L.wqkv, 3 * H, 0, part * H, L.bqkv, s));
    DP_TRY(pack_block(b + (size_t)(i++) * 2 * WBLK_BYTES, L.wo, H, 0, 0, L.bo, s));
    for (int part = 0; part < 2; ++part) DP_TRY(pack_block(b + (size_t)(i++) * 2 * WBLK_BYTES, L.w1, 2 * H, 0, part * H, L.b1, s));
    for (int part = 0; part < 2; ++part) DP_TRY(pack_block(b + (size_t)(i++) * 2 * WBLK_BYTES, L.w2, H, part * H, 0, nullptr, s));
    for (int part = 0; part < 3; ++part) DP_TRY(pack_block(b + (size_t)(i++) * 2 * WBLK_BYTES, L.wc1, H, part * H, 0, part == 0 ? L.bc1 : nullptr, s));
    for (int part = 0; part < 3; ++part) DP_TRY(pack_block(b + (size_t)(i++) * 2 * WBLK_BYTES, L.wc2, H, part * H, 0, part == 0 ? L.bc2 : nullptr, s));
  }
  m->tcx_packed = true;
  return DP_OK;
}

int tcx_run(dp_model* m, const EngineCall& c, cudaStream_t s) {
  DP_TRY(tcx_ensure_packed(m, s));
  DP_TRY(smem_opt_in<tcx_kernel>(m->device, SMEM_BYTES));
  TcxArgs a{};
  a.w = m->dw.get<Weights>(); a.wpack = m->tcx_blocks.get<uint8_t>(); a.n_layer = m->d.n_layer; a.c_in = m->d.c_in; a.c_out = m->d.c_out;
  a.forward_only = c.forward_only; a.has_temb = m->d.has_temb; a.emit_uvxyz = c.emit_uvxyz;
  a.x_in = c.x_in; a.x_is_repeated = c.x_is_repeated; a.out = c.out;
  a.n_rows = c.n_pose * c.n_hyp; a.n_pose = c.n_pose; a.n_steps = c.n_steps;
  a.temb = m->temb.get<float>(); a.noise = c.noise; a.key = c.key; a.mask = c.mask; a.steps_dev = c.steps_dev;
  const long n_tiles = (a.n_rows + TP - 1) / TP;
  const int grid = (int)(n_tiles < m->sm_count ? n_tiles : m->sm_count);
  tcx_kernel<<<grid, kThreads, SMEM_BYTES, s>>>(a, *c.inl);
  count_launch();
  DP_CUDA(cudaGetLastError());
  record_launch(m, grid, kThreads, SMEM_BYTES, TP, DP_ENGINE_TCX, n_tiles);
  return DP_OK;
}

}  // namespace dp
