// fp32 engine: one persistent kernel runs the whole DDIM loop (every step, every layer) for a tile of
// pose-hypotheses per CTA with all activations resident in shared memory.  Every contraction is an fp32
// FMA chain, so this engine is the on-device bit-level reference for the tensor-core engines and the only one for
// the configurations they do not cover (hid_dim != 96, n_head != 4, coordinates wider than 5).
//
// Reference semantics restated here (paths relative to the reference repository):
//   GCNdiff.forward            models/gcndiff.py:101-113      GCNpose.forward   models/gcnpose.py:101-113
//   _ResChebGC_diff.forward    models/gcndiff.py:48-53        _ResChebGC        models/ChebConv.py:154-165
//   ChebConv.forward           models/ChebConv.py:74-88       _GraphConv        models/ChebConv.py:145-151
//   GraAttenLayer/Sublayer     models/GraFormer.py:80-81,94-96
//   LayerNorm                  models/GraFormer.py:67-70      attention         models/GraFormer.py:99-140
//   GraphNet / LAM_Gconv       models/GraFormer.py:174-201
//   get_timestep_embedding     models/gcndiff.py:15-33        generalized_steps common/utils_diff.py:46-67
#include <cmath>
#include "dp_internal.h"

namespace dp {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kRB = 9;       // rows of the activation tile owned by one warp task in the GEMMs
constexpr int NP = 17;       // joints
constexpr int NPP = 292;     // padded 17*17 matrix in shared memory
constexpr int kMaxP = 4;     // pose-hypotheses per tile

enum Epi { EPI_STORE = 0, EPI_RELU = 1, EPI_RELU_TEMB = 2, EPI_ADD = 3, EPI_RELU_ADD = 4, EPI_NOBIAS = 5 };

struct SimtArgs {
  const Weights* w;
  Dims d;
  const float* x_in;
  int x_is_repeated;
  float* out;
  long n_rows;   // pose-hypotheses (sampling) or samples (forward)
  long n_pose;
  int n_steps;
  int forward_only;
  const float* temb;   // [n_steps | n_rows][n_layer][hid]
  const float* noise;  // [n_steps][n_rows][17][c] or NULL
  NoiseKey key;        // key.on: z from the keyed stream instead (noise is NULL)
  const unsigned char* mask;
  const dp_step* steps_dev;
  int P;
  float* xs_traj;      // sampler: x_t after each step and the x0 of that update, [n_steps][n_rows][17][c], or NULL
  float* x0_traj;
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// out[r][n0..] (op)= in[r][0..K) @ W[K][N] (+bias).  A warp task owns kRB rows x (32*CL) consecutive outputs;
// lane owns outputs n0+lane+32j, so weight reads are coalesced and activation reads are smem broadcasts.
template <int CL, int EPI>
__device__ void gemm_tile(const float* __restrict__ in, int ldin, int K, const float* __restrict__ W, int N,
                          const float* __restrict__ bias, float* out, int ldout, int R, const float* __restrict__ extra) {
  constexpr int H = 32 * CL;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nblk = (R + kRB - 1) / kRB, nchunk = N / H;
  for (int task = warp; task < nblk * nchunk; task += kWarps) {
    const int rb = task % nblk, ch = task / nblk;
    const int r0 = rb * kRB, n0 = ch * H;
    float acc[kRB][CL];
#pragma unroll
    for (int i = 0; i < kRB; ++i)
#pragma unroll
      for (int j = 0; j < CL; ++j) acc[i][j] = 0.f;
    const float* arow[kRB];
#pragma unroll
    for (int i = 0; i < kRB; ++i) arow[i] = in + (size_t)min(r0 + i, R - 1) * ldin;
    const float* wp = W + n0 + lane;
#pragma unroll 2
    for (int k = 0; k < K; k += 4) {
      float wv[4][CL];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int j = 0; j < CL; ++j) wv[kk][j] = __ldg(wp + (size_t)(k + kk) * N + 32 * j);
#pragma unroll
      for (int i = 0; i < kRB; ++i) {
        const float4 a = *reinterpret_cast<const float4*>(arow[i] + k);
#pragma unroll
        for (int j = 0; j < CL; ++j) {
          acc[i][j] = fmaf(a.x, wv[0][j], acc[i][j]);
          acc[i][j] = fmaf(a.y, wv[1][j], acc[i][j]);
          acc[i][j] = fmaf(a.z, wv[2][j], acc[i][j]);
          acc[i][j] = fmaf(a.w, wv[3][j], acc[i][j]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < CL; ++j) {
      const int n = n0 + lane + 32 * j;
      const float b = (EPI == EPI_NOBIAS) ? 0.f : __ldg(bias + n);
      const float ex = (EPI == EPI_RELU_TEMB) ? __ldg(extra + n) : 0.f;
#pragma unroll
      for (int i = 0; i < kRB; ++i) {
        const int r = r0 + i;
        if (r < R) {
          float v = acc[i][j] + b;
          float* o = out + (size_t)r * ldout + n;
          if (EPI == EPI_STORE || EPI == EPI_NOBIAS) *o = v;
          else if (EPI == EPI_RELU) *o = fmaxf(v, 0.f);
          else if (EPI == EPI_RELU_TEMB) *o = fmaxf(v, 0.f) + ex;
          else if (EPI == EPI_ADD) *o += v;
          else *o += fmaxf(v, 0.f);
        }
      }
    }
  }
}

// LayerNorm with unbiased std and eps added to std (GraFormer.py:67-70); one warp per row.
template <int CL>
__device__ void layer_norm_rows(const float* X, float* out, int R, const float* __restrict__ a, const float* __restrict__ b) {
  constexpr int H = 32 * CL;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float av[CL], bv[CL];
#pragma unroll
  for (int j = 0; j < CL; ++j) { av[j] = __ldg(a + lane + 32 * j); bv[j] = __ldg(b + lane + 32 * j); }
  for (int r = warp; r < R; r += kWarps) {
    float v[CL], s = 0.f;
#pragma unroll
    for (int j = 0; j < CL; ++j) { v[j] = X[(size_t)r * H + lane + 32 * j]; s += v[j]; }
    const float mean = warp_sum(s) / (float)H;
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < CL; ++j) { v[j] -= mean; q += v[j] * v[j]; }
    const float sd = sqrtf(warp_sum(q) / (float)(H - 1));
    const float den = sd + 1e-6f;
#pragma unroll
    for (int j = 0; j < CL; ++j) out[(size_t)r * H + lane + 32 * j] = (av[j] * v[j]) / den + bv[j];
  }
}

// out[p*17+i][c] (op)= sum_j M[i][j] in[p*17+j][c]  (per-pose 17x17 aggregation over C channels)
template <bool ADD_BIAS_RESID>
__device__ void aggregate(const float* M, const float* in, int ldin, int C, float* out, int ldout, int R,
                          const float* __restrict__ bias) {
  for (int idx = threadIdx.x; idx < R * C; idx += kThreads) {
    const int r = idx / C, c = idx - r * C;
    const int p = r / NP, i = r - p * NP;
    const float* src = in + (size_t)p * NP * ldin + c;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < NP; ++j) acc = fmaf(M[i * NP + j], src[(size_t)j * ldin], acc);
    if (ADD_BIAS_RESID) out[(size_t)r * ldout + c] += acc + __ldg(bias + c);
    else out[(size_t)r * ldout + c] = acc;
  }
}

// dst[r] = [ src[r] | (T1 src)[r] | (T2 src)[r] ]  -- the ChebConv input panel with T0 = I (ChebConv.py:74-112)
__device__ void cheb_concat(const float* t1, const float* t2, const float* src, int ldsrc, int C, float* dst, int lddst, int R) {
  for (int idx = threadIdx.x; idx < R * C; idx += kThreads) {
    const int r = idx / C, c = idx - r * C;
    const int p = r / NP, i = r - p * NP;
    const float* s = src + (size_t)p * NP * ldsrc + c;
    float a1 = 0.f, a2 = 0.f;
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const float v = s[(size_t)j * ldsrc];
      a1 = fmaf(t1[i * NP + j], v, a1);
      a2 = fmaf(t2[i * NP + j], v, a2);
    }
    float* d = dst + (size_t)r * lddst + c;
    d[0] = s[(size_t)i * ldsrc];
    d[C] = a1;
    d[2 * C] = a2;
  }
}

// softmax(q k^T / sqrt(dk), key mask) v for every (pose, head, query joint); qkv rows are [q | k | v] (3H wide).
__device__ void attention_rows(const float* qkv, int H, int n_head, float* out, int npose, const float* maskf) {
  const int dk = H / n_head;
  const float scale = sqrtf((float)dk);
  const int ld = 3 * H;
  for (int task = threadIdx.x; task < npose * n_head * NP; task += kThreads) {
    const int p = task / (n_head * NP);
    const int rem = task - p * n_head * NP;
    const int h = rem / NP, i = rem - h * NP;
    const float* q = qkv + (size_t)(p * NP + i) * ld + h * dk;
    const float* kb = qkv + (size_t)(p * NP) * ld + H + h * dk;
    const float* vb = kb + H;
    float sc[NP];
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const float* kj = kb + (size_t)j * ld;
      float s = 0.f;
      for (int dd = 0; dd < dk; ++dd) s = fmaf(q[dd], kj[dd], s);
      s = s / scale;
      if (maskf[j] == 0.f) s = -1e9f;
      sc[j] = s;
      mx = fmaxf(mx, s);
    }
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < NP; ++j) { sc[j] = expf(sc[j] - mx); sum += sc[j]; }
    const float inv = 1.0f / sum;
#pragma unroll
    for (int j = 0; j < NP; ++j) sc[j] *= inv;
    float* o = out + (size_t)(p * NP + i) * H + h * dk;
    for (int dd = 0; dd < dk; ++dd) {
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < NP; ++j) acc = fmaf(sc[j], vb[(size_t)j * ld + dd], acc);
      o[dd] = acc;
    }
  }
}

template <int CL>
__global__ void __launch_bounds__(kThreads, 1) simt_kernel(SimtArgs a, StepsArg inl) {
  constexpr int H = 32 * CL;
  extern __shared__ __align__(16) float smem[];
  const Dims d = a.d;
  const int P = a.P, RMAX = P * NP;
  float* X = smem;                        // [R][H]   residual stream
  float* B0 = X + (size_t)RMAX * H;       // [R][H]
  float* B1 = B0 + (size_t)RMAX * H;      // [R][3H]
  float* B2 = B1 + (size_t)RMAX * 3 * H;  // [R][H]
  float* xt = B2 + (size_t)RMAX * H;      // [R][8]   current x_t
  float* ep = xt + (size_t)RMAX * 8;      // [R][8]   eps / model output
  float* t1 = ep + (size_t)RMAX * 8;      // 3 padded 17x17 matrices + key mask
  float* t2 = t1 + NPP;
  float* lh = t2 + NPP;
  float* maskf = lh + NPP;                // [32]

  const Weights& w = *a.w;
  for (int i = threadIdx.x; i < NP * NP; i += kThreads) { t1[i] = __ldg(w.t1 + i); t2[i] = __ldg(w.t2 + i); }
  if (threadIdx.x < 32) maskf[threadIdx.x] = (threadIdx.x < NP && a.mask && a.mask[threadIdx.x] == 0) ? 0.f : 1.f;
  __syncthreads();

  const int cin = d.c_in, cout = d.c_out;
  const long n_tiles = (a.n_rows + P - 1) / P;
  for (long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long g0 = tile * P;
    const int npose = (int)min((long)P, a.n_rows - g0);
    const int R = npose * NP;

    for (int idx = threadIdx.x; idx < R * cin; idx += kThreads) {
      const int r = idx / cin, c = idx - r * cin;
      const long g = g0 + r / NP;
      const long src = a.x_is_repeated ? g : (g % a.n_pose);
      xt[r * 8 + c] = a.x_in[(src * NP + (r % NP)) * cin + c];
    }
    __syncthreads();

    for (int step = 0; step < a.n_steps; ++step) {
      // ---- input ChebConv: X = [x | T1 x | T2 x] Win + b   (gcndiff.py:108)
      cheb_concat(t1, t2, xt, 8, cin, B1, 3 * cin, R);
      __syncthreads();
      for (int idx = threadIdx.x; idx < R * H; idx += kThreads) {
        const int r = idx / H, n = idx - r * H;
        float acc = __ldg(w.bin + n);
        for (int k = 0; k < 3 * cin; ++k) acc = fmaf(B1[r * 3 * cin + k], __ldg(w.win + k * H + n), acc);
        X[idx] = acc;
      }
      __syncthreads();

      for (int l = 0; l < d.n_layer; ++l) {
        const LayerW& L = w.layer[l];
        for (int i = threadIdx.x; i < NP * NP; i += kThreads) lh[i] = __ldg(L.lhat + i);
        // ---- x = x + attn(LN0(x))   (GraFormer.py:95, :127-140)
        layer_norm_rows<CL>(X, B0, R, L.ln0_a, L.ln0_b);
        __syncthreads();
        gemm_tile<CL, EPI_STORE>(B0, H, H, L.wqkv, 3 * H, L.bqkv, B1, 3 * H, R, nullptr);
        __syncthreads();
        attention_rows(B1, H, d.n_head, B0, npose, maskf);
        __syncthreads();
        gemm_tile<CL, EPI_ADD>(B0, H, H, L.wo, H, L.bo, X, H, R, nullptr);
        __syncthreads();
        // ---- x = x + GraphNet(LN1(x))   (GraFormer.py:96, :180-201); fc2(Lhat h) == Lhat (h W2^T) + b2
        layer_norm_rows<CL>(X, B0, R, L.ln1_a, L.ln1_b);
        __syncthreads();
        aggregate<false>(lh, B0, H, H, B2, H, R, nullptr);
        __syncthreads();
        gemm_tile<CL, EPI_RELU>(B2, H, H, L.w1, 2 * H, L.b1, B1, 2 * H, R, nullptr);
        __syncthreads();
        gemm_tile<CL, EPI_NOBIAS>(B1, 2 * H, 2 * H, L.w2, H, nullptr, B0, H, R, nullptr);
        __syncthreads();
        aggregate<true>(lh, B0, H, H, X, H, R, L.b2);
        __syncthreads();
        // ---- x = x + GC2(GC1(x) + temb_l)   (gcndiff.py:48-53; ChebConv.py:145-151)
        cheb_concat(t1, t2, X, H, H, B1, 3 * H, R);
        __syncthreads();
        if (d.has_temb) {
          // temb row: the step (sampling, batch-invariant t) or the sample (forward, per-sample t).
          // Rows of one tile may have different temb rows in forward mode, so that mode adds it afterwards.
          if (!a.forward_only) {
            const float* te = a.temb + ((size_t)step * d.n_layer + l) * H;
            gemm_tile<CL, EPI_RELU_TEMB>(B1, 3 * H, 3 * H, L.wc1, H, L.bc1, B0, H, R, te);
          } else {
            gemm_tile<CL, EPI_RELU>(B1, 3 * H, 3 * H, L.wc1, H, L.bc1, B0, H, R, nullptr);
            __syncthreads();
            for (int idx = threadIdx.x; idx < R * H; idx += kThreads) {
              const int r = idx / H, n = idx - r * H;
              B0[idx] += __ldg(a.temb + ((size_t)(g0 + r / NP) * d.n_layer + l) * H + n);
            }
          }
        } else {
          gemm_tile<CL, EPI_RELU>(B1, 3 * H, 3 * H, L.wc1, H, L.bc1, B0, H, R, nullptr);
        }
        __syncthreads();
        cheb_concat(t1, t2, B0, H, H, B1, 3 * H, R);
        __syncthreads();
        gemm_tile<CL, EPI_RELU_ADD>(B1, 3 * H, 3 * H, L.wc2, H, L.bc2, X, H, R, nullptr);
        __syncthreads();
      }

      // ---- output ChebConv   (gcndiff.py:112)
      cheb_concat(t1, t2, X, H, H, B1, 3 * H, R);
      __syncthreads();
      for (int idx = threadIdx.x; idx < R * cout; idx += kThreads) {
        const int r = idx / cout, n = idx - r * cout;
        float acc = 0.f;
        const float* row = B1 + (size_t)r * 3 * H;
        for (int k = 0; k < 3 * H; ++k) acc = fmaf(row[k], __ldg(w.wout + k * cout + n), acc);
        ep[r * 8 + n] = acc + __ldg(w.bout + n);
      }
      __syncthreads();

      if (!a.forward_only) {
        // ---- DDIM update, operation order of common/utils_diff.py:59-65 without FMA contraction
        const dp_step st = a.steps_dev ? a.steps_dev[step] : inl.s[step];
        for (int idx = threadIdx.x; idx < R * cin; idx += kThreads) {
          const int r = idx / cin, c = idx - r * cin;
          const float et = ep[r * 8 + c], xv = xt[r * 8 + c];
          const float x0 = __fdiv_rn(__fsub_rn(xv, __fmul_rn(et, st.sqrt_1m_at)), st.sqrt_at);
          float nx = __fmul_rn(st.sqrt_an, x0);
          const size_t ot = ((size_t)step * a.n_rows + g0) * NP * cin + idx;   // element of the [n_steps][n_rows] arrays
          if (a.noise) {
            const float z = a.noise[ot];
            nx = __fadd_rn(nx, __fmul_rn(st.c1, z));
          } else if (a.key.on) {
            // hypothesis-major row g = h * n_pose + b
            const long g = g0 + r / NP, h = g / a.n_pose;
            const float z = philox_normal(a.key, a.key.step_offset + (uint32_t)step, a.key.pose_offset + (uint32_t)(g - h * a.n_pose),
                                          (uint32_t)h, (uint32_t)((r % NP) * cin + c));
            nx = __fadd_rn(nx, __fmul_rn(st.c1, z));
          }
          nx = __fadd_rn(nx, __fmul_rn(st.c2, et));
          xt[r * 8 + c] = nx;
          if (a.xs_traj) a.xs_traj[ot] = nx;
          if (a.x0_traj) a.x0_traj[ot] = x0;
        }
        __syncthreads();
      }
    }

    const float* res = a.forward_only ? ep : xt;
    for (int idx = threadIdx.x; idx < R * cout; idx += kThreads) {
      const int r = idx / cout, c = idx - r * cout;
      a.out[(size_t)g0 * NP * cout + idx] = res[r * 8 + c];
    }
    __syncthreads();
  }
}

// Time-embedding table: out[i][l][:] = temb_proj_l(swish(dense1(swish(dense0(sincos(t_i))))))
// (gcndiff.py:15-33, :103-106, :51).  One CTA evaluates kTB timesteps so weight reads are shared.
// kTB = 4 for a sampler schedule (a handful of timesteps: latency matters), 12 for per-sample timesteps of a forward call
// (thousands: every CTA streams the 0.7 MB of embedding weights from L2, so more timesteps per CTA = fewer passes).  The
// arithmetic per timestep is the same in both (one accumulator chain per timestep): results are bit-identical.
template <int kTB>
__global__ void temb_kernel(const Weights* wp, Dims d, const float* __restrict__ t_dev, int t_stride, StepsArg inl,
                            long n_t, float* __restrict__ out) {
  extern __shared__ float sm[];
  const int H = d.hid, E = 4 * H;
  float* emb = sm;            // [kTB][H]
  float* h1 = emb + kTB * H;  // [kTB][E]
  float* h2 = h1 + kTB * E;   // [kTB][E]
  const Weights& w = *wp;
  const long i0 = (long)blockIdx.x * kTB;
  const int nt = (int)min((long)kTB, n_t - i0);
  const int half = H / 2;
  const float c = (float)(-(log(10000.0) / (double)(half - 1)));
  for (int idx = threadIdx.x; idx < kTB * H; idx += blockDim.x) {
    const int b = idx / H, k = idx - b * H;
    float v = 0.f;
    if (b < nt) {
      const float t = t_dev ? t_dev[(size_t)(i0 + b) * t_stride] : inl.s[i0 + b].t;
      const int kk = k < half ? k : k - half;
      const float f = expf((float)kk * c);
      const float e = t * f;
      v = k < half ? sinf(e) : cosf(e);
    }
    emb[idx] = v;
  }
  __syncthreads();
  for (int n = threadIdx.x; n < E; n += blockDim.x) {
    float acc[kTB];
#pragma unroll
    for (int b = 0; b < kTB; ++b) acc[b] = __ldg(w.bd0 + n);
#pragma unroll 8
    for (int k = 0; k < H; ++k) {
      const float wv = __ldg(w.wd0 + (size_t)k * E + n);
#pragma unroll
      for (int b = 0; b < kTB; ++b) acc[b] = fmaf(emb[b * H + k], wv, acc[b]);
    }
#pragma unroll
    for (int b = 0; b < kTB; ++b) h1[b * E + n] = acc[b] / (1.0f + expf(-acc[b]));  // swish
  }
  __syncthreads();
  for (int n = threadIdx.x; n < E; n += blockDim.x) {
    float acc[kTB];
#pragma unroll
    for (int b = 0; b < kTB; ++b) acc[b] = __ldg(w.bd1 + n);
#pragma unroll 8
    for (int k = 0; k < E; ++k) {
      const float wv = __ldg(w.wd1 + (size_t)k * E + n);
#pragma unroll
      for (int b = 0; b < kTB; ++b) acc[b] = fmaf(h1[b * E + k], wv, acc[b]);
    }
#pragma unroll
    for (int b = 0; b < kTB; ++b) h2[b * E + n] = acc[b] / (1.0f + expf(-acc[b]));  // swish before temb_proj
  }
  __syncthreads();
  for (int o = threadIdx.x; o < d.n_layer * H; o += blockDim.x) {
    const int l = o / H, n = o - l * H;
    const LayerW& L = w.layer[l];
    float acc[kTB];
#pragma unroll
    for (int b = 0; b < kTB; ++b) acc[b] = __ldg(L.bt + n);
#pragma unroll 8
    for (int k = 0; k < E; ++k) {
      const float wv = __ldg(L.wt + (size_t)k * H + n);
#pragma unroll
      for (int b = 0; b < kTB; ++b) acc[b] = fmaf(h2[b * E + k], wv, acc[b]);
    }
    for (int b = 0; b < nt; ++b) out[((size_t)(i0 + b) * d.n_layer + l) * H + n] = acc[b];
  }
}

size_t simt_smem_bytes(int H, int P) {
  const size_t R = (size_t)P * NP;
  return (R * (6 * H + 16) + 3 * NPP + 32) * sizeof(float);
}

template <int CL>
int launch_simt(dp_model* m, const SimtArgs& a, const StepsArg& inl, cudaStream_t s) {
  const size_t smem = simt_smem_bytes(32 * CL, a.P);
  DP_TRY(smem_opt_in<simt_kernel<CL>>(m->device, 227 * 1024));
  const long n_tiles = (a.n_rows + a.P - 1) / a.P;
  const int grid = (int)min((long)m->sm_count, n_tiles);
  simt_kernel<CL><<<grid, kThreads, smem, s>>>(a, inl);
  count_launch();
  DP_CUDA(cudaGetLastError());
  record_launch(m, grid, kThreads, (long)smem, a.P, DP_ENGINE_FP32, n_tiles);
  return DP_OK;
}

int dispatch_simt(dp_model* m, const SimtArgs& a, const StepsArg& inl, cudaStream_t s) {
  switch (m->d.hid / 32) {
    case 1: return launch_simt<1>(m, a, inl, s);
    case 2: return launch_simt<2>(m, a, inl, s);
    case 3: return launch_simt<3>(m, a, inl, s);
    case 4: return launch_simt<4>(m, a, inl, s);
  }
  set_error("fp32 engine: unsupported hid_dim");
  return DP_ERR_UNSUPPORTED;
}

int pick_tile(const dp_model* m, long n_rows) {
  // Fill every SM before making tiles taller: small batches are latency runs (SURVEY.md 8e).
  long p = (n_rows + m->sm_count - 1) / m->sm_count;
  if (p < 1) p = 1;
  if (p > kMaxP) p = kMaxP;
  while (simt_smem_bytes(m->d.hid, (int)p) > 227 * 1024 && p > 1) --p;
  return (int)p;
}

}  // namespace

int simt_temb(dp_model* m, const float* t_dev, int t_stride, const StepsArg* inl, long n_t, cudaStream_t s) {
  if (!m->d.has_temb || n_t == 0) return DP_OK;
  const Dims& d = m->d;
  DP_TRY(m->temb.reserve((size_t)n_t * d.n_layer * d.hid * sizeof(float)));
  float* temb = m->temb.get<float>();
  StepsArg dummy{};
  const int H = d.hid;
  if (n_t >= 64) {
    constexpr int kTB = 12;
    const size_t smem = (size_t)kTB * (H + 8 * H) * sizeof(float);      // 41.5 KB at hid = 96 (48 KB without opt-in: hid <= 111)
    if (smem <= 48 * 1024) {
      temb_kernel<kTB><<<(unsigned)((n_t + kTB - 1) / kTB), 4 * H, smem, s>>>(m->dw.get<Weights>(), d, t_dev, t_stride, inl ? *inl : dummy, n_t, temb);
      count_launch();
      DP_CUDA(cudaGetLastError());
      return DP_OK;
    }
  }
  constexpr int kTB = 4;
  const size_t smem = (size_t)kTB * (H + 8 * H) * sizeof(float);
  const long grid = (n_t + kTB - 1) / kTB;
  temb_kernel<kTB><<<(unsigned)grid, 4 * H, smem, s>>>(m->dw.get<Weights>(), d, t_dev, t_stride, inl ? *inl : dummy, n_t, temb);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

int simt_run(dp_model* m, const EngineCall& c, cudaStream_t s) {
  SimtArgs a{};
  a.w = m->dw.get<Weights>(); a.d = m->d; a.x_in = c.x_in; a.x_is_repeated = c.x_is_repeated; a.out = c.out;
  a.n_rows = c.n_pose * c.n_hyp; a.n_pose = c.n_pose; a.n_steps = c.n_steps; a.forward_only = c.forward_only;
  a.temb = m->temb.get<float>(); a.noise = c.noise; a.key = c.key; a.mask = c.mask; a.steps_dev = c.steps_dev;
  a.xs_traj = c.xs_traj; a.x0_traj = c.x0_traj;
  a.P = pick_tile(m, a.n_rows);
  return dispatch_simt(m, a, *c.inl, s);
}

}  // namespace dp
