// C ABI of libdiffpose_b200.so: handle lifetime, weight packing, engine dispatch.
// See include/diffpose_b200.h for the contract and the reference interfaces each entry point replaces.
#include <atomic>
#include <cmath>
#include <cstring>
#include <new>
#include "dp_internal.h"
#include "dp_tc_layout.cuh"

namespace dp {

static thread_local std::string g_err;
static std::atomic<long> g_launches{0};

void set_error(const std::string& msg) { g_err = msg; }
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// dst[k*ld + col0 + n] = src[n*K + k]: a torch.nn.Linear weight [N][K] becomes an input-major [K][N] panel.
__global__ void pack_transpose_kernel(float* __restrict__ dst, const float* __restrict__ src, int K, int N, int ld,
                                      int col0) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= K * N) return;
  int k = idx / N, n = idx - k * N;
  dst[(size_t)k * ld + col0 + n] = src[(size_t)n * K + k];
}

__global__ void pack_copy_kernel(float* __restrict__ dst, const float* __restrict__ src, int rows, int cols, int ld,
                                 int col0) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  int r = idx / cols, c = idx - r * cols;
  dst[(size_t)r * ld + col0 + c] = src[idx];
}

// GraFormer.py:174-178: D_j = (sum_i A[i][j] + 1e-5)^-1/2 ; Lhat[i][j] = D_i * A[i][j] * D_j.
__global__ void pack_lhat_kernel(float* __restrict__ dst, const float* __restrict__ a_hat, int n) {
  __shared__ float d[32];
  int j = threadIdx.x;
  if (j < n) {
    float s = 0.f;
    for (int i = 0; i < n; ++i) s += a_hat[i * n + j];
    d[j] = 1.0f / sqrtf(s + 1e-5f);
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < n * n; idx += blockDim.x) {
    int i = idx / n, jj = idx - i * n;
    dst[idx] = d[i] * a_hat[idx] * d[jj];
  }
}

struct Carver {
  float* base;
  size_t off = 0;
  explicit Carver(float* b) : base(b) {}
  float* take(size_t n) {
    float* p = base ? base + off : nullptr;
    off += (n + 31) & ~size_t(31);  // 128-byte aligned panels
    return p;
  }
};

// Lays the packed fp32 blob out; with base == nullptr only measures it.
static size_t carve(Weights& w, const Dims& d, float* base) {
  Carver c(base);
  const int H = d.hid, P = d.n_pts * d.n_pts;
  w.win = c.take((size_t)3 * d.c_in * H);
  w.bin = c.take(H);
  w.wout = c.take((size_t)3 * H * d.c_out);
  w.bout = c.take(d.c_out);
  w.t1 = c.take(P);
  w.t2 = c.take(P);
  w.t1m = c.take(P);
  w.t2m = c.take(P);
  w.t1s = c.take(d.n_pts);
  w.t2s = c.take(d.n_pts);
  w.wd0 = c.take((size_t)H * 4 * H);
  w.bd0 = c.take(4 * H);
  w.wd1 = c.take((size_t)16 * H * H);
  w.bd1 = c.take(4 * H);
  for (int l = 0; l < d.n_layer; ++l) {
    LayerW& L = w.layer[l];
    L.ln0_a = c.take(H); L.ln0_b = c.take(H);
    L.wqkv = c.take((size_t)3 * H * H); L.bqkv = c.take(3 * H);
    L.wo = c.take((size_t)H * H); L.bo = c.take(H);
    L.ln1_a = c.take(H); L.ln1_b = c.take(H);
    L.lhat = c.take(P);
    L.w1 = c.take((size_t)2 * H * H); L.b1 = c.take(2 * H);
    L.w2 = c.take((size_t)2 * H * H); L.b2 = c.take(H);
    L.wc1 = c.take((size_t)3 * H * H); L.bc1 = c.take(H);
    L.wc2 = c.take((size_t)3 * H * H); L.bc2 = c.take(H);
    L.wt = c.take((size_t)4 * H * H); L.bt = c.take(H);
  }
  return c.off;
}

static long param_count(const Dims& d) {
  const long H = d.hid, P = (long)d.n_pts * d.n_pts;
  long n = 3L * d.c_in * H + H;
  long per = 2 * (3 * H * H + H) + 4 * (H * H + H) + P + (2 * H * H + 2 * H) + (2 * H * H + H) + 4 * H;
  if (d.has_temb) per += 4 * H * H + H;
  n += per * d.n_layer;
  n += 3L * H * d.c_out + d.c_out;
  if (d.has_temb) n += (4 * H * H + 4 * H) + (16 * H * H + 4 * H);
  return n;
}

static inline float* mut(const float* p) { return const_cast<float*>(p); }

// The Chebyshev matrices of a row-normalised skeleton adjacency have entries such as 1/3 that fp16 cannot hold, and
// rounding them biases every channel of every pose the same way.  Factor each row i as scale_i * (integers): the
// integer row is exact in fp16, so the tensor cores apply the matrix exactly and the epilogue multiplies by the fp32
// scale.  A row without such a factor (arbitrary adjacency) keeps scale 1 and is rounded as before.
static void integerise_rows(const std::vector<float>& g, int n, std::vector<float>& m, std::vector<float>& scale) {
  m.assign((size_t)n * n, 0.f);
  scale.assign(n, 1.f);
  for (int i = 0; i < n; ++i) {
    // accept q only when r/q reproduces every entry within a FIXED absolute tolerance on g itself, 1e-6 max(1, |g|): wide
    // enough for the fp32 rounding of the host-side 2 L L - I (a 17-term fp32 dot product; 2^-22 measurably rejects rows of
    // the H36M skeleton and brings the fp16-rounding bias back: 0.07 mm MPJPE), and 100x tighter than what a rejected row
    // gets instead (its entries rounded to fp16, 2^-12 relative) -- so accepting can only move the engine towards fp32
    int best = 0;
    for (int q = 1; q <= 4096 && !best; ++q) {
      bool ok = true;
      for (int j = 0; j < n && ok; ++j) {
        const double gv = (double)g[i * n + j], r = std::nearbyint(gv * q);
        ok = std::fabs(gv - r / q) <= 1e-6 * std::fmax(1.0, std::fabs(gv)) && std::fabs(r) <= 2048.0;
      }
      if (ok) best = q;
    }
    if (best) {
      scale[i] = 1.0f / (float)best;
      for (int j = 0; j < n; ++j) m[i * n + j] = (float)std::nearbyint((double)g[i * n + j] * best);
    } else {
      for (int j = 0; j < n; ++j) m[i * n + j] = g[i * n + j];
    }
  }
}

static int launch_transpose(float* dst, const float* src, int K, int N, int ld, int col0, cudaStream_t s) {
  int total = K * N;
  pack_transpose_kernel<<<(total + 255) / 256, 256, 0, s>>>(dst, src, K, N, ld, col0);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}
static int launch_copy(float* dst, const float* src, int rows, int cols, int ld, int col0, cudaStream_t s) {
  int total = rows * cols;
  pack_copy_kernel<<<(total + 255) / 256, 256, 0, s>>>(dst, src, rows, cols, ld, col0);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

static int pack_fp32(dp_model* m, const float* p, const float* adj_host, cudaStream_t s) {
  const Dims& d = m->d;
  const int H = d.hid, NP = d.n_pts, P = NP * NP;
  const Weights& w = m->hw;

  DP_TRY(launch_copy(mut(w.win), p, 3 * d.c_in, H, H, 0, s)); p += 3 * d.c_in * H;
  DP_TRY(launch_copy(mut(w.bin), p, 1, H, H, 0, s)); p += H;
  for (int l = 0; l < d.n_layer; ++l) {
    const LayerW& L = w.layer[l];
    DP_TRY(launch_copy(mut(L.wc1), p, 3 * H, H, H, 0, s)); p += 3 * H * H;
    DP_TRY(launch_copy(mut(L.bc1), p, 1, H, H, 0, s)); p += H;
    DP_TRY(launch_copy(mut(L.wc2), p, 3 * H, H, H, 0, s)); p += 3 * H * H;
    DP_TRY(launch_copy(mut(L.bc2), p, 1, H, H, 0, s)); p += H;
    if (d.has_temb) {
      DP_TRY(launch_transpose(mut(L.wt), p, 4 * H, H, H, 0, s)); p += 4 * H * H;
      DP_TRY(launch_copy(mut(L.bt), p, 1, H, H, 0, s)); p += H;
    }
    for (int i = 0; i < 3; ++i) {
      DP_TRY(launch_transpose(mut(L.wqkv), p, H, H, 3 * H, i * H, s)); p += H * H;
      DP_TRY(launch_copy(mut(L.bqkv), p, 1, H, 3 * H, i * H, s)); p += H;
    }
    DP_TRY(launch_transpose(mut(L.wo), p, H, H, H, 0, s)); p += H * H;
    DP_TRY(launch_copy(mut(L.bo), p, 1, H, H, 0, s)); p += H;
    pack_lhat_kernel<<<1, 32, 0, s>>>(mut(L.lhat), p, NP);
    count_launch();
    DP_CUDA(cudaGetLastError());
    p += P;
    DP_TRY(launch_transpose(mut(L.w1), p, H, 2 * H, 2 * H, 0, s)); p += 2 * H * H;
    DP_TRY(launch_copy(mut(L.b1), p, 1, 2 * H, 2 * H, 0, s)); p += 2 * H;
    DP_TRY(launch_transpose(mut(L.w2), p, 2 * H, H, H, 0, s)); p += 2 * H * H;
    DP_TRY(launch_copy(mut(L.b2), p, 1, H, H, 0, s)); p += H;
    DP_TRY(launch_copy(mut(L.ln0_a), p, 1, H, H, 0, s)); p += H;
    DP_TRY(launch_copy(mut(L.ln0_b), p, 1, H, H, 0, s)); p += H;
    DP_TRY(launch_copy(mut(L.ln1_a), p, 1, H, H, 0, s)); p += H;
    DP_TRY(launch_copy(mut(L.ln1_b), p, 1, H, H, 0, s)); p += H;
  }
  DP_TRY(launch_copy(mut(w.wout), p, 3 * H, d.c_out, d.c_out, 0, s)); p += 3 * H * d.c_out;
  DP_TRY(launch_copy(mut(w.bout), p, 1, d.c_out, d.c_out, 0, s)); p += d.c_out;
  if (d.has_temb) {
    DP_TRY(launch_transpose(mut(w.wd0), p, H, 4 * H, 4 * H, 0, s)); p += 4 * H * H;
    DP_TRY(launch_copy(mut(w.bd0), p, 1, 4 * H, 4 * H, 0, s)); p += 4 * H;
    DP_TRY(launch_transpose(mut(w.wd1), p, 4 * H, 4 * H, 4 * H, 0, s)); p += 16 * H * H;
    DP_TRY(launch_copy(mut(w.bd1), p, 1, 4 * H, 4 * H, 0, s)); p += 4 * H;
  }

  // Chebyshev basis on the host, fp32 like the reference (models/ChebConv.py:90-130):
  // D = diag(rowsum^-1/2), L = I - D A D, T1 = L, T2 = 2 L L - I.
  std::vector<float> dg(NP), lap(P), t2(P);
  for (int i = 0; i < NP; ++i) {
    float rs = 0.f;
    for (int j = 0; j < NP; ++j) rs += adj_host[i * NP + j];
    dg[i] = 1.0f / std::sqrt(rs);
  }
  for (int i = 0; i < NP; ++i)
    for (int j = 0; j < NP; ++j) lap[i * NP + j] = (i == j ? 1.f : 0.f) - (dg[i] * adj_host[i * NP + j]) * dg[j];
  for (int i = 0; i < NP; ++i)
    for (int j = 0; j < NP; ++j) {
      float acc = 0.f;
      for (int k = 0; k < NP; ++k) acc += lap[i * NP + k] * lap[k * NP + j];
      t2[i * NP + j] = 2.f * acc - (i == j ? 1.f : 0.f);
    }
  DP_CUDA(cudaMemcpyAsync(mut(w.t1), lap.data(), P * sizeof(float), cudaMemcpyHostToDevice, s));
  DP_CUDA(cudaMemcpyAsync(mut(w.t2), t2.data(), P * sizeof(float), cudaMemcpyHostToDevice, s));
  std::vector<float> t1m, t1s, t2m, t2s;
  integerise_rows(lap, NP, t1m, t1s);
  integerise_rows(t2, NP, t2m, t2s);
  DP_CUDA(cudaMemcpyAsync(mut(w.t1m), t1m.data(), P * sizeof(float), cudaMemcpyHostToDevice, s));
  DP_CUDA(cudaMemcpyAsync(mut(w.t2m), t2m.data(), P * sizeof(float), cudaMemcpyHostToDevice, s));
  DP_CUDA(cudaMemcpyAsync(mut(w.t1s), t1s.data(), NP * sizeof(float), cudaMemcpyHostToDevice, s));
  DP_CUDA(cudaMemcpyAsync(mut(w.t2s), t2s.data(), NP * sizeof(float), cudaMemcpyHostToDevice, s));
  DP_CUDA(cudaMemcpyAsync(m->dw.get<Weights>(), &m->hw, sizeof(Weights), cudaMemcpyHostToDevice, s));
  // the host vectors above go out of scope: finish the copies first (pack is not on the hot path)
  DP_CUDA(cudaStreamSynchronize(s));
  return DP_OK;
}

}  // namespace dp

using namespace dp;

// The handle's buffers live on the device that was current at dp_create: a call made with another device current would
// launch there with pointers into this one (ADVICE r1).  Refuse instead of faulting.
static int check_device(dp_handle h, const char* what) {
  int cur = -1;
  DP_CUDA(cudaGetDevice(&cur));
  if (cur != h->device) {
    set_error(std::string(what) + ": the handle was created on device " + std::to_string(h->device) + " but device " + std::to_string(cur) +
              " is current (create one handle per device; the Python shim re-creates it after model.to())");
    return DP_ERR_STATE;
  }
  return DP_OK;
}

// engine that runs a forward call: AUTO -> the split-precision engine (a forward output is not damped by a DDIM schedule,
// so it gets the accurate path), explicit settings are honoured
static int forward_engine(dp_handle h) {
  if (h->engine == DP_ENGINE_FP32 || !tc_supported(h->d)) return DP_ENGINE_FP32;
  if (h->engine == DP_ENGINE_TCG) return DP_ENGINE_TCG;
  return DP_ENGINE_TCX;
}

static int run_engine(dp_handle h, int eng, const EngineCall& c, cudaStream_t s) {
  if (eng == DP_ENGINE_TCG) return tc2_run(h, c, s);
  if (eng == DP_ENGINE_TCX) return tcx_run(h, c, s);
  return simt_run(h, c, s);
}

// GCNdiff.forward / GCNpose.forward (models/gcndiff.py:101-113, models/gcnpose.py:101-113): one pass with per-sample
// timesteps, in chunks that bound the per-sample embedding table (chunk * n_layer * hid floats).  That table goes into
// the buffer the sampler caches its per-step table in, so that cache is dropped.  emit_uvxyz (tcx only): out is
// [n][n_pts][c_in + c_out] = [uv | xyz - xyz_root] (runners/diffpose_frame.py:337-343).
static int forward_chunks(dp_handle h, int eng, const float* x, const float* t, const unsigned char* mask, float* out, long n,
                          bool emit_uvxyz, cudaStream_t s) {
  const Dims& d = h->d;
  const long chunk = 1L << 16;
  const int wd = emit_uvxyz ? d.c_in + d.c_out : d.c_out;
  const StepsArg none{};
  if (d.has_temb) h->temb_t.clear();
  for (long o = 0; o < n; o += chunk) {
    const long nn = (n - o < chunk) ? (n - o) : chunk;
    if (d.has_temb) DP_TRY(simt_temb(h, t + o, 1, nullptr, nn, s));
    EngineCall c;
    c.x_in = x + (size_t)o * d.n_pts * d.c_in; c.x_is_repeated = 1; c.out = out + (size_t)o * d.n_pts * wd;
    c.n_pose = nn; c.inl = &none; c.mask = mask; c.forward_only = true;
    c.emit_uvxyz = emit_uvxyz;
    DP_TRY(run_engine(h, eng, c, s));
  }
  return DP_OK;
}

extern "C" {

int dp_create(dp_handle* out, int n_pts, int c_in, int c_out, int hid, int n_layer, int n_head, int has_temb) {
  DP_REQUIRE(out != nullptr, "dp_create: out is NULL");
  *out = nullptr;
  DP_REQUIRE(n_pts == kMaxPts, "dp_create: kernels are built for the 17-joint Human3.6M skeleton (n_pts must be 17)");
  DP_REQUIRE(c_in >= 1 && c_in <= kMaxCoord && c_out >= 1 && c_out <= kMaxCoord, "dp_create: coords_dim must be in 1..8");
  DP_REQUIRE(hid >= 32 && hid <= 128 && hid % 32 == 0, "dp_create: hid_dim must be 32, 64, 96 or 128");
  DP_REQUIRE(n_layer >= 1 && n_layer <= kMaxLayers, "dp_create: num_layer must be in 1..16");
  DP_REQUIRE(n_head >= 1 && hid % n_head == 0 && hid / n_head <= 64, "dp_create: n_head must divide hid_dim with d_k <= 64");
  DP_REQUIRE(!has_temb || c_in == c_out, "dp_create: the diffusion denoiser needs coords_dim[0] == coords_dim[1]");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_error("dp_create: no CUDA device is visible; this library has no CPU path");
    return DP_ERR_CUDA;
  }
  dp_model* m = new (std::nothrow) dp_model();
  DP_REQUIRE(m != nullptr, "dp_create: out of host memory");
  m->d = Dims{n_pts, c_in, c_out, hid, n_layer, n_head, has_temb ? 1 : 0};
  m->n_params = param_count(m->d);
  Weights tmp{};
  m->blob_floats = carve(tmp, m->d, nullptr);
  cudaError_t e = cudaGetDevice(&m->device);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, m->device);
  if (e == cudaSuccess && (m->blob.reserve(m->blob_floats * sizeof(float)) != DP_OK || m->dw.reserve(sizeof(Weights)) != DP_OK))
    e = cudaErrorMemoryAllocation;
  if (e == cudaSuccess) e = cudaMemset(m->blob.get<float>(), 0, m->blob_floats * sizeof(float));
  if (e != cudaSuccess) {
    set_error(std::string("dp_create: ") + cudaGetErrorString(e));
    delete m;
    return DP_ERR_CUDA;
  }
  carve(m->hw, m->d, m->blob.get<float>());
  *out = m;
  return DP_OK;
}

long dp_param_count(dp_handle h) { return h ? h->n_params : -1; }

int dp_pack(dp_handle h, const float* params, long n_floats, const float* adj_host, void* stream) {
  DP_REQUIRE(h && params && adj_host, "dp_pack: NULL argument");
  if (n_floats != h->n_params) {
    set_error("dp_pack: expected " + std::to_string(h->n_params) + " floats, got " + std::to_string(n_floats));
    return DP_ERR_INVALID;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  DP_TRY(check_device(h, "dp_pack"));
  DP_TRY(pack_fp32(h, params, adj_host, s));
  h->tcx_packed = false;                      // the split-precision blocks are rebuilt lazily, on that engine's next use
  if (tc_supported(h->d)) DP_TRY(tc2_pack(h, s));
  h->temb_t.clear();
  h->packed = true;
  return DP_OK;
}

int dp_set_engine(dp_handle h, int engine) {
  DP_REQUIRE(h, "dp_set_engine: NULL handle");
  DP_REQUIRE(engine == DP_ENGINE_AUTO || engine == DP_ENGINE_FP32 || engine == DP_ENGINE_TCX || engine == DP_ENGINE_TCG, "dp_set_engine: unknown engine");
  if ((engine == DP_ENGINE_TCX || engine == DP_ENGINE_TCG) && !tc_supported(h->d)) {
    set_error("dp_set_engine: the tensor-core engines need hid_dim=96, n_head=4, n_pts=17 and coords_dim <= 5");
    return DP_ERR_UNSUPPORTED;
  }
  h->engine = engine;
  return DP_OK;
}

int dp_get_engine(dp_handle h) {
  if (!h) return DP_ERR_INVALID;
  if (h->engine == DP_ENGINE_FP32 || !tc_supported(h->d)) return DP_ENGINE_FP32;
  if (h->engine == DP_ENGINE_TCX) return DP_ENGINE_TCX;
  return DP_ENGINE_TCG;   // AUTO = the fp16-operand tensor-core engine (its error is damped by the DDIM schedule)
}

int dp_get_forward_engine(dp_handle h) {
  if (!h) return DP_ERR_INVALID;
  return forward_engine(h);
}

int dp_forward(dp_handle h, const float* x, const float* t, const unsigned char* mask, float* out, long n, void* stream) {
  DP_REQUIRE(h && x && out, "dp_forward: NULL argument");
  DP_REQUIRE(n >= 0, "dp_forward: negative batch");
  if (!h->packed) { set_error("dp_forward: dp_pack has not been called"); return DP_ERR_STATE; }
  DP_REQUIRE(!h->d.has_temb || t != nullptr, "dp_forward: t is required for the diffusion denoiser");
  if (n == 0) return DP_OK;
  DP_TRY(check_device(h, "dp_forward"));
  return forward_chunks(h, forward_engine(h), x, t, mask, out, n, false, static_cast<cudaStream_t>(stream));
}

int dp_lift(dp_handle h, const float* uv, const unsigned char* mask, float* out_uvxyz, long n, void* stream) {
  DP_REQUIRE(h && uv && out_uvxyz, "dp_lift: NULL argument");
  DP_REQUIRE(n >= 0, "dp_lift: negative batch");
  DP_REQUIRE(!h->d.has_temb, "dp_lift: the handle must be a GCNpose lifter (has_temb = 0)");
  if (!h->packed) { set_error("dp_lift: dp_pack has not been called"); return DP_ERR_STATE; }
  if (n == 0) return DP_OK;
  DP_TRY(check_device(h, "dp_lift"));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int eng = forward_engine(h);
  if (eng == DP_ENGINE_TCX) return forward_chunks(h, eng, uv, nullptr, mask, out_uvxyz, n, true, s);   // glue fused into the kernel's store
  const Dims& d = h->d;
  DP_TRY(h->lift_scratch.reserve((size_t)n * d.n_pts * d.c_out * sizeof(float)));
  float* xyz = h->lift_scratch.get<float>();
  DP_TRY(forward_chunks(h, eng, uv, nullptr, mask, xyz, n, false, s));
  return lift_glue_launch(uv, xyz, out_uvxyz, n, d.n_pts, d.c_in, d.c_out, s);
}

// The keyed stream of a call (dp_philox.cuh); the pose index is one 32-bit counter word.
static int make_key(const dp_noise_key* k, long n_pose, const char* what, NoiseKey* out) {
  if (k->pose_offset < 0 || k->step_offset < 0 || n_pose > (1L << 32) || k->pose_offset > (1L << 32) - n_pose) {
    set_error(std::string(what) + ": the key needs pose_offset >= 0, step_offset >= 0 and pose_offset + n_pose <= 2^32");
    return DP_ERR_INVALID;
  }
  out->k0 = (uint32_t)(k->seed & 0xffffffffull); out->k1 = (uint32_t)(k->seed >> 32);
  out->pose_offset = (uint32_t)k->pose_offset; out->step_offset = (uint32_t)k->step_offset; out->on = 1;
  return DP_OK;
}

static int sample_impl(dp_handle h, const float* x_in, int x_is_repeated, float* x_out, long n_pose, int n_hyp,
                       const dp_step* steps_host, int n_steps, const float* noise, const dp_noise_key* key, const unsigned char* mask,
                       int mean_over_hyp, const float* targets_xyz, const int* group, int n_groups, double* sums, float* xs_traj,
                       float* x0_traj, void* stream) {
  DP_REQUIRE(h && x_in && x_out && steps_host, "dp_sample: NULL argument");
  DP_REQUIRE(n_pose >= 0 && n_hyp >= 1 && n_steps >= 1, "dp_sample: n_pose >= 0, n_hyp >= 1, n_steps >= 1 required");
  DP_REQUIRE(h->d.has_temb, "dp_sample: handle was created with has_temb = 0 (GCNpose has no sampler)");
  DP_REQUIRE(!(noise && key), "dp_sample: give either a noise tensor or a noise key, not both");
  DP_REQUIRE(!group || targets_xyz, "dp_sample: group ids need targets_xyz");
  DP_REQUIRE(!group || n_groups >= 1, "dp_sample: group ids need n_groups >= 1");
  if (targets_xyz != nullptr) {
    DP_REQUIRE(sums != nullptr, "dp_sample: targets_xyz needs sums");
    DP_REQUIRE(h->d.c_out >= 3, "dp_sample: the model's output needs at least the three xyz coordinates");
    DP_REQUIRE(n_hyp == 1 || mean_over_hyp, "dp_sample: with n_hyp > 1 the metrics are those of the hypothesis mean (set mean_over_hyp)");
  }
  NoiseKey nk{};
  if (key != nullptr) {
    DP_TRY(make_key(key, n_pose, "dp_sample", &nk));
    // every c1 = 0 (eta = 0): the noise term is skipped, as with a NULL noise pointer
    bool any = false;
    for (int i = 0; i < n_steps; ++i) any = any || steps_host[i].c1 != 0.f;
    nk.on = any ? 1 : 0;
  }
  if (!h->packed) { set_error("dp_sample: dp_pack has not been called"); return DP_ERR_STATE; }
  if (n_pose == 0) return DP_OK;
  DP_TRY(check_device(h, "dp_sample"));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const Dims& d = h->d;

  StepsArg inl{};
  const dp_step* steps_dev = nullptr;
  if (n_steps <= kMaxInlineSteps) {
    std::memcpy(inl.s, steps_host, n_steps * sizeof(dp_step));
  } else {
    // long schedules (> 64 steps) live in a device buffer that is uploaded when the schedule CHANGES, not per call; the
    // upload reads the handle's own copy, and the one synchronisation below only happens on such a change
    const bool same = h->steps.get<dp_step>() != nullptr && h->steps_host.size() == (size_t)n_steps &&
                      std::memcmp(h->steps_host.data(), steps_host, n_steps * sizeof(dp_step)) == 0;
    if (!same) {
      DP_TRY(h->steps.reserve((size_t)n_steps * sizeof(dp_step)));
      h->steps_host.assign(steps_host, steps_host + n_steps);
      DP_CUDA(cudaMemcpyAsync(h->steps.get<dp_step>(), h->steps_host.data(), n_steps * sizeof(dp_step), cudaMemcpyHostToDevice, s));
      DP_CUDA(cudaStreamSynchronize(s));
    }
    steps_dev = h->steps.get<dp_step>();
  }
  // batch-invariant time embeddings: one row per step (models/gcndiff.py:103-106, :51).  The table depends only
  // on the weights and the schedule, so it is kept across calls until either changes.
  {
    bool same = (long)h->temb_t.size() == n_steps;
    for (int i = 0; same && i < n_steps; ++i) same = (h->temb_t[i] == steps_host[i].t);
    if (!same) {
      DP_TRY(simt_temb(h, steps_dev ? &steps_dev->t : nullptr, sizeof(dp_step) / sizeof(float), &inl, n_steps, s));
      if (tc_supported(d)) DP_TRY(tc2_tau(h, n_steps, s));
      h->temb_t.resize(n_steps);
      for (int i = 0; i < n_steps; ++i) h->temb_t[i] = steps_host[i].t;
    }
  }

  EngineCall c;
  c.x_in = x_in; c.x_is_repeated = x_is_repeated; c.out = x_out; c.n_pose = n_pose; c.n_hyp = n_hyp;
  c.n_steps = n_steps; c.steps_dev = steps_dev; c.inl = &inl; c.noise = noise; c.key = nk; c.mask = mask;
  c.xs_traj = xs_traj; c.x0_traj = x0_traj;   // hypothesis rows, written by every engine before any mean
  const bool mean = mean_over_hyp && n_hyp > 1;
  const int eng = dp_get_engine(h);
  // default engine: the hypothesis mean -- and, with targets_xyz, the MPJPE / P-MPJPE sums -- are fused into the kernel's
  // final store (one launch, no [H*B] scratch)
  if (eng == DP_ENGINE_TCG) {
    c.mean_over_hyp = mean; c.gt = targets_xyz; c.group = group; c.n_groups = n_groups; c.sums = sums;
    return tc2_run(h, c, s);
  }
  const int row_floats = d.n_pts * d.c_out;
  if (mean) {
    DP_TRY(h->hyp_scratch.reserve((size_t)n_pose * n_hyp * row_floats * sizeof(float)));
    c.out = h->hyp_scratch.get<float>();
  }
  DP_TRY(run_engine(h, eng, c, s));
  if (mean) DP_TRY(hyp_mean_launch(c.out, x_out, n_pose, n_hyp, row_floats, s));
  if (targets_xyz != nullptr) DP_TRY(metrics_launch(x_out, d.c_out, d.c_out - 3, targets_xyz, n_pose, d.n_pts, group, n_groups, sums, nullptr, s));
  return DP_OK;
}

int dp_sample(dp_handle h, const float* x_in, int x_is_repeated, float* x_out, long n_pose, int n_hyp,
              const dp_step* steps_host, int n_steps, const float* noise, const dp_noise_key* key, const unsigned char* mask,
              int mean_over_hyp, const float* targets_xyz, double* sums, void* stream) {
  return sample_impl(h, x_in, x_is_repeated, x_out, n_pose, n_hyp, steps_host, n_steps, noise, key, mask, mean_over_hyp, targets_xyz,
                     nullptr, 1, sums, nullptr, nullptr, stream);
}

int dp_sample_grouped(dp_handle h, const float* x_in, int x_is_repeated, float* x_out, long n_pose, int n_hyp,
                      const dp_step* steps_host, int n_steps, const float* noise, const dp_noise_key* key, const unsigned char* mask,
                      int mean_over_hyp, const float* targets_xyz, const int* group, int n_groups, double* sums, void* stream) {
  return sample_impl(h, x_in, x_is_repeated, x_out, n_pose, n_hyp, steps_host, n_steps, noise, key, mask, mean_over_hyp, targets_xyz,
                     group, n_groups, sums, nullptr, nullptr, stream);
}

int dp_sample_trajectory(dp_handle h, const float* x_in, int x_is_repeated, float* x_out, long n_pose, int n_hyp,
                         const dp_step* steps_host, int n_steps, const float* noise, const dp_noise_key* key, const unsigned char* mask,
                         int mean_over_hyp, float* xs_traj, float* x0_traj, void* stream) {
  return sample_impl(h, x_in, x_is_repeated, x_out, n_pose, n_hyp, steps_host, n_steps, noise, key, mask, mean_over_hyp, nullptr,
                     nullptr, 1, nullptr, xs_traj, x0_traj, stream);
}

int dp_noise_fill(const dp_noise_key* key, int n_steps, long n_pose, int n_hyp, int n_pts, int c, float* out, void* stream) {
  DP_REQUIRE(key, "dp_noise_fill: NULL key");
  DP_REQUIRE(n_steps >= 0 && n_pose >= 0 && n_hyp >= 1 && n_pts >= 1 && c >= 1, "dp_noise_fill: n_steps >= 0, n_pose >= 0, n_hyp >= 1, n_pts >= 1, c >= 1 required");
  NoiseKey nk{};
  DP_TRY(make_key(key, n_pose, "dp_noise_fill", &nk));
  if (n_steps == 0 || n_pose == 0) return DP_OK;
  DP_REQUIRE(out, "dp_noise_fill: NULL output");
  return noise_fill_launch(nk, n_steps, n_pose, n_hyp, n_pts * c, out, static_cast<cudaStream_t>(stream));
}

int dp_metrics(const float* pred, int pred_stride, int pred_offset, const float* gt, long n, int n_pts,
               const int* group, int n_groups, double* sums, float* per_pose, void* stream) {
  DP_REQUIRE(pred && gt && sums, "dp_metrics: NULL argument");
  DP_REQUIRE(n_pts == kMaxPts, "dp_metrics: n_pts must be 17");
  DP_REQUIRE(pred_stride >= 3 && pred_offset >= 0 && pred_offset + 3 <= pred_stride, "dp_metrics: bad pred stride/offset");
  DP_REQUIRE(!group || n_groups >= 1, "dp_metrics: group ids need n_groups >= 1");
  if (n <= 0) return n == 0 ? DP_OK : DP_ERR_INVALID;
  return metrics_launch(pred, pred_stride, pred_offset, gt, n, n_pts, group, n_groups, sums, per_pose, static_cast<cudaStream_t>(stream));
}

int dp_metrics_hyp(const float* pred, int pred_stride, int pred_offset, int n_hyp, const float* gt, long n, int n_pts, const int* group,
                   int n_groups, double* sums, float* mean_out, float* per_hyp, void* stream) {
  DP_REQUIRE(pred && gt && sums, "dp_metrics_hyp: NULL argument");
  DP_REQUIRE(n_hyp >= 1, "dp_metrics_hyp: n_hyp >= 1 required");
  DP_REQUIRE(n_pts == kMaxPts, "dp_metrics_hyp: n_pts must be 17");
  DP_REQUIRE(pred_stride >= 3 && pred_offset >= 0 && pred_offset + 3 <= pred_stride, "dp_metrics_hyp: bad pred stride/offset");
  DP_REQUIRE(!group || n_groups >= 1, "dp_metrics_hyp: group ids need n_groups >= 1");
  if (n <= 0) return n == 0 ? DP_OK : DP_ERR_INVALID;
  return metrics_hyp_launch(pred, pred_stride, pred_offset, n_hyp, gt, n, group, n_groups, sums, mean_out, per_hyp,
                            static_cast<cudaStream_t>(stream));
}

int dp_selftest_umma(const void* smem_image, int image_bytes, const dp_mma_op* ops_host, int n_ops, float* tmem_out, int ncols,
                     void* stream) {
  DP_REQUIRE(smem_image && ops_host && tmem_out, "dp_selftest_umma: NULL argument");
  return tc_lab(smem_image, image_bytes, ops_host, n_ops, tmem_out, ncols, nullptr, 0, 0, static_cast<cudaStream_t>(stream));
}

int dp_selftest_umma_ts(const void* smem_image, int image_bytes, const void* tmem_image, int tmem_col0, int tmem_ncols,
                        const dp_mma_op* ops_host, int n_ops, float* tmem_out, int ncols, void* stream) {
  DP_REQUIRE(smem_image && tmem_image && ops_host && tmem_out, "dp_selftest_umma_ts: NULL argument");
  return tc_lab(smem_image, image_bytes, ops_host, n_ops, tmem_out, ncols, tmem_image, tmem_col0, tmem_ncols, static_cast<cudaStream_t>(stream));
}

int dp_selftest_cycles(long long* out2) {
  DP_REQUIRE(out2, "dp_selftest_cycles: NULL argument");
  tc_lab_cycles(out2);
  return DP_OK;
}

int dp_set_trace(dp_handle h, long long* dev_buf, int capacity) {
  DP_REQUIRE(h, "dp_set_trace: NULL handle");
  DP_REQUIRE(capacity >= 0 && (dev_buf != nullptr || capacity == 0), "dp_set_trace: bad buffer");
  h->trace = capacity > 0 ? dev_buf : nullptr;
  h->trace_cap = capacity;
  return DP_OK;
}

// ---------------------------------------------------------------------------------------------- host-resident batches
struct dp_hstream {
  dp_handle h = nullptr;
  long max_pose = 0;
  int n_hyp = 1, mean = 0, depth = 0, head = 0;
  size_t in_floats = 0, out_floats = 0;
  cudaStream_t s_in = nullptr, s_out = nullptr;
  DevBuf x_dev[16], out_dev[16], gt_dev[16], grp_dev[16];   // per slot (depth <= 16): input, result, and (evaluation) the targets and
                                                           // group ids of the batch
  std::vector<cudaEvent_t> ev_in, ev_done, ev_out;
};

int dp_hstream_create(dp_hstream_t* out, dp_handle h, long max_pose, int n_hyp, int mean_over_hyp, int depth) {
  DP_REQUIRE(out && h, "dp_hstream_create: NULL argument");
  *out = nullptr;
  DP_REQUIRE(max_pose >= 1 && n_hyp >= 1 && depth >= 1 && depth <= 16, "dp_hstream_create: max_pose >= 1, n_hyp >= 1, 1 <= depth <= 16 required");
  DP_REQUIRE(h->d.has_temb, "dp_hstream_create: the handle must be a GCNdiff denoiser (the sampler runs on it)");
  DP_TRY(check_device(h, "dp_hstream_create"));
  dp_hstream* s = new (std::nothrow) dp_hstream();
  DP_REQUIRE(s != nullptr, "dp_hstream_create: out of host memory");
  s->h = h; s->max_pose = max_pose; s->n_hyp = n_hyp; s->mean = (mean_over_hyp && n_hyp > 1) ? 1 : 0; s->depth = depth;
  const size_t row = (size_t)h->d.n_pts * h->d.c_in;
  s->in_floats = (size_t)max_pose * row;
  s->out_floats = (size_t)max_pose * (s->mean ? 1 : n_hyp) * row;
  cudaError_t e = cudaStreamCreateWithFlags(&s->s_in, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->s_out, cudaStreamNonBlocking);
  for (int i = 0; i < depth && e == cudaSuccess; ++i) {
    cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr;
    if (s->x_dev[i].reserve(s->in_floats * sizeof(float)) != DP_OK || s->out_dev[i].reserve(s->out_floats * sizeof(float)) != DP_OK ||
        s->gt_dev[i].reserve((size_t)max_pose * h->d.n_pts * 3 * sizeof(float)) != DP_OK || s->grp_dev[i].reserve((size_t)max_pose * sizeof(int)) != DP_OK)
      e = cudaErrorMemoryAllocation;
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&e0, cudaEventDisableTiming);
    if (e == cudaSuccess) { s->ev_in.push_back(e0); e = cudaEventCreateWithFlags(&e1, cudaEventDisableTiming); }
    if (e == cudaSuccess) { s->ev_done.push_back(e1); e = cudaEventCreateWithFlags(&e2, cudaEventDisableTiming); }
    if (e == cudaSuccess) s->ev_out.push_back(e2);
  }
  if (e != cudaSuccess) {
    set_error(std::string("dp_hstream_create: ") + cudaGetErrorString(e));
    dp_hstream_destroy(s);
    return DP_ERR_CUDA;
  }
  *out = s;
  return DP_OK;
}

int dp_hstream_submit(dp_hstream_t s, const float* x_host, const float* targets_host, double* sums_dev, long n_pose, const dp_step* steps_host,
                      int n_steps, const float* noise_dev, const dp_noise_key* key, const unsigned char* mask_dev, float* out_host,
                      void* stream, int* slot_out) {
  return dp_hstream_submit_grouped(s, x_host, targets_host, nullptr, 1, sums_dev, n_pose, steps_host, n_steps, noise_dev, key, mask_dev,
                                   out_host, stream, slot_out);
}

int dp_hstream_submit_grouped(dp_hstream_t s, const float* x_host, const float* targets_host, const int* groups_host, int n_groups,
                              double* sums_dev, long n_pose, const dp_step* steps_host, int n_steps, const float* noise_dev,
                              const dp_noise_key* key, const unsigned char* mask_dev, float* out_host, void* stream, int* slot_out) {
  DP_REQUIRE(s && x_host && out_host && steps_host && slot_out, "dp_hstream_submit: NULL argument");
  DP_REQUIRE(n_pose >= 1 && n_pose <= s->max_pose, "dp_hstream_submit: batch exceeds the max_pose this stream was created for");
  // the combinations dp_sample refuses, refused before the copies below are enqueued
  DP_REQUIRE(!(noise_dev && key), "dp_hstream_submit: give either a noise tensor or a noise key, not both");
  DP_REQUIRE(!targets_host || (sums_dev && (s->n_hyp == 1 || s->mean)),
             "dp_hstream_submit: targets_host needs sums_dev and, with n_hyp > 1, a stream created with mean_over_hyp");
  DP_REQUIRE(!groups_host || targets_host, "dp_hstream_submit: groups_host needs targets_host");
  DP_REQUIRE(!groups_host || n_groups >= 1, "dp_hstream_submit: groups_host needs n_groups >= 1");
  DP_TRY(check_device(s->h, "dp_hstream_submit"));
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  const int k = s->head;
  const size_t row = (size_t)s->h->d.n_pts * s->h->d.c_in;
  const size_t in_bytes = (size_t)n_pose * row * sizeof(float), out_bytes = (size_t)n_pose * (s->mean ? 1 : s->n_hyp) * row * sizeof(float);
  // H2D on the copy-in stream, once the kernel that last read this slot's input has finished
  DP_CUDA(cudaStreamWaitEvent(s->s_in, s->ev_done[k], 0));
  DP_CUDA(cudaMemcpyAsync(s->x_dev[k].get<float>(), x_host, in_bytes, cudaMemcpyHostToDevice, s->s_in));
  if (targets_host != nullptr)
    DP_CUDA(cudaMemcpyAsync(s->gt_dev[k].get<float>(), targets_host, (size_t)n_pose * s->h->d.n_pts * 3 * sizeof(float), cudaMemcpyHostToDevice, s->s_in));
  if (groups_host != nullptr)
    DP_CUDA(cudaMemcpyAsync(s->grp_dev[k].get<int>(), groups_host, (size_t)n_pose * sizeof(int), cudaMemcpyHostToDevice, s->s_in));
  DP_CUDA(cudaEventRecord(s->ev_in[k], s->s_in));
  // the sampler on the caller's stream, once the input is there and the slot's previous result has left the device
  DP_CUDA(cudaStreamWaitEvent(cs, s->ev_in[k], 0));
  DP_CUDA(cudaStreamWaitEvent(cs, s->ev_out[k], 0));
  DP_TRY(sample_impl(s->h, s->x_dev[k].get<float>(), 0, s->out_dev[k].get<float>(), n_pose, s->n_hyp, steps_host, n_steps, noise_dev, key,
                     mask_dev, s->mean, targets_host != nullptr ? s->gt_dev[k].get<float>() : nullptr,
                     groups_host != nullptr ? s->grp_dev[k].get<int>() : nullptr, n_groups, sums_dev, nullptr, nullptr, stream));
  DP_CUDA(cudaEventRecord(s->ev_done[k], cs));
  // D2H on the copy-out stream
  DP_CUDA(cudaStreamWaitEvent(s->s_out, s->ev_done[k], 0));
  DP_CUDA(cudaMemcpyAsync(out_host, s->out_dev[k].get<float>(), out_bytes, cudaMemcpyDeviceToHost, s->s_out));
  DP_CUDA(cudaEventRecord(s->ev_out[k], s->s_out));
  *slot_out = k;
  s->head = (k + 1) % s->depth;
  return DP_OK;
}

int dp_hstream_wait(dp_hstream_t s, int slot) {
  DP_REQUIRE(s && slot >= 0 && slot < s->depth, "dp_hstream_wait: bad slot");
  DP_CUDA(cudaEventSynchronize(s->ev_out[slot]));
  return DP_OK;
}

void dp_hstream_destroy(dp_hstream_t s) {
  if (!s) return;
  if (s->s_in) cudaStreamSynchronize(s->s_in);
  if (s->s_out) cudaStreamSynchronize(s->s_out);
  for (cudaEvent_t e : s->ev_in) cudaEventDestroy(e);
  for (cudaEvent_t e : s->ev_done) cudaEventDestroy(e);
  for (cudaEvent_t e : s->ev_out) cudaEventDestroy(e);
  if (s->s_in) cudaStreamDestroy(s->s_in);
  if (s->s_out) cudaStreamDestroy(s->s_out);
  delete s;
}

long dp_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int dp_last_launch_info(dp_handle h, long* out6) {
  DP_REQUIRE(h && out6, "dp_last_launch_info: NULL argument");
  for (int i = 0; i < 6; ++i) out6[i] = h->last_launch[i];
  return DP_OK;
}

const char* dp_last_error(void) { return g_err.c_str(); }
const char* dp_version(void) { return "diffpose_b200 0.5 (sm_100a)"; }
int dp_device(dp_handle h) { return h ? h->device : DP_ERR_INVALID; }

void dp_destroy(dp_handle h) { delete h; }

}  // extern "C"
