// Internal declarations shared by the translation units of libdiffpose_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>
#include "../../include/diffpose_b200.h"
#include "../../include/diffpose_b200_diag.h"
#include "dp_philox.cuh"

namespace dp {

constexpr int kMaxLayers = 16;
constexpr int kMaxPts = 17;       // the kernels are written for the 17-joint Human3.6M skeleton
constexpr int kMaxCoord = 8;      // c_in / c_out upper bound (uvxyz = 5)

struct Dims {
  int n_pts, c_in, c_out, hid, n_layer, n_head, has_temb;
};

// fp32 weights of one GraAttenLayer + _ResChebGC(_diff) pair, every matrix stored [K][N] row-major
// (K = input feature, N = output feature) so that a warp reads consecutive output features.
struct LayerW {
  const float *ln0_a, *ln0_b;   // atten_layers.l.sublayer.0.norm
  const float *wqkv, *bqkv;     // [hid][3hid] = linears.0|1|2 side by side
  const float *wo, *bo;         // [hid][hid]   linears.3
  const float *ln1_a, *ln1_b;   // sublayer.1.norm
  const float *lhat;            // [n_pts][n_pts]  D A_hat D  (GraFormer.py:174-178)
  const float *w1, *b1;         // [hid][2hid]  feed_forward.gconv1.fc
  const float *w2, *b2;         // [2hid][hid]  feed_forward.gconv2.fc
  const float *wc1, *bc1;       // [3hid][hid]  gconv_layers.l.gconv1.gconv  (k = cheb_order*hid + c)
  const float *wc2, *bc2;       // [3hid][hid]  gconv_layers.l.gconv2.gconv
  const float *wt, *bt;         // [4hid][hid]  gconv_layers.l.temb_proj (has_temb)
};

struct Weights {
  const float *win, *bin;       // [3c_in][hid]
  const float *wout, *bout;     // [3hid][c_out]
  const float *t1, *t2;         // Chebyshev T1 = L, T2 = 2L^2 - I, [n_pts][n_pts]
  const float *t1m, *t2m;       // the same matrices factored as diag(t?s) * t?m with fp16-exact t?m when the rows allow it
  const float *t1s, *t2s;       //   (row scales [n_pts]); used by the tensor-core engine, see integerise_rows in dp_api.cu
  const float *wd0, *bd0;       // [hid][4hid]  temb.dense.0
  const float *wd1, *bd1;       // [4hid][4hid] temb.dense.1
  LayerW layer[kMaxLayers];
};

void set_error(const std::string& msg);
void count_launch(int n = 1);

#define DP_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      dp::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                           \
      return DP_ERR_CUDA;                                                                          \
    }                                                                                              \
  } while (0)

#define DP_REQUIRE(cond, msg)                                                                      \
  do {                                                                                             \
    if (!(cond)) {                                                                                 \
      dp::set_error(std::string(msg));                                                             \
      return DP_ERR_INVALID;                                                                       \
    }                                                                                              \
  } while (0)

#define DP_TRY(expr)              \
  do {                            \
    int _rc = (expr);             \
    if (_rc != DP_OK) return _rc; \
  } while (0)

// DDIM step scalars travel as a by-value kernel argument (no host->device copy, graph friendly).
constexpr int kMaxInlineSteps = 64;
struct StepsArg {
  dp_step s[kMaxInlineSteps];
};

// A grow-only device allocation that frees itself.  reserve() keeps the block when it is large enough; otherwise it frees
// it, contents and all, before allocating the new one (at least 4 KB).  If cudaMalloc fails the buffer is left empty, so
// the next reserve() allocates again instead of handing out a freed pointer.
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { if (p_) cudaFree(p_); }
  template <class T>
  T* get() const { return static_cast<T*>(p_); }
  int reserve(size_t bytes) {
    if (p_ && bytes_ >= bytes) return DP_OK;
    if (p_) cudaFree(p_);
    p_ = nullptr; bytes_ = 0;
    if (bytes < 4096) bytes = 4096;
    void* p = nullptr;
    DP_CUDA(cudaMalloc(&p, bytes));
    p_ = p; bytes_ = bytes;
    return DP_OK;
  }

 private:
  void* p_ = nullptr;
  size_t bytes_ = 0;
};

// One engine launch: a sampler call, or one chunk of a forward call (forward_only).  dp_api.cu decides which engine runs
// and which tails it fuses, and sets only the fields that engine implements; the rest keep these defaults.
struct EngineCall {
  const float* x_in = nullptr;
  int x_is_repeated = 0;         // 1: x_in holds all n_pose * n_hyp rows; 0: one row per pose, read for every hypothesis
  float* out = nullptr;
  long n_pose = 0;
  int n_hyp = 1;
  int n_steps = 1;
  const dp_step* steps_dev = nullptr;   // the handle's step table when n_steps > kMaxInlineSteps, else NULL
  const StepsArg* inl = nullptr;        // the step scalars otherwise (zero for a forward call)
  const float* noise = nullptr;
  NoiseKey key{};                       // key.on: the noise is the keyed stream (dp_philox.cuh) and `noise` is NULL
  const unsigned char* mask = nullptr;
  bool forward_only = false;
  float* xs_traj = nullptr;      // sampler, every engine: x_t after step k and the x0 of that update, [n_steps][n_pose * n_hyp]
  float* x0_traj = nullptr;      //   [n_pts][c] hypothesis-major (dp_sample_trajectory); either may be NULL
  // fused by tcg only
  bool mean_over_hyp = false;    // out is [n_pose, n_pts, c], the mean over each pose's hypotheses
  const float* gt = nullptr;     // fused evaluation tail, see dp_sample's targets_xyz
  const int* group = nullptr;    //   and dp_sample_grouped's group ids: sums is then [n_groups][3]
  int n_groups = 1;
  double* sums = nullptr;
  // fused by tcx only
  bool emit_uvxyz = false;       // forward of GCNpose: out is [n, n_pts, c_in + c_out] = [uv | xyz - xyz_root] (dp_lift)
};

// Opts `Kernel` into `bytes` of dynamic shared memory once per device (function attributes are per device).
template <auto Kernel>
int smem_opt_in(int device, int bytes) {
  static bool done[64] = {};
  bool& d = done[device & 63];
  if (!d) {
    DP_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    d = true;
  }
  return DP_OK;
}

}  // namespace dp

// The opaque handle.
struct dp_model {
  dp::Dims d{};
  int device = 0;
  int sm_count = 0;
  int engine = DP_ENGINE_AUTO;
  bool packed = false;
  long n_params = 0;

  dp::DevBuf blob;                // packed fp32 weights
  size_t blob_floats = 0;
  dp::Weights hw{};               // host copy of the device pointers
  dp::DevBuf dw;                  // the same struct in device memory

  dp::DevBuf temb;                // [n_rows][n_layer][hid] fp32 time-embedding table scratch
  std::vector<float> temb_t;      // timesteps the table currently holds (sampler schedule cache; empty = invalid)
  dp::DevBuf steps;               // device copy of the step scalars, only used when n_steps > kMaxInlineSteps
  std::vector<dp_step> steps_host;   // what `steps` currently holds (a long schedule is uploaded once, not per call)
  dp::DevBuf hyp_scratch;         // [n_pose*n_hyp, n_pts, c] fp32: hypothesis mean of the engines that do not fuse it (fp32, tcx)
  dp::DevBuf lift_scratch;        // [n, n_pts, c_out] fp32: dp_lift on the engines that do not fuse the glue

  dp::DevBuf tc2_blocks;          // default tensor-core engine: fp16 weight blocks, io blocks, per-layer parameters (dp_pack)
  dp::DevBuf tc2_tau;             //   and the GC2 bias blocks of the cached sampler schedule
  dp::DevBuf tcx_blocks;          // split-precision engine: hi/lo fp16 weight blocks, packed lazily
  bool tcx_packed = false;        //   from the current fp32 blob (cleared by dp_pack, set on the engine's next use)
  long last_launch[6] = {0, 0, 0, 0, 0, 0};
  long long* trace = nullptr;     // caller-owned device buffer for the hand-over timestamps (dp_set_trace)
  int trace_cap = 0;
};

namespace dp {
// dp_last_launch_info: grid, block, dynamic shared memory, poses per tile, engine, tiles of the last engine launch
inline void record_launch(dp_model* m, long grid, long threads, long smem, long tile_poses, int engine, long n_tiles) {
  long* l = m->last_launch;
  l[0] = grid; l[1] = threads; l[2] = smem; l[3] = tile_poses; l[4] = engine; l[5] = n_tiles;
}
// The engines: each fills its kernel arguments from the call and launches.  A sampler call reads m->temb as the table of
// its schedule, a forward call as the per-sample table of its chunk (simt_temb).
int simt_run(dp_model* m, const EngineCall& c, cudaStream_t s);
int tcx_run(dp_model* m, const EngineCall& c, cudaStream_t s);
int tc2_run(dp_model* m, const EngineCall& c, cudaStream_t s);
// dp_simt.cu
// time-embedding table [n_t][n_layer][hid]: t comes from t_dev[i*t_stride] or, when t_dev is NULL, from inl.s[i].t
int simt_temb(dp_model* m, const float* t_dev, int t_stride, const StepsArg* inl, long n_t, cudaStream_t s);
// dp_lab.cu
int tc_lab(const void* image_dev, int image_bytes, const dp_mma_op* ops_host, int n_ops, float* out_dev, int ncols,
           const void* tmem_image_dev, int tmem_col0, int tmem_ncols, cudaStream_t s);
void tc_lab_cycles(long long* out2);
// dp_tc2.cu
int tc2_pack(dp_model* m, cudaStream_t s);
// after simt_temb filled m->temb for a sampler schedule: the same embeddings as GC2 bias blocks of the tcg engine
int tc2_tau(dp_model* m, int n_steps, cudaStream_t s);
// dp_metrics.cu
// group != NULL: pose i adds to sums[3 * group[i] ..] of [n_groups][3], and nothing when group[i] is outside [0, n_groups)
int metrics_launch(const float* pred, int pred_stride, int pred_offset, const float* gt, long n, int n_pts,
                   const int* group, int n_groups, double* sums, float* per_pose, cudaStream_t s);
// dp_metrics_hyp: pred [n_hyp][n][n_pts][pred_stride] hypothesis-major; sums [n_groups][8] (group = NULL: row 0)
int metrics_hyp_launch(const float* pred, int pred_stride, int pred_offset, int n_hyp, const float* gt, long n, const int* group,
                       int n_groups, double* sums, float* mean_out, float* per_hyp, cudaStream_t s);
int hyp_mean_launch(const float* x, float* out, long n_pose, int n_hyp, int row_floats, cudaStream_t s);
// out[n][n_pts][c_in + c_out] = [uv | xyz - xyz[root]] (runners/diffpose_frame.py:337-343 with out-of-place root-centring)
int lift_glue_launch(const float* uv, const float* xyz, float* out, long n, int n_pts, int c_in, int c_out, cudaStream_t s);
// out[k][h * n_pose + p][e] = philox_normal(key, step_offset + k, pose_offset + p, h, e), e < row_floats (dp_noise_fill)
int noise_fill_launch(const NoiseKey& key, int n_steps, long n_pose, int n_hyp, int row_floats, float* out, cudaStream_t s);
}  // namespace dp
