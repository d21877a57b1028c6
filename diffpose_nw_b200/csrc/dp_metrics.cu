// Evaluation kernels that follow the sampler: hypothesis mean, MPJPE and Procrustes-aligned MPJPE.
//   hypothesis mean   runners/diffpose_frame.py:382
//   mpjpe             common/loss.py:7-13 (after root-centring, runners/diffpose_frame.py:384-386)
//   p_mpjpe           common/loss.py:25-64 == common/utils.py:155-187 (numpy float64 SVD in the reference;
//                     here one warp per pose: fp32 shuffle reductions for the centring / cross-covariance, a one-sided
//                     Jacobi SVD of the 3x3 matrix in fp32 registers, fp64 for the partial sums over poses)
#include "dp_internal.h"
#include "dp_metrics_dev.cuh"

namespace dp {
namespace {

using metric::NP;

__global__ void hyp_mean_kernel(const float* __restrict__ x, float* __restrict__ out, long n_pose, int n_hyp,
                                int row_floats) {
  const long total = n_pose * row_floats;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int h = 0; h < n_hyp; ++h) s += x[(size_t)h * total + i];
    out[i] = s / (float)n_hyp;
  }
}

// One WARP per pose: lane j < 17 owns joint j of the prediction and the target; every per-pose sum is a warp shuffle
// reduction, and the 3x3 SVD -- a register-only Jacobi iteration -- runs redundantly on all lanes (no divergence, no
// local-memory arrays).  A block of 8 warps handles 8 poses, so 1024 poses already
// spread over 128 CTAs (the first version ran one thread per pose with 34x3 doubles of local memory on 8 CTAs: 44 us
// per 1024 poses, half a sampler launch).
constexpr int kMetricWarps = 8;
__global__ void __launch_bounds__(kMetricWarps * 32) metrics_kernel(const float* __restrict__ pred, int ps, int po, const float* __restrict__ gt, long n,
                                                                    double* __restrict__ sums, float* __restrict__ per_pose) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // programmatic dependent launch (the evaluation loop alternates sampler and metrics kernels on one stream): this grid may
  // have been launched while the sampler that produces `pred` was draining -- wait for its results, and let the next
  // sampler launch begin its own set-up right away
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  double e1s = 0.0, e2s = 0.0, cnt = 0.0;      // this warp's partial sums (identical on every lane)
  for (long i = (long)blockIdx.x * kMetricWarps + warp; i < n; i += (long)gridDim.x * kMetricWarps) {
    const int j = lane < NP ? lane : 0;
    const float* p = pred + (size_t)i * NP * ps + po + j * ps;
    const float* g = gt + (size_t)i * NP * 3 + j * 3;
    float pv[3], gv[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) { pv[c] = p[c]; gv[c] = g[c]; }
    float e1f, e2f;
    metric::pose_errors(pv, gv, lane, e1f, e2f);
    const double e1 = (double)e1f, e2 = (double)e2f;
    e1s += e1; e2s += e2; cnt += 1.0;
    if (per_pose && lane == 0) { per_pose[2 * i] = (float)e1; per_pose[2 * i + 1] = (float)e2; }
  }
  // block reduction -> one atomic per block and quantity
  __shared__ double red[3][kMetricWarps];
  if (lane == 0) { red[0][warp] = e1s; red[1][warp] = e2s; red[2][warp] = cnt; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double s = 0.0;
    for (int w = 0; w < kMetricWarps; ++w) s += red[threadIdx.x][w];
    if (s != 0.0) atomicAdd(sums + threadIdx.x, s);
  }
}

// The same per pose, keyed by group (dp_metrics / dp_sample_grouped with group ids): pose i adds to row group[i] of sums
// [n_groups][3], and to nothing when the id is outside [0, n_groups).  Each warp carries the sums of its current run of
// equal ids in registers and flushes them with three atomics when the id changes and after its last pose: a batch that
// comes in runs of one action (as the reference's loader delivers them) costs about as many atomics as metrics_kernel.
__global__ void __launch_bounds__(kMetricWarps * 32, 2) metrics_grouped_kernel(const float* __restrict__ pred, int ps, int po, const float* __restrict__ gt,
                                                                            long n, const int* __restrict__ group, int n_groups,
                                                                            double* __restrict__ sums, float* __restrict__ per_pose) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  asm volatile("griddepcontrol.wait;" ::: "memory");            // as in metrics_kernel
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  double e1s = 0.0, e2s = 0.0, cnt = 0.0;      // the current run's partial sums (identical on every lane)
  int run = -1;                                 // and its id
  for (long i = (long)blockIdx.x * kMetricWarps + warp; i < n; i += (long)gridDim.x * kMetricWarps) {
    const int gi = __ldg(group + i);
    const int j = lane < NP ? lane : 0;
    const float* p = pred + (size_t)i * NP * ps + po + j * ps;
    const float* g = gt + (size_t)i * NP * 3 + j * 3;
    float pv[3], gv[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) { pv[c] = p[c]; gv[c] = g[c]; }
    float e1f, e2f;
    metric::pose_errors(pv, gv, lane, e1f, e2f);
    if (gi != run) {
      if (lane == 0 && cnt != 0.0 && (unsigned)run < (unsigned)n_groups) {
        atomicAdd(sums + 3 * run, e1s); atomicAdd(sums + 3 * run + 1, e2s); atomicAdd(sums + 3 * run + 2, cnt);
      }
      run = gi; e1s = e2s = cnt = 0.0;
    }
    const double e1 = (double)e1f, e2 = (double)e2f;
    e1s += e1; e2s += e2; cnt += 1.0;
    if (per_pose && lane == 0) { per_pose[2 * i] = (float)e1; per_pose[2 * i + 1] = (float)e2; }
  }
  if (lane == 0 && cnt != 0.0 && (unsigned)run < (unsigned)n_groups) {
    atomicAdd(sums + 3 * run, e1s); atomicAdd(sums + 3 * run + 1, e2s); atomicAdd(sums + 3 * run + 2, cnt);
  }
}

// NaN-propagating minimum (numpy's min): fminf would drop a NaN P-MPJPE of a zero-extent hypothesis
__device__ __forceinline__ float nan_min(float m, float x) { return (x < m || x != x) ? x : m; }

constexpr int kHypCols = 8;
// lane k < 8 adds column k of a run's sums to its row (a select chain, not an indexed load: acc stays in registers)
__device__ __forceinline__ void flush_hyp(const double (&acc)[kHypCols], int run, int n_groups, double* sums, int lane) {
  if (acc[2] == 0.0 || (unsigned)run >= (unsigned)n_groups || lane >= kHypCols) return;
  double v = acc[0];
#pragma unroll
  for (int k = 1; k < kHypCols; ++k) v = lane == k ? acc[k] : v;
  atomicAdd(sums + (size_t)kHypCols * run + lane, v);
}
// Multi-hypothesis evaluation (dp_metrics_hyp; the eight columns are defined in include/diffpose_b200.h).  One warp per
// pose, lane j < 17 owning joint j: the warp walks the H hypothesis rows of its pose in h order and carries in registers
// the fp32 running sum of the mean pose, the per-hypothesis minima, each lane's minimum joint distance and the fp64 sums
// of the average hypothesis.  Every per-hypothesis error is pose_errors on that row, the same bits dp_metrics gives it.
// Group sums are flushed per run of equal ids, as in metrics_grouped_kernel (no ids: one run per warp, into row 0).
__global__ void __launch_bounds__(kMetricWarps * 32) metrics_hyp_kernel(const float* __restrict__ pred, int ps, int po, int n_hyp,
                                                                        const float* __restrict__ gt, long n, const int* __restrict__ group,
                                                                        int n_groups, double* __restrict__ sums, float* __restrict__ mean_out,
                                                                        float* __restrict__ per_hyp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  asm volatile("griddepcontrol.wait;" ::: "memory");            // as in metrics_kernel
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const bool live = lane < NP;
  const int j = live ? lane : 0;
  const size_t hyp_stride = (size_t)n * NP * ps;               // floats between hypothesis h and h + 1 of a pose
  double acc[kHypCols] = {};                                     // the current run's sums (identical on every lane)
  int run = -1;
  for (long i = (long)blockIdx.x * kMetricWarps + warp; i < n; i += (long)gridDim.x * kMetricWarps) {
    const int gi = group != nullptr ? __ldg(group + i) : 0;
    const float* g = gt + (size_t)i * NP * 3 + j * 3;
    float g0[3], msum[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < 3; ++c) g0[c] = g[c];
    float best1 = INFINITY, best2 = INFINITY, jmin = INFINITY;
    double avg1 = 0.0, avg2 = 0.0;
    const float* row = pred + (size_t)i * NP * ps + po + j * ps;
    for (int h = 0; h < n_hyp; ++h, row += hyp_stride) {
      float pv[3], gv[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) { pv[c] = row[c]; gv[c] = g0[c]; msum[c] += pv[c]; }
      float e1, e2;
      metric::pose_errors(pv, gv, lane, e1, e2);                // leaves pv, gv root-centred
      // this joint's distance, with pose_errors' own operations on the same root-centred values
      float d2 = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float df = pv[c] - gv[c];
        d2 += df * df;
      }
      jmin = nan_min(jmin, sqrtf(d2));
      best1 = nan_min(best1, e1); best2 = nan_min(best2, e2);
      avg1 += (double)e1; avg2 += (double)e2;
      if (per_hyp && lane == 0) {
        const size_t r = (size_t)h * n + i;
        per_hyp[2 * r] = e1; per_hyp[2 * r + 1] = e2;
      }
    }
    // the hypothesis mean, in hyp_mean_kernel's order: summed from h = 0 upwards, one division
    float mv[3], gv[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) { mv[c] = msum[c] / (float)n_hyp; gv[c] = g0[c]; }
    if (mean_out != nullptr && live) {
      float* o = mean_out + (size_t)i * NP * ps + j * ps;
      const float* p = pred + (size_t)i * NP * ps + j * ps;
      for (int c = 0; c < ps; ++c) {
        if (c >= po && c < po + 3) { o[c] = c == po ? mv[0] : (c == po + 1 ? mv[1] : mv[2]); continue; }
        float s = 0.f;                                           // the channels outside xyz (uv of uvxyz)
        for (int h = 0; h < n_hyp; ++h) s += p[(size_t)h * hyp_stride + c];
        o[c] = s / (float)n_hyp;
      }
    }
    float m1, m2;
    metric::pose_errors(mv, gv, lane, m1, m2);
    // J-best: pose_errors' MPJPE reduction (shuffle tree, one division) over the per-joint minima
    float jb = live ? jmin : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) jb += __shfl_xor_sync(0xffffffffu, jb, o);
    jb = jb / (float)NP;
    if (gi != run) {
      flush_hyp(acc, run, n_groups, sums, lane);
      run = gi;
#pragma unroll
      for (int k = 0; k < kHypCols; ++k) acc[k] = 0.0;
    }
    acc[0] += (double)m1; acc[1] += (double)m2; acc[2] += 1.0;
    acc[3] += (double)best1; acc[4] += (double)best2; acc[5] += (double)jb;
    acc[6] += avg1 / n_hyp; acc[7] += avg2 / n_hyp;
  }
  flush_hyp(acc, run, n_groups, sums, lane);
}

// [uv | xyz - xyz[root]]: the glue between the lifter and the sampler for the engines whose forward kernel does not
// write it directly (runners/diffpose_frame.py:337-343 with the intended out-of-place root-centring)
__global__ void lift_glue_kernel(const float* __restrict__ uv, const float* __restrict__ xyz, float* __restrict__ out, long n, int n_pts,
                                 int c_in, int c_out) {
  const int wd = c_in + c_out;
  const long total = n * n_pts * wd;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long row = i / wd;
    const int c = (int)(i - row * wd);
    const long pose = row / n_pts;
    out[i] = c < c_in ? uv[row * c_in + c] : __fsub_rn(xyz[row * c_out + (c - c_in)], xyz[pose * n_pts * c_out + (c - c_in)]);
  }
}

}  // namespace

int metrics_launch(const float* pred, int pred_stride, int pred_offset, const float* gt, long n, int n_pts,
                   const int* group, int n_groups, double* sums, float* per_pose, cudaStream_t s) {
  (void)n_pts;
  long grid = (n + kMetricWarps - 1) / kMetricWarps;
  if (grid > 148 * 8) grid = 148 * 8;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kMetricWarps * 32); cfg.dynamicSmemBytes = 0; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (group != nullptr) DP_CUDA(cudaLaunchKernelEx(&cfg, metrics_grouped_kernel, pred, pred_stride, pred_offset, gt, n, group, n_groups, sums, per_pose));
  else DP_CUDA(cudaLaunchKernelEx(&cfg, metrics_kernel, pred, pred_stride, pred_offset, gt, n, sums, per_pose));
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

int metrics_hyp_launch(const float* pred, int pred_stride, int pred_offset, int n_hyp, const float* gt, long n, const int* group,
                       int n_groups, double* sums, float* mean_out, float* per_hyp, cudaStream_t s) {
  long grid = (n + kMetricWarps - 1) / kMetricWarps;
  if (grid > 148 * 8) grid = 148 * 8;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kMetricWarps * 32); cfg.dynamicSmemBytes = 0; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // chains behind the sampler, as metrics_launch
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  DP_CUDA(cudaLaunchKernelEx(&cfg, metrics_hyp_kernel, pred, pred_stride, pred_offset, n_hyp, gt, n, group, group ? n_groups : 1, sums,
                             mean_out, per_hyp));
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

int hyp_mean_launch(const float* x, float* out, long n_pose, int n_hyp, int row_floats, cudaStream_t s) {
  const long total = n_pose * row_floats;
  long grid = (total + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  hyp_mean_kernel<<<(unsigned)grid, 256, 0, s>>>(x, out, n_pose, n_hyp, row_floats);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

int lift_glue_launch(const float* uv, const float* xyz, float* out, long n, int n_pts, int c_in, int c_out, cudaStream_t s) {
  const long total = n * n_pts * (c_in + c_out);
  long grid = (total + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  lift_glue_kernel<<<(unsigned)grid, 256, 0, s>>>(uv, xyz, out, n, n_pts, c_in, c_out);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

}  // namespace dp
