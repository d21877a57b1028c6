// dp_noise_fill: the keyed noise stream of the sampler kernels (dp_philox.cuh) written out in the layout of dp_sample's
// `noise` argument, so that a keyed call can be reproduced through the noise pointer and a reference fed the same draws.
#include "dp_internal.h"

namespace dp {
namespace {

// out[k][h * n_pose + p][e]: one thread per element, each evaluating the same philox_normal the sampler kernels inline
__global__ void noise_fill_kernel(NoiseKey key, int n_steps, long n_pose, int n_hyp, int row_floats, float* __restrict__ out) {
  const long n_rows = n_pose * n_hyp;
  const long total = (long)n_steps * n_rows * row_floats;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long q = i / row_floats;
    const int e = (int)(i - q * row_floats);
    const long k = q / n_rows, row = q - k * n_rows;
    const long h = row / n_pose, p = row - h * n_pose;
    out[i] = philox_normal(key, key.step_offset + (uint32_t)k, key.pose_offset + (uint32_t)p, (uint32_t)h, (uint32_t)e);
  }
}

}  // namespace

int noise_fill_launch(const NoiseKey& key, int n_steps, long n_pose, int n_hyp, int row_floats, float* out, cudaStream_t s) {
  const long total = (long)n_steps * n_pose * n_hyp * row_floats;
  if (total == 0) return DP_OK;
  long grid = (total + 255) / 256;
  if (grid > 148 * 16) grid = 148 * 16;
  noise_fill_kernel<<<(unsigned)grid, 256, 0, s>>>(key, n_steps, n_pose, n_hyp, row_floats, out);
  count_launch();
  DP_CUDA(cudaGetLastError());
  return DP_OK;
}

}  // namespace dp
