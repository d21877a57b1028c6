/*
 * diffpose_b200.h -- C ABI of libdiffpose_b200.so: the B200 (sm_100a) implementation of DiffPose's
 * frame-based reverse-diffusion sampling path (GCNdiff denoiser + DDIM loop).
 *
 * The reference (nwicakson/diffpose-nw) is pure Python/PyTorch and has no FFI layer; its boundary for this
 * path is three Python call signatures.  Each entry point below names the reference interface it replaces
 * (paths relative to the reference repository root).  INTEGRATION.md shows the ctypes stub a reference
 * maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative dp_status otherwise; dp_last_error() returns a
 *     thread-local, human readable description of the last failure.  Nothing here calls abort().
 *   - all tensor pointers are DEVICE pointers to contiguous fp32 unless the name ends in _host.
 *   - the library borrows caller memory for the duration of a call; it owns only its packed weights and
 *     scratch, released by dp_destroy().
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  dp_forward, dp_lift, dp_sample and
 *     dp_metrics only enqueue work on it.  Exceptions, all off the per-batch path: dp_pack synchronises the stream once
 *     (it stages host-side graph matrices); dp_sample synchronises once when a schedule of MORE than 64 steps changes
 *     (the new step table is uploaded from the handle's own copy); scratch buffers (time-embedding table, hypothesis
 *     scratch of the non-default engines) grow with cudaMalloc the first time a larger batch or schedule is seen, and the
 *     first dp_forward / dp_lift after a dp_pack builds the split-precision weight blocks of DP_ENGINE_TCX (pack kernels
 *     on `stream`; one cudaMalloc the very first time).
 *     A call that neither grows a buffer nor changes a long schedule is CUDA-graph capturable.
 *   - a handle belongs to the device that was current at dp_create; calls made with another device current return
 *     DP_ERR_STATE.  One host thread per handle; one process per GPU.
 */
#ifndef DIFFPOSE_B200_H
#define DIFFPOSE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dp_model* dp_handle;

enum dp_status {
  DP_OK = 0,
  DP_ERR_INVALID = -1,     /* bad argument / unsupported shape */
  DP_ERR_CUDA = -2,        /* a CUDA runtime call failed       */
  DP_ERR_STATE = -3,       /* e.g. dp_forward before dp_pack   */
  DP_ERR_UNSUPPORTED = -4  /* the requested engine cannot run this configuration */
};

/* Which kernel family executes the denoiser / lifter. */
enum dp_engine {
  DP_ENGINE_AUTO = 0,  /* dp_sample: DP_ENGINE_TCG; dp_forward / dp_lift: DP_ENGINE_TCX (a forward output is not damped
                          by a DDIM schedule, so it takes the accurate path); fp32 when the configuration is outside
                          the tensor-core engines' limits (hid_dim=96, n_head=4, n_pts=17, coords_dim <= 5)          */
  DP_ENGINE_FP32 = 1,  /* fp32 FMA persistent kernel: every contraction in fp32 (bit-level reference)                */
  DP_ENGINE_TCX = 2,   /* split-precision tcgen05 kernel: dense projections as three fp16 products per K step
                          (A_hi W_hi + A_lo W_hi + A_hi W_lo, fp32 accumulation in TMEM), everything else fp32 on the
                          CUDA cores: <= 2e-5 from the fp32 reference                                                */
  DP_ENGINE_TCG = 3    /* the fast tcgen05 kernel (sampler default): every contraction on the tensor cores with fp16
                          operands (11-bit significand, as TF32) -- projections, 17x17 graph operators, attention,
                          in/out convolutions -- residual stream in TMEM, dedicated MMA-issuer warp.  fp16 operand
                          range: activations beyond +-65504 SATURATE (they never become inf/NaN)                     */
};

/* One DDIM step.  The scalars are evaluated by the caller with the reference's own fp32 tensor ops
 * (common/utils_diff.py:55-64) so that no re-derivation on the device can drift from them. */
typedef struct dp_step {
  float t;          /* timestep value fed to the denoiser (common/utils_diff.py:53,58)           */
  float sqrt_at;    /* sqrt(abar_t)                         (:59)                                 */
  float sqrt_1m_at; /* sqrt(1 - abar_t)                     (:59)                                 */
  float sqrt_an;    /* sqrt(abar_next)                      (:65)                                 */
  float c1;         /* eta * sqrt((1-at/an)(1-an)/(1-at))   (:61-63)                              */
  float c2;         /* sqrt((1-an) - c1^2)                  (:64)                                 */
} dp_step;

/* Replaces the constructors GCNdiff(adj, config) (models/gcndiff.py:56-98) and GCNpose(adj, config)
 * (models/gcnpose.py:56-98).  n_pts = config.model.n_pts, (c_in, c_out) = config.model.coords_dim,
 * hid = hid_dim, n_layer = num_layer, n_head = n_head; has_temb = 1 for GCNdiff, 0 for GCNpose. */
int dp_create(dp_handle* out, int n_pts, int c_in, int c_out, int hid, int n_layer, int n_head, int has_temb);

/* Number of fp32 values dp_pack expects (the state_dict flattened in the canonical order below). */
long dp_param_count(dp_handle h);

/* Replaces model.load_state_dict(states[0]) (runners/diffpose_frame.py:131-132) + the per-call graph
 * algebra of ChebConv.get_laplacian/cheb_polynomial (models/ChebConv.py:90-130) and
 * LAM_Gconv.laplacian_batch (models/GraFormer.py:174-178), which are evaluated once here.
 *
 * params: device pointer to the parameters, each tensor flattened in PyTorch (row-major) layout and
 * concatenated in this order (names are the reference state_dict keys):
 *   gconv_input.weight [3,1,c_in,hid], gconv_input.bias [hid]
 *   for l in 0..n_layer-1:
 *     gconv_layers.l.gconv1.gconv.weight [3,1,hid,hid], .bias [hid]
 *     gconv_layers.l.gconv2.gconv.weight [3,1,hid,hid], .bias [hid]
 *     (has_temb only) gconv_layers.l.temb_proj.weight [hid,4hid], .bias [hid]
 *     atten_layers.l.self_attn.linears.{0,1,2,3}.weight [hid,hid] each followed by its .bias [hid]
 *     atten_layers.l.feed_forward.A_hat [n_pts,n_pts]
 *     atten_layers.l.feed_forward.gconv1.fc.weight [2hid,hid], .bias [2hid]
 *     atten_layers.l.feed_forward.gconv2.fc.weight [hid,2hid], .bias [hid]
 *     atten_layers.l.sublayer.0.norm.a_2 [hid], .b_2 [hid], atten_layers.l.sublayer.1.norm.a_2, .b_2
 *   gconv_output.weight [3,1,hid,c_out], gconv_output.bias [c_out]
 *   (has_temb only) temb.dense.0.weight [4hid,hid], .bias [4hid], temb.dense.1.weight [4hid,4hid], .bias [4hid]
 * adj_host: host pointer, [n_pts*n_pts] fp32, the row-normalised adjacency (models/ChebConv.py:36-48). */
int dp_pack(dp_handle h, const float* params, long n_floats, const float* adj_host, void* stream);

/* Select the engine for subsequent dp_forward/dp_sample calls (default DP_ENGINE_AUTO). */
int dp_set_engine(dp_handle h, int engine);
/* Engine that dp_sample / dp_forward (and dp_lift) would use with the current setting: DP_ENGINE_FP32, _TCX or _TCG. */
int dp_get_engine(dp_handle h);
int dp_get_forward_engine(dp_handle h);
/* CUDA device ordinal the handle was created on. */
int dp_device(dp_handle h);

/* Replaces GCNdiff.forward(x, mask, t, cemd) (models/gcndiff.py:101-113; call sites
 * common/utils_diff.py:58, runners/diffpose_frame.py:225) and GCNpose.forward(x, mask)
 * (models/gcnpose.py:101-113; call site runners/diffpose_frame.py:337).
 *   x [n,n_pts,c_in], t [n] (per-sample timesteps; ignored/NULL when has_temb = 0),
 *   mask: [n_pts] bytes on the device (non-zero = key visible) or NULL (= all visible),
 *   out [n,n_pts,c_out]. */
int dp_forward(dp_handle h, const float* x, const float* t, const unsigned char* mask, float* out, long n, void* stream);

/* Replaces the glue between the two stages of the evaluation loop (runners/diffpose_frame.py:337-343):
 *     output_xyz = model_pose(input_2d, src_mask); output_xyz[:, :, :] -= output_xyz[:, :1, :];
 *     output_uvxyz = torch.cat([input_2d, output_xyz], dim=2)
 * in ONE launch on a GCNpose handle (has_temb = 0): uv [n,n_pts,c_in] -> out_uvxyz [n,n_pts,c_in+c_out] =
 * [uv | xyz - xyz[root]].  The root-centring is done OUT OF PLACE (the intended semantics; the reference's aliased
 * in-place form leaves joints 1..16 unchanged on CPU and races on CUDA, SURVEY.md 8a quirk 4). */
int dp_lift(dp_handle h, const float* uv, const unsigned char* mask, float* out_uvxyz, long n, void* stream);

/* Keyed noise: the sampler kernels draw z themselves from a counter-based stream, so a call needs no noise tensor and the
 * value every (pose, hypothesis, step, element) receives does not depend on how the work is split into calls, batches,
 * tiles or ranks.  The stream (this definition is part of the ABI):
 *   Philox4x32-10 (Salmon et al., SC'11; the round function and constants of Random123 / cuRAND Philox4_32_10)
 *   key      (seed & 0xffffffff, seed >> 32)
 *   counter  (e >> 2, s, b, h) as 32-bit words c0..c3, for element e = joint * c + coord (c = 5 for uvxyz) of
 *            global pose b = pose_offset + local pose, hypothesis h, step s = step_offset + k (k = execution index in
 *            the call, 0 = the first, largest t)
 *   normal   with output words x0..x3, l = e & 3, m = l >> 1:
 *            u1 = ((x[2m] >> 8) + 1) 2^-24 in (0, 1],  u2 = (x[2m+1] >> 8) 2^-24 in [0, 1),
 *            z = sqrtf(-2 logf(u1)) * (l even ? cospif(2 u2) : sinpif(2 u2)), every operation IEEE-rounded fp32.
 * Offset rules: a caller that splits one logical call into pieces gives each piece the global index of its first pose as
 * pose_offset (a rank: the start of its shard; a batch loop: the start of the batch), so the pieces together draw what one
 * call over all poses would.  A caller that runs the steps of one schedule as separate calls gives the call that runs
 * step k step_offset = k.  The pose index is one 32-bit word: pose_offset < 0, step_offset < 0 or
 * pose_offset + n_pose > 2^32 return DP_ERR_INVALID.  Different seeds (including seeds that differ only in their high
 * 32 bits) are different streams. */
typedef struct dp_noise_key {
  unsigned long long seed;
  long pose_offset;
  int step_offset;
} dp_noise_key;

/* Replaces generalized_steps(x, src_mask, seq, model, b, eta=...) (common/utils_diff.py:46-67) plus the
 * hypothesis handling around it (runners/diffpose_frame.py:342 `.repeat(test_times,1,1)` and :382
 * `mean(reshape(test_times,-1,17,5),0)`), in ONE persistent launch for all T steps.
 *   x_in      [n_rows_in,n_pts,c] with n_rows_in = n_pose*n_hyp if x_is_repeated else n_pose
 *             (the library reads pose b for every hypothesis h when x_is_repeated = 0);
 *   x_out     [n_pose*n_hyp,n_pts,c] hypothesis-major (index h*n_pose+b) when mean_over_hyp = 0,
 *             [n_pose,n_pts,c] when mean_over_hyp = 1 (DP_ENGINE_TCG folds the mean into the kernel's final store:
 *             one launch, no [n_pose*n_hyp] intermediate);
 *   steps_host T entries in execution order (largest t first);
 *   noise     [T,n_pose*n_hyp,n_pts,c] host-drawn N(0,1) replacing randn_like (:65), or NULL;
 *   key       the keyed stream above in place of a noise tensor, or NULL: no [T,n_pose*n_hyp,n_pts,c] buffer, and the
 *             key travels by value in the kernel arguments.  Not together with noise (DP_ERR_INVALID).  With neither,
 *             the noise term is skipped (exact when every c1 = 0, i.e. eta = 0); when every c1 = 0 a key has no effect;
 *   mask      as in dp_forward;
 *   targets_xyz, sums  NULL, or the fused evaluation: dp_metrics on the result, in the same launch on DP_ENGINE_TCG -- the
 *             body of the evaluation loop (runners/diffpose_frame.py:365-387: generalized_steps, hypothesis mean,
 *             root-centring, mpjpe, p_mpjpe).  Every pose the kernel finishes (after the hypothesis mean when n_hyp > 1,
 *             which then requires mean_over_hyp = 1) adds its MPJPE to sums[0], its P-MPJPE to sums[1] and 1 to sums[2]
 *             from the tile it was computed in -- one warp per pose in the tile's tail, one atomic per CTA -- instead of a
 *             second kernel re-reading x_out.  targets_xyz [n_pose,n_pts,3], sums: 3 doubles on the device (accumulated
 *             into; the caller zeroes them); targets_xyz requires sums.  Other engines run the sampler and dp_metrics
 *             back to back. */
int dp_sample(dp_handle h, const float* x_in, int x_is_repeated, float* x_out, long n_pose, int n_hyp,
              const dp_step* steps_host, int n_steps, const float* noise, const dp_noise_key* key, const unsigned char* mask,
              int mean_over_hyp, const float* targets_xyz, double* sums, void* stream);

/* Writes the keyed stream as out [n_steps][n_hyp*n_pose][n_pts][c] (hypothesis-major: row h*n_pose + p is pose
 * pose_offset + p, hypothesis h; step k is s = step_offset + k) -- the layout of dp_sample's `noise`.  So
 * dp_sample(noise = out) equals dp_sample(key) bit for bit. */
int dp_noise_fill(const dp_noise_key* key, int n_steps, long n_pose, int n_hyp, int n_pts, int c, float* out, void* stream);

/* Batches that live in HOST memory.  Replaces the copy-in / sample / copy-out sequence of the evaluation loop
 * (runners/diffpose_frame.py:333-335 `input_2d.to(self.device)` ..., :365 generalized_steps, :387 `.cpu()`), which the
 * reference runs strictly one after the other, by a ring of `depth` slots: the host->device copy of batch i+1 and the
 * device->host copy of batch i-1 run on the library's own copy streams while batch i is in the sampler kernel.
 *   create : device buffers, two copy streams and the events of `depth` slots for batches of up to max_pose poses,
 *            n_hyp hypotheses per pose (kernel-side repeat), optionally averaged (mean_over_hyp) -- all allocation
 *            happens here, none per batch;
 *   submit : x_host [n_pose,n_pts,c] and out_host ([n_pose*n_hyp,...] or [n_pose,...] with the mean) should be PINNED
 *            host memory (pageable memory works but serialises); enqueues copy-in, dp_sample on `stream`, copy-out and
 *            returns immediately; *slot identifies the batch.  noise_dev, key and mask_dev as in dp_sample (noise_dev and
 *            mask_dev on the device; each optional, noise_dev and key not both).  key->pose_offset numbers the batch's
 *            first pose: giving each batch the count of poses submitted before it draws what one keyed dp_sample over
 *            all batches would.  With targets_host [n_pose,n_pts,3] (pinned; requires sums_dev, 3 doubles on the device)
 *            the evaluation is fused in as in dp_sample: the targets travel with the batch and the kernel adds the batch's
 *            MPJPE / P-MPJPE sums to sums_dev -- the whole body of the evaluation loop (runners/diffpose_frame.py:333-387)
 *            per batch: two H2D copies, one launch, one D2H copy.  A refused combination enqueues nothing.
 *            A slot is reused after `depth` submits: wait for its result before that.
 *   wait   : blocks the host until the result of `slot` is in its out_host.
 * Results complete in submission order. */
typedef struct dp_hstream* dp_hstream_t;
int dp_hstream_create(dp_hstream_t* out, dp_handle h, long max_pose, int n_hyp, int mean_over_hyp, int depth);
int dp_hstream_submit(dp_hstream_t s, const float* x_host, const float* targets_host, double* sums_dev, long n_pose,
                      const dp_step* steps_host, int n_steps, const float* noise_dev, const dp_noise_key* key,
                      const unsigned char* mask_dev, float* out_host, void* stream, int* slot);
int dp_hstream_wait(dp_hstream_t s, int slot);
void dp_hstream_destroy(dp_hstream_t s);

/* Replaces mpjpe (common/loss.py:7-13) and p_mpjpe (common/loss.py:25-64, common/utils.py:155-187) as used
 * at runners/diffpose_frame.py:382-387: root-centres both inputs out of place, then accumulates
 * sums[0] += sum_pose mean_joint |pred-gt|, sums[1] += sum_pose P-MPJPE(pose), sums[2] += n.
 *   pred [n,n_pts,pred_stride] with xyz at column pred_offset (2 for uvxyz, 0 for xyz), gt [n,n_pts,3],
 *   sums: 3 doubles on the device (caller zeroes them; per-rank partials feed one all-reduce),
 *   per_pose: optional [n,2] fp32 device output (mpjpe, p_mpjpe per pose) or NULL. */
int dp_metrics(const float* pred, int pred_stride, int pred_offset, const float* gt, long n, int n_pts,
               double* sums, float* per_pose, void* stream);

/* Number of kernels this library has launched in this process (bench.py reports it as gpu_launches). */
long dp_launch_count(void);

/* Description of the kernel the last dp_sample/dp_forward launched: grid, block, dynamic smem bytes,
 * poses per tile, engine.  out6 is a host array of 6 longs. */
int dp_last_launch_info(dp_handle h, long* out6);

const char* dp_last_error(void);
const char* dp_version(void);
void dp_destroy(dp_handle h);

#ifdef __cplusplus
}
#endif
#endif /* DIFFPOSE_B200_H */
