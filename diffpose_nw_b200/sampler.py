"""Reverse-diffusion sampler: drop-in for the reference's common/utils_diff.py.

`generalized_steps(x, src_mask, seq, model, b, eta=...)` keeps the reference name, argument order and return
convention (`(xs, x0_preds)`; the runner uses `[0][-1]`, runners/diffpose_frame.py:365-366) but executes the
whole T-step loop in one persistent CUDA kernel launch through `dp_sample` (include/diffpose_b200.h).

Host-side pieces kept in Python because they are tiny and must use the reference's exact fp32 tensor ops:
`get_beta_schedule` (utils_diff.py:7-37), `compute_alpha` (:40-43) and the per-step scalars (:55-64).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from .metrics import _group_ids, _group_sums, _hyp_sums, _metrics_hyp
from .model import FusedGCNdiff


def get_beta_schedule(beta_schedule, *, beta_start, beta_end, num_diffusion_timesteps):
    """float64 numpy schedule; names and formulas of the reference (common/utils_diff.py:7-37)."""
    n = num_diffusion_timesteps
    if beta_schedule == "quad":
        betas = np.linspace(beta_start ** 0.5, beta_end ** 0.5, n, dtype=np.float64) ** 2
    elif beta_schedule == "linear":
        betas = np.linspace(beta_start, beta_end, n, dtype=np.float64)
    elif beta_schedule == "const":
        betas = beta_end * np.ones(n, dtype=np.float64)
    elif beta_schedule == "jsd":
        betas = 1.0 / np.linspace(n, 1, n, dtype=np.float64)
    elif beta_schedule == "sigmoid":
        grid = np.linspace(-6, 6, n)
        betas = (1 / (np.exp(-grid) + 1)) * (beta_end - beta_start) + beta_start
    else:
        raise NotImplementedError(beta_schedule)
    assert betas.shape == (n,)
    return betas


def compute_alpha(beta, t):
    """abar_t = cumprod(1 - [0, beta])[t + 1] as [n,1,1] (common/utils_diff.py:40-43); abar_{-1} = 1."""
    beta = torch.cat([torch.zeros(1, device=beta.device, dtype=beta.dtype), beta], dim=0)
    return (1 - beta).cumprod(dim=0).index_select(0, t + 1).view(-1, 1, 1)


def make_seq(skip_type, test_num_diffusion_timesteps, test_timesteps):
    """Timestep subsequence of test_hyber (runners/diffpose_frame.py:310-317)."""
    if skip_type == "uniform":
        skip = test_num_diffusion_timesteps // test_timesteps
        return list(range(0, test_num_diffusion_timesteps, skip))
    if skip_type == "quad":
        seq = np.linspace(0, np.sqrt(test_num_diffusion_timesteps * 0.8), test_timesteps) ** 2
        return [int(s) for s in list(seq)]
    raise NotImplementedError(skip_type)


def ddim_steps(b, seq, eta=0.0):
    """Per-step scalars in execution order, computed with the same fp32 CPU tensor ops the reference applies
    (common/utils_diff.py:55-64) -- c2 cancels catastrophically for eta near 1, so it is never re-derived
    on the device.  Returns a ctypes array of DpStep."""
    b = torch.as_tensor(b).detach().to("cpu", torch.float32)
    seq = [int(s) for s in seq]
    if len(seq) == 0:
        raise RuntimeError("generalized_steps: empty timestep sequence")
    if max(seq) + 1 > b.numel() or min(seq) < 0:
        raise RuntimeError(f"generalized_steps: timestep {max(seq)} is outside the {b.numel()}-entry beta schedule")
    seq_next = [-1] + seq[:-1]
    steps = (_lib.DpStep * len(seq))()
    for k, (i, j) in enumerate(zip(reversed(seq), reversed(seq_next))):
        at = compute_alpha(b, torch.tensor([i], dtype=torch.long))
        an = compute_alpha(b, torch.tensor([j], dtype=torch.long))
        c1 = eta * ((1 - at / an) * (1 - an) / (1 - at)).sqrt()
        c2 = ((1 - an) - c1 ** 2).sqrt()
        steps[k] = _lib.DpStep(float(i), at.sqrt().item(), (1 - at).sqrt().item(), an.sqrt().item(),
                               float(c1.item()), float(c2.item()))
    return steps


NOISE_CHUNK_BYTES = 2 << 30    # device-drawn noise held at any one time by `sample` (eta > 0, no caller noise)

_STEP_CACHE = {}      # (betas identity, seq, eta) -> (DpStep array, betas kept alive); a handful of schedules per process


def cached_ddim_steps(b, seq, eta):
    """`ddim_steps` once per (beta schedule, sequence, eta).  The reference runner keeps `self.betas` on the GPU
    (runners/diffpose_frame.py:49-50) and calls the sampler per batch: deriving the scalars each time would cost a
    device->host copy (a stream synchronisation) plus T small CPU tensor programs per call -- more than the kernel
    itself for the 2-step evaluation schedules."""
    if not torch.is_tensor(b):
        return ddim_steps(b, seq, eta)
    key = (b.data_ptr(), b._version, b.numel(), str(b.device), b.dtype, tuple(int(s) for s in seq), float(eta))
    hit = _STEP_CACHE.get(key)
    if hit is None:
        if len(_STEP_CACHE) >= 16:
            _STEP_CACHE.clear()
        hit = (ddim_steps(b, seq, eta), b)
        _STEP_CACHE[key] = hit
    return hit[0]


def _unwrap(model):
    inner = getattr(model, "module", model)   # torch.nn.DataParallel wrapper (runners/diffpose_frame.py:127)
    if not isinstance(inner, FusedGCNdiff):
        raise RuntimeError("generalized_steps: model must be a diffpose_nw_b200.FusedGCNdiff (there is no eager fallback)")
    return inner


def sample(model, x, src_mask, seq, b, eta=0.0, noise=None, n_hyp=1, repeat_input=False, mean_over_hyp=False,
           steps=None, targets=None, sums=None, seed=None, pose_offset=0, step_offset=0, groups=None, xs_out=None, x0_out=None,
           hyp_sums=None):
    """Run the DDIM loop on the device and return x_T.

    x: [n_hyp*n_pose,17,c] hypothesis-major (what `.repeat(test_times,1,1)` produces), or [n_pose,17,c] with
    `repeat_input=True` to let the kernel read each pose n_hyp times instead of materialising the repeat.
    noise: optional [T, n_hyp*n_pose, 17, c] standard-normal draws replacing `torch.randn_like` (:65).
    seed: draw the noise inside the kernel from the keyed stream (`dp_sample`'s key, include/diffpose_b200.h) instead: one
    launch, no noise tensor, and every pose receives the same draws however the work is split, as long as each piece
    passes the global index of its first pose as `pose_offset` (and a call that runs step k of a schedule alone passes
    `step_offset=k`).  `philox_noise` writes the same stream out.  Not together with `noise`; no effect when eta = 0.
    Without `noise` and `seed`, eta > 0 draws with torch.randn, in chunks of at most NOISE_CHUNK_BYTES.
    mean_over_hyp: fuse `mean(reshape(n_hyp,-1,17,c),0)` (runners/diffpose_frame.py:382) after the loop.
    targets, sums: fused evaluation (`dp_sample` with targets_xyz): targets [n_pose,17,3] on the device and a CUDA fp64 tensor of 3
    partial sums `[sum mpjpe, sum p_mpjpe, n]` that every finished pose is added to in the same launch (:384-387); with
    n_hyp > 1 this needs mean_over_hyp.  Without them nothing is evaluated.
    groups: with targets, an int32 tensor [n_pose] of group ids (e.g. `action_groups`); `sums` is then [n_groups,3] and each
    pose adds to the row of its id, in the same launch on the default engine (`dp_sample_grouped`).  An id outside
    [0, n_groups) adds to nothing.
    xs_out, x0_out: optional CUDA fp32 tensors [T, n_hyp*n_pose, 17, c] (hypothesis-major, like `noise`) that receive the
    denoising path from the same launch (`dp_sample_trajectory`): xs_out[k] is x_t after step k and x0_out[k] the x0
    prediction that step's update used -- the sampler's own values, before any hypothesis mean.  Either may be given
    alone.  Not together with `targets`.
    hyp_sums: with targets, the multi-hypothesis evaluation in place of `sums`: a CUDA fp64 tensor [8] (or [n_groups,8] with
    `groups`) that receives the columns of `hyp_error_sums` -- mean-pose, best-of-H, per-joint best and average-hypothesis
    MPJPE / P-MPJPE and the count.  The sampler writes all n_hyp rows of each pose and `dp_metrics_hyp` scores them: two
    launches, whatever the engine.  The result is the hypothesis mean with mean_over_hyp (written by that second launch,
    equal to the sampler's own mean bit for bit), else the n_hyp rows.  Not together with `sums` or a trajectory.
    """
    m = _unwrap(model)
    xc = m._check_x(x, m._c_in)
    dev = xc.device
    m._ensure_packed(dev)
    rows = xc.shape[0]
    if repeat_input:
        n_pose = rows
    else:
        if rows % n_hyp:
            raise RuntimeError(f"x has {rows} rows, not a multiple of n_hyp={n_hyp}")
        n_pose = rows // n_hyp
    if steps is None:
        steps = cached_ddim_steps(b, seq, eta)
    T = len(steps)
    total = n_pose * n_hyp
    c = m._c_in
    nz = None
    draw = False
    key = None
    if seed is not None and noise is not None:
        raise RuntimeError("sample: pass either seed= (keyed in-kernel noise) or noise=, not both")
    traj = xs_out is not None or x0_out is not None
    if hyp_sums is not None:
        if sums is not None:
            raise RuntimeError("sample: pass either sums= (hypothesis mean) or hyp_sums= (multi-hypothesis evaluation), not both")
        if targets is None:
            raise RuntimeError("sample: hyp_sums= needs targets=")
        if traj:
            raise RuntimeError("sample: a trajectory (xs_out= / x0_out=) is not stored together with hyp_sums=")
    if traj and targets is not None:
        raise RuntimeError("sample: a trajectory (xs_out= / x0_out=) is not stored together with the fused evaluation (targets=)")
    for name, buf in (("xs_out", xs_out), ("x0_out", x0_out)):
        if buf is None:
            continue
        if not torch.is_tensor(buf) or buf.device != dev or buf.dtype is not torch.float32 or not buf.is_contiguous():
            raise RuntimeError(f"{name} must be a contiguous float32 tensor on {dev}")
        if tuple(buf.shape) != (T, total, m.n_pts, c):
            raise RuntimeError(f"{name} must be [{T},{total},{m.n_pts},{c}], got {tuple(buf.shape)}")
    if seed is not None:
        if any(s.c1 != 0.0 for s in steps):   # eta = 0: the seed has no effect, the call is the unkeyed one
            key = _lib.noise_key(seed, pose_offset, step_offset)
    elif noise is not None:
        nz = torch.as_tensor(noise, device=dev).detach().to(torch.float32).contiguous()
        if tuple(nz.shape) != (T, total, m.n_pts, c):
            raise RuntimeError(f"noise must be [{T},{total},{m.n_pts},{c}], got {tuple(nz.shape)}")
    elif any(s.c1 != 0.0 for s in steps):
        draw = True        # eta > 0 without caller noise: N(0,1) draws in place of the reference's per-step randn_like (:65)
    out_rows = n_pose if mean_over_hyp else total
    out = torch.empty(out_rows, m.n_pts, c, device=dev, dtype=torch.float32)
    if total == 0:
        return out
    mb = m._mask_bytes(src_mask, dev)
    lib = _lib.load()
    mask_ptr = mb.data_ptr() if mb is not None else None
    tg = gid = None
    n_groups = 1
    if groups is not None and targets is None:
        raise RuntimeError("sample: groups= needs targets= and sums=")
    if hyp_sums is not None:
        hyp_sums, gid, n_groups = _hyp_sums(hyp_sums, groups, None, n_pose, dev, "sample")
    elif targets is not None:
        if groups is not None:
            if sums is None:
                raise RuntimeError("grouped evaluation needs `sums`: a CUDA float64 tensor [n_groups,3]")
            sums, n_groups = _group_sums(sums, None, dev, "sample")
            gid = _group_ids(groups, n_pose, dev, "sample")
        elif sums is None or not sums.is_cuda or sums.dtype is not torch.float64 or sums.numel() != 3:
            raise RuntimeError("fused evaluation needs `sums`: a CUDA float64 tensor of 3 elements")
        if n_hyp > 1 and not mean_over_hyp:
            raise RuntimeError("fused evaluation with n_hyp > 1 evaluates the hypothesis mean: pass mean_over_hyp=True")
    if targets is not None:
        tg = targets.detach().to(device=dev, dtype=torch.float32).contiguous()
        if tuple(tg.shape) != (n_pose, m.n_pts, 3):
            raise RuntimeError(f"targets must be [{n_pose},{m.n_pts},3], got {tuple(tg.shape)}")

    def ptr(t):
        return None if t is None else t.data_ptr()

    def launch(x_t, out_t, n_p, nz_t, repeated, lo=0, xs_t=None, x0_t=None):
        if hyp_sums is not None:
            # every hypothesis row from the sampler (into out_t itself when it holds them), then the evaluation, which also
            # writes the mean
            mean = mean_over_hyp and n_hyp > 1
            rows = torch.empty(n_p * n_hyp, m.n_pts, c, device=dev, dtype=torch.float32) if mean else out_t
            stream = torch.cuda.current_stream(dev).cuda_stream
            rc = lib.dp_sample_grouped(m._handle, x_t.data_ptr(), 1 if repeated else 0, rows.data_ptr(), n_p, n_hyp, steps, T, ptr(nz_t),
                                       key, mask_ptr, 0, None, None, 1, None, stream)
            if rc != 0:
                _lib.check(rc, "dp_sample")
            _metrics_hyp(lib, rows, c, n_hyp, tg[lo:lo + n_p], n_p, None if gid is None else gid[lo:lo + n_p], n_groups, hyp_sums,
                         out_t if mean else None, None, stream)
            return
        if traj:
            rc = lib.dp_sample_trajectory(m._handle, x_t.data_ptr(), 1 if repeated else 0, out_t.data_ptr(), n_p, n_hyp, steps, T,
                                          ptr(nz_t), key, mask_ptr, 1 if mean_over_hyp else 0, ptr(xs_t), ptr(x0_t),
                                          torch.cuda.current_stream(dev).cuda_stream)
            if rc != 0:
                _lib.check(rc, "dp_sample_trajectory")
            return
        rc = lib.dp_sample_grouped(m._handle, x_t.data_ptr(), 1 if repeated else 0, out_t.data_ptr(), n_p, n_hyp, steps, T,
                                   nz_t.data_ptr() if nz_t is not None else None, key, mask_ptr, 1 if mean_over_hyp else 0,
                                   None if tg is None else tg[lo:lo + n_p].data_ptr(), None if gid is None else gid[lo:lo + n_p].data_ptr(),
                                   n_groups, None if tg is None else sums.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        if rc != 0:
            _lib.check(rc, "dp_sample")

    def run():
        if not draw:
            return launch(xc, out, n_pose, nz, not repeat_input, 0, xs_out, x0_out)
        # Device-drawn noise is needed as [T, rows, 17, c] by the kernel (it runs all T steps of a tile in one go).  The
        # reference holds one step's draw at a time; to keep memory bounded like that, a large call is cut into pose chunks
        # whose noise fits NOISE_CHUNK_BYTES (the chunks are independent: poses are).  The random STREAM differs from the
        # reference's (same distribution, different draws for a given seed) -- pass `noise=` for comparable results.
        row_bytes = m.n_pts * c * 4
        per_chunk = max(1, NOISE_CHUNK_BYTES // (T * row_bytes * n_hyp))
        if per_chunk >= n_pose:
            return launch(xc, out, n_pose, torch.randn(T, total, m.n_pts, c, device=dev, dtype=torch.float32), not repeat_input, 0,
                          xs_out, x0_out)
        xv = xc if repeat_input else xc.view(n_hyp, n_pose, m.n_pts, c)
        ov = out if mean_over_hyp else out.view(n_hyp, n_pose, m.n_pts, c)
        buf = torch.empty(T, per_chunk * n_hyp, m.n_pts, c, device=dev, dtype=torch.float32)
        # a trajectory is hypothesis-major over all poses: each chunk writes its own and is scattered like `out`
        trv = [None if t is None else t.view(T, n_hyp, n_pose, m.n_pts, c) for t in (xs_out, x0_out)]
        for lo in range(0, n_pose, per_chunk):
            hi = min(n_pose, lo + per_chunk)
            k = hi - lo
            nzc = buf[:, : k * n_hyp] if k == per_chunk else torch.empty(T, k * n_hyp, m.n_pts, c, device=dev, dtype=torch.float32)
            nzc.normal_()
            x_c = xv[lo:hi] if repeat_input else xv[:, lo:hi].reshape(k * n_hyp, m.n_pts, c).contiguous()
            tr_c = [None if t is None else torch.empty(T, k * n_hyp, m.n_pts, c, device=dev, dtype=torch.float32) for t in trv]
            if mean_over_hyp:
                launch(x_c, ov[lo:hi], k, nzc, not repeat_input, lo, *tr_c)
            else:
                o_c = torch.empty(k * n_hyp, m.n_pts, c, device=dev, dtype=torch.float32)
                launch(x_c, o_c, k, nzc, not repeat_input, lo, *tr_c)
                ov[:, lo:hi] = o_c.view(n_hyp, k, m.n_pts, c)
            for t, t_c in zip(trv, tr_c):
                if t is not None:
                    t[:, :, lo:hi] = t_c.view(T, n_hyp, k, m.n_pts, c)

    if torch.cuda.current_device() == dev.index:      # the usual case: no device switch on the per-batch path
        run()
    else:
        with torch.cuda.device(dev):
            run()
    return out


def generalized_steps(x, src_mask, seq, model, b, **kwargs):
    """Drop-in for common/utils_diff.py:46-67.

    Returns `(xs, x0_preds)` with `xs = [x, x_T]` and `x0_preds = []`: the fused kernel keeps the intermediate
    x_t / x0 on chip (the only consumer in the reference takes `[0][-1]`).  Pass `return_all=True` to get the
    full per-step lists, `xs = [x, x_1, ..., x_T]` and one x0 prediction per step: the values the sampler itself computed,
    stored from the same single launch (`sample(xs_out=, x0_out=)`), at the cost of two [T, n, 17, c] buffers.
    Extra keyword `noise=[T,n,17,c]` supplies the per-step normal draws; `seed=` draws them in the kernel from the keyed
    stream instead (see `sample`), the same stream with and without `return_all`.
    """
    eta = kwargs.get("eta", 0)
    noise = kwargs.get("noise", None)
    seed = kwargs.get("seed", None)
    with torch.no_grad():
        if not kwargs.get("return_all", False):
            return [x, sample(model, x, src_mask, seq, b, eta=eta, noise=noise, seed=seed)], []
        m = _unwrap(model)
        shape = (len(seq), x.shape[0], m.n_pts, m._c_in)
        xs_out = torch.empty(shape, device=x.device, dtype=torch.float32)
        x0_out = torch.empty(shape, device=x.device, dtype=torch.float32)
        sample(model, x, src_mask, seq, b, eta=eta, noise=noise, seed=seed, xs_out=xs_out, x0_out=x0_out)
        return [x] + list(xs_out.unbind(0)), list(x0_out.unbind(0))


def philox_noise(seed, n_steps, n_pose, n_hyp=1, *, pose_offset=0, step_offset=0, device=None, n_pts=17, c=5):
    """The keyed noise stream of `sample(seed=...)` as a CUDA tensor [n_steps, n_hyp*n_pose, n_pts, c] (hypothesis-major, the
    layout of `noise=`), written by `dp_noise_fill`: `sample(..., noise=philox_noise(seed, T, n, H, pose_offset=o))` equals
    `sample(..., seed=seed, pose_offset=o)` bit for bit."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise RuntimeError("philox_noise: the stream is written on a CUDA device (diffpose_nw_b200 has no CPU path)")
    out = torch.empty(n_steps, n_hyp * n_pose, n_pts, c, device=dev, dtype=torch.float32)
    lib = _lib.load()
    key = _lib.noise_key(seed, pose_offset, step_offset)
    with torch.cuda.device(dev):
        rc = lib.dp_noise_fill(ctypes.byref(key), n_steps, n_pose, n_hyp, n_pts, c, out.data_ptr() if out.numel() else None,
                               torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "dp_noise_fill")
    return out
