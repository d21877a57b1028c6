"""Evaluation metrics that follow the sampler, computed on the GPU by `dp_metrics`.

Replaces `mpjpe` (reference common/loss.py:7-13) and `p_mpjpe` (common/loss.py:25-64, per-pose form
common/utils.py:155-187) as the runner uses them (runners/diffpose_frame.py:382-387), without the
`.cpu().numpy()` SVD round trip.  Per-rank partial sums `[sum mpjpe, sum p_mpjpe, count]` (fp64) are what the
multi-GPU driver all-reduces.  With group ids (for Human3.6M: each pose's action) the sums are `[n_groups, 3]`, one row per
group: the per-action table of `test_calculation` (common/utils.py:103-152), see `pipeline.reduce_action_errors`.
`hyp_error_sums` scores H hypotheses per pose at once: best-of-H, per-joint best and average-hypothesis errors beside
those of the hypothesis mean (`dp_metrics_hyp`, `pipeline.reduce_hyp_errors`).
"""
from __future__ import annotations

import torch

from . import _lib


def _group_sums(sums, n_groups, device, what, cols=3):
    """The `[n_groups, cols]` CUDA fp64 sums of a grouped evaluation: `sums` checked, or zeros when it is None.  Returns
    (sums, n_groups)."""
    if sums is None:
        if n_groups is None or int(n_groups) < 1:
            raise RuntimeError(f"{what}: grouped sums need n_groups >= 1 (or a [n_groups,{cols}] `sums` tensor)")
        return torch.zeros(int(n_groups), cols, device=device, dtype=torch.float64), int(n_groups)
    if (not sums.is_cuda or sums.dtype is not torch.float64 or sums.dim() != 2 or sums.shape[1] != cols or sums.shape[0] < 1
            or not sums.is_contiguous() or (n_groups is not None and sums.shape[0] != n_groups)):
        raise RuntimeError(f"{what}: grouped evaluation needs `sums`: a contiguous CUDA float64 tensor [n_groups,{cols}]")
    return sums, sums.shape[0]


def _hyp_sums(sums, groups, n_groups, n, device, what):
    """The CUDA fp64 sums of a multi-hypothesis evaluation, `[8]` or, with group ids, `[n_groups, 8]` (zeros when `sums` is
    None), and the ids checked as in `_group_ids`.  Returns (sums, ids or None, n_groups)."""
    if groups is not None:
        sums, n_groups = _group_sums(sums, n_groups, device, what, cols=HYP_COLS)
        return sums, _group_ids(groups, n, device, what), n_groups
    if sums is None:
        return torch.zeros(HYP_COLS, device=device, dtype=torch.float64), None, 1
    if not sums.is_cuda or sums.dtype is not torch.float64 or tuple(sums.shape) != (HYP_COLS,) or not sums.is_contiguous():
        raise RuntimeError(f"{what}: multi-hypothesis sums must be a contiguous CUDA float64 tensor of {HYP_COLS} elements")
    return sums, None, 1


def _metrics_hyp(lib, pred, stride, n_hyp, gt, n, gid, n_groups, sums, mean_out, per_hyp, stream):
    """One `dp_metrics_hyp` call on contiguous device tensors (pred hypothesis-major, xyz in the last three columns)."""
    rc = lib.dp_metrics_hyp(pred.data_ptr(), stride, stride - 3, n_hyp, gt.data_ptr(), n, 17, None if gid is None else gid.data_ptr(),
                            n_groups, sums.data_ptr(), None if mean_out is None else mean_out.data_ptr(),
                            None if per_hyp is None else per_hyp.data_ptr(), stream)
    if rc != 0:
        _lib.check(rc, "dp_metrics_hyp")


def _group_ids(groups, n, device, what):
    """Group ids as a contiguous int32 tensor [n] on `device` (moved there like the targets, never converted from another
    dtype: a cast could wrap an out-of-range id into range)."""
    if not torch.is_tensor(groups) or groups.dtype is not torch.int32 or tuple(groups.shape) != (n,):
        raise RuntimeError(f"{what}: groups must be an int32 tensor [{n}]")
    return groups.to(device=device).contiguous()


def pose_error_sums(pred, target, sums=None, per_pose=False, groups=None, n_groups=None):
    """pred [n,17,3] (xyz) or [n,17,5] (uvxyz: xyz = columns 2:5); target [n,17,3]; metres.

    Both are root-centred out of place (intended semantics of diffpose_frame.py:384-385).  Returns
    (sums, per_pose) where sums is a CUDA fp64 tensor [sum_pose mpjpe, sum_pose p_mpjpe, n] (accumulated into
    the tensor passed as `sums` if any) and per_pose is [n,2] fp32 or None.
    groups: int32 [n] group id per pose (e.g. `action_groups` of the loader's action names).  The sums are then
    [n_groups,3] (n_groups from `sums` when it is given), row g over the poses whose id is g; a pose whose id is outside
    [0, n_groups) adds to nothing (pad ids: -1).  per_pose is the same with or without groups.
    """
    if not (pred.is_cuda and target.is_cuda):
        raise RuntimeError("diffpose_nw_b200.metrics runs on CUDA only (no CPU fallback)")
    if pred.dim() != 3 or pred.shape[1] != 17 or pred.shape[2] not in (3, 5):
        raise RuntimeError(f"pred must be [n,17,3] or [n,17,5], got {tuple(pred.shape)}")
    n = pred.shape[0]
    if tuple(target.shape) != (n, 17, 3):
        raise RuntimeError(f"target must be [{n},17,3], got {tuple(target.shape)}")
    dev = pred.device
    p = pred.detach().to(torch.float32).contiguous()
    g = target.detach().to(device=dev, dtype=torch.float32).contiguous()
    stride = p.shape[2]
    gid = None
    if groups is not None:
        sums, n_groups = _group_sums(sums, n_groups, dev, "pose_error_sums")
        gid = _group_ids(groups, n, dev, "pose_error_sums")
    elif sums is None:
        sums = torch.zeros(3, device=dev, dtype=torch.float64)
    pp = torch.empty(n, 2, device=dev, dtype=torch.float32) if per_pose else None
    if n:
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.load().dp_metrics(p.data_ptr(), stride, stride - 3, g.data_ptr(), n, 17,
                                              None if gid is None else gid.data_ptr(), 1 if gid is None else n_groups,
                                              sums.data_ptr(), pp.data_ptr() if pp is not None else None, stream), "dp_metrics")
    return sums, pp


# Columns of the multi-hypothesis sums (dp_metrics_hyp, include/diffpose_b200.h): mean-pose MPJPE / P-MPJPE, count,
# best-of-H MPJPE / P-MPJPE, per-joint best MPJPE, average-hypothesis MPJPE / P-MPJPE.
HYP_COLS = 8


def hyp_error_sums(pred, target, sums=None, groups=None, n_groups=None, per_hyp=False, mean_out=False):
    """Multi-hypothesis MPJPE / P-MPJPE of H hypotheses per pose in one launch (`dp_metrics_hyp`).

    pred [H,n,17,c] or [H*n,17,c] hypothesis-major (what `sample(mean_over_hyp=False)` returns), c = 3 (xyz) or 5 (uvxyz,
    xyz = columns 2:5); target [n,17,3]; metres, root-centred out of place.  Returns (sums, per_hyp, mean): sums a CUDA fp64
    tensor [8] (accumulated into `sums` when given) whose columns are
      0, 1  MPJPE / P-MPJPE of the hypothesis mean,  2  the count,
      3, 4  best-of-H (minimum over hypotheses of each error on its own; a NaN P-MPJPE propagates),
      5     per-joint best MPJPE (each joint takes its closest hypothesis),
      6, 7  average hypothesis (the expected error of one sample),
    each summed over poses; per_hyp [H,n,2] fp32 (MPJPE, P-MPJPE of every hypothesis, as `pose_error_sums` gives them) or
    None; mean [n,17,c] (the hypothesis mean, as `sample(mean_over_hyp=True)` returns it) or None.
    groups: int32 [n] ids as in `pose_error_sums`: the sums are then [n_groups,8], one row per group (see `reduce_hyp_errors`).
    """
    if not (pred.is_cuda and target.is_cuda):
        raise RuntimeError("diffpose_nw_b200.metrics runs on CUDA only (no CPU fallback)")
    if target.dim() != 3 or tuple(target.shape[1:]) != (17, 3):
        raise RuntimeError(f"target must be [n,17,3], got {tuple(target.shape)}")
    n = target.shape[0]
    if pred.dim() == 4:
        H = pred.shape[0]
        if pred.shape[1] != n:
            raise RuntimeError(f"pred [H,n,17,c] must have n={n} poses, got {tuple(pred.shape)}")
    elif pred.dim() == 3 and n > 0 and pred.shape[0] % n == 0:
        H = pred.shape[0] // n
    else:
        raise RuntimeError(f"pred must be [H,{n},17,c] or [H*{n},17,c], got {tuple(pred.shape)}")
    if H < 1 or pred.shape[-2] != 17 or pred.shape[-1] not in (3, 5):
        raise RuntimeError(f"pred must be [H,n,17,3|5] or [H*n,17,3|5] with H >= 1, got {tuple(pred.shape)}")
    dev = pred.device
    c = pred.shape[-1]
    p = pred.detach().to(torch.float32).contiguous()
    g = target.detach().to(device=dev, dtype=torch.float32).contiguous()
    sums, gid, n_groups = _hyp_sums(sums, groups, n_groups, n, dev, "hyp_error_sums")
    ph = torch.empty(H, n, 2, device=dev, dtype=torch.float32) if per_hyp else None
    mo = torch.empty(n, 17, c, device=dev, dtype=torch.float32) if mean_out else None
    if n:
        with torch.cuda.device(dev):
            _metrics_hyp(_lib.load(), p, c, H, g, n, gid, n_groups, sums, mo, ph, torch.cuda.current_stream(dev).cuda_stream)
    return sums, ph, mo


def mpjpe(pred, target):
    """Mean per-joint position error of root-centred poses (scalar CUDA tensor, same unit as the inputs)."""
    s, _ = pose_error_sums(pred, target)
    return (s[0] / s[2]).to(torch.float32)


def p_mpjpe(pred, target):
    """Procrustes-aligned MPJPE, mean over poses (scalar CUDA tensor)."""
    s, _ = pose_error_sums(pred, target)
    return (s[1] / s[2]).to(torch.float32)
