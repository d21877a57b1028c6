"""Evaluation metrics that follow the sampler, computed on the GPU by `dp_metrics`.

Replaces `mpjpe` (reference common/loss.py:7-13) and `p_mpjpe` (common/loss.py:25-64, per-pose form
common/utils.py:155-187) as the runner uses them (runners/diffpose_frame.py:382-387), without the
`.cpu().numpy()` SVD round trip.  Per-rank partial sums `[sum mpjpe, sum p_mpjpe, count]` (fp64) are what the
multi-GPU driver all-reduces.  With group ids (for Human3.6M: each pose's action) the sums are `[n_groups, 3]`, one row per
group: the per-action table of `test_calculation` (common/utils.py:103-152), see `pipeline.reduce_action_errors`.
"""
from __future__ import annotations

import torch

from . import _lib


def _group_sums(sums, n_groups, device, what):
    """The `[n_groups, 3]` CUDA fp64 sums of a grouped evaluation: `sums` checked, or zeros when it is None.  Returns
    (sums, n_groups)."""
    if sums is None:
        if n_groups is None or int(n_groups) < 1:
            raise RuntimeError(f"{what}: grouped sums need n_groups >= 1 (or a [n_groups,3] `sums` tensor)")
        return torch.zeros(int(n_groups), 3, device=device, dtype=torch.float64), int(n_groups)
    if (not sums.is_cuda or sums.dtype is not torch.float64 or sums.dim() != 2 or sums.shape[1] != 3 or sums.shape[0] < 1
            or not sums.is_contiguous() or (n_groups is not None and sums.shape[0] != n_groups)):
        raise RuntimeError(f"{what}: grouped evaluation needs `sums`: a contiguous CUDA float64 tensor [n_groups,3]")
    return sums, sums.shape[0]


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


def mpjpe(pred, target):
    """Mean per-joint position error of root-centred poses (scalar CUDA tensor, same unit as the inputs)."""
    s, _ = pose_error_sums(pred, target)
    return (s[0] / s[2]).to(torch.float32)


def p_mpjpe(pred, target):
    """Procrustes-aligned MPJPE, mean over poses (scalar CUDA tensor)."""
    s, _ = pose_error_sums(pred, target)
    return (s[1] / s[2]).to(torch.float32)
