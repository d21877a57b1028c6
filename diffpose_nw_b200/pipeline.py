"""Evaluation pipeline around the sampler: the device-side equivalent of the body of `test_hyber`
(reference runners/diffpose_frame.py:330-391) and its multi-GPU sharding.

    uv --GCNpose--> xyz --root-centre, cat--> uvxyz --H hypotheses x T DDIM steps--> mean over H --> MPJPE / P-MPJPE

Poses are independent, so ranks take contiguous pose ranges, keep all hypotheses of a pose on the same rank and
exchange nothing inside the loop; one all-reduce of three fp64 partial sums ends the evaluation
(SURVEY.md section 8e).  The per-action table (common/utils.py:103-152, 247-271) is the same with one row of sums per
action: group ids travel with the targets, and one all-reduce of [15, 3] ends it (`reduce_action_errors`).  With several
hypotheses per pose, `hyp_sums` / `hyp_metrics=True` score all of them ([8] or [15, 8] sums, `reduce_hyp_errors`).
"""
from __future__ import annotations

import ctypes
from typing import NamedTuple

import torch

from . import _lib
from .metrics import HYP_COLS, _group_sums, pose_error_sums
from .sampler import sample

# The 15 Human3.6M actions in the order of the reference's define_actions (common/utils.py), which is the row order of the
# per-action sums; they are the names of the processed H36M files the reference's loader reads.
H36M_ACTIONS = ("Directions", "Discussion", "Eating", "Greeting", "Phoning", "Photo", "Posing", "Purchases", "Sitting",
                "SittingDown", "Smoking", "Waiting", "WalkDog", "Walking", "WalkTogether")


def action_groups(actions, names=H36M_ACTIONS):
    """The loader's per-sample action strings -> int32 CPU tensor of row indices into `names`.  A name is cut at its first
    space as mpjpe_by_action_p1/p2 do (common/utils.py:103-152), so "Walking 1" is "Walking".  An unknown name raises
    ValueError.  Move the result to the device (or pin it, for HostStream) like the targets."""
    index = {a: i for i, a in enumerate(names)}
    ids = []
    for a in actions:
        name = a.split(" ", 1)[0]
        if name not in index:
            raise ValueError(f"unknown action {a!r} (known: {', '.join(names)})")
        ids.append(index[name])
    return torch.tensor(ids, dtype=torch.int32)


def shard_range(n, rank, world):
    """Contiguous, balanced pose range [lo, hi) of `rank` out of `world`."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def lift_and_refine(model_diff, x_uvxyz=None, *, model_pose=None, input_2d=None, src_mask=None, seq, betas, eta=0.0,
                    test_times=1, noise=None, targets=None, sums=None, seed=None, pose_offset=0, groups=None, hyp_sums=None):
    """Two-stage inference for one batch.  Give either `x_uvxyz` [B,17,5] or (`model_pose`, `input_2d` [B,17,2]).
    Returns the hypothesis-averaged uvxyz [B,17,5].  With `targets` [B,17,3] and `sums` (CUDA fp64 [3]) the MPJPE / P-MPJPE
    partial sums of the batch are accumulated by the sampler launch itself (`dp_sample` with targets_xyz).  `seed` draws the noise in
    the kernel (keyed stream, see `sample`); `pose_offset` is the global index of the batch's first pose.  `groups` (int32
    [B], with targets): per-group sums, `sums` is then [n_groups,3] (see `sample`).  `hyp_sums` (CUDA fp64 [8] or
    [n_groups,8], with targets and in place of `sums`): the multi-hypothesis evaluation of `sample(hyp_sums=)`."""
    if x_uvxyz is None:
        # lift + out-of-place root-centring (SURVEY.md 8a quirk 4) + concat in ONE launch (dp_lift); the sampler below is
        # the second and last launch of the batch (kernel-side repeat, hypothesis mean fused into its final store)
        x_uvxyz = getattr(model_pose, "module", model_pose).lift(input_2d, src_mask)
    return sample(model_diff, x_uvxyz, src_mask, seq, betas, eta=eta, noise=noise, n_hyp=test_times,
                  repeat_input=True, mean_over_hyp=True, targets=targets, sums=sums, seed=seed, pose_offset=pose_offset, groups=groups,
                  hyp_sums=hyp_sums)


def evaluate_shard(model_diff, x_uvxyz, targets_3d, *, src_mask=None, seq, betas, eta=0.0, test_times=1, noise=None,
                   batch_size=None, model_pose=None, input_2d=None, seed=None, pose_offset=0, groups=None, n_groups=None,
                   hyp_metrics=False):
    """Sample this rank's poses and return fp64 partial sums [sum mpjpe, sum p_mpjpe, n] (metres) on the device.
    With `seed` the noise is the keyed stream and `pose_offset` the global index of this shard's first pose (the `lo` of
    `shard_range`): every pose then draws the same noise whatever the number of ranks or the batch size.
    With `groups` (int32 [n], e.g. `action_groups`) and `n_groups` the sums are [n_groups,3], one row per group, ready for
    `reduce_action_errors`.
    With `hyp_metrics=True` every hypothesis is scored (`sample(hyp_sums=)`): the sums are [8] or [n_groups,8] with the
    columns of `hyp_error_sums`, ready for `reduce_hyp_errors`."""
    n = targets_3d.shape[0]
    dev = targets_3d.device
    cols = HYP_COLS if hyp_metrics else 3
    if groups is not None:
        sums, _ = _group_sums(None, n_groups, dev, "evaluate_shard", cols=cols)
    else:
        sums = torch.zeros(cols, device=dev, dtype=torch.float64)
    bs = batch_size or max(n, 1)
    for lo in range(0, n, bs):
        hi = min(n, lo + bs)
        nz = None
        if noise is not None:   # noise is [T, H*n, 17, 5] hypothesis-major over this shard
            T = noise.shape[0]
            nz = noise.reshape(T, test_times, n, 17, -1)[:, :, lo:hi].reshape(T, test_times * (hi - lo), 17, -1)
        # sampler + metrics of the batch in one launch (two with the lifter in front)
        lift_and_refine(model_diff, None if x_uvxyz is None else x_uvxyz[lo:hi], model_pose=model_pose,
                        input_2d=None if input_2d is None else input_2d[lo:hi], src_mask=src_mask, seq=seq,
                        betas=betas, eta=eta, test_times=test_times, noise=nz, targets=targets_3d[lo:hi],
                        sums=None if hyp_metrics else sums, hyp_sums=sums if hyp_metrics else None,
                        seed=seed, pose_offset=pose_offset + lo, groups=None if groups is None else groups[lo:hi])
    return sums


def reduce_metrics(sums, group=None):
    """All-reduce the per-rank partial sums (NCCL on GPUs, gloo in CPU tests) and return
    (mpjpe_mm, p_mpjpe_mm, n) as python floats -- the AverageMeter values of diffpose_frame.py:386-387."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    s = sums.detach().cpu()
    n = float(s[2])
    if n == 0:
        return float("nan"), float("nan"), 0.0
    return float(s[0]) / n * 1000.0, float(s[1]) / n * 1000.0, n


def reduce_action_errors(sums, names=H36M_ACTIONS, group=None):
    """The per-action table of test_hyber (common/utils.py:247-271 print_error_action after test_calculation) from grouped
    partial sums [G,3] (`evaluate_shard(groups=...)`, `sample(groups=...)`): ONE all-reduce of the [G,3] tensor across the
    process group (in place, as reduce_metrics does), then, in millimetres,
      table     {name: (mpjpe_mm, p_mpjpe_mm, n)} for the G = len(names) rows; an action without poses is (nan, nan, 0);
      protocol  (protocol #1, protocol #2): the mean over the actions that have poses, each action weighted equally as
                print_error_action does (the reference would count an action without poses as 0; see DESIGN.md);
      totals    (mpjpe_mm, p_mpjpe_mm, n) weighted by pose, what reduce_metrics gives for the summed rows (the
                AverageMeter line of runners/diffpose_frame.py:386-387).
    Returns (table, protocol, totals) as python floats."""
    import torch.distributed as dist
    if sums.dim() != 2 or sums.shape != (len(names), 3):
        raise RuntimeError(f"reduce_action_errors: sums must be [{len(names)},3] (one row per name), got {tuple(sums.shape)}")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    s = sums.detach().double().cpu()
    nan = float("nan")
    table = {}
    for name, (e1, e2, n) in zip(names, s.tolist()):
        table[name] = (e1 / n * 1000.0, e2 / n * 1000.0, n) if n > 0 else (nan, nan, 0.0)
    have = [v for v in table.values() if v[2] > 0]
    protocol = (sum(v[0] for v in have) / len(have), sum(v[1] for v in have) / len(have)) if have else (nan, nan)
    tot = s.sum(0).tolist()
    totals = (tot[0] / tot[2] * 1000.0, tot[1] / tot[2] * 1000.0, tot[2]) if tot[2] > 0 else (nan, nan, 0.0)
    return table, protocol, totals


class HypErrors(NamedTuple):
    """Multi-hypothesis errors in millimetres, in the column order of the sums (`hyp_error_sums`)."""
    mean_mpjpe: float        # of the hypothesis mean
    mean_p_mpjpe: float
    n: float                 # poses
    best_mpjpe: float        # best-of-H
    best_p_mpjpe: float
    jbest_mpjpe: float       # per-joint best
    avg_mpjpe: float         # average hypothesis
    avg_p_mpjpe: float


def _hyp_row(row):
    n = row[2]
    if n <= 0:
        nan = float("nan")
        return HypErrors(nan, nan, 0.0, nan, nan, nan, nan, nan)
    mm = [v / n * 1000.0 for v in row]
    return HypErrors(mm[0], mm[1], n, *mm[3:])


def reduce_hyp_errors(sums, names=None, group=None):
    """Multi-hypothesis sums [8] or [G,8] (`hyp_error_sums`, `sample(hyp_sums=)`, `evaluate_shard(hyp_metrics=True)`) ->
    millimetres: ONE all-reduce of the tensor across the process group (in place, as reduce_metrics does), then
      without names  the totals over all rows, a HypErrors (pose-weighted; nan when there are no poses);
      with names     (table, protocol, totals) as reduce_action_errors: table {name: HypErrors} for the G = len(names) rows
                     (an action without poses is all nan with n = 0), protocol the mean of each column over the actions that
                     have poses, each action weighted equally (n = their poses), and totals as above.
    Returns python floats."""
    import torch.distributed as dist
    if sums.shape[-1:] != (HYP_COLS,) or sums.dim() not in (1, 2) or (names is not None and tuple(sums.shape) != (len(names), HYP_COLS)):
        want = f"[{len(names)},{HYP_COLS}] (one row per name)" if names is not None else f"[{HYP_COLS}] or [G,{HYP_COLS}]"
        raise RuntimeError(f"reduce_hyp_errors: sums must be {want}, got {tuple(sums.shape)}")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    s = sums.detach().double().cpu().reshape(-1, HYP_COLS)
    totals = _hyp_row(s.sum(0).tolist())
    if names is None:
        return totals
    table = {name: _hyp_row(row) for name, row in zip(names, s.tolist())}
    have = [v for v in table.values() if v.n > 0]
    if have:
        protocol = HypErrors(*[sum(v[k] for v in have) / len(have) if k != 2 else sum(v.n for v in have) for k in range(HYP_COLS)])
    else:
        protocol = _hyp_row([0.0] * HYP_COLS)
    return table, protocol, totals


class HostStream:
    """Batches that live in HOST memory, sampled at device speed: the H2D copy of batch i+1 and the D2H copy of
    batch i-1 run on their own CUDA streams while batch i is in the sampler kernel (the reference's loop,
    runners/diffpose_frame.py:330-366, copies, computes and reads back strictly one after the other).  The ring itself --
    device buffers, copy streams, events, the three enqueues per batch -- lives in the C library (`dp_hstream_*`,
    include/diffpose_b200.h); one `submit` is one C call.

        hs = HostStream(model_diff, batch=1024, seq=seq, betas=betas, test_times=1)
        for uvxyz_cpu in loader:            # pinned [B,17,5] fp32 tensors
            done = hs.submit(uvxyz_cpu)     # -> the result of an EARLIER batch (pinned host tensor) or None
        for out in hs.drain(): ...

    Results come back in submission order.  `depth` batches are in flight; every buffer is allocated once.  A returned
    tensor aliases a ring buffer and stays valid for the next `depth` submits.

    eta > 0 needs `seed`: the kernel then draws the noise from the keyed stream (`dp_hstream_submit`'s key), and the poses
    of consecutive batches are numbered like one big call, so the results equal one `sample(seed=...)` over all batches.
    """

    def __init__(self, model_diff, batch, seq, betas, eta=0.0, test_times=1, src_mask=None, depth=3, device=None, seed=None):
        import collections
        from .sampler import ddim_steps
        self.model = getattr(model_diff, "module", model_diff)
        self.dev = torch.device(device) if device is not None else self.model._device()
        if self.dev.type != "cuda":
            raise RuntimeError("HostStream needs the model on a CUDA device (diffpose_nw_b200 has no CPU path)")
        self.B, self.H, self.depth = batch, test_times, depth
        self.steps = ddim_steps(betas, seq, eta)
        self.T = len(self.steps)
        self._keyed = seed is not None and any(s.c1 != 0.0 for s in self.steps)
        if any(s.c1 != 0.0 for s in self.steps) and seed is None:
            raise RuntimeError("HostStream takes no noise tensor: use eta = 0, or pass seed= for keyed in-kernel noise")
        self.seed = seed
        self.n_submitted = 0                       # poses submitted so far: the default pose_offset of the next batch
        self.model._ensure_packed(self.dev)
        self._lib = _lib.load()
        self._mask = self.model._mask_bytes(src_mask, self.dev)
        self._mask_ptr = self._mask.data_ptr() if self._mask is not None else None
        c = self.model._c_in
        self.hs = ctypes.c_void_p()
        with torch.cuda.device(self.dev):
            _lib.check(self._lib.dp_hstream_create(ctypes.byref(self.hs), self.model._handle, batch, test_times, 1 if test_times > 1 else 0, depth),
                       "dp_hstream_create")
        self._handle_used = self.model._handle
        self.out_host = [torch.empty(batch, 17, c).pin_memory() for _ in range(2 * depth)]
        self._hpos = 0
        self._slot = ctypes.c_int(0)
        self._slot_ref = ctypes.byref(self._slot)
        self._pending = collections.deque()        # (slot, host buffer, rows, input tensor kept alive until its copy has run)

    def _collect(self):
        slot, hb, n = self._pending.popleft()[:3]
        rc = self._lib.dp_hstream_wait(self.hs, slot)
        if rc != 0:
            _lib.check(rc, "dp_hstream_wait")
        return self.out_host[hb][:n]

    def submit(self, x_host, targets_host=None, sums=None, pose_offset=None, groups_host=None):
        """Queue one pinned host batch [n<=B,17,c] (fp32, contiguous).  Returns the oldest finished result when the ring is
        full, else None.  With `targets_host` [n,17,3] (pinned fp32) and `sums` (CUDA fp64 [3]) the batch's MPJPE / P-MPJPE
        partial sums are accumulated by the sampler launch itself (`dp_hstream_submit` with targets_host).  With a seed, `pose_offset`
        is the global index of the batch's first pose; it defaults to the number of poses submitted before.
        `groups_host` (pinned int32 [n], with targets_host): group ids that travel with the targets; `sums` is then CUDA
        fp64 [n_groups,3] and each pose adds to the row of its id (`dp_hstream_submit_grouped`)."""
        n = x_host.shape[0]
        if n > self.B:
            raise RuntimeError(f"batch of {n} poses exceeds the {self.B} this HostStream was built for")
        if x_host.is_cuda or x_host.dtype is not torch.float32 or not x_host.is_contiguous():
            raise RuntimeError("HostStream.submit takes a contiguous fp32 HOST tensor (pinned for overlap)")
        if self.model._handle is not self._handle_used:
            raise RuntimeError("the model was moved or re-created after this HostStream was built: build a new one")
        self.model._ensure_packed(self.dev)           # weights edited since the last batch are re-packed (same rules as sample())
        ret = self._collect() if len(self._pending) == self.depth else None
        hb = self._hpos
        self._hpos = (hb + 1) % len(self.out_host)
        stream = torch.cuda.current_stream(self.dev).cuda_stream
        if targets_host is not None:
            if (targets_host.is_cuda or targets_host.dtype is not torch.float32 or not targets_host.is_contiguous()
                    or tuple(targets_host.shape) != (n, 17, 3)):
                raise RuntimeError(f"targets_host must be a contiguous fp32 HOST tensor [{n},17,3]")
            if groups_host is not None:
                if (groups_host.is_cuda or groups_host.dtype is not torch.int32 or not groups_host.is_contiguous()
                        or tuple(groups_host.shape) != (n,)):
                    raise RuntimeError(f"groups_host must be a contiguous int32 HOST tensor [{n}]")
                if sums is None:
                    raise RuntimeError("grouped evaluation needs `sums`: a CUDA float64 tensor [n_groups,3]")
                sums, n_groups = _group_sums(sums, None, self.dev, "HostStream.submit")
            elif sums is None or not sums.is_cuda or sums.dtype is not torch.float64 or sums.numel() != 3:
                raise RuntimeError("fused evaluation needs `sums`: a CUDA float64 tensor of 3 elements")
        elif groups_host is not None:
            raise RuntimeError("HostStream.submit: groups_host needs targets_host and sums")
        key = _lib.noise_key(self.seed, self.n_submitted if pose_offset is None else pose_offset) if self._keyed else None
        rc = self._lib.dp_hstream_submit_grouped(self.hs, x_host.data_ptr(), None if targets_host is None else targets_host.data_ptr(),
                                                 None if groups_host is None else groups_host.data_ptr(),
                                                 1 if groups_host is None else n_groups,
                                                 None if targets_host is None else sums.data_ptr(), n, self.steps, self.T, None, key,
                                                 self._mask_ptr, self.out_host[hb].data_ptr(), stream, self._slot_ref)
        if rc != 0:
            _lib.check(rc, "dp_hstream_submit")
        self._pending.append((self._slot.value, hb, n, x_host, targets_host, groups_host))
        self.n_submitted += n
        return ret

    def drain(self):
        """Wait for and return (in order) the results still in flight; the returned tensors alias the ring buffers."""
        outs = []
        while self._pending:
            outs.append(self._collect())
        return outs

    def __del__(self):
        try:
            if getattr(self, "hs", None) is not None and self.hs.value:
                self._lib.dp_hstream_destroy(self.hs)
                self.hs = None
        except Exception:
            pass
