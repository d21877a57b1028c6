"""Restatement of the reference's per-action evaluation (float64 numpy / torch, CPU), which the grouped sums are compared
against:
  define_error_list, AccumLoss      common/utils.py (the table and its accumulators; AccumLoss.avg starts at 0)
  mpjpe_by_action_p1 / _p2          common/utils.py:103-152, called through test_calculation at runners/diffpose_frame.py:391
  print_error_action                common/utils.py:247-271 (per-action mean x 1000, then the mean over actions)
on top of the oracle's per-pose metrics (oracle/diffpose_oracle.py `mpjpe` restated per pose, `p_mpjpe_per_pose`).
"""
import numpy as np
import torch

from oracle import diffpose_oracle as O

ACTIONS = ("Directions", "Discussion", "Eating", "Greeting", "Phoning", "Photo", "Posing", "Purchases", "Sitting",
           "SittingDown", "Smoking", "Waiting", "WalkDog", "Walking", "WalkTogether")


class AccumLoss:
    def __init__(self):
        self.val, self.avg, self.sum, self.count = 0, 0, 0, 0

    def update(self, val, n=1):
        self.val = val
        self.sum += val
        self.count += n
        self.avg = self.sum / self.count


def _action_name(a):
    end = a.find(" ")
    return a[:end] if end != -1 else a


def per_pose_errors(pred, target):
    """(mpjpe, p_mpjpe) per pose in float64 of root-centred [n,17,3] poses: common/loss.py:7-13 per pose, common/utils.py:155-187."""
    p = torch.as_tensor(pred, dtype=torch.float64)
    t = torch.as_tensor(target, dtype=torch.float64)
    return torch.norm(p - t, dim=-1).mean(dim=-1).numpy(), O.p_mpjpe_per_pose(p.numpy(), t.numpy())


def mpjpe_by_action(pred, target, actions, error_sum):
    """mpjpe_by_action_p1 and _p2 on one batch: a batch of one action adds mean * n with count n (the whole-batch branch),
    a mixed batch adds every pose to its own action (the per-sample branch)."""
    d1, d2 = per_pose_errors(pred, target)
    n = len(actions)
    if len(set(actions)) == 1:
        name = _action_name(actions[0])
        error_sum[name]["p1"].update(float(np.mean(d1)) * n, n)
        error_sum[name]["p2"].update(float(np.mean(d2)) * n, n)
    else:
        for i in range(n):
            name = _action_name(actions[i])
            error_sum[name]["p1"].update(float(d1[i]), 1)
            error_sum[name]["p2"].update(float(d2[i]), 1)
    return error_sum


def action_error_table(pred, target, actions, names=ACTIONS, batch_size=None):
    """The reference's per-action table of root-centred poses pred, target [n,17,3] with the loader's action strings, the
    batches of `batch_size` poses going through mpjpe_by_action one after the other.  Returns (table, protocol):
    table {name: (mpjpe_mm, p_mpjpe_mm, n)}, protocol (#1, #2) the mean of the per-action values over the actions.
    An action without poses is (nan, nan, 0) and left out of the mean; the reference's AccumLoss would report avg = 0
    for it and print_error_action would average that 0 in (a documented difference, DESIGN.md section 4.5)."""
    error_sum = {a: {"p1": AccumLoss(), "p2": AccumLoss()} for a in names}
    n = len(actions)
    bs = batch_size or max(n, 1)
    for lo in range(0, n, bs):
        hi = min(n, lo + bs)
        mpjpe_by_action(pred[lo:hi], target[lo:hi], list(actions[lo:hi]), error_sum)
    table = {}
    for a in names:
        e = error_sum[a]
        table[a] = (e["p1"].avg * 1000.0, e["p2"].avg * 1000.0, e["p1"].count) if e["p1"].count else (np.nan, np.nan, 0)
    have = [v for v in table.values() if v[2] > 0]
    protocol = (float(np.mean([v[0] for v in have])), float(np.mean([v[1] for v in have]))) if have else (np.nan, np.nan)
    return table, protocol
