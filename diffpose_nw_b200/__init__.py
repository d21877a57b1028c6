"""diffpose_nw_b200 -- B200 (sm_100a) implementation of DiffPose's frame-based DDIM sampling path.

Host-side mirror of the reference interface (nwicakson/diffpose-nw):
    FusedGCNdiff / FusedGCNpose   <- models/gcndiff.py::GCNdiff, models/gcnpose.py::GCNpose
    EMAHelper                     <- models/ema.py
    generalized_steps, get_beta_schedule, compute_alpha   <- common/utils_diff.py
    adj_mx_from_edges             <- models/ChebConv.py
    mpjpe, p_mpjpe                <- common/loss.py
All arithmetic runs in libdiffpose_b200.so (C ABI: include/diffpose_b200.h).  No CPU fallback.
"""
from .graph import H36M_EDGES, adj_mx_from_edges
from .model import EMAHelper, FusedGCNdiff, FusedGCNpose
from .sampler import compute_alpha, ddim_steps, generalized_steps, get_beta_schedule, make_seq, philox_noise, sample
from .metrics import mpjpe, p_mpjpe, pose_error_sums
from .pipeline import HostStream, evaluate_shard, lift_and_refine, reduce_metrics, shard_range

__all__ = ["H36M_EDGES", "adj_mx_from_edges", "FusedGCNdiff", "FusedGCNpose", "EMAHelper", "compute_alpha", "ddim_steps",
           "generalized_steps", "get_beta_schedule", "make_seq", "philox_noise", "sample", "mpjpe", "p_mpjpe", "pose_error_sums",
           "HostStream", "evaluate_shard", "lift_and_refine", "reduce_metrics", "shard_range"]
