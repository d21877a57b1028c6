"""CPU: the host side of the multi-hypothesis evaluation -- the reduction of [8] / [G, 8] sums to millimetres and the
per-action table (one all-reduce, also over 2 gloo ranks), dp_metrics_hyp's argument refusals, and no CPU fallback."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import diffpose_nw_b200 as D
from diffpose_nw_b200 import _lib


def _row(mean, best, jbest, avg, n):
    """One [8] row of sums for n poses whose errors (metres) are the given per-pose values."""
    return torch.tensor([mean[0] * n, mean[1] * n, n, best[0] * n, best[1] * n, jbest * n, avg[0] * n, avg[1] * n],
                        dtype=torch.float64)


def test_reduce_hyp_errors_totals():
    s = _row((0.05, 0.025), (0.04, 0.02), 0.03, (0.06, 0.03), 4)
    got = D.reduce_hyp_errors(s.clone())
    assert isinstance(got, D.HypErrors) and got.n == 4
    assert got == pytest.approx(D.HypErrors(50.0, 25.0, 4.0, 40.0, 20.0, 30.0, 60.0, 30.0))
    # [G, 8] without names: the pose-weighted totals over the rows
    two = torch.stack([s, _row((0.1, 0.05), (0.08, 0.04), 0.07, (0.12, 0.06), 12)])
    got = D.reduce_hyp_errors(two.clone())
    assert got.n == 16 and got.mean_mpjpe == pytest.approx((0.2 + 1.2) / 16 * 1000) and got.jbest_mpjpe == pytest.approx((0.12 + 0.84) / 16 * 1000)
    empty = D.reduce_hyp_errors(torch.zeros(8, dtype=torch.float64))
    assert empty.n == 0 and all(np.isnan(v) for k, v in empty._asdict().items() if k != "n")
    with pytest.raises(RuntimeError, match=r"\[8\] or \[G,8\]"):
        D.reduce_hyp_errors(torch.zeros(3, dtype=torch.float64))


def test_reduce_hyp_errors_per_action():
    sums = torch.zeros(15, 8, dtype=torch.float64)
    sums[0] = _row((0.05, 0.025), (0.04, 0.02), 0.03, (0.06, 0.03), 4)
    sums[13] = _row((0.1, 0.05), (0.08, 0.04), 0.07, (0.12, 0.06), 30)
    table, protocol, totals = D.reduce_hyp_errors(sums.clone(), D.H36M_ACTIONS)
    assert table["Directions"] == pytest.approx((50.0, 25.0, 4.0, 40.0, 20.0, 30.0, 60.0, 30.0))
    assert table["Walking"] == pytest.approx((100.0, 50.0, 30.0, 80.0, 40.0, 70.0, 120.0, 60.0))
    for a in D.H36M_ACTIONS:
        if a not in ("Directions", "Walking"):
            assert table[a].n == 0 and all(np.isnan(v) for k, v in table[a]._asdict().items() if k != "n")
    # each action with poses counts once (as reduce_action_errors weighs them), the empty ones not at all
    assert protocol == pytest.approx((75.0, 37.5, 34.0, 60.0, 30.0, 50.0, 90.0, 45.0))
    assert totals == D.reduce_hyp_errors(sums.clone())
    assert totals.best_mpjpe == pytest.approx((0.16 + 2.4) / 34 * 1000)
    # columns 0-2 are the [G, 3] sums of the hypothesis mean: the same table as reduce_action_errors
    t3, p3, tot3 = D.reduce_action_errors(sums[:, :3].clone())
    assert p3 == pytest.approx(protocol[:2]) and tot3 == pytest.approx(totals[:3])
    for a in ("Directions", "Walking"):
        assert t3[a] == pytest.approx(table[a][:3])
    _, protocol, totals = D.reduce_hyp_errors(torch.zeros(15, 8, dtype=torch.float64), D.H36M_ACTIONS)
    assert np.isnan(protocol.mean_mpjpe) and np.isnan(totals.avg_p_mpjpe) and totals.n == 0
    with pytest.raises(RuntimeError, match=r"\[15,8\]"):
        D.reduce_hyp_errors(torch.zeros(14, 8, dtype=torch.float64), D.H36M_ACTIONS)


def test_metrics_hyp_arguments_refused_before_any_launch():
    """Every refusal returns DP_ERR_INVALID before the library touches a device (so it holds on a machine without one)."""
    lib = _lib.load()
    P = 4096                                   # never dereferenced: each call is refused first

    def call(pred=P, stride=5, offset=2, n_hyp=5, gt=P, n=10, n_pts=17, group=None, n_groups=1, sums=P):
        return lib.dp_metrics_hyp(pred, stride, offset, n_hyp, gt, n, n_pts, group, n_groups, sums, None, None, None)

    for kw, msg in [(dict(n_hyp=0), b"n_hyp"), (dict(n_hyp=-2), b"n_hyp"), (dict(n_pts=16), b"n_pts"),
                    (dict(offset=3), b"stride"), (dict(stride=2, offset=0), b"stride"), (dict(offset=-1), b"stride"),
                    (dict(pred=None), b"NULL"), (dict(gt=None), b"NULL"), (dict(sums=None), b"NULL"),
                    (dict(group=P, n_groups=0), b"n_groups"), (dict(n=-1), b"")]:
        assert call(**kw) == -1, kw
        assert msg in lib.dp_last_error(), kw
    assert call(n=0) == 0                      # an empty batch enqueues nothing


def test_no_cpu_fallback():
    pred, gt = torch.zeros(2, 3, 17, 3), torch.zeros(3, 17, 3)
    with pytest.raises(RuntimeError, match="CUDA only"):
        D.hyp_error_sums(pred, gt)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_sums(rank):
    """Rank r's [15, 8] partial sums: rank 0 holds Directions and half of Walking, rank 1 the other half and Eating."""
    s = torch.zeros(15, 8, dtype=torch.float64)
    if rank == 0:
        s[0] = _row((0.05, 0.025), (0.04, 0.02), 0.03, (0.06, 0.03), 4)
        s[13] = _row((0.1, 0.05), (0.08, 0.04), 0.07, (0.12, 0.06), 10)
    else:
        s[13] = _row((0.2, 0.1), (0.16, 0.08), 0.14, (0.24, 0.12), 10)
        s[2] = _row((0.03, 0.02), (0.02, 0.01), 0.01, (0.04, 0.03), 7)
    return s


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        q.put((rank, D.reduce_hyp_errors(_rank_sums(rank), D.H36M_ACTIONS)))
    finally:
        dist.destroy_process_group()


def test_two_rank_hyp_table_equals_single_process():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    table, protocol, totals = D.reduce_hyp_errors(_rank_sums(0) + _rank_sums(1), D.H36M_ACTIONS)
    assert table["Walking"] == pytest.approx((150.0, 75.0, 20.0, 120.0, 60.0, 105.0, 180.0, 90.0))
    for _, (got, got_protocol, got_totals) in res:          # every rank holds the single-process table
        for a in D.H36M_ACTIONS:
            np.testing.assert_allclose(got[a], table[a], rtol=1e-12)
        assert got_protocol == pytest.approx(protocol, rel=1e-12)
        assert got_totals == pytest.approx(totals, rel=1e-12)
