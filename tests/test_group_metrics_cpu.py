"""CPU: the host side of the per-action evaluation -- action names to group ids, the reduction of [G, 3] grouped sums to
the reference's per-action table (one all-reduce, also over 2 gloo ranks), and the restatement of that table."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import diffpose_nw_b200 as D
from oracle import diffpose_oracle as O
import _action_oracle as A


def test_action_names_and_normalisation():
    assert D.H36M_ACTIONS == A.ACTIONS and len(set(D.H36M_ACTIONS)) == 15
    ids = D.action_groups(["Walking 1", "Walking", "WalkDog 1", "Directions", "SittingDown 2", "WalkTogether"])
    assert ids.dtype is torch.int32 and ids.tolist() == [13, 13, 12, 0, 9, 14]
    assert D.action_groups([]).shape == (0,)
    assert D.action_groups(["b x", "a"], names=("a", "b")).tolist() == [1, 0]
    with pytest.raises(ValueError, match="unknown action"):
        D.action_groups(["Walking", "Jumping 1"])
    with pytest.raises(ValueError, match="unknown action"):
        D.action_groups([" Walking"])         # the text before the first space is empty


def test_reduce_action_errors_on_hand_made_sums():
    sums = torch.zeros(15, 3, dtype=torch.float64)
    sums[0] = torch.tensor([0.2, 0.1, 4.0], dtype=torch.float64)       # 50 mm, 25 mm over 4 poses
    sums[13] = torch.tensor([3.0, 1.5, 30.0], dtype=torch.float64)     # 100 mm, 50 mm over 30 poses
    table, (p1, p2), totals = D.reduce_action_errors(sums.clone(), D.H36M_ACTIONS)
    assert table["Directions"] == pytest.approx((50.0, 25.0, 4.0))
    assert table["Walking"] == pytest.approx((100.0, 50.0, 30.0))
    empty = [a for a in D.H36M_ACTIONS if a not in ("Directions", "Walking")]
    assert all(np.isnan(table[a][0]) and np.isnan(table[a][1]) and table[a][2] == 0 for a in empty)
    assert (p1, p2) == pytest.approx((75.0, 37.5))               # each action counts once, the empty ones not at all
    assert totals == pytest.approx(D.reduce_metrics(sums.sum(0)))  # pose-weighted: 3.2 / 34 m
    assert totals[0] == pytest.approx(3200.0 / 34)
    t, prot, tot = D.reduce_action_errors(torch.zeros(15, 3, dtype=torch.float64))
    assert np.isnan(prot[0]) and np.isnan(tot[0]) and tot[2] == 0
    with pytest.raises(RuntimeError, match=r"\[15,3\]"):
        D.reduce_action_errors(torch.zeros(14, 3, dtype=torch.float64))


def _poses_and_actions(n, seed):
    pred = O.root_centre(O.synthetic_poses(n, seed=seed)[:, :, 2:])
    tgt = O.root_centre(O.synthetic_targets(O.synthetic_poses(n, seed=seed), seed=seed + 1))
    rng = np.random.default_rng(seed)
    # six runs of one action each, as the loader delivers them, with the loader's subaction suffixes; nine actions have no poses
    runs = rng.choice(15, size=6, replace=False)
    lens = np.diff(np.sort(np.r_[0, rng.choice(np.arange(1, n), size=5, replace=False), n]))
    acts = [f"{A.ACTIONS[a]}{'' if k % 2 else ' 1'}" for k, (a, m) in enumerate(zip(runs, lens)) for _ in range(m)]
    return pred, tgt, acts


@pytest.mark.parametrize("batch_size", [None, 7, 64])
def test_action_error_table_against_direct_restatement(batch_size):
    """None: one mixed batch (the per-sample branch); 7 and 64: most batches hold one action (the whole-batch branch),
    the ones across a run boundary mix two."""
    n = 300
    pred, tgt, acts = _poses_and_actions(n, 11)
    table, protocol = A.action_error_table(pred, tgt, acts, batch_size=batch_size)
    ids = D.action_groups(acts).numpy()
    d1, d2 = A.per_pose_errors(pred, tgt)
    cnt = np.bincount(ids, minlength=15)
    with np.errstate(invalid="ignore", divide="ignore"):
        m1 = np.bincount(ids, weights=d1, minlength=15) / cnt * 1000
        m2 = np.bincount(ids, weights=d2, minlength=15) / cnt * 1000
    for g, a in enumerate(A.ACTIONS):
        assert table[a][2] == cnt[g]
        if cnt[g]:
            assert table[a][:2] == pytest.approx((m1[g], m2[g]), rel=1e-12)
        else:
            assert np.isnan(table[a][0]) and np.isnan(table[a][1])
    assert protocol == pytest.approx((m1[cnt > 0].mean(), m2[cnt > 0].mean()), rel=1e-12)
    # the grouped sums these pose errors make give the same table through reduce_action_errors
    sums = torch.zeros(15, 3, dtype=torch.float64)
    sums.index_add_(0, torch.from_numpy(ids).long(), torch.from_numpy(np.stack([d1, d2, np.ones(n)], 1)))
    got, got_protocol, totals = D.reduce_action_errors(sums)
    for a in A.ACTIONS:
        np.testing.assert_allclose(got[a], table[a], rtol=1e-12)
    assert got_protocol == pytest.approx(protocol, rel=1e-12)
    assert totals == pytest.approx((d1.mean() * 1000, d2.mean() * 1000, n), rel=1e-12)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        pred, tgt, acts = _poses_and_actions(n, 21)
        lo, hi = D.shard_range(n, rank, world)
        # per-rank grouped partial sums as the device produces them: row g = [sum mpjpe, sum p_mpjpe, count] of action g
        d1, d2 = A.per_pose_errors(pred[lo:hi], tgt[lo:hi])
        ids = D.action_groups(acts[lo:hi]).long()
        sums = torch.zeros(15, 3, dtype=torch.float64)
        sums.index_add_(0, ids, torch.from_numpy(np.stack([d1, d2, np.ones(hi - lo)], 1)))
        q.put((rank, D.reduce_action_errors(sums)))
    finally:
        dist.destroy_process_group()


def test_two_rank_action_table_equals_single_process():
    n, world = 101, 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    pred, tgt, acts = _poses_and_actions(n, 21)
    table, protocol = A.action_error_table(pred, tgt, acts)
    d1, d2 = A.per_pose_errors(pred, tgt)
    for _, (got, got_protocol, totals) in res:       # every rank holds the single-process table
        for a in A.ACTIONS:
            np.testing.assert_allclose(got[a], table[a], rtol=1e-12)
        assert got_protocol == pytest.approx(protocol, rel=1e-12)
        assert totals == pytest.approx((d1.mean() * 1000, d2.mean() * 1000, n), rel=1e-12)
