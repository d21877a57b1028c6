"""GPU (-m gpu): group-keyed evaluation sums (dp_metrics with group ids, dp_sample_grouped, dp_hstream_submit_grouped).

The grouped rows are checked against the kernel's own per-pose errors and the oracle's, bucketed by group on the host;
the fused grouped tail against the sampler followed by grouped dp_metrics on every engine; then what the ids are for:
out-of-range ids that add to nothing, shards and batches, the host-memory ring, refused arguments and graph replay."""
import ctypes

import numpy as np
import pytest
import torch

import diffpose_nw_b200 as D
from diffpose_nw_b200 import _lib
from oracle import diffpose_oracle as O
from _cases import betas

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

DEV = torch.device("cuda:0")
INT_MAX = 2 ** 31 - 1


def _model(engine="tcg"):
    torch.manual_seed(0)
    m = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config())
    sd = O.perturb_state_dict({k: v.detach().clone() for k, v in m.state_dict().items()}, seed=21, scale=0.02)
    m.load_state_dict(sd)
    return m.to(DEV).eval().set_engine(engine)


def _ids(n, G, kind, seed=0):
    """int32 [n] ids in [0, G): sorted runs (as a loader delivers a test set), random, or a single group."""
    rng = np.random.default_rng(seed)
    if kind == "single":
        ids = np.full(n, G - 1)
    elif kind == "random":
        ids = rng.integers(0, G, n)
    else:
        ids = np.sort(rng.integers(0, G, n))
    return torch.from_numpy(ids.astype(np.int32))


def _bucket(ids, values, G):
    """float64 [G, 3]: per group the sums of the two value columns and the count (ids outside [0, G) dropped)."""
    ids = np.asarray(ids, dtype=np.int64)
    v = np.asarray(values, dtype=np.float64)
    ok = (ids >= 0) & (ids < G)
    out = np.zeros((G, 3))
    for c in range(2):
        out[:, c] = np.bincount(ids[ok], weights=v[ok, c], minlength=G)
    out[:, 2] = np.bincount(ids[ok], minlength=G)
    return out


def _eval_set(n, seed):
    g = torch.Generator().manual_seed(seed)
    gt = torch.randn(n, 17, 3, generator=g) * 0.3
    pred = gt + torch.randn(n, 17, 3, generator=g) * 0.05
    pred[::7, :, 0] *= -1.0                      # mirrored predictions: the reflection branch of P-MPJPE
    return pred, gt


# ------------------------------------------------------------------------------------------------ dp_metrics grouped
@pytest.mark.parametrize("n", [1, 37, 2 * 148 * 8 * 8 + 13])    # 2 x 9472 + 13: three grid-stride passes, the last ragged
@pytest.mark.parametrize("G", [1, 15, 1000])
@pytest.mark.parametrize("kind", ["runs", "random", "single"])
def test_metrics_grouped_vs_oracle(n, G, kind):
    pred, gt = _eval_set(n, 100 + n)
    ids = _ids(n, G, kind, seed=n + G)
    flat, pp_flat = D.pose_error_sums(pred.to(DEV), gt.to(DEV), per_pose=True)
    sums, pp = D.pose_error_sums(pred.to(DEV), gt.to(DEV), per_pose=True, groups=ids.to(DEV), n_groups=G)
    torch.cuda.synchronize()
    assert sums.shape == (G, 3) and sums.dtype is torch.float64
    assert torch.equal(pp, pp_flat)                                            # per-pose errors unchanged
    got = sums.cpu().numpy()
    # against the kernel's own per-pose errors, summed per group in float64
    np.testing.assert_allclose(got, _bucket(ids, pp.cpu().numpy(), G), rtol=1e-12, atol=0)
    # against the oracle (common/loss.py restated in float64), at the bound of test_metrics_kernel_many_poses_vs_oracle
    p, t = O.root_centre(pred), O.root_centre(gt)
    want_m = (p - t).norm(dim=-1).mean(dim=-1).double().numpy()
    want_p = O.p_mpjpe_per_pose(p.numpy(), t.numpy())
    want = _bucket(ids, np.stack([want_m, want_p], 1), G)
    assert (got[:, 2] == want[:, 2]).all()
    assert np.abs(got[:, :2] - want[:, :2]).max() < 1e-4
    # the rows add up to the ungrouped sums
    np.testing.assert_allclose(got.sum(0), flat.cpu().numpy(), rtol=1e-12)
    if G == 1:
        np.testing.assert_allclose(got[0], flat.cpu().numpy(), rtol=1e-12)
    # accumulates into a given [G, 3] tensor
    D.pose_error_sums(pred.to(DEV), gt.to(DEV), sums=sums, groups=ids.to(DEV))
    np.testing.assert_allclose(sums.cpu().numpy(), 2 * got, rtol=1e-12)


def test_out_of_range_ids_add_to_nothing():
    """Ids -1, G and INT_MAX add to nothing: guard rows around the [G, 3] block stay zero, in dp_metrics and in the fused
    tail of the default engine."""
    G, n = 15, 301
    pred, gt = _eval_set(n, 5)
    ids = _ids(n, G, "random", seed=3)
    ids[::5] = -1
    ids[1::7] = G
    ids[2::11] = INT_MAX
    ids[3::13] = -INT_MAX - 1
    bad = (ids < 0) | (ids >= G)
    assert bad.sum() > 50
    big = torch.zeros(G + 2, 3, device=DEV, dtype=torch.float64)
    _, pp = D.pose_error_sums(pred.to(DEV), gt.to(DEV), sums=big[1:G + 1], per_pose=True, groups=ids.to(DEV))
    torch.cuda.synchronize()
    b = big.cpu().numpy()
    assert (b[0] == 0).all() and (b[G + 1] == 0).all()
    np.testing.assert_allclose(b[1:G + 1], _bucket(ids, pp.cpu().numpy(), G), rtol=1e-12)
    assert b[1:G + 1, 2].sum() == n - bad.sum()
    # fused: a batch padded with -1 and with ids beyond the table
    m = _model("tcg")
    x = O.synthetic_poses(n, seed=9).to(DEV)
    tg = O.synthetic_targets(x.cpu(), seed=10).to(DEV)
    out = D.sample(m, x, None, [0, 12], betas())
    _, pp = D.pose_error_sums(out, tg, per_pose=True)
    big.zero_()
    D.sample(m, x, None, [0, 12], betas(), targets=tg, sums=big[1:G + 1], groups=ids.to(DEV))
    torch.cuda.synchronize()
    b = big.cpu().numpy()
    assert (b[0] == 0).all() and (b[G + 1] == 0).all()
    np.testing.assert_allclose(b[1:G + 1], _bucket(ids, pp.cpu().numpy(), G), rtol=1e-12)


def test_grouped_arguments_are_checked():
    lib = _lib.load()
    pred, gt = (t.to(DEV) for t in _eval_set(10, 1))
    ids = _ids(10, 15, "random").to(DEV)
    sums = torch.zeros(15, 3, device=DEV, dtype=torch.float64)
    assert lib.dp_metrics(pred.data_ptr(), 3, 0, gt.data_ptr(), 10, 17, ids.data_ptr(), 0, sums.data_ptr(), None, None) == -1
    assert b"n_groups" in lib.dp_last_error()
    torch.cuda.synchronize()
    assert sums.abs().max().item() == 0
    with pytest.raises(RuntimeError, match="int32"):
        D.pose_error_sums(pred, gt, groups=ids.long(), n_groups=15)
    with pytest.raises(RuntimeError, match="int32"):
        D.pose_error_sums(pred, gt, groups=ids[:9], n_groups=15)
    with pytest.raises(RuntimeError, match="n_groups"):
        D.pose_error_sums(pred, gt, groups=ids)
    with pytest.raises(RuntimeError, match=r"\[n_groups,3\]"):
        D.pose_error_sums(pred, gt, sums=torch.zeros(3, device=DEV, dtype=torch.float64), groups=ids)
    m = _model("tcg")
    x = O.synthetic_poses(10, seed=2).to(DEV)
    with pytest.raises(RuntimeError, match="targets"):
        D.sample(m, x, None, [0, 12], betas(), sums=sums, groups=ids)
    with pytest.raises(RuntimeError, match=r"\[n_groups,3\]"):
        D.sample(m, x, None, [0, 12], betas(), targets=gt, sums=torch.zeros(3, device=DEV, dtype=torch.float64), groups=ids)


# ------------------------------------------------------------------------------------------------ fused == two launches
@pytest.mark.parametrize("engine", ["auto", "tcx", "fp32"])
@pytest.mark.parametrize("n,Hh", [(1, 1), (37, 1), (300, 1), (23, 5), (150, 3), (9, 10), (2100, 1)])
def test_fused_grouped_equals_sampler_then_grouped_metrics(engine, n, Hh):
    """dp_sample_grouped accumulates per group what dp_sample followed by grouped dp_metrics does: ragged batches, several
    tiles per CTA (n = 2100), poses completing across tile boundaries (hypothesis mean), accumulation over calls."""
    m = _model(engine)
    seq = [0, 6]
    G = 15
    x = O.synthetic_poses(n, seed=90 + n).to(DEV)
    tgt = O.synthetic_targets(x.cpu(), seed=91).to(DEV)
    ids = _ids(n, G, "random" if n % 2 else "runs", seed=n).to(DEV)
    g = torch.Generator().manual_seed(92)
    noise = torch.randn(len(seq), Hh * n, 17, 5, generator=g).to(DEV)
    kw = dict(eta=1.0, noise=noise, n_hyp=Hh, repeat_input=True, mean_over_hyp=Hh > 1)
    flat = torch.zeros(3, device=DEV, dtype=torch.float64)
    plain = D.sample(m, x, None, seq, betas(), targets=tgt, sums=flat, **kw)
    want, _ = D.pose_error_sums(plain, tgt, groups=ids, n_groups=G)
    sums = torch.zeros(G, 3, device=DEV, dtype=torch.float64)
    l0 = _lib.launch_count()
    fused = D.sample(m, x, None, seq, betas(), targets=tgt, sums=sums, groups=ids, **kw)
    n_launch = _lib.launch_count() - l0
    torch.cuda.synchronize()
    assert torch.equal(fused, plain)                          # x_out bit-identical to the ungrouped call
    np.testing.assert_allclose(sums.cpu().numpy(), want.cpu().numpy(), rtol=1e-12)
    np.testing.assert_allclose(sums.sum(0).cpu().numpy(), flat.cpu().numpy(), rtol=1e-12)
    assert sums[:, 2].sum().item() == n
    if engine == "auto":
        assert m.engine() == "tcg" and n_launch == 1
    D.sample(m, x, None, seq, betas(), targets=tgt, sums=sums, groups=ids, **kw)          # accumulates
    np.testing.assert_allclose(sums.cpu().numpy(), 2 * want.cpu().numpy(), rtol=1e-12)


# ------------------------------------------------------------------------------------------------ keyed noise + groups
def test_keyed_shards_and_batches_per_group():
    m = _model("tcg")
    n, H, G = 50, 3, 15
    x = O.synthetic_poses(n, seed=6).to(DEV)
    tgt = O.synthetic_targets(x.cpu(), seed=7).to(DEV)
    ids = _ids(n, G, "runs", seed=8).to(DEV)
    kw = dict(seq=[0, 12], betas=betas(), eta=1.0, test_times=H, seed=1234, n_groups=G)
    whole = D.evaluate_shard(m, x, tgt, groups=ids, **kw)
    assert whole.shape == (G, 3)
    batched = D.evaluate_shard(m, x, tgt, groups=ids, batch_size=7, **kw)
    parts = torch.zeros(G, 3, device=DEV, dtype=torch.float64)
    for r in range(2):
        lo, hi = D.shard_range(n, r, 2)
        parts += D.evaluate_shard(m, x[lo:hi].contiguous(), tgt[lo:hi].contiguous(), groups=ids[lo:hi], pose_offset=lo, **kw)
    np.testing.assert_allclose(batched.cpu().numpy(), whole.cpu().numpy(), rtol=1e-9)
    np.testing.assert_allclose(parts.cpu().numpy(), whole.cpu().numpy(), rtol=1e-9)
    # and the rows are those of the x_T the whole call samples
    out = D.lift_and_refine(m, x, seq=[0, 12], betas=betas(), eta=1.0, test_times=H, seed=1234)
    ref, _ = D.pose_error_sums(out, tgt, groups=ids, n_groups=G)
    np.testing.assert_allclose(whole.cpu().numpy(), ref.cpu().numpy(), rtol=1e-9)
    table, protocol, totals = D.reduce_action_errors(whole.clone())
    assert totals[2] == n and np.isfinite(protocol).all()


# ------------------------------------------------------------------------------------------------ host-resident batches
def test_host_stream_grouped_equals_one_call():
    m = _model("tcg")
    seq, H, G = [0, 12], 2, 15
    sizes = [64, 64, 10, 64, 33]
    xs = [O.synthetic_poses(k, seed=80 + i) for i, k in enumerate(sizes)]
    tgs = [O.synthetic_targets(x, seed=90 + i) for i, x in enumerate(xs)]
    ids = _ids(sum(sizes), G, "runs", seed=4)
    x_all, t_all = torch.cat(xs).to(DEV), torch.cat(tgs).to(DEV)
    s_want = torch.zeros(G, 3, device=DEV, dtype=torch.float64)
    want = D.sample(m, x_all, None, seq, betas(), n_hyp=H, repeat_input=True, mean_over_hyp=True, targets=t_all, sums=s_want,
                    groups=ids.to(DEV)).cpu()
    hs = D.HostStream(m, batch=64, seq=seq, betas=betas(), test_times=H)
    sums = torch.zeros(G, 3, device=DEV, dtype=torch.float64)
    got, lo = [], 0
    for x, t in zip(xs, tgs):
        r = hs.submit(x.pin_memory(), t.pin_memory(), sums, groups_host=ids[lo:lo + len(x)].clone().pin_memory())
        lo += len(x)
        if r is not None:
            got.append(r.clone())
    got += [t.clone() for t in hs.drain()]
    torch.cuda.synchronize()
    assert torch.equal(torch.cat(got), want)
    np.testing.assert_allclose(sums.cpu().numpy(), s_want.cpu().numpy(), rtol=1e-12)
    with pytest.raises(RuntimeError, match="groups_host"):
        hs.submit(xs[0].pin_memory(), None, None, groups_host=ids[:64].clone())


def test_refused_grouped_combinations_leave_handle_and_ring_usable():
    """dp_sample_grouped and dp_hstream_submit_grouped refuse group ids without targets and n_groups < 1 with ids, with
    DP_ERR_INVALID and without enqueueing anything; the next valid call on the same handle and ring gives the expected
    result and the refused submits took no ring slot."""
    lib = _lib.load()
    m = _model("tcg")
    n, seq, G = 40, [0, 12], 15
    x = O.synthetic_poses(n, seed=12).to(DEV)
    tg = O.synthetic_targets(x.cpu(), seed=13).to(DEV)
    ids = _ids(n, G, "random", seed=14).to(DEV)
    want = D.sample(m, x, None, seq, betas())
    want_sums, _ = D.pose_error_sums(want, tg, groups=ids, n_groups=G)
    steps = D.ddim_steps(betas(), seq, 0.0)
    T, h = len(steps), m._handle
    stream = torch.cuda.current_stream(DEV).cuda_stream
    out = torch.zeros_like(x)
    sums = torch.zeros(G, 3, device=DEV, dtype=torch.float64)

    def sample(targets, group, n_groups):
        return lib.dp_sample_grouped(h, x.data_ptr(), 1, out.data_ptr(), n, 1, steps, T, None, None, None, 0, targets, group, n_groups,
                                     sums.data_ptr(), stream)

    assert sample(None, ids.data_ptr(), G) == -1 and b"dp_sample: " in lib.dp_last_error() and b"targets" in lib.dp_last_error()
    assert sample(tg.data_ptr(), ids.data_ptr(), 0) == -1 and b"n_groups" in lib.dp_last_error()
    assert sample(tg.data_ptr(), ids.data_ptr(), -3) == -1
    torch.cuda.synchronize()
    assert out.abs().max().item() == 0 and sums.abs().max().item() == 0
    assert sample(tg.data_ptr(), ids.data_ptr(), G) == 0
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    np.testing.assert_allclose(sums.cpu().numpy(), want_sums.cpu().numpy(), rtol=1e-12)

    xh, th, ih = x.cpu().pin_memory(), tg.cpu().pin_memory(), ids.cpu().pin_memory()
    oh = torch.zeros(n, 17, 5).pin_memory()
    slot = ctypes.c_int(-1)
    ring = ctypes.c_void_p()
    try:
        assert lib.dp_hstream_create(ctypes.byref(ring), h, 64, 1, 0, 2) == 0

        def submit(targets, groups, n_groups):
            return lib.dp_hstream_submit_grouped(ring, xh.data_ptr(), targets, groups, n_groups, sums.data_ptr(), n, steps, T, None, None,
                                                 None, oh.data_ptr(), stream, ctypes.byref(slot))

        assert submit(None, ih.data_ptr(), G) == -1 and b"dp_hstream_submit: " in lib.dp_last_error()
        assert submit(th.data_ptr(), ih.data_ptr(), 0) == -1 and b"n_groups" in lib.dp_last_error()
        assert slot.value == -1
        sums.zero_()
        assert submit(th.data_ptr(), ih.data_ptr(), G) == 0
        assert slot.value == 0                     # the refused submits did not take a slot
        assert lib.dp_hstream_wait(ring, slot.value) == 0
        torch.cuda.synchronize()
        assert torch.equal(oh, want.cpu())
        np.testing.assert_allclose(sums.cpu().numpy(), want_sums.cpu().numpy(), rtol=1e-12)
    finally:
        if ring.value:
            lib.dp_hstream_destroy(ring)


# ------------------------------------------------------------------------------------------------ CUDA graphs
def test_grouped_call_in_cuda_graph():
    """A grouped fused call is captured into a CUDA graph; replaying it after rewriting the static id buffer moves the
    counts to the new groups."""
    m = _model("tcg")
    n, G = 300, 15
    x = O.synthetic_poses(n, seed=5).to(DEV)
    tgt = O.synthetic_targets(x.cpu()).to(DEV)
    ids = _ids(n, G, "runs", seed=1).to(DEV)
    kw = dict(n_hyp=3, repeat_input=True, mean_over_hyp=True)
    sums = torch.zeros(G, 3, device=DEV, dtype=torch.float64)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        want = D.sample(m, x, None, [0, 12], betas(), targets=tgt, sums=sums, groups=ids, **kw)    # warms every cache
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    first = sums.clone()
    sums.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = D.sample(m, x, None, [0, 12], betas(), targets=tgt, sums=sums, groups=ids, **kw)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    np.testing.assert_allclose(sums.cpu().numpy(), first.cpu().numpy(), rtol=1e-12)
    new_ids = torch.from_numpy((G - 1 - ids.cpu().numpy()).astype(np.int32))
    ids.copy_(new_ids)
    sums.zero_()
    g.replay()
    torch.cuda.synchronize()
    np.testing.assert_allclose(sums.cpu().numpy(), first.cpu().numpy()[::-1], rtol=1e-12)
