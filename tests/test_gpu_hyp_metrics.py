"""GPU (-m gpu): multi-hypothesis evaluation (dp_metrics_hyp, hyp_error_sums, sample(hyp_sums=), evaluate_shard(hyp_metrics=)).

dp_metrics_hyp against a float64 oracle per pose; against the existing kernels bit for bit (per-hypothesis errors, the
hypothesis mean, H = 1); the orderings J-best <= best <= average, NaN propagation and out-of-range ids; then through the
sampler on every engine: the mean it returns, the mean-pose columns against the existing evaluation, shards and batches,
and graph replay.  Per-pose values are read from a call with one group per pose (row b = pose b's eight values)."""
import functools

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
H_MAX = 33
INT_MAX = 2 ** 31 - 1
M_COLS, P_COLS = [0, 3, 5, 6], [1, 4, 7]       # MPJPE-like and P-MPJPE-like columns


def _model(engine="tcg"):
    torch.manual_seed(0)
    m = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config())
    sd = O.perturb_state_dict({k: v.detach().clone() for k, v in m.state_dict().items()}, seed=21, scale=0.02)
    m.load_state_dict(sd)
    return m.to(DEV).eval().set_engine(engine)


@functools.lru_cache(maxsize=None)
def _hyp_set(n, c=3):
    """pred [H_MAX, n, 17, c] (xyz in the last three columns), gt [n, 17, 3]: hypotheses spread around the target at
    different scales, some mirrored (the reflection branch of P-MPJPE)."""
    g = torch.Generator().manual_seed(1000 + n)
    gt = torch.randn(n, 17, 3, generator=g) * 0.3
    scale = 0.02 + 0.08 * torch.rand(H_MAX, n, 1, 1, generator=g)
    xyz = gt + torch.randn(H_MAX, n, 17, 3, generator=g) * scale
    xyz[1::3, ::7, :, 0] *= -1.0
    pred = torch.cat([torch.rand(H_MAX, n, 17, c - 3, generator=g), xyz], -1) if c > 3 else xyz
    return pred, gt


@functools.lru_cache(maxsize=None)
def _oracle_hyp(n):
    """float64 per hypothesis: e1 [H_MAX, n], e2 [H_MAX, n], joint distances d [H_MAX, n, 17]."""
    pred, gt = _hyp_set(n)
    t = O.root_centre(gt.double())
    d = np.stack([(O.root_centre(pred[h].double()) - t).norm(dim=-1).numpy() for h in range(H_MAX)])
    e2 = np.stack([O.p_mpjpe_per_pose(O.root_centre(pred[h]).numpy(), O.root_centre(gt).numpy()) for h in range(H_MAX)])
    return d.mean(-1), e2, d


def _oracle_cols(n, H):
    """float64 [n, 8] per pose: the eight columns of include/diffpose_b200.h."""
    pred, gt = _hyp_set(n)
    e1, e2, d = (a[:H] for a in _oracle_hyp(n))
    m = pred[:H].double().mean(0)
    mt, gr = O.root_centre(m), O.root_centre(gt.double())
    out = np.zeros((n, 8))
    out[:, 0] = (mt - gr).norm(dim=-1).mean(-1).numpy()
    out[:, 1] = O.p_mpjpe_per_pose(mt.numpy(), gr.numpy())
    out[:, 2] = 1
    out[:, 3], out[:, 4] = e1.min(0), e2.min(0)
    out[:, 5] = d.min(0).mean(-1)
    out[:, 6], out[:, 7] = e1.mean(0), e2.mean(0)
    return out


def _per_pose(pred, gt, **kw):
    """[n, 8] per-pose values: one group per pose, so each row is written by exactly one pose (0 + v = v)."""
    n = gt.shape[0]
    ids = torch.arange(n, dtype=torch.int32, device=DEV)
    s, ph, mo = D.hyp_error_sums(pred, gt, groups=ids, n_groups=n, **kw)
    return s, ph, mo


def _mean_rows(rows):
    """The hypothesis mean of [H, ...] rows in hyp_mean_kernel's order: summed from h = 0 upwards, one IEEE division (by a
    tensor: torch multiplies by the reciprocal of a scalar divisor)."""
    s = torch.zeros_like(rows[0])
    for h in range(rows.shape[0]):
        s = s + rows[h]
    return s / torch.full_like(s, rows.shape[0])


def _bucket(ids, rows, G):
    ids = np.asarray(ids, dtype=np.int64)
    ok = (ids >= 0) & (ids < G)
    return np.stack([np.bincount(ids[ok], weights=rows[ok, k], minlength=G) for k in range(rows.shape[1])], 1)


# ------------------------------------------------------------------------------------------------ against float64
@pytest.mark.parametrize("n", [1, 37, 2 * 148 * 8 * 8 + 13])    # 2 x 9472 + 13: three grid-stride passes, the last ragged
@pytest.mark.parametrize("H", [1, 2, 5, 10, 33])
@pytest.mark.parametrize("G", [1, 15])
def test_metrics_hyp_vs_oracle(n, H, G):
    pred, gt = _hyp_set(n)
    p, g = pred[:H].to(DEV), gt.to(DEV)
    per, _, _ = _per_pose(p, g)
    got = per.cpu().numpy()
    want = _oracle_cols(n, H)
    assert (got[:, 2] == 1).all()
    # the bound of test_metrics_kernel_many_poses_vs_oracle, per pose
    np.testing.assert_allclose(got[:, M_COLS], want[:, M_COLS], rtol=0, atol=2e-7)
    np.testing.assert_allclose(got[:, P_COLS], want[:, P_COLS], rtol=0, atol=1e-6)
    # grouped sums = the per-pose rows bucketed in float64; [H*n] input = [H, n] input
    ids = torch.from_numpy(np.random.default_rng(n + H).integers(0, G, n).astype(np.int32))
    sums, _, _ = D.hyp_error_sums(p.reshape(H * n, 17, 3), g, groups=ids.to(DEV), n_groups=G)
    np.testing.assert_allclose(sums.cpu().numpy(), _bucket(ids, got, G), rtol=1e-12)
    flat, _, _ = D.hyp_error_sums(p, g)
    assert flat.shape == (8,) and flat[2].item() == n
    np.testing.assert_allclose(flat.cpu().numpy(), got.sum(0), rtol=1e-12)


# ------------------------------------------------------------------------------------------------ against existing bits
@pytest.mark.parametrize("H", [1, 5, 10])
@pytest.mark.parametrize("c", [3, 5])
def test_metrics_hyp_bits_equal_existing_kernels(H, c):
    n = 301
    pred, gt = _hyp_set(n, c)
    p, g = pred[:H].to(DEV), gt.to(DEV)
    per, ph, mo = _per_pose(p, g, per_hyp=True, mean_out=True)
    for h in range(H):                                        # dp_metrics' per_pose on slice h
        _, pp = D.pose_error_sums(p[h], g, per_pose=True)
        assert torch.equal(ph[h], pp), h
    assert torch.equal(mo, _mean_rows(p))
    mean_sums, mean_pp = D.pose_error_sums(mo, g, per_pose=True)
    got = per.cpu().numpy()
    assert np.array_equal(got[:, :2], mean_pp.double().cpu().numpy())           # columns 0, 1: dp_metrics on the mean
    if H == 1:
        for k in (3, 5, 6):
            assert np.array_equal(got[:, k], got[:, 0]), k
        for k in (4, 7):
            assert np.array_equal(got[:, k], got[:, 1]), k
        flat, _, _ = D.hyp_error_sums(p, g)
        np.testing.assert_allclose(flat[:3].cpu().numpy(), mean_sums.cpu().numpy(), rtol=1e-12)
        assert flat[2].item() == n


# ------------------------------------------------------------------------------------------------ invariants
def test_orderings_nan_and_guard_rows():
    n, H, G = 2000, 10, 15
    pred, gt = _hyp_set(n)
    p, g = pred[:H].clone(), gt.clone()
    p[4, 17] = 0.2                                            # a zero-extent hypothesis: its P-MPJPE is NaN
    p, g = p.to(DEV), g.to(DEV)
    per, ph, _ = _per_pose(p, g, per_hyp=True)
    got = per.cpu().numpy()
    assert np.isnan(ph[4, 17, 1].item()) and np.isfinite(ph[4, 17, 0].item())
    assert np.isnan(got[17, 4]) and np.isnan(got[17, 7])      # best and average P-MPJPE propagate the NaN
    assert np.isfinite(got[17, [0, 1, 2, 3, 5, 6]]).all()
    ok = np.isfinite(got).all(1)
    assert ok.sum() == n - 1
    g_ok = got[ok]
    assert (g_ok[:, 5] <= g_ok[:, 3]).all() and (g_ok[:, 3] <= g_ok[:, 6]).all() and (g_ok[:, 4] <= g_ok[:, 7]).all()
    assert (g_ok[:, 5] < g_ok[:, 6]).any()
    # on the sums, without the NaN pose, up to fp64 reordering
    keep = torch.arange(n) != 17
    kd = keep.to(DEV)
    s, _, _ = D.hyp_error_sums(p[:, kd], g[kd])
    s = s.cpu().numpy()
    assert s[5] <= s[3] * (1 + 1e-12) and s[3] <= s[6] * (1 + 1e-12) and s[4] <= s[7] * (1 + 1e-12)
    # ids -1, G and beyond add to nothing: guard rows around the [G, 8] block stay zero
    ids = torch.from_numpy(np.sort(np.random.default_rng(3).integers(0, G, n)).astype(np.int32))
    ids[::5] = -1
    ids[1::7] = G
    ids[2::11] = INT_MAX
    ids[3::13] = -INT_MAX - 1
    bad = (ids < 0) | (ids >= G)
    big = torch.zeros(G + 2, 8, device=DEV, dtype=torch.float64)
    D.hyp_error_sums(p[:, kd], g[kd], sums=big[1:G + 1], groups=ids[keep].to(DEV))
    b = big.cpu().numpy()
    assert (b[0] == 0).all() and (b[G + 1] == 0).all()
    np.testing.assert_allclose(b[1:G + 1], _bucket(ids[keep], got[ok], G), rtol=1e-12)
    assert b[1:G + 1, 2].sum() == (~bad[keep]).sum().item()


def test_python_arguments_are_checked():
    pred, gt = (t.to(DEV) for t in _hyp_set(10))
    with pytest.raises(RuntimeError, match=r"\[H\*10,17,c\]"):
        D.hyp_error_sums(pred[:3].reshape(30, 17, 3)[:29], gt)
    with pytest.raises(RuntimeError, match="n=10"):
        D.hyp_error_sums(pred[:3, :9], gt)
    with pytest.raises(RuntimeError, match="8 elements"):
        D.hyp_error_sums(pred[:3], gt, sums=torch.zeros(3, device=DEV, dtype=torch.float64))
    ids = torch.zeros(10, dtype=torch.int32, device=DEV)
    with pytest.raises(RuntimeError, match=r"\[n_groups,8\]"):
        D.hyp_error_sums(pred[:3], gt, sums=torch.zeros(15, 3, device=DEV, dtype=torch.float64), groups=ids)
    with pytest.raises(RuntimeError, match="int32"):
        D.hyp_error_sums(pred[:3], gt, groups=ids.long(), n_groups=15)
    m = _model("tcg")
    x = O.synthetic_poses(10, seed=2).to(DEV)
    hs = torch.zeros(8, device=DEV, dtype=torch.float64)
    kw = dict(n_hyp=3, repeat_input=True, mean_over_hyp=True)
    with pytest.raises(RuntimeError, match="not both"):
        D.sample(m, x, None, [0, 12], betas(), targets=gt, sums=torch.zeros(3, device=DEV, dtype=torch.float64), hyp_sums=hs, **kw)
    with pytest.raises(RuntimeError, match="needs targets"):
        D.sample(m, x, None, [0, 12], betas(), hyp_sums=hs, **kw)
    xs = torch.empty(2, 30, 17, 5, device=DEV)
    with pytest.raises(RuntimeError, match="trajectory"):
        D.sample(m, x, None, [0, 12], betas(), targets=gt, hyp_sums=hs, xs_out=xs, **kw)
    assert hs.abs().max().item() == 0


# ------------------------------------------------------------------------------------------------ through the sampler
@pytest.mark.parametrize("engine", ["auto", "tcx", "fp32"])
def test_sampler_hyp_eval_configs2_shape(engine):
    """configs[2] shape (1024 x H=5, seq [0, 12], eta = 1, keyed noise): the mean returned through dp_metrics_hyp equals the
    sampler's own mean, the mean-pose columns equal the existing evaluation, the H rows equal sample(mean_over_hyp=False)."""
    m = _model(engine)
    n, H, G, seq = 1024, 5, 15, [0, 12]
    x = O.synthetic_poses(n, seed=31).to(DEV)
    tg = O.synthetic_targets(x.cpu(), seed=32).to(DEV)
    ids = torch.from_numpy(np.sort(np.random.default_rng(5).integers(0, G, n)).astype(np.int32)).to(DEV)
    kw = dict(eta=1.0, n_hyp=H, repeat_input=True, seed=99, pose_offset=7)
    want = D.sample(m, x, None, seq, betas(), mean_over_hyp=True, **kw)
    rows = D.sample(m, x, None, seq, betas(), mean_over_hyp=False, **kw)
    s3 = torch.zeros(G, 3, device=DEV, dtype=torch.float64)
    D.sample(m, x, None, seq, betas(), mean_over_hyp=True, targets=tg, sums=s3, groups=ids, **kw)
    hs = torch.zeros(G, 8, device=DEV, dtype=torch.float64)
    l0 = _lib.launch_count()
    got = D.sample(m, x, None, seq, betas(), mean_over_hyp=True, targets=tg, hyp_sums=hs, groups=ids, **kw)
    if engine == "auto":
        assert m.engine() == "tcg" and _lib.launch_count() - l0 == 2          # the sampler, then dp_metrics_hyp
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    np.testing.assert_allclose(hs[:, :3].cpu().numpy(), s3.cpu().numpy(), rtol=1e-12)
    assert torch.equal(hs[:, 2], s3[:, 2]) and hs[:, 2].sum().item() == n
    direct, _, _ = D.hyp_error_sums(rows, tg, groups=ids, n_groups=G)
    np.testing.assert_allclose(hs.cpu().numpy(), direct.cpu().numpy(), rtol=1e-12)
    # without the mean: the H rows come back, the same sums
    hs2 = torch.zeros(G, 8, device=DEV, dtype=torch.float64)
    got_rows = D.sample(m, x, None, seq, betas(), mean_over_hyp=False, targets=tg, hyp_sums=hs2, groups=ids, **kw)
    assert torch.equal(got_rows, rows)
    np.testing.assert_allclose(hs2.cpu().numpy(), hs.cpu().numpy(), rtol=1e-12)


def test_sampler_hyp_eval_chunked_device_noise(monkeypatch):
    """eta > 0 without noise or seed: the torch-drawn noise is cut into pose chunks; every chunk is evaluated."""
    from diffpose_nw_b200 import sampler
    m = _model("tcg")
    n, H = 50, 3
    x = O.synthetic_poses(n, seed=41).to(DEV)
    tg = O.synthetic_targets(x.cpu(), seed=42).to(DEV)
    D.sample(m, x, None, [0, 12], betas())                   # packs the weights and caches the schedule: no launches below
    monkeypatch.setattr(sampler, "NOISE_CHUNK_BYTES", 2 * H * 17 * 5 * 4 * 7)     # 7 poses per chunk: 8 chunks
    for mean in (True, False):
        hs = torch.zeros(8, device=DEV, dtype=torch.float64)
        l0 = _lib.launch_count()
        torch.manual_seed(3)
        out = D.sample(m, x, None, [0, 12], betas(), eta=1.0, n_hyp=H, repeat_input=True, mean_over_hyp=mean, targets=tg, hyp_sums=hs)
        assert _lib.launch_count() - l0 == 16
        rows = out if not mean else None
        if mean:
            torch.manual_seed(3)
            rows = D.sample(m, x, None, [0, 12], betas(), eta=1.0, n_hyp=H, repeat_input=True)
            assert torch.equal(out, _mean_rows(rows.view(H, n, 17, 5)))
        want, _, _ = D.hyp_error_sums(rows, tg)
        np.testing.assert_allclose(hs.cpu().numpy(), want.cpu().numpy(), rtol=1e-12)
        assert hs[2].item() == n


def test_evaluate_shard_hyp_metrics_shards_and_batches():
    m = _model("tcg")
    n, H, G = 50, 5, 15
    x = O.synthetic_poses(n, seed=6).to(DEV)
    tgt = O.synthetic_targets(x.cpu(), seed=7).to(DEV)
    ids = torch.from_numpy(np.sort(np.random.default_rng(8).integers(0, G, n)).astype(np.int32)).to(DEV)
    kw = dict(seq=[0, 12], betas=betas(), eta=1.0, test_times=H, seed=1234, hyp_metrics=True)
    for groups in (None, ids):
        gk = dict(groups=groups, n_groups=G) if groups is not None else {}
        whole = D.evaluate_shard(m, x, tgt, **kw, **gk)
        assert whole.shape == ((G, 8) if groups is not None else (8,))
        batched = D.evaluate_shard(m, x, tgt, batch_size=7, **kw, **gk)
        parts = torch.zeros_like(whole)
        for r in range(2):
            lo, hi = D.shard_range(n, r, 2)
            gs = dict(gk, groups=groups[lo:hi]) if groups is not None else {}
            parts += D.evaluate_shard(m, x[lo:hi].contiguous(), tgt[lo:hi].contiguous(), pose_offset=lo, **kw, **gs)
        np.testing.assert_allclose(batched.cpu().numpy(), whole.cpu().numpy(), rtol=1e-12)
        np.testing.assert_allclose(parts.cpu().numpy(), whole.cpu().numpy(), rtol=1e-12)
        # the mean-pose columns are the existing evaluation's
        flat = D.evaluate_shard(m, x, tgt, **dict(kw, hyp_metrics=False), **gk)
        np.testing.assert_allclose(whole[..., :3].cpu().numpy(), flat.cpu().numpy(), rtol=1e-12)
    table, protocol, totals = D.reduce_hyp_errors(whole.clone(), D.H36M_ACTIONS)
    assert totals.n == n and totals.jbest_mpjpe <= totals.best_mpjpe <= totals.avg_mpjpe
    assert np.isfinite(protocol).all()


def test_hyp_eval_in_cuda_graph():
    m = _model("tcg")
    n, G = 300, 15
    x = O.synthetic_poses(n, seed=5).to(DEV)
    tgt = O.synthetic_targets(x.cpu()).to(DEV)
    ids = torch.from_numpy(np.sort(np.random.default_rng(1).integers(0, G, n)).astype(np.int32)).to(DEV)
    kw = dict(n_hyp=3, repeat_input=True, mean_over_hyp=True, eta=1.0, seed=11)
    hs = torch.zeros(G, 8, device=DEV, dtype=torch.float64)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        want = D.sample(m, x, None, [0, 12], betas(), targets=tgt, hyp_sums=hs, groups=ids, **kw)    # warms every cache
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    first = hs.clone()
    hs.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = D.sample(m, x, None, [0, 12], betas(), targets=tgt, hyp_sums=hs, groups=ids, **kw)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    np.testing.assert_allclose(hs.cpu().numpy(), first.cpu().numpy(), rtol=1e-12)
    g.replay()
    torch.cuda.synchronize()
    np.testing.assert_allclose(hs.cpu().numpy(), 2 * first.cpu().numpy(), rtol=1e-12)
