"""GPU (-m gpu): keyed in-kernel noise (the key of dp_sample and dp_hstream_submit, dp_noise_fill).

dp_noise_fill is checked against the numpy restatement (oracle/philox.py).  Every keyed call is then checked bit for bit
against the same call fed dp_noise_fill's tensor through `noise=`, which carries the oracle parity of the noise path
(test_gpu_parity, test_gpu_pipeline) over to the keyed path.  Then the properties the stream exists for: results that do
not depend on how the poses are split into shards, batches or host-stream submits, one launch, no noise tensor, graph
capture."""
import ctypes

import numpy as np
import pytest
import torch

import diffpose_nw_b200 as D
from diffpose_nw_b200 import _lib
from oracle import diffpose_oracle as O
from oracle import philox as P
from _cases import betas

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

DEV = torch.device("cuda:0")
ENGINES = ["fp32", "tcx", "tcg"]


def _model(engine="tcg"):
    torch.manual_seed(0)
    m = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config())
    sd = O.perturb_state_dict({k: v.detach().clone() for k, v in m.state_dict().items()}, seed=21, scale=0.02)
    m.load_state_dict(sd)
    return m.to(DEV).eval().set_engine(engine)


_LONG_BETAS = torch.from_numpy(D.get_beta_schedule("linear", beta_start=1e-4, beta_end=2e-2, num_diffusion_timesteps=200)).float()


def _schedule(T):
    """(seq, betas) with T steps: T = 70 goes through the device step table (more than 64 steps)."""
    if T == 2:
        return [0, 12], betas()
    return list(range(0, 2 * T, 2)), _LONG_BETAS


def _poses(n, seed):
    return O.synthetic_poses(n, seed=seed).to(DEV)


def _ulp_close(got, want, ulps=4):
    got = np.asarray(got, dtype=np.float32)
    tol = ulps * np.spacing(np.abs(want).astype(np.float32))
    bad = np.abs(got.astype(np.float64) - want) > tol
    assert not bad.any(), f"{bad.sum()} of {bad.size} values beyond {ulps} ulp, worst at {np.argmax(np.abs(got - want))}"


# ------------------------------------------------------------------------------------------------ dp_noise_fill
@pytest.mark.parametrize("seed,T,n,H,po,so", [
    (0, 2, 37, 1, 0, 0),
    (0x0123456789ABCDEF, 3, 37, 5, (1 << 32) - 37, 4),
    ((1 << 63) + 5, 1, 9, 5, 12345, 70),
    (-3, 2, 1, 1, 1000000, 3),
])
def test_noise_fill_matches_restatement(seed, T, n, H, po, so):
    got = D.philox_noise(seed, T, n, H, pose_offset=po, step_offset=so, device=DEV).cpu().numpy()
    want = P.noise(seed, T, n, H, pose_offset=po, step_offset=so)
    assert got.shape == want.shape == (T, H * n, 17, 5)
    _ulp_close(got, want)


def test_noise_fill_known_values():
    z = D.philox_noise(0, 1, 1, device=DEV).view(-1)[:6].cpu().numpy()
    np.testing.assert_allclose(z, [0.991138, -0.924663, -0.617609, -0.482068, -0.153638, 0.180826], atol=2e-6)
    z = D.philox_noise(0x0123456789ABCDEF, 1, 1, 5, pose_offset=1000000, step_offset=3, device=DEV)[0, 4].reshape(-1)
    np.testing.assert_allclose(z[[0, 1, 84]].cpu().numpy(), [-0.449827, -0.401344, -0.664848], atol=2e-6)


def test_noise_key_range_is_checked():
    lib = _lib.load()
    out = torch.empty(2, 10, 17, 5, device=DEV)
    for po, so, n in [(-1, 0, 10), (0, -1, 10), ((1 << 32) - 9, 0, 10), (1 << 40, 0, 10)]:
        key = _lib.DpNoiseKey(7, po, so)
        assert lib.dp_noise_fill(ctypes.byref(key), 2, n, 1, 17, 5, out.data_ptr(), None) == -1
    key = _lib.DpNoiseKey(7, (1 << 32) - 10, 0)
    assert lib.dp_noise_fill(ctypes.byref(key), 2, 10, 1, 17, 5, out.data_ptr(), None) == 0
    m = _model("tcg")
    seq = [0, 12]
    x = _poses(10, 1)
    with pytest.raises(RuntimeError, match="pose_offset"):
        D.sample(m, x, None, seq, betas(), eta=1.0, seed=1, pose_offset=(1 << 32) - 9)
    with pytest.raises(RuntimeError, match="pose_offset"):
        D.sample(m, x, None, seq, betas(), eta=1.0, seed=1, pose_offset=-1)
    with pytest.raises(RuntimeError, match="not both"):
        D.sample(m, x, None, seq, betas(), eta=1.0, seed=1, noise=torch.zeros(2, 10, 17, 5, device=DEV))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------- keyed == materialised
# (n, H, mean_over_hyp, repeat_input, T, partial mask, fused evaluation, pose_offset)
CASES = [
    (1, 1, False, False, 2, False, False, 0),
    (37, 5, True, True, 2, True, False, 5),
    (37, 5, False, False, 70, False, False, 0),
    (37, 5, False, True, 2, False, False, 123),
    (1037, 1, False, True, 2, False, True, 0),
    (1037, 5, True, True, 2, True, True, 4000000000),
    (1037, 5, True, False, 70, False, False, 0),
    (37, 1, False, False, 70, True, True, 9),
]


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("case", CASES, ids=lambda c: "n%d_H%d_mean%d_rep%d_T%d_mask%d_eval%d" % c[:7])
def test_keyed_equals_materialised(engine, case):
    n, H, mean, rep, T, part_mask, ev, po = case
    m = _model(engine)
    seq, b = _schedule(T)
    x = _poses(n, 3) if rep else _poses(n, 3).repeat(H, 1, 1) + 0.01 * torch.randn(H * n, 17, 5, device=DEV)
    mask = None
    if part_mask:
        mask = torch.ones(1, 1, 17, dtype=torch.bool, device=DEV)
        mask[..., [3, 9, 14]] = False
    seed = 0xDEADBEEF12345678
    kw = dict(eta=1.0, n_hyp=H, repeat_input=rep, mean_over_hyp=mean)
    tg = s1 = s2 = None
    if ev:
        tg = O.synthetic_targets(_poses(n, 3).cpu(), seed=4).to(DEV)
        s1 = torch.zeros(3, device=DEV, dtype=torch.float64)
        s2 = torch.zeros(3, device=DEV, dtype=torch.float64)
    keyed = D.sample(m, x, mask, seq, b, seed=seed, pose_offset=po, targets=tg, sums=s1, **kw)
    nz = D.philox_noise(seed, T, n, H, pose_offset=po, device=DEV)
    mat = D.sample(m, x, mask, seq, b, noise=nz, targets=tg, sums=s2, **kw)
    torch.cuda.synchronize()
    assert m.engine() == engine
    assert torch.equal(keyed, mat), f"max |keyed - materialised| = {(keyed - mat).abs().max().item():.3e}"
    assert keyed.abs().max().item() > 0
    if ev:
        np.testing.assert_allclose(s1.cpu().numpy(), s2.cpu().numpy(), rtol=1e-12)
        assert s1[2].item() == n


def test_seed_without_effect_at_eta_zero():
    m = _model("tcg")
    x = _poses(50, 5)
    a = D.sample(m, x, None, [0, 12], betas(), eta=0.0)
    b = D.sample(m, x, None, [0, 12], betas(), eta=0.0, seed=99)
    assert torch.equal(a, b)


# ------------------------------------------------------------------------------------- shard and batch invariance
@pytest.mark.parametrize("engine", ENGINES)
def test_shards_and_batches_draw_the_same_noise(engine):
    m = _model(engine)
    n, H, seq, seed = 50, 3, [0, 12], 1234
    x = _poses(n, 6)
    tgt = O.synthetic_targets(x.cpu(), seed=7).to(DEV)
    kw = dict(seq=seq, betas=betas(), eta=1.0, test_times=H, seed=seed)
    whole = D.lift_and_refine(m, x, **kw)
    parts = []
    for r in range(3):
        lo, hi = D.shard_range(n, r, 3)
        parts.append(D.lift_and_refine(m, x[lo:hi].contiguous(), pose_offset=lo, **kw))
    assert torch.equal(torch.cat(parts), whole)
    # a different split without the offsets draws other noise (the test can fail)
    assert not torch.equal(D.lift_and_refine(m, x[17:].contiguous(), **kw), whole[17:])
    s_whole = D.evaluate_shard(m, x, tgt, **kw)
    s_parts = torch.zeros(3, device=DEV, dtype=torch.float64)
    for r in range(3):
        lo, hi = D.shard_range(n, r, 3)
        s_parts += D.evaluate_shard(m, x[lo:hi].contiguous(), tgt[lo:hi].contiguous(), pose_offset=lo, **kw)
    s_batch = D.evaluate_shard(m, x, tgt, batch_size=7, **kw)
    np.testing.assert_allclose(s_parts.cpu().numpy(), s_whole.cpu().numpy(), rtol=1e-9)
    np.testing.assert_allclose(s_batch.cpu().numpy(), s_whole.cpu().numpy(), rtol=1e-9)
    # the sums are those of the x_T the whole call returned
    ref, _ = D.pose_error_sums(whole, tgt)
    np.testing.assert_allclose(s_whole.cpu().numpy(), ref.cpu().numpy(), rtol=1e-9)


# ------------------------------------------------------------------------------------- host-resident batches
@pytest.mark.parametrize("with_targets", [False, True])
def test_host_stream_keyed_equals_one_call(with_targets):
    m = _model("tcg")
    seq, seed, H = [0, 12], 77, 2
    sizes = [64, 64, 10, 64, 33]
    xs = [O.synthetic_poses(k, seed=80 + i) for i, k in enumerate(sizes)]
    tgs = [O.synthetic_targets(x, seed=90 + i) for i, x in enumerate(xs)]
    x_all, t_all = torch.cat(xs).to(DEV), torch.cat(tgs).to(DEV)
    s_want = torch.zeros(3, device=DEV, dtype=torch.float64)
    want = D.sample(m, x_all, None, seq, betas(), eta=1.0, n_hyp=H, repeat_input=True, mean_over_hyp=True, seed=seed,
                    targets=t_all if with_targets else None, sums=s_want if with_targets else None).cpu()
    with pytest.raises(RuntimeError, match="eta = 0"):
        D.HostStream(m, batch=64, seq=seq, betas=betas(), eta=1.0, test_times=H)
    hs = D.HostStream(m, batch=64, seq=seq, betas=betas(), eta=1.0, test_times=H, seed=seed)
    sums = torch.zeros(3, device=DEV, dtype=torch.float64)
    got = []
    for x, t in zip(xs, tgs):
        r = hs.submit(x.pin_memory(), t.pin_memory() if with_targets else None, sums if with_targets else None)
        if r is not None:
            got.append(r.clone())
    got += [t.clone() for t in hs.drain()]
    assert torch.equal(torch.cat(got), want)
    if with_targets:
        np.testing.assert_allclose(sums.cpu().numpy(), s_want.cpu().numpy(), rtol=1e-12)


# ------------------------------------------------------------------------------------- refused argument combinations
def test_refused_combinations_leave_handle_and_ring_usable():
    """dp_sample and dp_hstream_submit take every option as an argument, so a caller can pass combinations they refuse:
    noise and key together, targets without sums, and (ring) targets with n_hyp > 1 but no mean.  Each returns
    DP_ERR_INVALID without enqueueing anything; the next valid call on the same handle and ring gives the expected result."""
    lib = _lib.load()
    m = _model("tcg")
    n, seq, seed = 40, [0, 12], 7
    x = _poses(n, 12)
    tg = O.synthetic_targets(x.cpu(), seed=13).to(DEV)
    want = D.sample(m, x, None, seq, betas(), eta=1.0, seed=seed)
    want_sums, _ = D.pose_error_sums(want, tg)
    steps = D.ddim_steps(betas(), seq, 1.0)
    T, h, key = len(steps), m._handle, _lib.noise_key(seed)
    nz = D.philox_noise(seed, T, n, device=DEV)
    stream = torch.cuda.current_stream(DEV).cuda_stream
    out = torch.zeros_like(x)
    sums = torch.zeros(3, device=DEV, dtype=torch.float64)

    def sample(noise, targets, sums_ptr):
        return lib.dp_sample(h, x.data_ptr(), 1, out.data_ptr(), n, 1, steps, T, noise, key, None, 0, targets, sums_ptr, stream)

    assert sample(nz.data_ptr(), None, None) == -1 and b"dp_sample: " in lib.dp_last_error() and b"not both" in lib.dp_last_error()
    assert sample(None, tg.data_ptr(), None) == -1 and b"dp_sample: " in lib.dp_last_error()
    torch.cuda.synchronize()
    assert out.abs().max().item() == 0
    assert sample(None, tg.data_ptr(), sums.data_ptr()) == 0
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    np.testing.assert_allclose(sums.cpu().numpy(), want_sums.cpu().numpy(), rtol=1e-12)

    xh, th = x.cpu().pin_memory(), tg.cpu().pin_memory()
    oh = torch.zeros(n, 17, 5).pin_memory()
    slot = ctypes.c_int(-1)
    rings = [ctypes.c_void_p(), ctypes.c_void_p()]
    try:
        assert lib.dp_hstream_create(ctypes.byref(rings[0]), h, 64, 1, 0, 2) == 0
        assert lib.dp_hstream_create(ctypes.byref(rings[1]), h, 64, 2, 0, 2) == 0     # two hypotheses, no mean

        def submit(ring, noise, targets, sums_ptr):
            return lib.dp_hstream_submit(ring, xh.data_ptr(), targets, sums_ptr, n, steps, T, noise, key, None, oh.data_ptr(),
                                         stream, ctypes.byref(slot))

        assert submit(rings[0], nz.data_ptr(), None, None) == -1
        assert b"dp_hstream_submit: " in lib.dp_last_error() and b"not both" in lib.dp_last_error()
        assert submit(rings[0], None, th.data_ptr(), None) == -1 and b"dp_hstream_submit: " in lib.dp_last_error()
        assert submit(rings[1], None, th.data_ptr(), sums.data_ptr()) == -1 and b"mean_over_hyp" in lib.dp_last_error()
        assert slot.value == -1
        sums.zero_()
        assert submit(rings[0], None, th.data_ptr(), sums.data_ptr()) == 0
        assert slot.value == 0                     # the refused submits did not take a slot
        assert lib.dp_hstream_wait(rings[0], slot.value) == 0
        torch.cuda.synchronize()
        assert torch.equal(oh, want.cpu())
        np.testing.assert_allclose(sums.cpu().numpy(), want_sums.cpu().numpy(), rtol=1e-12)
    finally:
        for r in rings:
            if r.value:
                lib.dp_hstream_destroy(r)


# ------------------------------------------------------------------------------------- per-step launches, determinism
@pytest.mark.parametrize("engine", ENGINES)
def test_return_all_keyed_equals_materialised(engine):
    m = _model(engine)
    seq, seed, n = [0, 6, 12, 18], 5, 40
    x = _poses(n, 8)
    xs_k, x0_k = D.generalized_steps(x, None, seq, m, betas(), eta=1.0, return_all=True, seed=seed)
    nz = D.philox_noise(seed, len(seq), n, device=DEV)
    xs_m, x0_m = D.generalized_steps(x, None, seq, m, betas(), eta=1.0, return_all=True, noise=nz)
    assert len(xs_k) == len(xs_m) == len(seq) + 1
    for a, b in zip(xs_k + x0_k, xs_m + x0_m):
        assert torch.equal(a, b)


def test_determinism_and_one_launch():
    m = _model("tcg")
    x = _poses(300, 9)
    kw = dict(eta=1.0, n_hyp=4, repeat_input=True, mean_over_hyp=True)
    a = D.sample(m, x, None, [0, 12], betas(), seed=42, **kw)
    l0 = _lib.launch_count()
    b = D.sample(m, x, None, [0, 12], betas(), seed=42, **kw)
    torch.cuda.synchronize()
    assert _lib.launch_count() - l0 == 1
    c = D.sample(m, x, None, [0, 12], betas(), seed=43, **kw)
    d = D.sample(m, x, None, [0, 12], betas(), seed=42 + (1 << 32), **kw)
    assert torch.equal(a, b)
    assert not torch.equal(a, c) and not torch.equal(a, d)


def test_keyed_call_holds_no_noise_tensor():
    """4096 poses x H = 10 x T = 50: a noise tensor would take 50 * 40960 * 85 * 4 B = 696 MB."""
    m = _model("tcg")
    seq = list(range(0, 50))
    b = torch.from_numpy(D.get_beta_schedule("linear", beta_start=1e-4, beta_end=2e-2, num_diffusion_timesteps=50)).float()
    x = _poses(4096, 10)
    D.sample(m, x[:8], None, seq, b, eta=1.0, seed=1, n_hyp=10, repeat_input=True, mean_over_hyp=True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(DEV)
    base = torch.cuda.memory_allocated(DEV)
    out = D.sample(m, x, None, seq, b, eta=1.0, seed=1, n_hyp=10, repeat_input=True, mean_over_hyp=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(DEV) - base
    print(f"keyed 4096 x 10 x 50: torch peak {peak / 2**20:.2f} MiB above the inputs")
    assert peak < 16 * 2**20
    assert torch.isfinite(out).all()


def test_keyed_call_in_cuda_graph():
    m = _model("tcg")
    x = _poses(100, 11)
    kw = dict(eta=1.0, n_hyp=3, repeat_input=True, mean_over_hyp=True, seed=31337, pose_offset=17)
    eager = D.sample(m, x, None, [0, 12], betas(), **kw)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        D.sample(m, x, None, [0, 12], betas(), **kw)      # warm-up on the capture stream: caches and buffers are in place
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = D.sample(m, x, None, [0, 12], betas(), **kw)
    out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)


# ------------------------------------------------------------------------------------- device-side statistics
def test_device_stream_statistics():
    S, H, B = 64, 4, 3085
    z = D.philox_noise(0xC0FFEE, S, B, H, device=DEV)        # [S, H*B, 17, 5]
    n = z.numel()
    assert n >= 1 << 26
    v = z.view(-1).double()
    mean, var = v.mean().item(), v.var().item()
    assert abs(mean) < 5 / np.sqrt(n)
    assert abs(var - 1.0) < 5 * np.sqrt(2.0 / n)
    c = v - mean
    skew = (c ** 3).mean().item() / var ** 1.5
    kurt = (c ** 4).mean().item() / var ** 2 - 3.0
    assert abs(skew) < 5 * np.sqrt(6.0 / n) and abs(kurt) < 5 * np.sqrt(24.0 / n)
    del c
    srt = torch.sort(z.view(-1))[0].double()
    cdf = torch.special.ndtr(srt)
    i = torch.arange(1, n + 1, device=DEV, dtype=torch.float64)
    ks = torch.maximum(i / n - cdf, cdf - (i - 1) / n).max().item()
    del srt, cdf, i
    assert ks * np.sqrt(n) < 2.5, f"KS statistic {ks:.3e} (sqrt(n) D = {ks * np.sqrt(n):.2f})"
    g = z.view(S, H, B, 85).double()

    def corr(a, b):
        a, b = a.reshape(-1), b.reshape(-1)
        a, b = a - a.mean(), b - b.mean()
        return ((a * b).mean() / (a.std() * b.std())).item(), a.numel()

    for name, (a, b) in {"e": (g[..., :-1], g[..., 1:]), "s": (g[:-1], g[1:]), "h": (g[:, :-1], g[:, 1:]),
                         "b": (g[:, :, :-1], g[:, :, 1:])}.items():
        r, m = corr(a, b)
        assert abs(r) < 5 / np.sqrt(m), f"neighbour correlation along {name}: {r:.2e}"
    del g
    # counter collisions: no two (b, h, s) rows are the same
    rows = z.view(-1, 85)[:, :8].contiguous().view(torch.int32)
    assert torch.unique(rows, dim=0).shape[0] == rows.shape[0]
