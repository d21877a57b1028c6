"""GPU (-m gpu): the evaluation pipeline around the sampler (body of test_hyber, runners/diffpose_frame.py:330-391):
BASELINE configs[4] semantics -- GCNpose lift, out-of-place root-centring, concat, H hypotheses, DDIM, hypothesis mean,
MPJPE / P-MPJPE partial sums -- against the oracle on a small batch; plus shard-equals-whole."""
import numpy as np
import pytest
import torch

import diffpose_nw_b200 as D
from oracle import diffpose_oracle as O
from _cases import betas

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


def _models():
    adj = D.adj_mx_from_edges()
    torch.manual_seed(0)
    diff = D.FusedGCNdiff(adj, O.default_config())
    sd_d = O.perturb_state_dict({k: v.detach().clone() for k, v in diff.state_dict().items()}, seed=21, scale=0.02)
    diff.load_state_dict(sd_d)
    torch.manual_seed(1)
    pose = D.FusedGCNpose(adj, O.default_config(coords_dim=[2, 3]))
    sd_p = O.perturb_state_dict({k: v.detach().clone() for k, v in pose.state_dict().items()}, seed=22, scale=0.02)
    pose.load_state_dict(sd_p)
    return adj, diff, sd_d, pose, sd_p


@pytest.mark.parametrize("engine", ["fp32", "auto", "tcg"])
def test_two_stage_pipeline_vs_oracle(engine):
    """auto (the default) = split-precision tensor-core lifter (tcx) + fp16-operand tensor-core sampler (tcg): within the
    north_star tolerance (1e-3 abs, 0.05 mm).  The sampler's fp16-operand error reaches x damped by the DDIM coefficients
    (a few 1e-5 here); the lifter's output IS the xyz input, undamped, which is why it runs on tcx.  "tcg" forces the
    fp16-operand engine for the lifter too: up to ~2e-3 with these random weights (|xyz| up to 2.6), reported, not default."""
    dev = torch.device("cuda:0")
    adj, diff, sd_d, pose, sd_p = _models()
    diff = diff.to(dev).set_engine(engine)
    pose = pose.to(dev).set_engine(engine)
    B, Hh, seq, eta = 23, 5, [0, 6], 1.0
    uv = O.synthetic_poses(B, seed=30)[:, :, :2].contiguous()
    tgt = O.synthetic_targets(O.synthetic_poses(B, seed=30), seed=31)
    g = torch.Generator().manual_seed(32)
    noise = torch.randn(len(seq), Hh * B, 17, 5, generator=g)
    mask = torch.ones(1, 1, 17, dtype=torch.bool)
    # oracle: the runner's glue restated with the intended (out-of-place) root-centring
    xyz = O.root_centre(O.gcnpose_forward(sd_p, adj, 5, 4, uv, mask))
    x = torch.cat([uv, xyz], dim=2).repeat(Hh, 1, 1)
    den = lambda xt, m, tt: O.gcndiff_forward(sd_d, adj, 5, 4, xt, m, tt)
    ref = O.hypothesis_mean(O.ddim_sample(x, mask, seq, den, betas(), eta=eta, noise=noise)[0][-1], Hh)
    ref_xyz = O.root_centre(ref[:, :, 2:])
    want = (O.mpjpe(ref_xyz, O.root_centre(tgt)).item() * 1000, float(O.p_mpjpe_per_pose(ref_xyz.numpy(), O.root_centre(tgt).numpy()).mean()) * 1000)
    # product
    l0 = D._lib.launch_count()
    out = D.lift_and_refine(diff, model_pose=pose, input_2d=uv.to(dev), src_mask=mask.to(dev), seq=seq, betas=betas(),
                            eta=eta, test_times=Hh, noise=noise.to(dev))
    n_launch = D._lib.launch_count() - l0
    tol = {"fp32": 2e-5, "auto": 1e-3, "tcg": 3e-3}[engine]
    err = (out.cpu() - ref).abs().max().item()
    print(f"two-stage / {engine}: max|dx|={err:.2e} launches (incl. one-time packing)={n_launch}")
    assert err < tol
    if engine == "auto":
        # second batch: everything is packed and cached -> exactly two launches (dp_lift, dp_sample)
        l0 = D._lib.launch_count()
        D.lift_and_refine(diff, model_pose=pose, input_2d=uv.to(dev), src_mask=mask.to(dev), seq=seq, betas=betas(),
                          eta=eta, test_times=Hh, noise=noise.to(dev))
        assert D._lib.launch_count() - l0 == 2
    sums = D.evaluate_shard(diff, None, tgt.to(dev), src_mask=mask.to(dev), seq=seq, betas=betas(), eta=eta, test_times=Hh,
                            noise=noise.to(dev), model_pose=pose, input_2d=uv.to(dev), batch_size=10)
    m, pm, cnt = D.reduce_metrics(sums)
    assert cnt == B and abs(m - want[0]) < 0.05 and abs(pm - want[1]) < 0.05


def test_shards_equal_whole():
    """Sharding over ranks never changes a pose's result: the union of 3 contiguous shards equals the unsharded run
    (the per-rank fp64 partial sums only differ by the order they are added in)."""
    dev = torch.device("cuda:0")
    adj, diff, sd_d, _, _ = _models()
    diff = diff.to(dev)
    n, Hh, seq = 50, 2, [0, 12]
    x = O.synthetic_poses(n, seed=40).to(dev)
    tgt = O.synthetic_targets(x.cpu(), seed=41).to(dev)
    whole = D.evaluate_shard(diff, x, tgt, seq=seq, betas=betas(), test_times=Hh)
    parts = torch.zeros(3, device=dev, dtype=torch.float64)
    for r in range(3):
        lo, hi = D.shard_range(n, r, 3)
        parts += D.evaluate_shard(diff, x[lo:hi].contiguous(), tgt[lo:hi].contiguous(), seq=seq, betas=betas(), test_times=Hh)
    np.testing.assert_allclose(parts.cpu().numpy(), whole.cpu().numpy(), rtol=1e-9)
    diff.set_engine("fp32")
    whole = D.evaluate_shard(diff, x, tgt, seq=seq, betas=betas(), test_times=Hh)
    parts = torch.zeros(3, device=dev, dtype=torch.float64)
    for r in range(3):
        lo, hi = D.shard_range(n, r, 3)
        parts += D.evaluate_shard(diff, x[lo:hi].contiguous(), tgt[lo:hi].contiguous(), seq=seq, betas=betas(), test_times=Hh)
    np.testing.assert_allclose(parts.cpu().numpy(), whole.cpu().numpy(), rtol=1e-9)


def test_eval_mode_weight_changes_are_picked_up():
    """eval() mode uses a cheap parameter fingerprint: load_state_dict, .to() and repack() must still invalidate the
    packed device copy, and training mode must see any in-place edit."""
    import diffpose_nw_b200 as D
    from oracle import diffpose_oracle as O
    from _cases import betas
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev).eval()
    x = O.synthetic_poses(64, seed=2).to(dev)
    a = D.generalized_steps(x, None, [0, 12], model, betas())[0][-1]
    sd = O.perturb_state_dict({k: v.detach().cpu().clone() for k, v in model.state_dict().items()}, seed=3)
    model.load_state_dict(sd)
    b = D.generalized_steps(x, None, [0, 12], model, betas())[0][-1]
    assert (a - b).abs().max().item() > 1e-3
    with torch.no_grad():
        model.atten_layers[2].self_attn.linears[1].weight.mul_(0.5)      # a middle parameter, edited in place
    model.repack()
    c = D.generalized_steps(x, None, [0, 12], model, betas())[0][-1]
    assert (b - c).abs().max().item() > 1e-5
    model.train()
    with torch.no_grad():
        model.atten_layers[2].self_attn.linears[1].weight.mul_(2.0)
    d = D.generalized_steps(x, None, [0, 12], model, betas())[0][-1]
    assert (b - d).abs().max().item() < 1e-5


def test_host_stream_matches_direct_calls():
    """HostStream (overlapped H2D / kernel / D2H ring) returns, in order, exactly what one-at-a-time calls return."""
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev).eval()
    seq = [0, 12]
    batches = [O.synthetic_poses(n, seed=60 + i).pin_memory() for i, n in enumerate([64, 64, 10, 64, 33, 64, 64])]
    want = [D.generalized_steps(b.to(dev), None, seq, model, betas())[0][-1].cpu() for b in batches]
    hs = D.HostStream(model, batch=64, seq=seq, betas=betas(), depth=3)
    got = []
    for b in batches:
        r = hs.submit(b)
        if r is not None:
            got.append(r.clone())
    got += [t.clone() for t in hs.drain()]
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g.shape == w.shape and torch.equal(g, w)
    with pytest.raises(RuntimeError, match="exceeds"):
        hs.submit(O.synthetic_poses(65).pin_memory())
    # hypotheses: kernel-side repeat + fused mean, through the same ring (eta = 0: HostStream draws no noise)
    want3 = [D.sample(model, b.to(dev), None, seq, betas(), n_hyp=3, repeat_input=True, mean_over_hyp=True).cpu() for b in batches[:4]]
    hs3 = D.HostStream(model, batch=64, seq=seq, betas=betas(), test_times=3, depth=2)
    got3 = []
    for b in batches[:4]:
        r = hs3.submit(b)
        if r is not None:
            got3.append(r.clone())
    got3 += [t.clone() for t in hs3.drain()]
    assert len(got3) == 4 and all(torch.equal(g, w) for g, w in zip(got3, want3))
    with pytest.raises(RuntimeError, match="eta = 0"):
        D.HostStream(model, batch=64, seq=seq, betas=betas(), eta=1.0)
    # evaluation fused into the ring: targets travel with each batch, the sums accumulate on the device
    tgts = [O.synthetic_targets(b, seed=70 + i).pin_memory() for i, b in enumerate(batches)]
    want_sums = torch.zeros(3, device=dev, dtype=torch.float64)
    for w, tg in zip(want, tgts):
        D.pose_error_sums(w.to(dev), tg.to(dev), sums=want_sums)
    sums = torch.zeros(3, device=dev, dtype=torch.float64)
    hs4 = D.HostStream(model, batch=64, seq=seq, betas=betas(), depth=3)
    got4 = []
    for b, tg in zip(batches, tgts):
        r = hs4.submit(b, tg, sums)
        if r is not None:
            got4.append(r.clone())
    got4 += [t.clone() for t in hs4.drain()]
    torch.cuda.synchronize()
    assert all(torch.equal(g, w) for g, w in zip(got4, want))
    np.testing.assert_allclose(sums.cpu().numpy(), want_sums.cpu().numpy(), rtol=1e-12)


def test_second_device_in_one_process():
    """A model on cuda:1 while cuda:0 is current (DataParallel-style use): per-device kernel attributes and device guards."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    torch.manual_seed(0)
    cfg = O.default_config()
    m0 = D.FusedGCNdiff(D.adj_mx_from_edges(), cfg).to("cuda:0").eval()
    torch.manual_seed(0)
    m1 = D.FusedGCNdiff(D.adj_mx_from_edges(), cfg).to("cuda:1").eval()
    x = O.synthetic_poses(30, seed=70)
    a = D.generalized_steps(x.to("cuda:0"), None, [0, 12], m0, betas())[0][-1]
    torch.cuda.set_device(0)
    b = D.generalized_steps(x.to("cuda:1"), None, [0, 12], m1, betas())[0][-1]
    assert b.device.index == 1 and torch.equal(a.cpu(), b.cpu())
    for eng in ("fp32", "tcx"):
        c = D.generalized_steps(x.to("cuda:1"), None, [0, 12], m1.set_engine(eng), betas())[0][-1]
        assert (c.cpu() - a.cpu()).abs().max().item() < 1e-3


@pytest.mark.parametrize("engine", ["auto", "fp32"])
@pytest.mark.parametrize("n,Hh", [(1, 1), (37, 1), (300, 1), (23, 5), (150, 3), (9, 10)])
def test_fused_evaluation_equals_sampler_then_metrics(engine, n, Hh):
    """dp_sample with targets_xyz (sampler + MPJPE / P-MPJPE partial sums in one launch on the default engine; one warp per
    finished pose in the tile's tail) accumulates exactly what dp_sample followed by dp_metrics does -- ragged batches, several tiles per
    CTA, hypothesis mean (poses completing across tile boundaries, H larger than a tile), accumulation over calls."""
    dev = torch.device("cuda:0")
    adj, diff, sd_d, _, _ = _models()
    diff = diff.to(dev).set_engine(engine).eval()
    seq = [0, 6]
    x = O.synthetic_poses(n, seed=90 + n).to(dev)
    tgt = O.synthetic_targets(x.cpu(), seed=91).to(dev)
    g = torch.Generator().manual_seed(92)
    noise = torch.randn(len(seq), Hh * n, 17, 5, generator=g).to(dev)
    kw = dict(eta=1.0, noise=noise, n_hyp=Hh, repeat_input=True, mean_over_hyp=Hh > 1)
    plain = D.sample(diff, x, None, seq, betas(), **kw)
    want, _ = D.pose_error_sums(plain, tgt)
    sums = torch.zeros(3, device=dev, dtype=torch.float64)
    l0 = D._lib.launch_count()
    fused = D.sample(diff, x, None, seq, betas(), targets=tgt, sums=sums, **kw)
    n_launch = D._lib.launch_count() - l0
    assert torch.equal(fused, plain)
    np.testing.assert_allclose(sums.cpu().numpy(), want.cpu().numpy(), rtol=1e-12)
    assert sums[2].item() == n
    if engine == "auto":
        assert n_launch == 1
    D.sample(diff, x, None, seq, betas(), targets=tgt, sums=sums, **kw)          # accumulates
    np.testing.assert_allclose(sums.cpu().numpy(), 2 * want.cpu().numpy(), rtol=1e-12)
    # against the oracle's metrics of the oracle's sample
    den = lambda xt, m, tt: O.gcndiff_forward(sd_d, adj, 5, 4, xt, m, tt)
    ref = O.hypothesis_mean(O.ddim_sample(x.cpu().repeat(Hh, 1, 1), None, seq, den, betas(), eta=1.0, noise=noise.cpu())[0][-1], Hh)
    m_ref = O.mpjpe(O.root_centre(ref[:, :, 2:]), O.root_centre(tgt.cpu())).item() * 1000
    assert abs(want[0].item() / n * 1000 - m_ref) < 0.05
    with pytest.raises(RuntimeError, match="mean_over_hyp"):
        D.sample(diff, x.repeat(2, 1, 1), None, seq, betas(), n_hyp=2, targets=tgt, sums=sums)


def test_sampler_call_is_cuda_graph_capturable():
    """include/diffpose_b200.h: a dp_sample call that neither grows a buffer nor changes a long schedule only enqueues work,
    so it can be captured into a CUDA graph (programmatic-dependent-launch attribute included) and replayed."""
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev).eval()
    seq = [0, 12]
    x = O.synthetic_poses(300, seed=5).to(dev)
    tgt = O.synthetic_targets(x.cpu()).to(dev)
    want = D.sample(model, x, None, seq, betas(), n_hyp=3, repeat_input=True, mean_over_hyp=True)     # also warms every cache
    sums = torch.zeros(3, device=dev, dtype=torch.float64)
    static_x = x.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        D.sample(model, static_x, None, seq, betas(), n_hyp=3, repeat_input=True, mean_over_hyp=True, targets=tgt, sums=sums)
    torch.cuda.current_stream().wait_stream(s)
    sums.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = D.sample(model, static_x, None, seq, betas(), n_hyp=3, repeat_input=True, mean_over_hyp=True, targets=tgt, sums=sums)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want) and sums[2].item() == 3 * 300
    static_x.copy_(x.flip(0))
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want.flip(0))
