"""Every model shape dp_create accepts, against a float64 oracle.

The library takes coords_dim 1..8, hid_dim 32/64/96/128, any n_head with d_k <= 64 and 1..16 layers on the fp32 engine,
and coords_dim <= 5 with hid 96 / 4 heads on the tensor-core engines (tcg, tcx).  Many branches of the kernels depend on
exactly these sizes: tcg splits each tile row's c output coordinates between two threads and indexes the keyed noise with
e = joint c + coord, packs the convolution blocks at panel position order * 5 + coordinate, pushes 2 + 14 L weight blocks
per step through a 4-stage ring (odd and even L wrap it differently) and takes xyz as the last three output columns in its
fused evaluation tail; tcx and the glue kernels carry c_in / c_out through their stores.  The golden cases run only c = 5
(lifter 2 -> 3) and L = 5 on tcx, so each shape here is compared with the oracle in float64 (`O.gcndiff_forward` /
`O.gcnpose_forward` on double weights and inputs; the time embedding stays fp32, as in the kernels).  tcg keeps the two
checks of test_gpu_sampler_eps: its rounding-point emulation under TCG_TOL and the oracle under the operand-precision
bound.

The shape lists cover each value at least once and name the risky combinations explicitly; weights are perturbed so that
LayerNorm, A_hat and the biases are not at identity.  Every probe comparison also measures the distance to the reference at
t + 1 and with 1 % on head 0 of one layer's v bias, and asserts that the bound rejects both.
"""
import time

import numpy as np
import pytest
import torch

import diffpose_nw_b200 as D
from oracle import diffpose_oracle as O
from oracle import philox as P
from oracle import tc_emulation as E
from _cases import betas
from test_gpu_noise import _ulp_close
from test_gpu_sampler_eps import (AMP, FWD_TOL, TCG_TOL, TP, _outside, _sched_70, _seq_mean, _stats, _tol, _x_steps,
                                  probe_steps, ref_loop)

torch.set_grad_enabled(False)

TCG_ORACLE_TOL = 3e-2      # tcg against the oracle with perturbed weights (test_gpu_tc, test_gpu_sampler_eps)
PROBE_TV = 12
MASKED = (3, 9, 14)        # joints hidden by the partial key mask

# (hid, n_head, c, n_layer).  Tensor-core engines: every coordinate width at L = 5, then even and deep stacks at c = 5.
TC_DIFF = [(96, 4, c, 5) for c in (1, 2, 3, 4, 5)] + [(96, 4, 5, L) for L in (2, 4, 16)]
# fp32: hid 32 (simt_kernel<1>), 64 (<2>), 128 (<4>); d_k = 1 (32 heads of hid 32), d_k = 32 and d_k = 64 (one head of
# 64, two of 128); c in {1, 3, 4, 8}; L in {1, 2, 16}.
FP32_DIFF = [(32, 1, 1, 1), (32, 32, 3, 2), (64, 1, 8, 16), (128, 2, 3, 16), (128, 2, 8, 1), (64, 1, 4, 2), (32, 32, 1, 16)]
DIFF_CASES = [("tcg", s) for s in TC_DIFF] + [("tcx", s) for s in TC_DIFF] + [("fp32", s) for s in FP32_DIFF]
LIFT_IO = [(2, 3), (1, 5), (5, 1), (3, 3), (5, 5), (4, 2)]
LIFT_CASES = [(e, io) for e in ("fp32", "tcx", "tcg") for io in LIFT_IO]


def _id(case):
    e, s = case
    return f"{e}-" + ("h%d_nh%d_c%d_L%d" % s if len(s) == 4 else "in%d_out%d" % s)


def dev():
    return torch.device("cuda:0")


def n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


# --------------------------------------------------------------------------- models, inputs, references
class _Lifter(D.FusedGCNpose):
    """GCNpose at any output width: the reference hard-codes 3 (gcnpose.py:91), the library takes c_out 1..8."""

    def _out_dim(self):
        return self.coords_dim[1]


def _model(cls, hid, heads, c_in, c_out, n_layer, seed=5):
    """Seeded default init plus O.perturb_state_dict.  Sixteen layers perturbed by the usual 0.05 amplify eps to |eps| ~ 150
    (2000 at hid 128): the fp16-operand error grows with it, and a few x + 0.1 eps steps leave the fp16 range.  At 0.03
    |eps| stays below ~ 20, as with 5 layers at 0.05."""
    adj = D.adj_mx_from_edges()
    torch.manual_seed(seed)
    model = cls(adj, O.default_config(hid_dim=hid, n_head=heads, coords_dim=[c_in, c_out], num_layer=n_layer))
    sd = O.perturb_state_dict({k: v.detach().clone() for k, v in model.state_dict().items()}, seed=13,
                              scale=0.03 if n_layer > 5 else 0.05)
    model.load_state_dict(sd)
    return adj, model, sd


def _diff(spec):
    hid, heads, c, n_layer = spec
    return _model(D.FusedGCNdiff, hid, heads, c, c, n_layer)


def _poses(n, c, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, 17, c, generator=g) * 2 - 1


def _mask():
    m = torch.ones(1, 1, 17, dtype=torch.bool)
    m[..., list(MASKED)] = False
    return m


def _bias_error(sd, n_layer, n_head):
    """1 % on head 0 of the v bias of layer min(2, L - 1)."""
    sd = dict(sd)
    key = f"atten_layers.{min(2, n_layer - 1)}.self_attn.linears.2.bias"
    b = sd[key].clone()
    b[:b.numel() // n_head] *= 1.01
    sd[key] = b
    return sd


def _f64(sd, adj):
    return {k: v.double() for k, v in sd.items()}, adj.double()


def _den64(sd, adj, n_layer, heads, mask):
    """eps(x, t [n]) in float64; the time embedding is formed in fp32 and cast, as the kernels form it."""
    sd64, adj64 = _f64(sd, adj)
    return lambda x, tt: O.gcndiff_forward(sd64, adj64, n_layer, heads, x.double(), mask, tt)


def _emu(sd, adj, n_layer, mask):
    return lambda x, tt: E.gcndiff_forward_tcg(sd, adj, n_layer, 4, x, mask, tt, p16=True, temb_in_gc2=True)


def _den(engine, sd, adj, n_layer, heads, mask):
    return _emu(sd, adj, n_layer, mask) if engine == "tcg" else _den64(sd, adj, n_layer, heads, mask)


def _targets(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 17, 3, generator=g) * 0.3 + torch.tensor([0.1, -0.2, 5.0])


def _metrics64(pred_xyz, tgt):
    """float64 per-pose MPJPE and P-MPJPE of root-centred prediction and target."""
    p, g = pred_xyz.double(), tgt.double()
    p, g = p - p[:, :1], g - g[:, :1]
    return (p - g).norm(dim=-1).mean(dim=-1).numpy(), O.p_mpjpe_per_pose(p.numpy(), g.numpy())


# --------------------------------------------------------------------------- 1. the float64 reference is pinned (CPU)
@pytest.mark.parametrize("spec", sorted(set(TC_DIFF + FP32_DIFF)), ids=lambda s: "h%d_nh%d_c%d_L%d" % s)
def test_float64_oracle_gcndiff(spec):
    """The float64 oracle agrees with the fp32 one within 1e-5 max(1, |ref|) at every denoiser shape of the matrices, and
    ref_loop in float64 with a probe step returns the float64 eps bit for bit."""
    hid, heads, c, n_layer = spec
    adj, _, sd = _diff((hid, heads, c, n_layer))
    x, mask = _poses(24, c, seed=11), _mask()
    tt = torch.arange(24, dtype=torch.float32) * 2
    ref = _den64(sd, adj, n_layer, heads, mask)(x, tt)
    assert ref.dtype == torch.float64
    f32 = O.gcndiff_forward(sd, adj, n_layer, heads, x, mask, tt)
    scale = max(1.0, ref.abs().max().item())
    err = (f32.double() - ref).abs().max().item()
    print(f"oracle h{hid} nh{heads} c{c} L{n_layer}: |fp32 - f64| = {err:.2e} (scale {scale:.2f})")
    assert err < 1e-5 * scale
    den = _den64(sd, adj, n_layer, heads, mask)
    x64 = x.double()
    assert torch.equal(ref_loop(x64, probe_steps([PROBE_TV]), den), den(x64, torch.full((24,), float(PROBE_TV))))


@pytest.mark.parametrize("io", LIFT_IO)
def test_float64_oracle_gcnpose(io):
    ci, co = io
    adj, _, sd = _model(_Lifter, 96, 4, ci, co, 5)
    x = _poses(24, ci, seed=12)
    sd64, adj64 = _f64(sd, adj)
    ref = O.gcnpose_forward(sd64, adj64, 5, 4, x.double(), _mask())
    f32 = O.gcnpose_forward(sd, adj, 5, 4, x, _mask())
    scale = max(1.0, ref.abs().max().item())
    assert ref.shape == (24, 17, co) and (f32.double() - ref).abs().max().item() < 1e-5 * scale


# --------------------------------------------------------------------------- 3. keyed noise layout at any width (CPU)
@pytest.mark.parametrize("c", [1, 3, 4, 8])
def test_noise_layout_any_width(c):
    """oracle/philox.py noise(c=) against the counter rule restated element by element: entry [k, h n + p, j, i] is the
    normal of (step k, pose p, hypothesis h, element j c + i)."""
    T, n, H, seed = 2, 3, 2, 0xABCDEF01 + c
    z = P.noise(seed, T, n, H, c=c, pose_offset=7, step_offset=1)
    assert z.shape == (T, H * n, 17, c)
    for k in range(T):
        for h in range(H):
            for p in range(n):
                for j in range(17):
                    for i in range(c):
                        want = P.normal(seed, 1 + k, 7 + p, h, j * c + i)
                        assert z[k, h * n + p, j, i] == want


# --------------------------------------------------------------------------- 2. forward eps (dp_forward, per-sample t)
@pytest.mark.gpu
@pytest.mark.parametrize("case", DIFF_CASES, ids=_id)
def test_forward_eps(case):
    engine, (hid, heads, c, n_layer) = case
    adj, model, sd = _diff((hid, heads, c, n_layer))
    model = model.to(dev()).set_engine(engine)
    n = TP * n_sm() + 1
    x, mask = _poses(n, c, seed=21), _mask()
    tt = torch.randint(0, 51, (n,), generator=torch.Generator().manual_seed(22)).float()
    out = model(x.to(dev()), mask.to(dev()), tt.to(dev()), 0).cpu()
    assert model.forward_engine() == engine
    ref = _den64(sd, adj, n_layer, heads, mask)(x, tt)
    scale = max(1.0, ref.abs().max().item())
    err = (out.double() - ref).abs().max().item()
    if engine != "tcg":
        print(f"forward {_id(case)}: |out - f64| = {err:.2e} (bound {FWD_TOL * scale:.2e})")
        assert err < FWD_TOL * scale
        return
    emu = E.gcndiff_forward_tcg(sd, adj, n_layer, 4, x, mask, tt, p16=True)
    e_emu = (out - emu).abs().max().item()
    print(f"forward {_id(case)}: |out - emu| = {e_emu:.2e} (bound {TCG_TOL[0] * scale:.2e})  |out - f64| = {err:.2e} "
          f"(bound {TCG_ORACLE_TOL * scale:.2e})")
    assert e_emu < TCG_TOL[0] * scale and err < TCG_ORACLE_TOL * scale


# --------------------------------------------------------------------------- 2./3. undamped eps and z + eps through probe steps
@pytest.mark.gpu
@pytest.mark.parametrize("case", DIFF_CASES, ids=_id)
def test_probe_eps(case):
    """eps(x, 12) through one probe step on 7 S + 1 poses with a partial key mask, within the engine's bound of its
    reference; the references at t + 1 and with 1 % on one head's v bias fall outside it.  Then a keyed probe step with
    c1 = 1 (z + eps) within the same bound of z_ref + eps_ref: a noise element drawn for another coordinate is O(1) off."""
    engine, (hid, heads, c, n_layer) = case
    adj, model, sd = _diff((hid, heads, c, n_layer))
    model = model.to(dev()).set_engine(engine)
    n = TP * n_sm() + 1
    x, mask = _poses(n, c, seed=31), _mask()
    xd, md = x.to(dev()), mask.to(dev())
    out = D.sample(model, xd, md, None, betas(), steps=probe_steps([PROBE_TV])).cpu()
    assert model.engine() == engine
    tt = torch.full((n,), float(PROBE_TV))
    den = _den(engine, sd, adj, n_layer, heads, mask)
    ref = den(x, tt)
    ref1 = den(x, tt + 1)
    refw = _den(engine, _bias_error(sd, n_layer, heads), adj, n_layer, heads, mask)(x, tt)
    scale = max(1.0, ref.abs().max().item())
    tol = _tol(engine, scale, n)
    st, st1, stw = _stats(out, ref), _stats(out, ref1), _stats(out, refw)
    print(f"probe {_id(case)}: vs {'emu' if engine == 'tcg' else 'f64'} max/rms/chmean={st[0]:.2e}/{st[1]:.2e}/{st[2]:.2e} "
          f"bound {tol[0]:.2e}/{tol[1]:.2e}/{tol[2]:.2e}  t+1: {st1[0]:.2e}/{st1[1]:.2e}/{st1[2]:.2e}  "
          f"1% v-bias: {stw[0]:.2e}/{stw[1]:.2e}/{stw[2]:.2e}")
    assert all(s < b for s, b in zip(st, tol)), f"{_id(case)}: eps off its reference {st} (bound {tol})"
    assert _outside(st1, tol), f"{_id(case)}: the bound cannot tell t from t+1"
    if hid // heads > 1:     # with d_k = 1, head 0 is one channel of 32: 1 % of it can stay inside the fp32 bound
        assert _outside(stw, tol), f"{_id(case)}: the bound cannot see a 1 % error on one head's v bias"
    if engine == "tcg":
        e_or = (out.double() - _den64(sd, adj, n_layer, heads, mask)(x, tt)).abs().max().item()
        print(f"   tcg vs f64: max={e_or:.2e} (bound {TCG_ORACLE_TOL * scale:.2e})")
        assert e_or < TCG_ORACLE_TOL * scale
    seed = 0x5EED0000 + c
    zo = D.sample(model, xd, md, None, betas(), steps=probe_steps([PROBE_TV], c1=1.0), seed=seed, pose_offset=3).cpu()
    z = torch.from_numpy(P.noise(seed, 1, n, 1, c=c, pose_offset=3)[0])
    stz = _stats(zo, (z + ref.double()).to(ref.dtype))
    print(f"   z + eps: max/rms/chmean={stz[0]:.2e}/{stz[1]:.2e}/{stz[2]:.2e}")
    assert all(s < b for s, b in zip(stz, tol)), f"{_id(case)}: z + eps off {stz} (bound {tol})"


# --------------------------------------------------------------------------- 2./3./4. two DDIM steps, keyed, H = 3, fused tail
def _group_ids(n, G, seed):
    ids = torch.randint(-1, G, (n,), generator=torch.Generator().manual_seed(seed), dtype=torch.int32)
    ids[: G + 1] = torch.arange(-1, G, dtype=torch.int32)
    return ids


@pytest.mark.gpu
@pytest.mark.parametrize("case", DIFF_CASES, ids=_id)
def test_keyed_two_steps_fused(case):
    """seq [0, 12], eta 1, keyed noise, H = 3, kernel-side repeat, fused hypothesis mean on 2 S + 3 poses.  The keyed call
    is bit-identical to the same call given `noise=philox_noise(..., c=c)`; the result is within the engine's bound of the
    in-order hypothesis mean of ref_loop on the float64 (tcg: emulated) eps with the float64 stream.  Where c >= 3, the
    fused evaluation's sums -- ungrouped and [G, 3] grouped with -1 padding ids -- equal float64 MPJPE / P-MPJPE of the
    last three columns of the returned tensor (the xyz rule of every engine) within n 1e-6 (pose scale)."""
    engine, (hid, heads, c, n_layer) = case
    adj, model, sd = _diff((hid, heads, c, n_layer))
    model = model.to(dev()).set_engine(engine)
    S, H, G = n_sm(), 3, 4
    n = 2 * S + 3
    x, mask = _poses(n, c, seed=41), _mask()
    xd, md = x.to(dev()), mask.to(dev())
    steps = D.ddim_steps(betas(), [0, 12], 1.0)
    seed = 0xC0DE0000 + 16 * c + n_layer
    kw = dict(n_hyp=H, repeat_input=True, mean_over_hyp=True, steps=steps)
    evaluated = c >= 3
    tgt = _targets(n, seed=42)
    ids = _group_ids(n, G, seed=43)
    ev = [dict(), dict()]
    if evaluated:
        ev = [dict(targets=tgt.to(dev()), sums=torch.zeros(3, dtype=torch.float64, device=dev())) for _ in range(2)]
    keyed = D.sample(model, xd, md, None, betas(), seed=seed, **kw, **ev[0])
    nz = D.philox_noise(seed, 2, n, H, c=c, device=dev())
    mat = D.sample(model, xd, md, None, betas(), noise=nz, **kw, **ev[1])
    assert keyed.shape == (n, 17, c)
    assert torch.equal(keyed, mat), f"{_id(case)}: keyed noise differs from dp_noise_fill's at c = {c}"
    zref = torch.from_numpy(P.noise(seed, 2, n, H, c=c))
    den = _den(engine, sd, adj, n_layer, heads, mask)
    x_in = x.repeat(H, 1, 1)
    ref = _seq_mean(ref_loop(x_in.double() if engine != "tcg" else x_in, steps, den,
                             zref if engine != "tcg" else zref.float()), H)
    out = keyed.cpu()
    scale = max(1.0, ref.abs().max().item())
    tol = _tol(engine, scale, n)
    st = _stats(out, ref)
    print(f"keyed2 {_id(case)}: max/rms/chmean={st[0]:.2e}/{st[1]:.2e}/{st[2]:.2e} (bound {tol[0]:.2e}/{tol[1]:.2e}/{tol[2]:.2e})")
    assert all(s < b for s, b in zip(st, tol)), f"{_id(case)}: {st} (bound {tol})"
    if not evaluated:
        return
    s1, s2 = ev[0]["sums"].cpu().numpy(), ev[1]["sums"].cpu().numpy()
    np.testing.assert_allclose(s1, s2, rtol=1e-12)
    m, pm = _metrics64(out[:, :, c - 3:], tgt)
    pscale = max(out[:, :, c - 3:].abs().max().item(), tgt.abs().max().item())
    print(f"   eval: |sum mpjpe - f64|={abs(s1[0] - m.sum()):.2e} |sum p_mpjpe - f64|={abs(s1[1] - pm.sum()):.2e} "
          f"(bound {n * 1e-6 * pscale:.2e})")
    assert s1[2] == n
    assert abs(s1[0] - m.sum()) < n * 1e-6 * pscale and abs(s1[1] - pm.sum()) < n * 1e-6 * pscale
    sg = torch.zeros(G, 3, dtype=torch.float64, device=dev())
    outg = D.sample(model, xd, md, None, betas(), seed=seed, **kw, targets=tgt.to(dev()), sums=sg, groups=ids.to(dev()))
    assert torch.equal(outg, keyed)
    sg = sg.cpu().numpy()
    for g in range(G):
        sel = (ids == g).numpy()
        assert sg[g, 2] == sel.sum()
        assert abs(sg[g, 0] - m[sel].sum()) < n * 1e-6 * pscale and abs(sg[g, 1] - pm[sel].sum()) < n * 1e-6 * pscale


# --------------------------------------------------------------------------- 2. 70 steps at L = 16: step table, 70 x 16 tembs
@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["tcx", "tcg"])
def test_deep_long_schedule(engine):
    """The `_x_steps` form of test_multi_step_probe at L = 16 on a 70-step permuted schedule (device step table, a 70 x 16
    time-embedding table), with a partial key mask: within AMP a T_active x the readout bound of ref_loop, and the same
    schedule with every t shifted by one outside it."""
    adj, model, sd = _diff((96, 4, 5, 16))
    model = model.to(dev()).set_engine(engine)
    mask = _mask()
    den = _den(engine, sd, adj, 16, 4, mask)
    ts, alpha, every, n = _sched_70(), 0.1, 10, 40
    x = _poses(n, 5, seed=51)
    xr = x if engine == "tcg" else x.double()
    steps, n_act = _x_steps(ts, alpha, every)
    out = D.sample(model, x.to(dev()), mask.to(dev()), None, betas(), steps=steps).cpu()
    ref = ref_loop(xr, steps, den)
    ref1 = ref_loop(xr, _x_steps([v + 1 for v in ts], alpha, every)[0], den)
    scale = max(1.0, ref.abs().max().item())
    bound = AMP * alpha * n_act * _tol(engine, scale, n)[0]
    st, st1 = _stats(out, ref), _stats(out, ref1)
    print(f"deep70 {engine}: max={st[0]:.2e} (bound {bound:.2e})  t+1: max={st1[0]:.2e}")
    assert torch.isfinite(out).all()
    assert st[0] < bound and st1[0] > bound


# --------------------------------------------------------------------------- 2. the GCNpose lifter at any (c_in, c_out)
@pytest.mark.gpu
@pytest.mark.parametrize("case", LIFT_CASES, ids=_id)
def test_lifter_shapes(case):
    """forward against float64 (tcg: its emulation and the oracle bound), and lift = [uv | xyz - xyz_root]: the uv columns
    are the input bit for bit, the xyz columns are the engine's own forward output root-centred bit for bit (fused into the
    kernel's store on tcx, the glue kernel elsewhere), and within the forward bound (doubled: two values) of float64."""
    engine, (ci, co) = case
    adj, model, sd = _model(_Lifter, 96, 4, ci, co, 5)
    model = model.to(dev()).set_engine(engine)
    n = TP * n_sm() + 1
    uv, mask = _poses(n, ci, seed=61), _mask()
    ud, md = uv.to(dev()), mask.to(dev())
    out = model(ud, md).cpu()
    assert out.shape == (n, 17, co) and model.forward_engine() == engine
    sd64, adj64 = _f64(sd, adj)
    ref = O.gcnpose_forward(sd64, adj64, 5, 4, uv.double(), mask)
    scale = max(1.0, ref.abs().max().item())
    err = (out.double() - ref).abs().max().item()
    if engine == "tcg":
        e_emu = (out - E.gcnpose_forward_tcg(sd, adj, 5, 4, uv, mask)).abs().max().item()
        print(f"lifter {_id(case)}: |out - emu| = {e_emu:.2e} (bound {TCG_TOL[0] * scale:.2e})  |out - f64| = {err:.2e}")
        assert e_emu < TCG_TOL[0] * scale and err < TCG_ORACLE_TOL * scale
        bound = 2 * TCG_ORACLE_TOL * scale
    else:
        print(f"lifter {_id(case)}: |out - f64| = {err:.2e} (bound {FWD_TOL * scale:.2e})")
        assert err < FWD_TOL * scale
        bound = 2 * FWD_TOL * scale
    lifted = model.lift(ud, md).cpu()
    assert lifted.shape == (n, 17, ci + co)
    assert torch.equal(lifted[:, :, :ci], uv)
    assert torch.equal(lifted[:, :, ci:], out - out[:, :1])
    assert (lifted[:, :, ci:].double() - O.root_centre(ref)).abs().max().item() < bound


# --------------------------------------------------------------------------- 3. dp_noise_fill at any width
@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 3, 4, 8])
def test_noise_fill_any_width(c):
    seed = 0x0123456789ABCDEF + c
    got = D.philox_noise(seed, 2, 37, 3, pose_offset=1000 + c, step_offset=5, c=c, device=dev()).cpu().numpy()
    want = P.noise(seed, 2, 37, 3, c=c, pose_offset=1000 + c, step_offset=5)
    assert got.shape == want.shape == (2, 3 * 37, 17, c)
    _ulp_close(got, want)


# --------------------------------------------------------------------------- 5. more than 2^31 elements in one call
BIG_N, BIG_H, SLICE = 2_600_000, 10, 1000


@pytest.mark.gpu
@pytest.mark.parametrize("engine,mean", [("tcg", True), ("tcg", False), ("tcx", True)])
def test_past_2_31_elements(engine, mean):
    """One keyed eta = 1 step on 2.6 M poses x H = 10 (26 M rows, 2.2e9 elements), kernel-side repeat: the first, a middle
    and the last 1000 poses are bit-identical to a call on those poses alone with pose_offset (keyed results do not
    depend on the split); with the fused mean and evaluation, sums[2] = n and sums[0:2] are pose_error_sums of the
    returned tensor.  Without the mean (tcg) the hypothesis-major output offset itself passes 2^31 elements."""
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev()).eval().set_engine(engine)
    n, H = BIG_N, BIG_H
    assert n * H * 17 * 5 > 2 ** 31
    steps = (D._lib.DpStep * 1)(D.ddim_steps(betas(), [0, 12], 1.0)[0])      # c1 > 0: the step draws noise
    assert steps[0].c1 > 0
    x = _poses(n, 5, seed=71).to(dev())
    seed = 0xB16B00B5
    kw = dict(n_hyp=H, repeat_input=True, mean_over_hyp=mean, steps=steps, seed=seed)
    ev = {}
    if mean:
        tgt = _targets(n, seed=72).to(dev())
        ev = dict(targets=tgt, sums=torch.zeros(3, dtype=torch.float64, device=dev()))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = D.sample(model, x, None, None, betas(), **kw, **ev)
    torch.cuda.synchronize()
    print(f"past 2^31 {engine} mean={mean}: {n} poses x {H} in {time.perf_counter() - t0:.2f} s")
    assert out.shape == ((n if mean else n * H), 17, 5)
    view = out if mean else out.view(H, n, 17, 5)
    for lo in (0, n // 2 - SLICE // 2, n - SLICE):
        part = D.sample(model, x[lo:lo + SLICE], None, None, betas(), pose_offset=lo, **kw)
        want = view[lo:lo + SLICE] if mean else view[:, lo:lo + SLICE].reshape(H * SLICE, 17, 5)
        assert torch.equal(part, want), f"{engine}: poses {lo}..{lo + SLICE} differ from a call on them alone"
    assert torch.isfinite(view[-1]).all()
    if mean:
        s = ev["sums"].cpu().numpy()
        ref, _ = D.pose_error_sums(out, tgt)
        assert s[2] == n
        np.testing.assert_allclose(s[:2], ref.cpu().numpy()[:2], rtol=1e-9)
