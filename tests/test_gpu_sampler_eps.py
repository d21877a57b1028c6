"""The sampler kernels' eps, read out undamped through probe steps.

A DDIM step reaches x_T only through `c2 - sqrt(abar_next) sqrt(1 - abar_t) / sqrt(abar_t)`, 0.01 ... 0.04 for the evaluation
schedules, so a comparison of x_T cannot see an eps error below ~2e-2.  Every engine applies a step's scalars literally, with
no FMA contraction (csrc/dp_tc2.cu, dp_tcx.cu, dp_simt.cu):

    x0 = (x - eps * sqrt_1m_at) / sqrt_at;   x' = sqrt_an * x0 (+ c1 * z) + c2 * eps

so a hand-made `DpStep` turns the sampler into a readout of what it computes:
    DpStep(t, 1, 0, 0, 0, 1)   -> eps(x, t), bit for bit;
    DpStep(t, 1, 0, 0, 1, 1)   -> z + eps (a wrong noise row is an O(1) error);
    DpStep(t, 1, 0, 1, 0, a)   -> x + a * eps (several steps, each step's eps weighted by a instead of ~0.01).
These run the sampler-only code paths -- the per-(step, layer) time-embedding blocks of tcg, the step table and its cache,
the rotated step loop, the device step table past 64 steps, the hypothesis remaps and the fused evaluation tail -- with the
eps error in full view, and compare it with the fp32 oracle (fp32, tcx) or the rounding-point emulation (tcg).

Each comparison also measures the distance to two deliberately wrong references (the denoiser at t+1, and a 1 % error on
head 0 of one layer's v bias) and asserts that the bound rejects them: the tests show they can fail.
"""
import copy

import numpy as np
import pytest
import torch

import diffpose_nw_b200 as D
from diffpose_nw_b200 import _lib
from oracle import diffpose_oracle as O
from oracle import tc_emulation as E
from _cases import betas, build_diff, mask_for, t

torch.set_grad_enabled(False)

TP = 7                       # tcg tile height in poses (model.last_launch()[3])
FWD_TOL = 2e-5               # fp32 / tcx eps against the oracle, x max(1, |ref|max) (DESIGN.md 5, the forward bound)
# tcg eps against its rounding-point emulation, x max(1, |emu|max): (max, RMS, largest |mean over poses and joints| of
# one output channel).  Measured on a B200 (test_eps_readout, 1037 poses, t in {0, 1, 6, 12, 25, 50}, golden weights
# A / B / D; worst over t and cases: 8.6e-4, 1.07e-4, 2.4e-6), so the margins are 2.3x, 1.9x, 4.1x.  The channel mean of
# pure rounding noise shrinks as 1 / sqrt(poses x joints); over a few poses its bound is 4 RMS bounds / sqrt(17 n) instead.
TCG_TOL = (2e-3, 2e-4, 1e-5)
TCG_ORACLE_TOL = {"A": 3e-3, "B": 3e-2, "D": 3e-2}       # tcg against the fp32 oracle (the forward tcg tests' bounds)
PROBE_T = (0, 1, 6, 12, 25, 50)
BIAS_KEY = "atten_layers.2.self_attn.linears.2.bias"    # v projection of layer 2; head 0 = channels 0 .. d_k - 1


def dev():
    return torch.device("cuda:0")


def n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


# --------------------------------------------------------------------------- helpers
def probe_steps(ts, sqrt_an=0.0, c1=0.0, c2=1.0):
    """DpStep array with sqrt_at = 1, sqrt_1m_at = 0: x0 = x, x' = sqrt_an * x (+ c1 * z) + c2 * eps(x, t) per step."""
    arr = (_lib.DpStep * len(ts))()
    for k, tv in enumerate(ts):
        arr[k] = _lib.DpStep(float(tv), 1.0, 0.0, float(sqrt_an), float(c1), float(c2))
    return arr


def ref_loop(x, steps, eps_fn, noise=None):
    """The kernels' step update in fp32 torch, same operation order.  eps_fn(x, t [n]) -> eps; noise [T, n, 17, c]."""
    for k, st in enumerate(steps):
        et = eps_fn(x, torch.full((x.shape[0],), st.t))
        x0 = (x - et * st.sqrt_1m_at) / st.sqrt_at
        nx = st.sqrt_an * x0
        if noise is not None:
            nx = nx + st.c1 * noise[k]
        x = nx + st.c2 * et
    return x


def _den(sd, adj, n_layer, mask, emulate):
    if emulate:
        return lambda x, tt: E.gcndiff_forward_tcg(sd, adj, n_layer, 4, x, mask, tt, p16=True, temb_in_gc2=True)
    return lambda x, tt: O.gcndiff_forward(sd, adj, n_layer, 4, x, mask, tt)


def _stats(out, ref):
    d = (out.cpu() - ref).double()
    return d.abs().max().item(), d.pow(2).mean().sqrt().item(), d.mean(dim=(0, 1)).abs().max().item()


def _outside(st, tol):
    return any(s > b for s, b in zip(st, tol))


def _tol(engine, scale, n_pose):
    """(max, RMS, channel-mean) bounds for n_pose distinct poses; fp32 / tcx bound the maximum only."""
    if engine != "tcg":
        return FWD_TOL * scale, float("inf"), float("inf")
    return TCG_TOL[0] * scale, TCG_TOL[1] * scale, max(TCG_TOL[2], 4 * TCG_TOL[1] / (17 * n_pose) ** 0.5) * scale


def _seq_mean(v, n_hyp):
    """Hypothesis mean as the kernels form it: running fp32 sum over h in order, then one division by H."""
    v = v.reshape(n_hyp, -1, *v.shape[1:])
    acc = v[0].clone()
    for h in range(1, n_hyp):
        acc = acc + v[h]
    return acc / n_hyp


def _bias_error(sd, n_head=4):
    sd = dict(sd)
    b = sd[BIAS_KEY].clone()
    dk = b.numel() // n_head
    b[:dk] *= 1.01
    sd[BIAS_KEY] = b
    return sd


def _pool(n, seed):
    return O.synthetic_poses(n, seed=seed)


_REF = {}


def _cached(key, fn):
    if key not in _REF:
        _REF[key] = fn()
    return _REF[key]


# --------------------------------------------------------------------------- 1. the reference loop is pinned (CPU)
@pytest.mark.parametrize("tag", ["B", "D"])
def test_ref_loop_reproduces_oracle_sampler(golden, tag):
    """ref_loop fed the real DDIM scalars reproduces O.ddim_sample and the reference's golden x_T bit for bit, and a probe
    step returns the oracle's eps bit for bit: the restatement used as the GPU tests' reference is the sampler itself."""
    cfg, adj, _, sd = build_diff(tag, golden)
    x, mask = t(golden, f"{tag}.x"), mask_for(tag, golden)
    seq, eta, noise = golden[f"{tag}.seq"].tolist(), float(golden[f"{tag}.eta"]), t(golden, f"{tag}.noise")
    den = _den(sd, adj, 5, mask, False)
    out = ref_loop(x, D.ddim_steps(betas(), seq, eta), den, noise)
    want = O.ddim_sample(x, mask, seq, lambda a, m, tt: O.gcndiff_forward(sd, adj, 5, 4, a, m, tt), betas(), eta=eta,
                         noise=noise)[0][-1]
    assert torch.equal(out, want)
    assert torch.equal(out, t(golden, f"{tag}.x_final"))
    for tv in (0, 17, 50):
        eps = den(x, torch.full((x.shape[0],), float(tv)))
        assert torch.equal(ref_loop(x, probe_steps([tv]), den), eps)
    z = torch.randn(1, *x.shape, generator=torch.Generator().manual_seed(1))
    assert torch.equal(ref_loop(x, probe_steps([9], c1=1.0), den, z), z[0] + den(x, torch.full((x.shape[0],), 9.0)))


# --------------------------------------------------------------------------- 2./3. eps readout per engine, with power checks
@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["fp32", "tcx", "tcg"])
@pytest.mark.parametrize("tag", ["A", "B", "D"])
def test_eps_readout(golden, tag, engine):
    """eps(x, t) read through one probe step on 7 S + 1 poses (S = SM count: one full wave of 7-pose tiles plus one pose),
    t in {0, 1, 6, 12, 25, 50}, golden weights A (default init), B (perturbed, partial key mask), D (perturbed).

    fp32 / tcx: within 2e-5 max(1, |ref|max) of the oracle, and within 1e-6 of the same engine's forward call (reported:
    bitwise or not).  tcg: max, RMS and largest per-channel mean of (kernel - emulation) within TCG_TOL x max(1, |emu|max),
    and within the forward tcg bound of the oracle.  Power: the same statistics against the reference evaluated at t+1 and
    against the reference with 1 % on head 0 of BIAS_KEY must fall outside the bound."""
    cfg, adj, model, sd = build_diff(tag, golden)
    model = model.to(dev()).set_engine(engine)
    mask = mask_for(tag, golden)
    n = TP * n_sm() + 1
    x = _pool(n, seed=101)
    emulate = engine == "tcg"
    sd_bad = _bias_error(sd)
    worst = [0.0, 0.0, 0.0]
    for tv in PROBE_T:
        out = D.sample(model, x.to(dev()), mask.to(dev()), None, betas(), steps=probe_steps([tv])).cpu()
        assert model.engine() == engine
        tt = torch.full((n,), float(tv))
        ref = _cached(("eps", tag, emulate, tv, n), lambda: _den(sd, adj, 5, mask, emulate)(x, tt))
        ref1 = _cached(("eps", tag, emulate, tv + 1, n), lambda: _den(sd, adj, 5, mask, emulate)(x, tt + 1))
        refw = _cached(("bias", tag, emulate, tv, n), lambda: _den(sd_bad, adj, 5, mask, emulate)(x, tt))
        scale = max(1.0, ref.abs().max().item())
        tol = _tol(engine, scale, n)
        st, st1, stw = _stats(out, ref), _stats(out, ref1), _stats(out, refw)
        print(f"eps {engine} {tag} t={tv}: scale={scale:.2f}  vs {'emu' if emulate else 'oracle'} max/rms/chmean="
              f"{st[0]:.2e}/{st[1]:.2e}/{st[2]:.2e}  t+1: {st1[0]:.2e}/{st1[1]:.2e}/{st1[2]:.2e}  "
              f"1% v-bias: {stw[0]:.2e}/{stw[1]:.2e}/{stw[2]:.2e}")
        worst = [max(w, s / scale) for w, s in zip(worst, st)]
        assert all(s < b for s, b in zip(st, tol)), f"{engine} {tag} t={tv}: eps off its reference {st} (bound {tol})"
        assert _outside(st1, tol), f"{engine} {tag} t={tv}: the bound cannot tell t from t+1"
        assert _outside(stw, tol), f"{engine} {tag} t={tv}: the bound cannot see a 1 % error on one head's v bias"
        if engine != "tcg":
            assert st1[0] > 4 * tol[0] and stw[0] > 4 * tol[0], f"{engine} {tag} t={tv}: power margin below 4x"
            fwd = model(x.to(dev()), mask.to(dev()), tt.to(dev()), 0).cpu()
            same = torch.equal(fwd, out)
            print(f"   {engine} sampler eps vs forward: max|d|={(fwd - out).abs().max().item():.2e} bitwise={same}")
            assert (fwd - out).abs().max().item() < 1e-6 * scale
        else:
            ro = _cached(("eps", tag, False, tv, n), lambda: _den(sd, adj, 5, mask, False)(x, tt))
            e_or = (out - ro).abs().max().item()
            print(f"   tcg vs oracle: max={e_or:.2e} (bound {TCG_ORACLE_TOL[tag] * scale:.2e})")
            assert e_or < TCG_ORACLE_TOL[tag] * scale
    print(f"eps {engine} {tag}: worst max/rms/chmean over t, relative to scale = {worst[0]:.2e}/{worst[1]:.2e}/{worst[2]:.2e}")


# --------------------------------------------------------------------------- 4. tile and CTA geometry
def _geometry_model(golden, engine, masked):
    cfg, adj, model, sd = build_diff("B", golden)
    mask = mask_for("B", golden) if masked else None
    return adj, model.to(dev()).set_engine(engine), sd, mask


def _pool_ref(golden, engine, masked, tv, n):
    emulate = engine == "tcg"

    def make():
        cfg, adj, _, sd = build_diff("B", golden)
        mask = mask_for("B", golden) if masked else None
        return _den(sd, adj, 5, mask, emulate)(_pool(n, seed=202), torch.full((n,), float(tv)))
    return _cached(("pool", emulate, masked, tv, n), make)


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("engine", ["fp32", "tcx", "tcg"])
def test_eps_readout_row_counts(golden, engine, masked):
    """Row counts around the tile (7 poses) and the first wave (7 S): every pose's readout is bitwise equal to its readout
    in a call with the rows permuted, and within the engine's bound of its reference."""
    S = n_sm()
    rows = [1, TP - 1, TP, TP + 1, TP * S - 1, TP * S, TP * S + 1, 3 * TP * S + 5]
    tv = 12
    adj, model, sd, mask = _geometry_model(golden, engine, masked)
    pool = _pool(rows[-1], seed=202)
    ref = _pool_ref(golden, engine, masked, tv, rows[-1])
    scale = max(1.0, ref.abs().max().item())      # of the weights, not of the first n poses
    md = mask.to(dev()) if mask is not None else None
    g = torch.Generator().manual_seed(3)
    for n in rows:
        x = pool[:n].to(dev())
        out = D.sample(model, x, md, None, betas(), steps=probe_steps([tv]))
        if engine == "tcg":
            assert model.last_launch()[3] == TP
        perm = torch.randperm(n, generator=g).to(dev())
        outp = D.sample(model, x[perm].contiguous(), md, None, betas(), steps=probe_steps([tv]))
        assert torch.equal(outp, out[perm]), f"{engine} n={n}: a pose's eps depends on its slot or tile"
        st, tol = _stats(out, ref[:n]), _tol(engine, scale, n)
        print(f"rows {engine} masked={masked} n={n}: max/rms/chmean={st[0]:.2e}/{st[1]:.2e}/{st[2]:.2e}")
        assert all(s < b for s, b in zip(st, tol)), f"{engine} n={n}: {st} (bound {tol})"


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["fp32", "tcx", "tcg"])
def test_hypotheses_noise_rows_and_mean(golden, engine):
    """Probe step z + eps (c1 = 1, host noise) with H hypotheses: n_hyp in {2, 3, 7, 10}, n_pose in {1, S-1, S, S+1, 2S+3},
    kernel-side repeat on and off, fused hypothesis mean on and off.  Row h n_pose + b must hold z[h n_pose + b] + eps(x_b)
    (a wrong noise row or input row is an O(1) error), the fused mean must be bit-identical to the in-order mean of the
    unfused output, and both must be within the engine's bound of the reference (z + eps_ref, summed over h, divided by H)."""
    S = n_sm()
    tv = 25
    n_max = 2 * S + 3
    adj, model, sd, mask = _geometry_model(golden, engine, True)
    md = mask.to(dev())
    pool = _pool(n_max, seed=303)
    eps_ref = _cached(("hyp", engine == "tcg", tv, n_max),
                      lambda: _den(sd, adj, 5, mask, engine == "tcg")(pool, torch.full((n_max,), float(tv))))
    scale = max(1.0, eps_ref.abs().max().item())
    steps = probe_steps([tv], c1=1.0)
    g = torch.Generator().manual_seed(4)
    worst = 0.0
    for H in (2, 3, 7, 10):
        for n in (1, S - 1, S, S + 1, n_max):
            x = pool[:n].to(dev())
            z = torch.randn(1, H * n, 17, 5, generator=g)
            zd = z.to(dev())
            ref = z[0] + eps_ref[:n].repeat(H, 1, 1)
            tol = _tol(engine, scale, n)
            full = D.sample(model, x.repeat(H, 1, 1), md, None, betas(), noise=zd, n_hyp=H, steps=steps)
            full_r = D.sample(model, x, md, None, betas(), noise=zd, n_hyp=H, repeat_input=True, steps=steps)
            assert torch.equal(full, full_r), f"{engine} H={H} n={n}: kernel-side repeat differs from the materialised one"
            st = _stats(full, ref)
            assert all(s < b for s, b in zip(st, tol)), f"{engine} H={H} n={n}: {st} (bound {tol})"
            mean_ref = _seq_mean(ref, H)
            unfused_mean = _seq_mean(full.cpu(), H)
            for rep in (False, True):
                xin = x if rep else x.repeat(H, 1, 1)
                fused = D.sample(model, xin, md, None, betas(), noise=zd, n_hyp=H, repeat_input=rep, mean_over_hyp=True,
                                 steps=steps)
                assert fused.shape == (n, 17, 5)
                assert torch.equal(fused.cpu(), unfused_mean), f"{engine} H={H} n={n} repeat={rep}: fused mean differs"
                stm = _stats(fused, mean_ref)
                assert all(s < b for s, b in zip(stm, tol)), f"{engine} H={H} n={n} repeat={rep}: mean {stm} (bound {tol})"
            worst = max(worst, st[0] / scale)
    print(f"hypotheses {engine}: worst max|z + eps - ref| / scale = {worst:.2e}")


# --------------------------------------------------------------------------- 5. several steps, step / layer indexing, caches
def _depth_model(n_layer):
    adj = D.adj_mx_from_edges()
    torch.manual_seed(5)
    model = D.FusedGCNdiff(adj, O.default_config(num_layer=n_layer))
    sd = O.perturb_state_dict({k: v.detach().clone() for k, v in model.state_dict().items()}, seed=13)
    model.load_state_dict(sd)
    return adj, model.to(dev()), sd


SCHED_5 = [50, 3, 27, 12, 0]


def _sched_70():
    return [int(v) for v in torch.randperm(70, generator=torch.Generator().manual_seed(7))]


def _x_steps(ts, alpha, every):
    """x' = x + alpha eps(x, t) on every `every`-th step, x' = x (c2 = 0) on the others: a long schedule whose error does
    not grow like (1 + alpha Lip(eps))^T, yet a step that reads another step's scalars or time embedding still moves x."""
    steps = probe_steps(ts, sqrt_an=1.0, c2=alpha)
    for k in range(len(ts)):
        if k % every != every - 1:
            steps[k].c2 = 0.0
    return steps, len(ts) // every


def _schedules(n_poses):
    """(t list, alpha, every, poses): 5 distinct unsorted t, every step active (a = 0.5); 70 permuted t -- past 64 steps the
    scalars come from the device step table -- with every 10th step active (a = 0.1)."""
    return ((SCHED_5, 0.5, 1, n_poses), (_sched_70(), 0.1, 10, 40))


AMP = 2.0    # allowance for the eps network's amplification of an input error over the active steps (perturbed weights)


@pytest.mark.gpu
@pytest.mark.parametrize("engine,n_layer", [("fp32", 5), ("tcx", 5), ("tcg", 1), ("tcg", 3), ("tcg", 5)])
def test_multi_step_probe(engine, n_layer):
    """Several probe steps x' = x + a eps(x, t_k) in one launch (the tcg time-embedding blocks are a [step][layer] table),
    against ref_loop on the oracle (fp32, tcx) or the emulation (tcg).  The eps network is not a contraction (perturbed
    weights amplify an input error), so the bound is AMP a T_active x max-bound of the readout; the power check runs the
    same schedule with every t shifted by one, which a table read for the wrong step resembles."""
    adj, model, sd = _depth_model(n_layer)
    model.set_engine(engine)
    emulate = engine == "tcg"
    den = _den(sd, adj, n_layer, None, emulate)
    for ts, alpha, every, n in _schedules(TP * n_sm() + 1):
        x = _pool(n, seed=404)
        steps, n_act = _x_steps(ts, alpha, every)
        out = D.sample(model, x.to(dev()), None, None, betas(), steps=steps)
        ref = _cached(("multi", emulate, n_layer, len(ts), n), lambda: ref_loop(x, steps, den))
        scale = max(1.0, ref.abs().max().item())
        tol = (AMP * alpha * n_act * _tol(engine, scale, n)[0], float("inf"), float("inf"))
        st = _stats(out, ref)
        ref1 = _cached(("multi+1", emulate, n_layer, len(ts), n), lambda: ref_loop(x, _x_steps([v + 1 for v in ts], alpha, every)[0], den))
        st1 = _stats(out, ref1)
        print(f"multi {engine} L={n_layer} T={len(ts)} active={n_act} a={alpha}: max/rms/chmean={st[0]:.2e}/{st[1]:.2e}/"
              f"{st[2]:.2e}  t+1: {st1[0]:.2e}/{st1[1]:.2e}/{st1[2]:.2e}  (bound {tol[0]:.2e}, scale {scale:.2f})")
        assert torch.isfinite(out).all()
        assert st[0] < tol[0], f"{engine} L={n_layer} T={len(ts)}: {st} (bound {tol})"
        assert st1[0] > tol[0]


@pytest.mark.gpu
def test_schedule_caches_across_calls():
    """The time-embedding table and its tcg blocks are cached on the handle, keyed on the steps' t; the > 64-step table on
    the schedule.  S1, then S2 (same length, other t), a forward call, S1 again, then tcg -> tcx -> tcg on S1 -- for a
    short and a long schedule: each result is bit-identical to a run on a fresh handle and within bound of ref_loop."""
    adj, model, sd = _depth_model(5)
    n = 2 * TP * n_sm() + 3
    x = _pool(n, seed=505)
    xd = x.to(dev())
    s2s = {5: [49, 4, 26, 13, 1], 70: [v + 1 for v in _sched_70()]}
    for s1, alpha, every, npo in _schedules(n):
        s2 = s2s[len(s1)]
        xs, xc = xd[:npo], x[:npo]
        plan = [("tcg", s1), ("tcg", s2), ("forward", None), ("tcg", s1), ("tcx", s1), ("tcg", s1)]
        for what, ts in plan:
            if what == "forward":
                model(xd, None, torch.full((n,), 33.0, device=dev()), 0)
                continue
            model.set_engine(what)
            steps, n_act = _x_steps(ts, alpha, every)
            out = D.sample(model, xs, None, None, betas(), steps=steps)
            fresh = D.sample(copy.deepcopy(model), xs, None, None, betas(), steps=steps)
            assert torch.equal(out, fresh), f"{what} T={len(ts)}: a cached table gave another result than a fresh handle"
            emulate = what == "tcg"
            ref = _cached(("cache", emulate, tuple(ts)), lambda: ref_loop(xc, steps, _den(sd, adj, 5, None, emulate)))
            scale = max(1.0, ref.abs().max().item())
            bound = AMP * alpha * n_act * _tol(what, scale, npo)[0]
            st = _stats(out, ref)
            print(f"cache {what} T={len(ts)} t0={ts[0]}: max/rms/chmean={st[0]:.2e}/{st[1]:.2e}/{st[2]:.2e} (bound {bound:.2e})")
            assert st[0] < bound, f"{what} T={len(ts)}: {st} (bound {bound})"


# --------------------------------------------------------------------------- 6. fused evaluation tail against float64
@pytest.mark.gpu
@pytest.mark.parametrize("n_mult", [1, 7])
@pytest.mark.parametrize("kind", ["configs2", "probe"])
@pytest.mark.parametrize("engine", ["fp32", "tcx", "tcg"])
def test_eval_sums_vs_float64(engine, kind, n_mult):
    """sample(..., targets=, sums=) on S and 7 S poses, targets in a camera frame (root near z = 5 m): MPJPE and P-MPJPE
    recomputed in float64 from the tensor the call returned agree with sums[0], sums[1] within n 1e-6 (pose scale), and
    sums[2] == n exactly.  configs2: seq [0, 6], eta 1, host noise, H = 5, kernel-side repeat, fused mean.  probe: one
    probe step, so the evaluated prediction is eps itself (scale ~ 3)."""
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev()).eval().set_engine(engine)
    n = n_mult * n_sm()
    x = _pool(n, seed=606)
    tgt = O.synthetic_targets(x) + torch.tensor([0.1, -0.2, 5.0])
    sums = torch.zeros(3, dtype=torch.float64, device=dev())
    if kind == "configs2":
        H = 5
        noise = torch.randn(2, H * n, 17, 5, generator=torch.Generator().manual_seed(9))
        out = D.sample(model, x.to(dev()), None, [0, 6], betas(), eta=1.0, noise=noise.to(dev()), n_hyp=H,
                       repeat_input=True, mean_over_hyp=True, targets=tgt.to(dev()), sums=sums)
    else:
        out = D.sample(model, x.to(dev()), None, None, betas(), steps=probe_steps([12]), targets=tgt.to(dev()), sums=sums)
    assert out.shape == (n, 17, 5)
    p = out.cpu()[:, :, 2:].double()
    g = tgt.double()
    p, g = p - p[:, :1], g - g[:, :1]
    m = (p - g).norm(dim=-1).mean(dim=-1).sum().item()
    pm = O.p_mpjpe_per_pose(p.numpy(), g.numpy()).sum()
    s = sums.cpu().numpy()
    scale = max(p.abs().max().item(), g.abs().max().item())
    print(f"eval {engine} {kind} n={n}: |sum mpjpe - f64|={abs(s[0] - m):.2e} |sum p_mpjpe - f64|={abs(s[1] - pm):.2e}"
          f" (bound {n * 1e-6 * scale:.2e})")
    assert s[2] == n
    assert abs(s[0] - m) < n * 1e-6 * scale and abs(s[1] - pm) < n * 1e-6 * scale
