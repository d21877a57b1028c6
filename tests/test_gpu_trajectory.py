"""GPU (-m gpu): the DDIM trajectory stored from inside the sampler launch (`sample(xs_out=, x0_out=)`,
`dp_sample_trajectory`, `generalized_steps(return_all=True)`).

xs_out[k] is x_t after step k and x0_out[k] the x0 prediction the update of step k used.  The checks:
  1. update-rule identity: with eps read back through a probe step at (xs[k], t_k), x0_out[k] and xs_out[k] are the
     kernels' update rule evaluated with torch fp32 ops on the device, bit for bit;
  2. one launch equals T single-step launches (keyed, step_offset = k), bit for bit, also on a 70-step table schedule;
  3. hypotheses: the trajectory does not depend on the fused mean, and x_out is the mean of its last step;
  4. oracle parity of every step;
  5. generalized_steps(return_all=True) is one launch, keyed equals materialised noise, and the chunked torch draw scatters
     its per-chunk trajectories into the caller's layout;
  6. offsets past 2^31 elements;
  7. partial buffers and the refused arguments.
Checks 1 and 2 rest on the batch-composition property (DESIGN.md 5): a pose's eps does not depend on which other poses
share its launch, tile or CTA.
"""
import ctypes

import pytest
import torch

import diffpose_nw_b200 as D
from diffpose_nw_b200 import _lib
from oracle import diffpose_oracle as O
from _cases import betas, build_diff, mask_for, t

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

DEV = torch.device("cuda:0")
ENGINES = ["fp32", "tcx", "tcg"]
TP = 7                      # tcg tile height in poses
FP32_TOL = 2e-5             # as tests/test_gpu_parity.py
TC_TOL_X = 1e-3
TCG_EPS_ORACLE_TOL_B = 3e-2   # tcg eps against the fp32 oracle on golden case B (test_eps_readout), x max(1, |eps|max)
_LONG_BETAS = torch.from_numpy(D.get_beta_schedule("linear", beta_start=1e-4, beta_end=2e-2, num_diffusion_timesteps=200)).float()


def n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _model(engine="tcg"):
    torch.manual_seed(0)
    m = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config())
    sd = O.perturb_state_dict({k: v.detach().clone() for k, v in m.state_dict().items()}, seed=21, scale=0.02)
    m.load_state_dict(sd)
    return m.to(DEV).eval().set_engine(engine)


def _poses(n, seed):
    return O.synthetic_poses(n, seed=seed).to(DEV)


def _bufs(T, rows):
    return torch.empty(T, rows, 17, 5, device=DEV), torch.empty(T, rows, 17, 5, device=DEV)


def _probe(ts):
    """sqrt_at = 1, sqrt_1m_at = 0, sqrt_an = 0, c1 = 0, c2 = 1: one step returns eps(x, t) undamped."""
    arr = (_lib.DpStep * len(ts))()
    for k, tv in enumerate(ts):
        arr[k] = _lib.DpStep(float(tv), 1.0, 0.0, 0.0, 0.0, 1.0)
    return arr


def _one(steps, k):
    return (_lib.DpStep * 1)(steps[k])


def _full(like, v):
    return torch.full_like(like, v)


def _seq_mean(v, n_hyp):
    """Hypothesis mean as the kernels form it: running fp32 sum over h in order, then one IEEE division by H (a tensor
    divisor: torch divides by a Python scalar through its reciprocal, which rounds differently)."""
    v = v.reshape(n_hyp, -1, *v.shape[1:])
    acc = v[0].clone()
    for h in range(1, n_hyp):
        acc = acc + v[h]
    return acc / _full(acc, float(n_hyp))


# ------------------------------------------------------------------------------------------- 1. update-rule identity
@pytest.mark.parametrize("engine", ENGINES)
def test_update_rule_identity(golden, engine):
    """x0_out[k] = (xs[k] - eps sqrt_1m_at) / sqrt_at and xs_out[k] = sqrt_an x0 + c1 z + c2 eps, every operation a separate
    IEEE-rounded torch fp32 op on the device, with eps read back through a probe step at (xs[k], t_k) and z from
    philox_noise: keyed eta = 1, T = 4, 7 S + 1 poses, a partial key mask."""
    m = _model(engine)
    mask = mask_for("B", golden).to(DEV)
    n, seed, seq = TP * n_sm() + 1, 31, [0, 6, 12, 18]
    x = _poses(n, 1)
    steps = D.ddim_steps(betas(), seq, 1.0)
    T = len(steps)
    xs_out, x0_out = _bufs(T, n)
    out = D.sample(m, x, mask, seq, betas(), eta=1.0, seed=seed, xs_out=xs_out, x0_out=x0_out)
    assert m.engine() == engine
    assert torch.equal(xs_out[T - 1], out)
    z = D.philox_noise(seed, T, n, device=DEV)
    xk = x
    for k, st in enumerate(steps):
        eps = D.sample(m, xk, mask, None, betas(), steps=_probe([st.t]))
        x0 = (xk - eps * _full(xk, st.sqrt_1m_at)) / _full(xk, st.sqrt_at)
        assert torch.equal(x0_out[k], x0), f"{engine} step {k}: x0 max|d|={(x0_out[k] - x0).abs().max().item():.3e}"
        nx = x0 * _full(xk, st.sqrt_an) + z[k] * _full(xk, st.c1)
        nx = nx + eps * _full(xk, st.c2)
        assert torch.equal(xs_out[k], nx), f"{engine} step {k}: x_t max|d|={(xs_out[k] - nx).abs().max().item():.3e}"
        xk = xs_out[k]


# -------------------------------------------------------------------------------- 2. one launch = T single-step launches
@pytest.mark.parametrize("engine,T", [("fp32", 4), ("tcx", 4), ("tcg", 4), ("tcg", 70), ("fp32", 70)])
def test_one_launch_equals_single_steps(engine, T):
    """The trajectory of one keyed call equals the chain of T single-step keyed calls (step_offset = k), x_t and x0, bit for
    bit; its last step is x_out.  T = 70 runs the full call from the device step table (more than 64 steps)."""
    m = _model(engine)
    n, seed = TP * n_sm() + 1 if T < 64 else 500, 77
    seq, b = ([0, 6, 12, 18], betas()) if T == 4 else (list(range(0, 2 * T, 2)), _LONG_BETAS)
    steps = D.ddim_steps(b, seq, 1.0)
    x = _poses(n, 2)
    xs_out, x0_out = _bufs(T, n)
    out = D.sample(m, x, None, None, b, steps=steps, seed=seed, xs_out=xs_out, x0_out=x0_out)
    assert torch.equal(xs_out[T - 1], out)
    xk = x
    x0_one = torch.empty(1, n, 17, 5, device=DEV)
    for k in range(T):
        nxt = D.sample(m, xk, None, None, b, steps=_one(steps, k), seed=seed, step_offset=k, x0_out=x0_one)
        assert torch.equal(xs_out[k], nxt), f"{engine} T={T} step {k}: max|d|={(xs_out[k] - nxt).abs().max().item():.3e}"
        assert torch.equal(x0_out[k], x0_one[0]), f"{engine} T={T} step {k}: x0 differs"
        xk = nxt


# ------------------------------------------------------------------------------------------------------ 3. hypotheses
@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("n_pose", [10, 7 * 148 + 3])
def test_hypotheses_and_fused_mean(engine, n_pose):
    """n_hyp = 5, kernel-side repeat: the trajectory with mean_over_hyp equals the one without, bit for bit, and x_out is the
    sequential fp32 mean of the last step's hypothesis rows (the order of the fused mean and hyp_mean_kernel)."""
    m = _model(engine)
    H, seq, seed = 5, [0, 6, 12], 5
    T = len(seq)
    x = _poses(n_pose, 3)
    kw = dict(eta=1.0, seed=seed, n_hyp=H, repeat_input=True)
    xs_m, x0_m = _bufs(T, n_pose * H)
    xs_p, x0_p = _bufs(T, n_pose * H)
    mean = D.sample(m, x, None, seq, betas(), mean_over_hyp=True, xs_out=xs_m, x0_out=x0_m, **kw)
    plain = D.sample(m, x, None, seq, betas(), xs_out=xs_p, x0_out=x0_p, **kw)
    assert torch.equal(xs_m, xs_p) and torch.equal(x0_m, x0_p)
    assert torch.equal(xs_p[T - 1], plain)
    assert torch.equal(mean, _seq_mean(xs_m[T - 1], H))
    # the materialised-noise call writes the same trajectory (the unkeyed TRAJ instantiation on tcg)
    nz = D.philox_noise(seed, T, n_pose, H, device=DEV)
    xs_n, x0_n = _bufs(T, n_pose * H)
    D.sample(m, x, None, seq, betas(), eta=1.0, noise=nz, n_hyp=H, repeat_input=True, mean_over_hyp=True, xs_out=xs_n, x0_out=x0_n)
    assert torch.equal(xs_n, xs_m) and torch.equal(x0_n, x0_m)


# ------------------------------------------------------------------------------------------------- 4. oracle parity
@pytest.mark.parametrize("engine", ["fp32", "tcg"])
def test_return_all_vs_oracle(golden, engine):
    """Golden case B (host noise, partial key mask): every xs[k] and x0_preds[k] of generalized_steps(return_all=True)
    against O.ddim_sample.  x0 = (x_t - eps sqrt_1m_at) / sqrt_at carries the engine's eps bound (fp32: FP32_TOL, tcg: the
    tcg eps-vs-oracle bound of test_eps_readout, 3e-2, each x max(1, |eps|max)) times max_k sqrt_1m_at / sqrt_at, plus the
    error x_t already carries into the step divided by min_k sqrt_at.  xs: fp32 FP32_TOL x max(1, |ref|max), tcg TC_TOL_X."""
    cfg, adj, model, sd = build_diff("B", golden)
    model = model.to(DEV).set_engine(engine)
    x, mask = t(golden, "B.x"), mask_for("B", golden)
    seq, eta, noise = golden["B.seq"].tolist(), float(golden["B.eta"]), t(golden, "B.noise")
    den = lambda a, mm, tt: O.gcndiff_forward(sd, adj, 5, 4, a, mm, tt)
    ref_xs, ref_x0 = O.ddim_sample(x, mask, seq, den, betas(), eta=eta, noise=noise)
    xs, x0 = D.generalized_steps(x.to(DEV), mask.to(DEV), seq, model, betas(), eta=eta, noise=noise.to(DEV), return_all=True)
    assert model.engine() == engine
    assert len(xs) == len(ref_xs) and len(x0) == len(ref_x0)
    steps = D.ddim_steps(betas(), seq, eta)
    eps_scale = max(1.0, max(den(a, mask, torch.full((a.shape[0],), st.t)).abs().max().item() for a, st in zip(ref_xs, steps)))
    ratio = max(st.sqrt_1m_at / st.sqrt_at for st in steps)
    min_sat = min(st.sqrt_at for st in steps)
    x_scale = max(1.0, max(a.abs().max().item() for a in ref_xs))
    tol_x = FP32_TOL * x_scale if engine == "fp32" else TC_TOL_X
    tol_x0 = (FP32_TOL if engine == "fp32" else TCG_EPS_ORACLE_TOL_B) * eps_scale * ratio + tol_x / min_sat
    print(f"{engine} bounds: xs {tol_x:.3e}; x0 {FP32_TOL if engine == 'fp32' else TCG_EPS_ORACLE_TOL_B:g} x {eps_scale:.2f} x "
          f"{ratio:.4f} + {tol_x:.1e} / {min_sat:.4f} = {tol_x0:.3e}")
    for k in range(len(ref_xs)):
        e = (xs[k].cpu() - ref_xs[k]).abs().max().item()
        print(f"{engine} xs[{k}]: max|d|={e:.2e}")
        assert e < tol_x
    for k in range(len(ref_x0)):
        e = (x0[k].cpu() - ref_x0[k]).abs().max().item()
        print(f"{engine} x0[{k}]: max|d|={e:.2e}")
        assert e < tol_x0


# ------------------------------------------------------------------------------------- 5. generalized_steps(return_all)
@pytest.mark.parametrize("engine", ENGINES)
def test_return_all_one_launch(engine):
    m = _model(engine)
    seq, seed, n = [0, 6, 12, 18], 9, 300
    x = _poses(n, 4)
    D.generalized_steps(x, None, seq, m, betas(), eta=1.0, seed=seed, return_all=True)      # warm-up: schedule tables
    torch.cuda.synchronize()
    before = _lib.launch_count()
    xs, x0 = D.generalized_steps(x, None, seq, m, betas(), eta=1.0, seed=seed, return_all=True)
    assert _lib.launch_count() - before == 1
    assert len(xs) == len(seq) + 1 and len(x0) == len(seq) and xs[0] is x
    assert torch.equal(xs[-1], D.generalized_steps(x, None, seq, m, betas(), eta=1.0, seed=seed)[0][-1])
    nz = D.philox_noise(seed, len(seq), n, device=DEV)
    xs_m, x0_m = D.generalized_steps(x, None, seq, m, betas(), eta=1.0, noise=nz, return_all=True)
    for a, b in zip(xs + x0, xs_m + x0_m):
        assert torch.equal(a, b)


@pytest.mark.parametrize("mean", [False, True])
def test_chunked_torch_draw_trajectory(monkeypatch, mean):
    """eta > 0 without seed / noise draws with torch in pose chunks: each chunk's trajectory lands in the caller's
    hypothesis-major rows.  The last step equals x_out (or its mean), and step 0's x0 is the update rule at x with eps read
    back through a probe step."""
    m = _model("tcg")
    H, n, seq = 3, 100, [0, 6, 12]
    T = len(seq)
    monkeypatch.setattr(D.sampler, "NOISE_CHUNK_BYTES", T * 17 * 5 * 4 * H * 30)   # 30 poses per chunk: 4 chunks
    x = _poses(n, 5)
    xs_out, x0_out = _bufs(T, n * H)
    before = _lib.launch_count()
    out = D.sample(m, x, None, seq, betas(), eta=1.0, n_hyp=H, repeat_input=True, mean_over_hyp=mean, xs_out=xs_out, x0_out=x0_out)
    torch.cuda.synchronize()
    assert _lib.launch_count() - before >= 4
    assert torch.equal(_seq_mean(xs_out[T - 1], H) if mean else xs_out[T - 1], out)
    st = D.ddim_steps(betas(), seq, 1.0)[0]
    xr = x.repeat(H, 1, 1)
    eps = D.sample(m, xr, None, None, betas(), steps=_probe([st.t]))
    assert torch.equal(x0_out[0], (xr - eps * _full(xr, st.sqrt_1m_at)) / _full(xr, st.sqrt_at))
    xs, x0 = D.generalized_steps(x, None, seq, m, betas(), eta=1.0, return_all=True)
    assert len(xs) == T + 1 and len(x0) == T and torch.isfinite(torch.stack(xs[1:])).all()


# ------------------------------------------------------------------------------------------------- 6. large offsets
def test_trajectory_past_2_31_elements():
    """One keyed tcg call on 400 k poses x 70 steps: each trajectory buffer holds 2.38e9 elements (9.5 GB).  Slices are
    bit-identical to calls on those poses alone with pose_offset, at every step, so offsets past 2^31 are right."""
    m = _model("tcg")
    n, T, seed, SLICE = 400_000, 70, 11, 1000
    steps = D.ddim_steps(_LONG_BETAS, list(range(0, 2 * T, 2)), 1.0)
    x = _poses(n, 6)
    xs_out, x0_out = _bufs(T, n)
    assert xs_out.numel() > 2 ** 31
    out = D.sample(m, x, None, None, _LONG_BETAS, steps=steps, seed=seed, xs_out=xs_out, x0_out=x0_out)
    assert torch.equal(xs_out[T - 1], out)
    for lo in (0, n // 2 + 3, n - SLICE):
        xs_p, x0_p = _bufs(T, SLICE)
        D.sample(m, x[lo:lo + SLICE], None, None, _LONG_BETAS, steps=steps, seed=seed, pose_offset=lo, xs_out=xs_p, x0_out=x0_p)
        assert torch.equal(xs_out[:, lo:lo + SLICE], xs_p), f"slice at {lo}"
        assert torch.equal(x0_out[:, lo:lo + SLICE], x0_p), f"slice at {lo}"


# --------------------------------------------------------------------------------------- 7. partial buffers, refusals
@pytest.mark.parametrize("engine", ENGINES)
def test_partial_buffers(engine):
    m = _model(engine)
    seq, n = [0, 6, 12], 50
    T = len(seq)
    x = _poses(n, 7)
    xs_f, x0_f = _bufs(T, n)
    D.sample(m, x, None, seq, betas(), eta=1.0, seed=3, xs_out=xs_f, x0_out=x0_f)
    xs_only = torch.full((T, n, 17, 5), float("nan"), device=DEV)
    D.sample(m, x, None, seq, betas(), eta=1.0, seed=3, xs_out=xs_only)
    x0_only = torch.full((T, n, 17, 5), float("nan"), device=DEV)
    D.sample(m, x, None, seq, betas(), eta=1.0, seed=3, x0_out=x0_only)
    assert torch.equal(xs_only, xs_f) and torch.equal(x0_only, x0_f)


def test_refusals_before_launch():
    m = _model("tcg")
    seq, n = [0, 6], 20
    x = _poses(n, 8)
    ok = torch.empty(2, n, 17, 5, device=DEV)
    bad = [torch.empty(3, n, 17, 5, device=DEV), torch.empty(2, n + 1, 17, 5, device=DEV),
           torch.empty(2, n, 17, 5, device=DEV, dtype=torch.float64), torch.empty(2, n, 17, 5),
           torch.empty(2, n, 5, 17, device=DEV).transpose(2, 3)]
    D.sample(m, x, None, seq, betas(), eta=1.0, seed=1, xs_out=ok)      # warm-up: schedule tables
    torch.cuda.synchronize()
    before = _lib.launch_count()
    for buf in bad:
        for kw in (dict(xs_out=buf), dict(x0_out=buf), dict(xs_out=ok, x0_out=buf)):
            with pytest.raises(RuntimeError):
                D.sample(m, x, None, seq, betas(), eta=1.0, seed=1, **kw)
    tg = O.synthetic_targets(x.cpu()).to(DEV)
    sums = torch.zeros(3, dtype=torch.float64, device=DEV)
    with pytest.raises(RuntimeError, match="fused evaluation"):
        D.sample(m, x, None, seq, betas(), eta=1.0, seed=1, targets=tg, sums=sums, xs_out=ok)
    assert _lib.launch_count() == before


def test_abi_refusal_leaves_buffers_and_handle():
    """dp_sample_trajectory with both a noise tensor and a key returns DP_ERR_INVALID and writes nothing; the next valid
    call on the same handle gives what sample() gives."""
    m = _model("tcg")
    seq, n, seed = [0, 6, 12], 64, 4
    T = len(seq)
    x = _poses(n, 9)
    want_xs, want_x0 = _bufs(T, n)
    want = D.sample(m, x, None, seq, betas(), eta=1.0, seed=seed, xs_out=want_xs, x0_out=want_x0)
    lib = _lib.load()
    steps = D.ddim_steps(betas(), seq, 1.0)
    nz = D.philox_noise(seed, T, n, device=DEV)
    key = _lib.noise_key(seed)
    out = torch.full((n, 17, 5), -7.0, device=DEV)
    xs_t = torch.full((T, n, 17, 5), -7.0, device=DEV)
    x0_t = torch.full((T, n, 17, 5), -7.0, device=DEV)
    stream = torch.cuda.current_stream(DEV).cuda_stream
    torch.cuda.synchronize()
    before = _lib.launch_count()
    rc = lib.dp_sample_trajectory(m._handle, x.data_ptr(), 0, out.data_ptr(), n, 1, steps, T, nz.data_ptr(), ctypes.byref(key),
                                  None, 0, xs_t.data_ptr(), x0_t.data_ptr(), stream)
    assert rc == -1 and _lib.launch_count() == before
    torch.cuda.synchronize()
    assert (xs_t == -7.0).all() and (x0_t == -7.0).all() and (out == -7.0).all()
    rc = lib.dp_sample_trajectory(m._handle, x.data_ptr(), 0, out.data_ptr(), n, 1, steps, T, None, ctypes.byref(key),
                                  None, 0, xs_t.data_ptr(), x0_t.data_ptr(), stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(out, want) and torch.equal(xs_t, want_xs) and torch.equal(x0_t, want_x0)
    # both pointers NULL: the call is dp_sample
    out2 = torch.empty_like(out)
    rc = lib.dp_sample_trajectory(m._handle, x.data_ptr(), 0, out2.data_ptr(), n, 1, steps, T, None, ctypes.byref(key),
                                  None, 0, None, None, stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(out2, want)
