"""CPU: host-side mirror of the reference interface (no kernels run here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import diffpose_nw_b200 as D
from diffpose_nw_b200 import _lib
from diffpose_nw_b200.model import _param_order
from oracle import diffpose_oracle as O
from _cases import betas

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_state_dict_layout_matches_reference():
    # SURVEY.md 8a "state_dict layout": names, shapes, count
    torch.manual_seed(0)
    m = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config())
    sd = m.state_dict()
    assert len(sd) == 123 and sum(v.numel() for v in sd.values()) == 1025674
    expect = {
        "gconv_input.weight": (3, 1, 5, 96), "gconv_input.bias": (1, 1, 96),
        "gconv_layers.4.gconv2.gconv.weight": (3, 1, 96, 96), "gconv_layers.0.gconv1.gconv.bias": (1, 1, 96),
        "gconv_layers.2.temb_proj.weight": (96, 384), "gconv_layers.2.temb_proj.bias": (96,),
        "atten_layers.3.self_attn.linears.3.weight": (96, 96), "atten_layers.3.self_attn.linears.0.bias": (96,),
        "atten_layers.0.feed_forward.A_hat": (17, 17), "atten_layers.0.feed_forward.gconv1.fc.weight": (192, 96),
        "atten_layers.0.feed_forward.gconv2.fc.weight": (96, 192), "atten_layers.1.sublayer.1.norm.a_2": (96,),
        "gconv_output.weight": (3, 1, 96, 5), "gconv_output.bias": (1, 1, 5),
        "temb.dense.0.weight": (384, 96), "temb.dense.1.weight": (384, 384), "temb.dense.1.bias": (384,),
    }
    for k, shp in expect.items():
        assert tuple(sd[k].shape) == shp, k
    assert "adj" not in sd                      # adj is a plain attribute in the reference
    assert sorted(_param_order(5, True)) == sorted(sd.keys())
    # seeded init reproduces the reference constructor (SURVEY.md 8c known answer)
    assert abs(sum(v.double().sum().item() for v in sd.values()) - 1124.303041338549) < 1e-9
    np.testing.assert_allclose(sd["gconv_input.weight"][0, 0, 0, :3].numpy(), [-0.0363363251, -0.0371922664, -0.0080873892], rtol=1e-6)
    # the reference deep-copies one attention block into every layer
    assert torch.equal(sd["atten_layers.0.self_attn.linears.0.weight"], sd["atten_layers.4.self_attn.linears.3.weight"])


def test_gcnpose_layout():
    m = D.FusedGCNpose(D.adj_mx_from_edges(), O.default_config(coords_dim=[2, 3]))
    sd = m.state_dict()
    assert tuple(sd["gconv_input.weight"].shape) == (3, 1, 2, 96) and tuple(sd["gconv_output.weight"].shape) == (3, 1, 96, 3)
    assert not any("temb_proj" in k for k in sd) and "temb.dense.0.weight" in sd
    assert sum(v.numel() for v in sd.values()) == 839432


def test_load_reference_style_checkpoint():
    cfg = O.default_config()
    torch.manual_seed(1)
    src = D.FusedGCNdiff(D.adj_mx_from_edges(), cfg)
    ckpt = [{"module." + k: v.clone() for k, v in src.state_dict().items()}, {}, 3, 100]   # runner's list format
    dst = D.FusedGCNdiff(D.adj_mx_from_edges(), cfg)
    dst.load_state_dict(ckpt[0])
    assert all(torch.equal(a, b) for a, b in zip(src.state_dict().values(), dst.state_dict().values()))
    with pytest.raises(RuntimeError):
        dst.load_state_dict({"bogus": torch.zeros(1)})


def test_ddim_steps_match_reference_scalars(golden):
    for tag in ["A", "A1", "B", "D"]:
        steps = D.ddim_steps(betas(), golden[f"{tag}.seq"].tolist(), float(golden[f"{tag}.eta"]))
        sc = golden[f"{tag}.scalars"]
        assert len(steps) == len(sc)
        for s, row in zip(steps, sc):
            tt, at, an, c1, c2 = row
            assert s.t == tt and s.c1 == np.float32(c1) and s.c2 == np.float32(c2)
            assert s.sqrt_at == np.sqrt(np.float32(at)) and s.sqrt_an == np.sqrt(np.float32(an))
            assert s.sqrt_1m_at == np.sqrt(np.float32(1) - np.float32(at))
    with pytest.raises(RuntimeError):
        D.ddim_steps(betas(), range(0, 500, 10), 0.0)       # argv default 500 would index past the 51 betas


def test_sequences_and_schedules(golden):
    assert D.make_seq("uniform", 24, 2) == [0, 12] and D.make_seq("uniform", 50, 50) == list(range(50))
    assert D.make_seq("quad", 24, 2) == O.eval_sequence("quad", 24, 2)
    with pytest.raises(NotImplementedError):
        D.make_seq("cosine", 24, 2)
    for kind in ["linear", "quad", "const", "jsd", "sigmoid"]:
        assert np.array_equal(D.get_beta_schedule(kind, beta_start=1e-4, beta_end=1e-3, num_diffusion_timesteps=51), golden[f"betas_{kind}"])
    with pytest.raises(NotImplementedError):
        D.get_beta_schedule("cosine", beta_start=1e-4, beta_end=1e-3, num_diffusion_timesteps=51)


def test_no_cpu_fallback():
    m = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config(hid_dim=32, num_layer=1, n_head=2))
    x = O.synthetic_poses(2)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m(x, None, torch.zeros(2), 0)
    with pytest.raises(RuntimeError, match="CUDA only"):
        D.generalized_steps(x, None, [0, 12], m, betas(), eta=0.0)
    with pytest.raises(RuntimeError, match="FusedGCNdiff"):
        D.generalized_steps(x, None, [0, 12], torch.nn.Linear(1, 1), betas())
    with pytest.raises(RuntimeError, match="CUDA only"):
        D.mpjpe(torch.zeros(1, 17, 3), torch.zeros(1, 17, 3))


def test_shard_range_partitions():
    for n in [0, 1, 7, 1024, 1000003]:
        for w in [1, 2, 3, 8]:
            spans = [D.shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1


def test_abi_library_exports_header_symbols():
    """The C-ABI library loads without a GPU and exports every function include/diffpose_b200.h (product ABI) and
    include/diffpose_b200_diag.h (diagnostics, kept apart) declare."""
    def names(fname):
        header = open(os.path.join(ROOT, "include", fname)).read()
        header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
        return set(re.findall(r"\b(dp_[a-z_0-9]+)\s*\(", header))
    product, diag = names("diffpose_b200.h"), names("diffpose_b200_diag.h")
    assert {"dp_create", "dp_pack", "dp_forward", "dp_lift", "dp_sample", "dp_metrics", "dp_destroy", "dp_last_error"} <= product
    assert diag == {"dp_selftest_umma", "dp_selftest_umma_ts", "dp_selftest_cycles", "dp_set_trace"} and not (diag & product)
    declared = product | diag
    assert declared == set(_lib.SIGNATURES), "binding table and headers disagree"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} missing from libdiffpose_b200.so"
    # one entry point per function, every option an argument: the former per-combination variants are not exported
    for name in [f"dp_{fn}_{opt}" for fn in ("sample", "hstream_submit") for opt in ("eval", "keyed")]:
        assert not hasattr(lib, name), f"{name} is still exported"
    lib.dp_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.dp_version()
    assert ctypes.sizeof(_lib.DpStep) == 24
    if not torch.cuda.is_available():
        # without a device the library must fail loudly, not fall back
        _lib.load()
        h = ctypes.c_void_p()
        rc = _lib.load().dp_create(ctypes.byref(h), 17, 5, 5, 96, 5, 4, 1)
        assert rc != 0 and b"CUDA" in _lib.load().dp_last_error()


def test_reference_checkpoint_list_and_ema(tmp_path):
    """runners/diffpose_frame.py:247-258 saves [state_dict (module.-prefixed), optimizer, epoch, step, ema_shadow];
    load_checkpoint takes states[0] like the reference's evaluation (:131-132) or the EMA shadow on request."""
    import torch
    import diffpose_nw_b200 as D
    from oracle import diffpose_oracle as O
    adj = D.adj_mx_from_edges()
    torch.manual_seed(3)
    src = D.FusedGCNdiff(adj, O.default_config())
    sd = {"module." + k: v.detach().clone() for k, v in src.state_dict().items()}
    shadow = {k: v.detach().clone() * 0.5 for k, v in src.named_parameters()}      # EMAHelper.shadow: no prefix
    path = tmp_path / "ckpt.pth"
    torch.save([sd, {"state": {}}, 7, 1234, shadow], path)
    torch.manual_seed(4)
    dst = D.FusedGCNdiff(adj, O.default_config())
    assert dst.load_checkpoint(str(path)) == (7, 1234)
    for k, v in src.state_dict().items():
        assert torch.equal(dst.state_dict()[k], v)
    dst.load_checkpoint(str(path), use_ema=True)
    for k, v in src.named_parameters():
        assert torch.equal(dict(dst.named_parameters())[k], v * 0.5)
    with pytest.raises(RuntimeError, match="no EMA shadow"):
        dst.load_checkpoint([sd, {}, 1, 2], use_ema=True)


def test_step_scalars_are_cached_per_schedule():
    """generalized_steps is called per batch with the same betas / seq / eta: the step scalars are derived once
    (no device->host copy of betas per call), and an in-place change of the schedule is noticed."""
    from diffpose_nw_b200 import sampler as S
    b = torch.from_numpy(S.get_beta_schedule("linear", beta_start=1e-4, beta_end=1e-3, num_diffusion_timesteps=51)).float()
    s1 = S.cached_ddim_steps(b, range(0, 24, 12), 0.0)
    s2 = S.cached_ddim_steps(b, [0, 12], 0)
    assert s1 is s2 and len(s1) == 2
    ref = S.ddim_steps(b, [0, 12], 0.0)
    assert all(abs(getattr(s1[k], f) - getattr(ref[k], f)) == 0 for k in range(2) for f in ("t", "sqrt_at", "sqrt_an", "c1", "c2"))
    assert S.cached_ddim_steps(b, [0, 12], 1.0) is not s1
    b.mul_(1.5)
    s3 = S.cached_ddim_steps(b, [0, 12], 0.0)
    assert s3 is not s1 and s3[0].sqrt_at != s1[0].sqrt_at


def test_ema_helper_and_copies_keep_no_stale_state():
    """The reference's EMAHelper.ema() writes parameters through `param.data.copy_` (models/ema.py:27-29), which bumps no
    autograd version counter -- so the package ships an EMAHelper that calls repack() itself.  Also: deepcopy / pickling a
    module must not share or carry the native handle (ADVICE r1)."""
    import copy
    import pickle
    adj = D.adj_mx_from_edges()
    torch.manual_seed(5)
    m = D.FusedGCNdiff(adj, O.default_config())
    p = m.atten_layers[2].self_attn.linears[1].weight
    v0 = p._version
    p.data.copy_(p.data * 2)                       # the idiom in question: invisible to _version
    assert p._version == v0
    ema = D.EMAHelper(mu=0.5)
    ema.register(m)
    with torch.no_grad():
        for q in m.parameters():
            q.add_(1.0)
    ema.update(m)                                   # shadow = 0.5 * (w + 1) + 0.5 * w
    m._packed_version = ("sentinel",)               # pretend the weights are packed
    ema.ema(m)
    assert m._packed_version is None, "EMAHelper.ema() must invalidate the packed device copy"
    want = p.detach().clone()
    m2 = ema.ema_copy(torch.nn.DataParallel(m))     # with a GPU visible, the module may now live on cuda:0
    assert isinstance(m2, torch.nn.DataParallel) and torch.equal(m2.module.atten_layers[2].self_attn.linears[1].weight.cpu(), want)
    assert set(ema.state_dict()) == {k for k, _ in m.named_parameters()}
    m._handle = "native pointer"
    c = copy.deepcopy(m)
    assert c._handle is None and c._packed_version is None and m._handle == "native pointer"
    assert torch.equal(c.gconv_input.weight, m.gconv_input.weight) and c.gconv_input.weight is not m.gconv_input.weight
    c2 = pickle.loads(pickle.dumps(m))
    assert c2._handle is None and torch.equal(c2.gconv_output.bias, m.gconv_output.bias)
    m._handle = None


def test_engine_names():
    m = D.FusedGCNpose(D.adj_mx_from_edges(), O.default_config(coords_dim=[2, 3]))
    for name in ("auto", "fp32", "tcx", "tcg"):
        m.set_engine(name)
    with pytest.raises(KeyError):
        m.set_engine("tc")                          # the first tensor-core engine is retired


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` runs without a GPU, prints ONE JSON line with the contract's keys, and carries exactly the
    `config` object the GPU arm prints for the same command line (the driver compares them)."""
    import json
    import subprocess
    import sys
    sys.path.insert(0, ROOT)
    import bench
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "poses/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["steps"] == 1 and d["warmup"] == 3
    assert d["config"] == bench.bench_config(bench.WORKLOADS["cpn1024"], 1)[0]
    assert set(d["config"]) == {"workload", "batch", "batch_is", "n_hyp", "T", "eta", "l2"}
    for name, wl in bench.WORKLOADS.items():      # every workload names a BASELINE config and a schedule inside the 51-entry beta table
        assert "configs[" in wl["name"] and max(wl["seq"]) < 51 and wl["batch"] >= 1


def test_bench_dump_outputs_stays_in_budget(tmp_path):
    """`bench.py --dump-outputs`: the files of all ranks together stay within 64 MB (headers included) even for the
    million-pose output of sweep1m; a larger array keeps the same seeded, sorted sample of rows in every run; a small one
    is written whole; names carry the rank suffix only when it is given."""
    import bench
    n = 1_000_000
    x = torch.arange(n, dtype=torch.float32)[:, None, None].expand(n, 17, 5)      # every value of a row is its index
    sums = torch.tensor([1.0, 2.0, 3.0], dtype=torch.float64)

    def written(d):
        return {f: os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)}

    for arrays in ({"x_T": x}, {"x_T": x, "metric_sums": sums}):
        runs = []
        for k in range(2):
            d = str(tmp_path / f"{len(arrays)}_{k}")
            bench.dump_outputs(d, arrays, bench.DUMP_BYTES)
            files = written(d)
            assert set(files) == {name + ".npy" for name in arrays} and sum(files.values()) <= bench.DUMP_BYTES
            runs.append(np.load(os.path.join(d, "x_T.npy")))
        a, b = runs
        assert a.dtype == np.float32 and a.shape[1:] == (17, 5) and 0.9 * bench.DUMP_BYTES / len(arrays) < a.nbytes
        assert np.array_equal(a, b)
        rows = a[:, 0, 0]
        assert (np.diff(rows) > 0).all() and (a == rows[:, None, None]).all()
        if "metric_sums" in arrays:
            s = np.load(os.path.join(str(tmp_path / "2_0"), "metric_sums.npy"))
            assert s.dtype == np.float64 and np.array_equal(s, sums.numpy())
    world = 4
    d = str(tmp_path / "ranks")
    for r in range(world):
        bench.dump_outputs(d, {"x_T": x}, bench.DUMP_BYTES // world, f"_rank{r}")
    files = written(d)
    assert set(files) == {f"x_T_rank{r}.npy" for r in range(world)} and sum(files.values()) <= bench.DUMP_BYTES
    small = torch.randn(1024, 17, 5)
    bench.dump_outputs(str(tmp_path / "small"), {"x_T": small}, bench.DUMP_BYTES)
    assert np.array_equal(np.load(str(tmp_path / "small" / "x_T.npy")), small.numpy())


def test_bench_rejects_bad_arguments(tmp_path):
    """No timed step (--steps 0) and a dump of the reference arm are argument errors, reported before any work."""
    import subprocess
    import sys
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "out")]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=300)
        assert out.returncode == 2 and "error:" in out.stderr and out.stdout == "", (extra, out.stderr[-500:])
    assert os.listdir(tmp_path) == []
