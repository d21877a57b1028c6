"""Multi-hypothesis evaluation against the mean-only fused evaluation, on one GPU
(python tools/hyp_eval_time.py [--out FILE] [--batches N] [--big-batches M] [--repeats R]).

Records the card, its power limit and max SM clock, then measures with CUDA events, arms alternated, R repeats:
  workloads  configs[2] (1024 poses x H=5 x T=2, seq [0, 12], eta=1, keyed noise, kernel-side repeat; N batches, inputs and
             targets rotating through a pool larger than the 126 MB L2) and the configs[3] slice (16384 poses x H=10 x T=50,
             eta=1, keyed; M batches);
  arms       mean_fused        sample(targets=, sums=, mean_over_hyp=True): the hypothesis mean's MPJPE / P-MPJPE, fused
                               into the sampler launch on the default engine (one launch);
             hyp_eval          sample(targets=, hyp_sums=, mean_over_hyp=True): the sampler writes all H rows, then
                               dp_metrics_hyp scores them and writes the mean (two launches);
             metrics_hyp_only  dp_metrics_hyp alone on device-resident hypotheses (the rows one sampler call wrote, so they
                               sit in L2 as they do right after the sampler).
Prints one JSON object (and writes it to --out when given).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import diffpose_nw_b200 as D  # noqa: E402
from diffpose_nw_b200 import _lib  # noqa: E402
from diffpose_nw_b200.metrics import _metrics_hyp  # noqa: E402
from oracle import diffpose_oracle as O  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, n, warm):
    """ms per batch over n batches (CUDA events around the window, after `warm` warm-up batches)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result to this file")
    ap.add_argument("--batches", type=int, default=2000, help="timed batches per arm and repeat, configs[2]")
    ap.add_argument("--big-batches", type=int, default=4, help="timed batches per arm and repeat, configs[3] slice")
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev).eval()
    res = {"card": card(), "engine": model.engine(), "torch": torch.__version__, "repeats": args.repeats}
    print("card:", res["card"], flush=True)
    b51 = torch.from_numpy(D.get_beta_schedule("linear", beta_start=1e-4, beta_end=1e-3, num_diffusion_timesteps=51)).float()
    lib = _lib.load()
    stream = torch.cuda.current_stream(dev).cuda_stream
    flat = torch.zeros(3, device=dev, dtype=torch.float64)
    hs = torch.zeros(8, device=dev, dtype=torch.float64)
    workloads = {
        "configs2_1024xH5xT2_keyed": dict(B=1024, H=5, seq=[0, 12], batches=args.batches, warm=20),
        "configs3_slice_16384xH10xT50_keyed": dict(B=16384, H=10, seq=list(range(50)), batches=args.big_batches, warm=1),
    }
    for name, wl in workloads.items():
        B, H = wl["B"], wl["H"]
        pool_n = max(2, int(126 * 2**20 * 1.1) // (B * 17 * 8 * 4) + 1)     # x [B,17,5] + targets [B,17,3] per batch
        xs = torch.stack([O.synthetic_poses(B, seed=10 + i) for i in range(2)]).to(dev)
        pool_x = xs.repeat(pool_n // 2 + 1, 1, 1, 1)[:pool_n].contiguous()
        pool_t = torch.stack([O.synthetic_targets(xs[i % 2].cpu(), seed=20 + i) for i in range(pool_n)]).to(dev)
        state = {"i": 0}

        def nxt():
            i = state["i"] = (state["i"] + 1) % pool_n
            return pool_x[i], pool_t[i]

        kw = dict(steps=D.ddim_steps(b51, wl["seq"], 1.0), eta=1.0, n_hyp=H, repeat_input=True, mean_over_hyp=True, seed=7)

        def mean_fused():
            x, t = nxt()
            D.sample(model, x, None, None, b51, targets=t, sums=flat, **kw)

        def hyp_eval():
            x, t = nxt()
            D.sample(model, x, None, None, b51, targets=t, hyp_sums=hs, **kw)

        rows = D.sample(model, pool_x[0], None, None, b51, **dict(kw, mean_over_hyp=False))
        t0 = pool_t[0]

        def metrics_hyp_only():
            _metrics_hyp(lib, rows, 5, H, t0, B, None, 1, hs, None, None, stream)

        arms = {"mean_fused": mean_fused, "hyp_eval": hyp_eval, "metrics_hyp_only": metrics_hyp_only}
        runs = {a: [] for a in arms}
        for rep in range(args.repeats):
            for a in (list(arms) if rep % 2 == 0 else list(reversed(list(arms)))):
                n = args.batches if a == "metrics_hyp_only" else wl["batches"]
                ms = timed(arms[a], n, 20 if a == "metrics_hyp_only" else wl["warm"])
                runs[a].append(ms)
                print(f"{name} {a}: {ms:.4f} ms/batch", flush=True)
        r = {a: {"ms_per_batch": v, "min": min(v), "max": max(v)} for a, v in runs.items()}
        r["timed_batches"] = {"sampler_arms": wl["batches"], "metrics_hyp_only": args.batches}
        r["l2"] = f"inputs and targets rotate through {pool_n} batches = {(pool_x.numel() + pool_t.numel()) * 4 / 2**20:.0f} MiB"
        r["hyp_eval_over_mean_fused"] = [h / m - 1.0 for h, m in zip(runs["hyp_eval"], runs["mean_fused"])]
        res[name] = r
        del pool_x, pool_t, rows
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
