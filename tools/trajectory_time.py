"""Cost of storing the DDIM trajectory from inside the sampler launch, on one GPU (python tools/trajectory_time.py [--out FILE]).

Records the card, its power limit and max SM clock, then measures with CUDA events (arms alternated, 3 repeats, each
timed as in tools/noise_time.py):
  1. configs[2] (1024 poses x H=5 x T=2, eta=1, keyed, kernel-side repeat, fused hypothesis mean) and the bench `sweep`
     shape (16384 x H=10 x T=50, same options): sample() without and with xs_out= / x0_out= (preallocated);
  2. generalized_steps(return_all=True) on 1024 poses at T=2 and T=50 (keyed, eta=1) against the per-step path it
     replaces, emulated with public calls: per step one single-step sample(steps=[step k], step_offset=k) and one forward
     call whose eps gives x0 = (x_t - eps sqrt(1 - abar_t)) / sqrt(abar_t).
Both arms of 2 are also compared: their xs must agree bit for bit, and the largest |x0 difference| is recorded (the old
path's x0 came from a separate forward call, on the default engine the split-precision one).
Prints one JSON object (and writes it to --out when given).
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

import diffpose_nw_b200 as D  # noqa: E402
from diffpose_nw_b200 import _lib  # noqa: E402
from noise_time import card, timed  # noqa: E402
from oracle import diffpose_oracle as O  # noqa: E402


def per_step_return_all(model, x, seq, b, seed):
    """generalized_steps(return_all=True) as it was before the trajectory was stored by the kernel: 2 T launches."""
    steps = D.ddim_steps(b, seq, 1.0)
    xs, x0_preds = [x], []
    for k in range(len(steps)):
        one = (_lib.DpStep * 1)(steps[k])
        xt = xs[-1]
        nxt = D.sample(model, xt, None, None, b, steps=one, seed=seed, step_offset=k)
        et = model(xt, None, torch.full((xt.shape[0],), steps[k].t, device=xt.device), 0)
        x0_preds.append((xt - et * steps[k].sqrt_1m_at) / steps[k].sqrt_at)
        xs.append(nxt)
    return xs, x0_preds


def spread(v):
    return {"ms_per_call": v, "min": min(v), "max": max(v), "spread_pct": 100 * (max(v) - min(v)) / min(v)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result to this file")
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev).eval()
    res = {"card": card(), "engine": model.engine(), "forward_engine": model.forward_engine(), "torch": torch.__version__}
    print("card:", res["card"], flush=True)
    b51 = torch.from_numpy(D.get_beta_schedule("linear", beta_start=1e-4, beta_end=1e-3, num_diffusion_timesteps=51)).float()

    # ---- 1. sample() with and without the trajectory
    shapes = {"configs2_1024xH5xT2": (1024, 5, [0, 6]), "sweep_16384xH10xT50": (16384, 10, list(range(50)))}
    res["sample"] = {}
    for name, (B, H, seq) in shapes.items():
        T = len(seq)
        x = O.synthetic_poses(B, seed=1).to(dev)
        steps = D.ddim_steps(b51, seq, 1.0)
        kw = dict(eta=1.0, n_hyp=H, repeat_input=True, mean_over_hyp=True, steps=steps, seed=1234)
        xs_out = torch.empty(T, B * H, 17, 5, device=dev)
        x0_out = torch.empty_like(xs_out)
        arms = {
            "plain": lambda: D.sample(model, x, None, None, b51, **kw),
            "trajectory": lambda: D.sample(model, x, None, None, b51, xs_out=xs_out, x0_out=x0_out, **kw),
        }
        same = torch.equal(arms["plain"](), arms["trajectory"]())
        runs = {a: [] for a in arms}
        for rep in range(args.repeats):
            for a in (list(arms) if rep % 2 == 0 else list(reversed(list(arms)))):
                ms, n = timed(arms[a])
                runs[a].append(ms)
                print(f"{name} {a}: {ms:.4f} ms/call over {n} calls", flush=True)
        r = {a: spread(v) for a, v in runs.items()}
        r["x_out_bit_identical"] = same
        r["trajectory_bytes_per_call"] = 2 * xs_out.numel() * 4
        r["cost_pct_min_to_min"] = 100 * (r["trajectory"]["min"] / r["plain"]["min"] - 1)
        res["sample"][name] = r
        del xs_out, x0_out

    # ---- 2. generalized_steps(return_all=True): one launch against 2 T launches
    res["return_all"] = {}
    B = 1024
    x = O.synthetic_poses(B, seed=2).to(dev)
    for T in (2, 50):
        seq = list(range(0, 50, 50 // T))[:T]
        arms = {
            "per_step_2T_launches": lambda: per_step_return_all(model, x, seq, b51, 7),
            "one_launch": lambda: D.generalized_steps(x, None, seq, model, b51, eta=1.0, seed=7, return_all=True),
        }
        old, new = arms["per_step_2T_launches"](), arms["one_launch"]()
        xs_same = all(torch.equal(a, b) for a, b in zip(old[0], new[0]))
        x0_diff = max((a - b).abs().max().item() for a, b in zip(old[1], new[1]))
        runs = {a: [] for a in arms}
        for rep in range(args.repeats):
            for a in (list(arms) if rep % 2 == 0 else list(reversed(list(arms)))):
                ms, n = timed(arms[a], min_calls=50)
                runs[a].append(ms)
                print(f"return_all 1024 poses T={T} {a}: {ms:.4f} ms/call over {n} calls", flush=True)
        r = {a: spread(v) for a, v in runs.items()}
        r["xs_bit_identical"] = xs_same
        r["x0_max_abs_diff_old_vs_new"] = x0_diff
        r["speedup_min_to_min"] = r["per_step_2T_launches"]["min"] / r["one_launch"]["min"]
        res["return_all"][f"1024xT{T}"] = r
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
