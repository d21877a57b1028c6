"""Group-keyed (per-action) evaluation against the ungrouped fused evaluation, on one GPU
(python tools/group_eval_time.py [--out FILE] [--batches N] [--repeats R]).

Records the card and its power limit, then measures with CUDA events, arms alternated, R repeats of N batches each:
  workloads  evalloop (1024 poses, H=1, T=2: bench.py's evaluation loop) device-resident and through HostStream from pinned
             host memory, and configs[2] (1024 poses x H=5 with the fused hypothesis mean, T=2, eta=1 with keyed noise)
             device-resident;
  arms       ungrouped fused (dp_sample with targets), grouped fused (dp_sample_grouped), and the sampler followed by grouped
             dp_metrics (two launches; device-resident workloads only), each grouped arm with 15 groups in sorted runs (as a
             loader delivers a test set) and with random ids (three atomics per pose, the worst case).
Device-resident inputs and targets rotate through a pool larger than the 126 MB L2.  Prints one JSON object (and writes it
to --out when given).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import diffpose_nw_b200 as D  # noqa: E402
from oracle import diffpose_oracle as O  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, n):
    """ms per batch over n batches (CUDA events around the window, after 20 warm-up batches)."""
    for _ in range(20):
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
    ap.add_argument("--batches", type=int, default=2000)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev).eval()
    res = {"card": card(), "engine": model.engine(), "torch": torch.__version__, "batches": args.batches, "repeats": args.repeats}
    print("card:", res["card"], flush=True)
    b51 = torch.from_numpy(D.get_beta_schedule("linear", beta_start=1e-4, beta_end=1e-3, num_diffusion_timesteps=51)).float()
    B, G = 1024, 15
    rng = np.random.default_rng(0)
    id_sets = {"runs": torch.from_numpy(np.sort(rng.integers(0, G, B)).astype(np.int32)),
               "random": torch.from_numpy(rng.integers(0, G, B).astype(np.int32))}
    pool_n = int(126 * 2**20 * 1.1) // (B * 17 * 8 * 4) + 1            # x [B,17,5] + targets [B,17,3] per batch
    xs = torch.stack([O.synthetic_poses(B, seed=10 + i) for i in range(4)]).to(dev)
    pool_x = xs.repeat(pool_n // 4 + 1, 1, 1, 1)[:pool_n].contiguous()
    pool_t = torch.stack([O.synthetic_targets(xs[i % 4].cpu(), seed=20 + i) for i in range(pool_n)]).to(dev)
    res["l2"] = f"inputs and targets rotate through {pool_n} batches = {(pool_x.numel() + pool_t.numel()) * 4 / 2**20:.0f} MiB"
    flat = torch.zeros(3, device=dev, dtype=torch.float64)
    grouped = torch.zeros(G, 3, device=dev, dtype=torch.float64)
    ids_dev = {k: v.to(dev) for k, v in id_sets.items()}
    state = {"i": 0}

    def nxt():
        i = state["i"] = (state["i"] + 1) % pool_n
        return pool_x[i], pool_t[i]

    workloads = {
        "evalloop_1024xH1xT2": dict(seq=[0, 12], eta=0.0, kw=dict(n_hyp=1)),
        "configs2_1024xH5xT2_mean_keyed": dict(seq=[0, 6], eta=1.0, kw=dict(n_hyp=5, repeat_input=True, mean_over_hyp=True, seed=7)),
    }
    res["device"] = {}
    for name, wl in workloads.items():
        steps = D.ddim_steps(b51, wl["seq"], wl["eta"])
        kw = dict(wl["kw"], steps=steps, eta=wl["eta"])

        def ungrouped():
            x, t = nxt()
            D.sample(model, x, None, None, b51, targets=t, sums=flat, **kw)

        def fused(k):
            def f():
                x, t = nxt()
                D.sample(model, x, None, None, b51, targets=t, sums=grouped, groups=ids_dev[k], **kw)
            return f

        def two_launch(k):
            def f():
                x, t = nxt()
                out = D.sample(model, x, None, None, b51, **kw)
                D.pose_error_sums(out, t, sums=grouped, groups=ids_dev[k])
            return f

        arms = {"ungrouped_fused": ungrouped, "grouped_fused_runs": fused("runs"), "grouped_fused_random": fused("random"),
                "sampler_then_grouped_metrics_runs": two_launch("runs"), "sampler_then_grouped_metrics_random": two_launch("random")}
        runs = {a: [] for a in arms}
        for rep in range(args.repeats):
            for a in (list(arms) if rep % 2 == 0 else list(reversed(list(arms)))):
                ms = timed(arms[a], args.batches)
                runs[a].append(ms)
                print(f"{name} {a}: {ms:.4f} ms/batch", flush=True)
        res["device"][name] = {a: {"ms_per_batch": v, "min": min(v), "max": max(v)} for a, v in runs.items()}

    # ---- evalloop through HostStream: pinned host batches, targets and ids travel with each batch
    seq = [0, 12]
    host_x = [O.synthetic_poses(B, seed=30 + i).pin_memory() for i in range(2)]
    host_t = [O.synthetic_targets(x, seed=40 + i).pin_memory() for i, x in enumerate(host_x)]
    host_ids = {k: v.clone().pin_memory() for k, v in id_sets.items()}
    hs = D.HostStream(model, batch=B, seq=seq, betas=b51, depth=3)

    def ring(k):
        def f():
            i = state["i"] = state["i"] + 1
            if k is None:
                hs.submit(host_x[i & 1], host_t[i & 1], flat)
            else:
                hs.submit(host_x[i & 1], host_t[i & 1], grouped, groups_host=host_ids[k])
        return f

    def ring_timed(fn, n):
        for _ in range(20):
            fn()
        hs.drain()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        hs.drain()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    arms = {"hoststream_ungrouped": ring(None), "hoststream_grouped_runs": ring("runs"), "hoststream_grouped_random": ring("random")}
    runs = {a: [] for a in arms}
    for rep in range(args.repeats):
        for a in (list(arms) if rep % 2 == 0 else list(reversed(list(arms)))):
            ms = ring_timed(arms[a], args.batches)
            runs[a].append(ms)
            print(f"evalloop hoststream {a}: {ms:.4f} ms/batch", flush=True)
    res["hoststream_evalloop_1024xH1xT2"] = {a: {"ms_per_batch": v, "min": min(v), "max": max(v)} for a, v in runs.items()}
    del hs
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
