"""Keyed in-kernel noise against tensor noise, on one GPU (python tools/noise_time.py [--out FILE]).

Records the card and its power limit, then measures with CUDA events:
  1. configs[2] (1024 poses x H=5 x T=2, eta=1) and the bench `sweep` shape (16384 x H=10 x T=50, eta=1), three arms per
     shape -- caller-provided preallocated noise (what bench.py times), noise=None (the torch chunked draw inside sample())
     and seed= (keyed) -- alternated, 3 repeats, each timed over at least 1 s and at least 200 calls (fewer when 200 calls
     would take more than 5 s: the sweep shape runs ~14 calls of ~0.37 s);
  2. the host-memory configs[2] loop: HostStream(seed=) against the serial copy -> sample(noise=None) -> copy;
  3. the peak device memory (torch allocator) of one 125k-pose x H=10 x T=50 call, keyed against the chunked draw.
Prints one JSON object (and writes it to --out when given).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import diffpose_nw_b200 as D  # noqa: E402
from oracle import diffpose_oracle as O  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, min_calls=200, min_s=1.0, max_s=5.0):
    """ms per call over at least min_s seconds, and at least min_calls calls unless they would take more than max_s
    (CUDA events around the whole window)."""
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    per = max((time.perf_counter() - t0) / 5, 1e-6)
    n = max(int(min_s / per) + 1, min(min_calls, int(max_s / per) + 1))
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result to this file")
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev).eval()
    res = {"card": card(), "engine": model.engine(), "torch": torch.__version__}
    print("card:", res["card"], flush=True)
    b51 = torch.from_numpy(D.get_beta_schedule("linear", beta_start=1e-4, beta_end=1e-3, num_diffusion_timesteps=51)).float()

    shapes = {"configs2_1024xH5xT2": (1024, 5, [0, 6]), "sweep_16384xH10xT50": (16384, 10, list(range(50)))}
    res["device"] = {}
    for name, (B, H, seq) in shapes.items():
        T = len(seq)
        x = O.synthetic_poses(B, seed=1).to(dev)
        steps = D.ddim_steps(b51, seq, 1.0)
        noise = torch.randn(T, B * H, 17, 5, device=dev)
        kw = dict(n_hyp=H, repeat_input=True, mean_over_hyp=True, steps=steps)
        arms = {
            "preallocated_noise": lambda: D.sample(model, x, None, None, b51, eta=1.0, noise=noise, **kw),
            "torch_draw": lambda: D.sample(model, x, None, None, b51, eta=1.0, **kw),
            "keyed": lambda: D.sample(model, x, None, None, b51, eta=1.0, seed=1234, **kw),
        }
        runs = {a: [] for a in arms}
        for rep in range(args.repeats):
            order = list(arms) if rep % 2 == 0 else list(reversed(list(arms)))
            for a in order:
                ms, n = timed(arms[a])
                runs[a].append(ms)
                print(f"{name} {a}: {ms:.4f} ms/call over {n} calls", flush=True)
        res["device"][name] = {a: {"ms_per_call": v, "min": min(v), "max": max(v),
                                   "spread_pct": 100 * (max(v) - min(v)) / min(v)} for a, v in runs.items()}
        del noise

    # ---- host-memory configs[2] loop
    B, H, seq = 1024, 5, [0, 6]
    steps = D.ddim_steps(b51, seq, 1.0)
    host_in = [O.synthetic_poses(B, seed=2 + i).pin_memory() for i in range(2)]
    host_out = [torch.empty(B, 17, 5).pin_memory() for _ in range(2)]
    xd = torch.empty(B, 17, 5, device=dev)
    hs = D.HostStream(model, batch=B, seq=seq, betas=b51, eta=1.0, test_times=H, seed=99)
    state = {"i": 0}

    def serial():
        i = state["i"] = state["i"] + 1
        xd.copy_(host_in[i & 1], non_blocking=True)
        o = D.sample(model, xd, None, None, b51, eta=1.0, n_hyp=H, repeat_input=True, mean_over_hyp=True, steps=steps)
        host_out[i & 1].copy_(o, non_blocking=True)

    def ring():
        i = state["i"] = state["i"] + 1
        hs.submit(host_in[i & 1])

    host = {"serial_copy_sample_copy": [], "hoststream_keyed": []}
    for rep in range(args.repeats):
        for a, fn in ([("serial_copy_sample_copy", serial), ("hoststream_keyed", ring)] if rep % 2 == 0 else
                      [("hoststream_keyed", ring), ("serial_copy_sample_copy", serial)]):
            for _ in range(10):
                fn()
            hs.drain(); torch.cuda.synchronize()
            n = 2000
            t0 = time.perf_counter()
            for _ in range(n):
                fn()
            hs.drain(); torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3 / n
            host[a].append(ms)
            print(f"host loop {a}: {ms:.4f} ms/batch over {n} batches", flush=True)
    res["host_loop_configs2"] = {a: {"ms_per_batch": v, "min": min(v), "max": max(v)} for a, v in host.items()}

    # ---- peak device memory of one 125k x H=10 x T=50 call
    B, H, seq = 125000, 10, list(range(50))
    steps = D.ddim_steps(b51, seq, 1.0)
    x = O.synthetic_poses(B, seed=3).to(dev)
    mem = {}
    for a, extra in (("keyed", dict(seed=5)), ("torch_draw", {})):
        D.sample(model, x[:64], None, None, b51, eta=1.0, n_hyp=H, repeat_input=True, mean_over_hyp=True, steps=steps, **extra)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        o = D.sample(model, x, None, None, b51, eta=1.0, n_hyp=H, repeat_input=True, mean_over_hyp=True, steps=steps, **extra)
        e1.record()
        torch.cuda.synchronize()
        mem[a] = {"peak_bytes_above_inputs": torch.cuda.max_memory_allocated(dev) - base, "ms": e0.elapsed_time(e1),
                  "finite": bool(torch.isfinite(o).all())}
        del o
        print(f"125k x 10 x 50 {a}: peak {mem[a]['peak_bytes_above_inputs'] / 2**20:.1f} MiB, {mem[a]['ms']:.1f} ms", flush=True)
    res["peak_memory_125k_H10_T50"] = mem
    del hs
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
