#!/usr/bin/env python
"""bench.py -- poses/sec of full DDIM sampling (H hypotheses x T steps) through diffpose_nw_b200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cpn1024|gt1024x5|sweep|sweep1m|twostage|evalloop]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

One "step" = one call of the hot path (`generalized_steps` -> dp_sample: all T DDIM steps of one batch in one
persistent kernel) on one batch of synthetic Human3.6M-shaped poses.  Default workload at every N (weak scaling: each
rank processes its own batch): BASELINE.json configs[1] -- human36m_diffpose_uvxyz_cpn.yml shape, batch 1024, 1 hypothesis,
seq = range(0,24,12) (T = 2), random-init weights.  The other BASELINE configs are --workload choices (gt1024x5 = configs[2],
strong-sharded over the ranks; sweep1m = configs[3] at any N; twostage = configs[4]).  Prints ONE JSON line on rank 0.

  value      device-timed throughput, inputs already resident in HBM (rotating through a pool larger than L2)
  e2e        same metric through the public API with pinned HOST buffers: H2D of x and D2H of x_T inside the timed region
  --steps K  the number of timed steps, in the device-timed region and again in the e2e one (host clock: K >= 200 steadies it)
  roofline   tensor bound: algorithmic FLOPs (24.65 MFLOP per pose-forward, SURVEY.md 8d) / dp_sample device time
  cpu_baseline  the oracle port (PyTorch CPU restatement of the reference) timed on the host cores, bounded sample
  --impl reference   the reference's CPU implementation of the path (oracle port; the reference is pure Python and
                     /root/reference does not exist on the GPU box) on all host threads, same config/metric.
  --dump-outputs DIR  after every measurement, write the arrays the last timed step returned to its caller as DIR/<name>.npy:
                     x_T (float32: the sampled poses; the hypothesis mean when H > 1) and, for evalloop, metric_sums (float64
                     [sum MPJPE, sum P-MPJPE, poses] accumulated over the K timed steps).  Inputs and weights are seeded, so two
                     builds run with the same arguments can be compared output for output.  At most 64 MB (64 000 000 bytes)
                     in all: a larger array keeps a fixed, seeded sample of its rows.  With N ranks every rank writes
                     <name>_rank<r>.npy.  Choose a DIR outside the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_POSE_FORWARD = 24.65e6          # minimal algorithmic work, SURVEY.md section 8d
ROW_BYTES = 17 * 5 * 4                   # one uvxyz pose, fp32
DUMP_BYTES = 64_000_000                  # --dump-outputs: all files of all ranks together, .npy headers included
NPY_HEADER_BYTES = 4096                  # room kept per file for its .npy header (128 bytes for these shapes)
METRIC = "poses/sec, full DDIM sampling (H hyps x T steps)"

WORKLOADS = {
    # BASELINE.json configs[1]: cpn.yml shape, batch 1024, H=1, config eval timesteps (2 of 24)
    "cpn1024": dict(batch=1024, n_hyp=1, seq=list(range(0, 24, 12)), eta=0.0,
                    name="configs[1]: human36m_diffpose_uvxyz_cpn.yml shape, batch 1024, H=1, seq=[0,12] (T=2), random-init"),
    # the same batches through the evaluation loop of runners/diffpose_frame.py:365-387: sampler, then MPJPE / P-MPJPE partial sums
    "evalloop": dict(batch=1024, n_hyp=1, seq=list(range(0, 24, 12)), eta=0.0, with_metrics=True,
                     name="configs[1] + metrics per batch: sampler (batch 1024, H=1, T=2) with the MPJPE / P-MPJPE sums of the batch fused into its tail (dp_sample_eval), as diffpose_frame.py:365-387"),
    # BASELINE.json configs[2]: gt.yml shape (seq [0,6]), test_times=5, ONE batch of 1024 poses sharded over the ranks (strong scaling)
    "gt1024x5": dict(batch=1024, n_hyp=5, seq=[0, 6], eta=1.0, scaling="strong",
                     name="configs[2]: human36m_diffpose_uvxyz_gt.yml shape, batch 1024 sharded over the ranks, H=5 (fused mean), seq=[0,6] (T=2), eta=1 with device noise, random-init"),
    # a slice of BASELINE.json configs[3] (1M x 10 x 50 sweep): same H and T, 16384 poses per step
    "sweep": dict(batch=16384, n_hyp=10, seq=list(range(0, 50)), eta=1.0,
                  name="slice of configs[3]: 16384 poses x H=10 x T=50 (seq=range(50)), eta=1 with device noise, random-init"),
    # one tenth of BASELINE.json configs[3] in a single call: 100 000 poses x H=10 x T=50 (17 GB of device-drawn noise)
    "sweep100k": dict(batch=100000, n_hyp=10, seq=list(range(0, 50)), eta=1.0,
                      name="tenth of configs[3]: 100000 poses x H=10 x T=50 (seq=range(50)), eta=1 with device noise, random-init"),
    # BASELINE.json configs[3] itself at ANY number of ranks: 1M poses x H=10 x T=50 in total, sharded (strong scaling); the noise
    # of a call is drawn in bounded chunks (sampler.sample: <= 2 GiB at a time)
    "sweep1m": dict(batch=1000000, n_hyp=10, seq=list(range(0, 50)), eta=1.0, scaling="strong", draw_noise=True,
                    name="configs[3]: 1M poses sharded over the ranks x H=10 x T=50 (seq=range(50)), eta=1 with device noise drawn per call, NCCL MPJPE reduction, random-init"),
    # BASELINE.json configs[4] per GPU: GCNpose lifts uv -> xyz, root-centre, concat, H=5 hypotheses refined by GCNdiff (gt.yml seq)
    "twostage": dict(batch=4096, n_hyp=5, seq=[0, 6], eta=0.0, two_stage=True,
                     name="configs[4]: GCNpose (uv->xyz) + GCNdiff refinement, batch 4096, H=5, seq=[0,6] (T=2), random-init"),
}


def load_peaks(timed_region_s):
    """bf16 peak the roofline is reported against: the burst figure for a kernel timed alone (< 1 s region), the sustained
    one for a kernel timed inside a long step (the board reaches its power cap)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    long_run = timed_region_s >= 1.0
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        burst = float(d.get("bf16_tflops", 1590.0))
        sus = float(d.get("bf16_tflops_sustained", burst))
        return dict(tflops=sus if long_run else burst, hbm=float(d.get("hbm_gbs", 6650.0)),
                    src="measured (MEASURED_PEAKS.json, bf16 %s)" % ("sustained: timed region >= 1 s" if long_run else "burst: timed region < 1 s"))
    return dict(tflops=1590.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per tc2_kernel launch of configs[1], read from the newest committed
    `ncu --set full` summary under profiles/ (tools/ncu_summary.py writes them); (None, why) when there is none."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_tcg_metrics.csv")))
    if not files:
        return None, "no profiles/*_ncu_tcg_metrics.csv"
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot, n = 0.0, 0
    with open(files[-1]) as f:
        for line in f:
            c = line.strip().split(",")
            if c[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and c[1] in mult:
                vals = [float(v) for v in c[2:] if v]
                tot += mult[c[1]] * sum(vals) / max(1, len(vals))
                n += 1
    if n != 2:
        return None, f"{os.path.basename(files[-1])}: dram counters missing"
    return int(round(tot)), f"ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per tc2_kernel launch (profiles/{os.path.basename(files[-1])})"


def l2_note(pool_n, batch_bytes):
    return (f"inputs rotate through a pool of {pool_n} distinct buffers = {pool_n * batch_bytes / 2**20:.0f} MiB (> 126 MiB L2), written once at set-up in "
            "order, so every timed step reads a batch that is not cache resident; weights (1.6 MB) stay L2-resident by design")


def dump_outputs(path, arrays, budget, suffix=""):
    """Write each tensor as path/<name><suffix>.npy, the files together at most `budget` bytes.  One whose data does not fit
    its share (less the room for its header) keeps a sorted sample of its rows drawn with a fixed seed, so the same
    arguments select the same rows in every run."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    share = budget // len(arrays) - NPY_HEADER_BYTES
    for name, t in arrays.items():
        a = t.cpu().numpy()
        if a.nbytes > share:
            row_bytes = a.nbytes // a.shape[0]
            keep = np.random.default_rng(0).choice(a.shape[0], max(0, share) // row_bytes, replace=False)
            a = a[np.sort(keep)]
        np.save(os.path.join(path, name + suffix + ".npy"), a)


def bench_config(wl, world):
    """The `config` object -- IDENTICAL in both arms (ours / reference) for the same command line."""
    B = wl["batch"]
    strong = wl.get("scaling") == "strong"
    batch_bytes = (B // world if strong else B) * ROW_BYTES
    pool_n = max(2, (int(126 * 2**20 * 1.1) + batch_bytes - 1) // batch_bytes)
    return {"workload": wl["name"], "batch": B, "batch_is": "total, sharded over the ranks" if strong else "per GPU", "n_hyp": wl["n_hyp"],
            "T": len(wl["seq"]), "eta": wl["eta"], "l2": l2_note(pool_n, batch_bytes)}, pool_n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the benchmark runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.t0, self.t1 = [], None, None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        inside = [r for (ts, r) in self.rows if self.t0 is not None and self.t0 - 0.05 <= ts <= self.t1 + 0.1]
        rows = inside or [r for (_, r) in self.rows]
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [c.strip() for c in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except Exception:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "in_timed_region": bool(inside), "power_w_max": max(pw) if pw else None}


def oracle_setup(wl, n):
    """Weights/inputs for the CPU legs: same architecture, seeds and synthetic distribution as the GPU arm."""
    import torch
    import diffpose_nw_b200 as D
    from oracle import diffpose_oracle as O
    cfg = O.default_config()
    adj = D.adj_mx_from_edges()
    torch.manual_seed(0)
    sd = {k: v.detach().clone() for k, v in D.FusedGCNdiff(adj, cfg).state_dict().items()}
    betas = torch.from_numpy(O.beta_schedule("linear", 1e-4, 1e-3, 51)).float()
    x = O.synthetic_poses(n, seed=1).repeat(wl["n_hyp"], 1, 1)
    den = lambda xt, m, tt: O.gcndiff_forward(sd, adj, 5, 4, xt, m, tt)
    mask = torch.ones(1, 1, 17, dtype=torch.bool)
    run = lambda: O.ddim_sample(x, mask, wl["seq"], den, betas, eta=wl["eta"])[0][-1]
    return run


def time_oracle(wl, n, budget_s, min_reps=2):
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    run = oracle_setup(wl, n)
    with torch.no_grad():
        run()
        reps, t0 = 0, time.perf_counter()
        while reps < min_reps or time.perf_counter() - t0 < budget_s:
            run()
            reps += 1
        dt = time.perf_counter() - t0
    return n * reps / dt, reps, dt


def run_reference(args, wl):
    """The reference arm: the reference's CPU implementation of the path (oracle port), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    steps, warm = args.steps, args.warmup
    # size the per-step sample so the whole run stays within ~2 minutes
    probe_n = 32
    rate, _, _ = time_oracle(wl, probe_n, 1.0, min_reps=1)
    per_step = 110.0 / max(1, steps + warm)
    n = int(max(8, min(wl["batch"], rate * per_step)))
    run = oracle_setup(wl, n)
    with torch.no_grad():
        for _ in range(warm):
            run()
        t0 = time.perf_counter()
        for _ in range(steps):
            run()
        dt = time.perf_counter() - t0
    val = n * steps / dt
    sample = f"{n}-pose slice of the {wl['batch']}-pose batch per step, H={wl['n_hyp']}, T={len(wl['seq'])}, {steps} steps after {warm} warm-up"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "poses/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": wl.get("scaling", "weak"), "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": bench_config(wl, int(os.environ.get("WORLD_SIZE", "1")))[0],
            "detail": {"device": "host CPU", "torch_threads": torch.get_num_threads()},
            "cpu_baseline": {"value": val, "unit": "poses/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4000)   # ~0.5 s timed region: enough nvidia-smi clock samples inside it
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cpn1024", choices=sorted(WORKLOADS))
    ap.add_argument("--engine", default="auto", choices=["auto", "fp32", "tcx", "tcg"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU arm's outputs; the reference arm times a slice sized by its own speed")
        return run_reference(args, wl)

    import torch
    import diffpose_nw_b200 as D
    from diffpose_nw_b200 import _lib
    from oracle import diffpose_oracle as O   # synthetic input generators + the cpu_baseline leg only

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (the product has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    torch.set_grad_enabled(False)

    B_total, H, seq, eta = wl["batch"], wl["n_hyp"], wl["seq"], wl["eta"]
    T = len(seq)
    strong = wl.get("scaling") == "strong"
    if strong:                       # one workload-sized batch per step, sharded: this rank's contiguous pose range
        lo, hi = D.shard_range(B_total, rank, world)
        B = hi - lo
    else:
        B = B_total
    cfg = O.default_config()
    torch.manual_seed(0)
    model = D.FusedGCNdiff(D.adj_mx_from_edges(), cfg).to(dev).set_engine(args.engine)
    model.eval()     # as the reference's evaluation loop does (runners/diffpose_frame.py:292-293)
    betas = torch.from_numpy(D.get_beta_schedule("linear", beta_start=1e-4, beta_end=1e-3, num_diffusion_timesteps=51)).float()
    steps_arr = D.ddim_steps(betas, seq, eta)

    # input pool larger than L2, written once in order: every timed step reads a batch that is not cache resident
    config, pool_n = bench_config(wl, world)
    batch_bytes = B * ROW_BYTES
    if B * pool_n > 4_000_000:       # bound the host-side generation for the million-pose workloads
        pool_n = 2
    base = O.synthetic_poses(min(B, 131072), seed=1 + rank)
    if base.shape[0] < B:
        base = base.repeat((B + base.shape[0] - 1) // base.shape[0], 1, 1)[:B].contiguous()
    g = torch.Generator().manual_seed(100 + rank)
    pool = torch.empty(pool_n, B, 17, 5, device=dev)
    base_dev = base.to(dev)
    for i in range(pool_n):
        pool[i] = base_dev + 0.01 * torch.randn(1, 17, 5, generator=g).to(dev)
    pool[:, :, 0, 2:] = 0
    noise = None
    if eta > 0 and not wl.get("draw_noise"):
        noise = torch.randn(T, B * H, 17, 5, device=dev)
    targets = O.synthetic_targets(base).to(dev)

    pose_model = None
    if wl.get("two_stage"):
        torch.manual_seed(1)
        pose_model = D.FusedGCNpose(D.adj_mx_from_edges(), O.default_config(coords_dim=[2, 3])).to(dev).set_engine(args.engine).eval()
        uv_pool = pool[:, :, :, :2].contiguous()
    msums = torch.zeros(3, device=dev, dtype=torch.float64)

    def step(i):
        if pose_model is not None:
            out = D.lift_and_refine(model, model_pose=pose_model, input_2d=uv_pool[i % pool_n], src_mask=None, seq=seq, betas=betas,
                                    eta=eta, test_times=H)
        elif wl.get("with_metrics"):      # sampler + MPJPE / P-MPJPE sums of the batch in one launch (dp_sample_eval)
            out = D.sample(model, pool[i % pool_n], None, seq, betas, eta=eta, noise=noise, n_hyp=H, repeat_input=True,
                           mean_over_hyp=(H > 1), steps=steps_arr, targets=targets, sums=msums)
        else:
            out = D.sample(model, pool[i % pool_n], None, seq, betas, eta=eta, noise=noise, n_hyp=H, repeat_input=True,
                           mean_over_hyp=(H > 1), steps=steps_arr)
        return out

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # benchmark hygiene for the short timed window (20 steps = 2 ms when the driver runs it, max over ranks): no Python GC
    # pause inside it, one core pair per rank (eight rank processes otherwise migrate over the same cores), no idle OpenMP pool
    import gc
    torch.set_num_threads(1)
    if world > 1 and hasattr(os, "sched_setaffinity"):
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            os.sched_setaffinity(0, set(cores[local * per:(local + 1) * per]) or set(cores))
        except OSError:
            pass
    sampler = ClockSampler(local) if rank == 0 else None
    gc.collect()
    gc.disable()
    # untimed set-up before the W declared warm-up steps: ~10 ms of the same calls, so that the board has left its idle
    # power state when the (possibly only 2 ms long) timed window starts -- clocks are sampled and reported below
    ramp = max(0, min(100, 200000 // max(1, B * H * T)))      # none for the long-step workloads
    for i in range(ramp):
        out = step(args.steps + i)
    for i in range(args.warmup):
        out = step(args.steps + i)
    barrier()
    # The barrier + synchronize leave the GPU idle (for milliseconds under NCCL), and its SM clock needs ~15 of these 0.1 ms
    # steps to come back (tools/first_steps.py: 148, 111, 111, 108, ... 102 us per step after an idle gap).  A lead-in of
    # untimed steps (3 ms) between the synchronisation and the first event hands the timed K steps a busy, full-clock GPU; the
    # timed region itself is exactly K steps between two CUDA events, followed by barrier + synchronize.
    lead_in = min(30, ramp)     # 10 were enough for one process; behind an 8-rank NCCL barrier the idle gap is longer (every rank measured
                                # 0.1004-0.1027 ms per step in the 20-step window against 0.0973 in a 2000-step run with 10)
    for i in range(lead_in):
        out = step(args.steps + args.warmup + i)
    timing_note = (f"{ramp} set-up + {args.warmup} warm-up steps, barrier + synchronize, {lead_in} untimed lead-in steps, CUDA event, "
                   f"{args.steps} timed steps, CUDA event, barrier + synchronize")
    if args.dump_outputs and wl.get("with_metrics"):
        msums.zero_()       # the dumped sums then cover exactly the K timed steps
    l0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler:
        sampler.t0 = time.time()
    ev0.record()
    for i in range(args.steps):
        out = step(i)
    ev1.record()
    barrier()
    if sampler:
        sampler.t1 = time.time()
    dump = None
    if args.dump_outputs:       # held on the device (the e2e leg adds to msums) and written after every measurement
        dump = {"x_T": out}
        if wl.get("with_metrics"):
            dump["metric_sums"] = msums.clone()
    gc.enable()
    launches = _lib.launch_count() - l0
    ms = ev0.elapsed_time(ev1)
    ms_ranks = [ms / args.steps]
    if dist is not None:
        tms = torch.tensor([ms], device=dev, dtype=torch.float64)
        allms = [torch.zeros_like(tms) for _ in range(world)]
        dist.all_gather(allms, tms)
        ms_ranks = [float(t.item()) / args.steps for t in allms]
        ms = max(float(t.item()) for t in allms)          # the job is as fast as its slowest rank
    poses_per_step = B_total if strong else world * B        # whole job
    value = poses_per_step * args.steps / (ms * 1e-3)

    # ---- end-to-end: pinned host buffers, H2D + D2H inside the timed region, public API (HostStream: the copies of
    #      neighbouring batches overlap the kernel of the current one; every step still moves its own input and output)
    two_stage = pose_model is not None
    out_rows = B if H > 1 else B * H
    e2e = None
    if B <= 131072:
        host_in = [torch.empty(B, 17, 5).pin_memory() for _ in range(2)]
        host_in[0].copy_(base); host_in[1].copy_(base)
        hs = D.HostStream(model, batch=B, seq=seq, betas=betas, eta=eta, test_times=H) if (eta == 0 and not two_stage) else None
        xd = torch.empty(B, 17, 5, device=dev)
        if two_stage:       # the two-stage pipeline takes 2D keypoints from the host: [B,17,2] in, refined [B,17,5] out
            host_uv = [base[:, :, :2].contiguous().pin_memory() for _ in range(2)]
            uvd = torch.empty(B, 17, 2, device=dev)
        host_out = [torch.empty(out_rows, 17, 5).pin_memory() for _ in range(2)]

        def e2e_serial(i):      # eta > 0 with device noise: plain copy -> sample -> copy (HostStream draws no noise itself)
            if two_stage:
                uvd.copy_(host_uv[i & 1], non_blocking=True)
                o = D.lift_and_refine(model, model_pose=pose_model, input_2d=uvd, src_mask=None, seq=seq, betas=betas, eta=eta, test_times=H)
                host_out[i & 1].copy_(o, non_blocking=True)
                return
            xd.copy_(host_in[i & 1], non_blocking=True)
            o = D.sample(model, xd, None, seq, betas, eta=eta, noise=noise, n_hyp=H, repeat_input=True, mean_over_hyp=(H > 1), steps=steps_arr,
                         targets=targets if wl.get("with_metrics") else None, sums=msums if wl.get("with_metrics") else None)
            host_out[i & 1].copy_(o, non_blocking=True)

        host_tg = targets.cpu().pin_memory() if (wl.get("with_metrics") and hs is not None) else None      # evaluation: targets travel with the batch
        hs_sums = msums if host_tg is not None else None
        # K batches, as in the device-timed region.  A host-clock window of 20 batches (2 ms) measures scheduling jitter of the
        # rank processes as much as the pipeline (8 ranks, max over ranks: 0.87 "efficiency" at 20 batches, 0.99 at 2000)
        e_steps = args.steps
        last = None
        for i in range(3):
            e2e_serial(i) if hs is None else hs.submit(host_in[i & 1], host_tg, hs_sums)
        if hs is not None:
            hs.drain()
        barrier()
        t0 = time.perf_counter()
        for i in range(e_steps):
            if hs is None:
                e2e_serial(i)
            else:
                r = hs.submit(host_in[i & 1], host_tg, hs_sums)
                last = r if r is not None else last
        if hs is not None:
            tail = hs.drain()
            last = tail[-1]
        torch.cuda.synchronize()
        e_ms = (time.perf_counter() - t0) * 1e3
        if dist is not None:
            tms = torch.tensor([e_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            e_ms = float(tms.item())
        assert torch.isfinite(last if last is not None else host_out[0]).all()
        e2e = {"value": poses_per_step * e_steps / (e_ms * 1e-3), "unit": "poses/s",
               "h2d_bytes_per_step": B * 17 * 2 * 4 if two_stage else B * ROW_BYTES + (B * 17 * 3 * 4 if host_tg is not None else 0),
               "d2h_bytes_per_step": out_rows * ROW_BYTES, "steps": e_steps, "ms_per_step": e_ms / e_steps,
               "how": "pinned host buffers; " + ("HostStream (H2D / kernel / D2H of neighbouring batches overlap)" if hs is not None else "copy -> call -> copy per step")}
    elif dist is not None:
        barrier()

    # ---- the evaluation tail: per-rank partial sums + one all-reduce (NCCL) -- not part of the timed sampler region
    sums, _ = D.pose_error_sums(out, targets)
    mp, pmp, cnt = D.reduce_metrics(sums)
    clocks = sampler.stop() if sampler else None

    if rank == 0:
        peaks = load_peaks(ms * 1e-3)
        per_launch_s = ms * 1e-3 / args.steps
        flops = B * H * T * FLOP_PER_POSE_FORWARD + (B * 25.2e6 if two_stage else 0.0)   # per GPU; + GCNpose: 25.2 MFLOP/pose (SURVEY.md 8a a14)
        achieved = flops / per_launch_s / 1e12
        hbm_bytes = B * ROW_BYTES + out_rows * ROW_BYTES + (T * B * H * ROW_BYTES if eta > 0 else 0)
        ll = model.last_launch()
        traffic, traffic_src = ncu_traffic() if (args.workload == "cpn1024" and model.engine() == "tcg") else (None, "measured for the cpn1024 workload only")
        line = {
            "metric": METRIC, "value": value, "unit": "poses/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f16 operands / f32 accumulate (tcgen05)" if model.engine() == "tcg" else ("f16 hi+lo operands / f32 accumulate (tcgen05)" if model.engine() == "tcx" else "f32"),
            "data": "synthetic",
            "config": config,
            "detail": {"timing": timing_note, "ms_per_step_by_rank": [round(v, 5) for v in ms_ranks], "engine": model.engine(), "lifter_engine": pose_model.forward_engine() if two_stage else None, "batch_this_rank": B,
                       "launch": {"grid": ll[0], "block": ll[1], "smem": ll[2], "poses_per_tile": ll[3], "tiles": ll[5]}},
            "e2e": e2e,
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peaks["src"],
                         "note": "per GPU: achieved = 24.65 MFLOP x poses x H x T (+ 25.2 MFLOP x poses for the lifter) per step / mean device time of a step",
                         "hbm_gbs": hbm_bytes / per_launch_s / 1e9},
            "clocks": clocks,
            "eval": {"mpjpe_mm": mp, "p_mpjpe_mm": pmp, "poses": cnt},
        }
        if world == 1 and not args.no_cpu_baseline:
            torch.set_num_threads(os.cpu_count() or 1)
            n_cpu = 256 if H * T <= 4 else 16
            v, reps, dt = time_oracle(wl, n_cpu, 12.0)
            line["cpu_baseline"] = {"value": v, "unit": "poses/s", "cores": os.cpu_count() or 1, "kind": "port",
                                    "sample": f"{n_cpu}-pose slice of the workload (H={H}, T={T}), {reps} reps in {dt:.1f} s after 1 warm-up, torch CPU threads={os.cpu_count()}"}
        print(json.dumps(line), flush=True)
    if dump is not None:
        dump_outputs(args.dump_outputs, dump, DUMP_BYTES // world, f"_rank{rank}" if world > 1 else "")
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
