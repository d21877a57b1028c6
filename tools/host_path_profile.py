"""Where the host time of one drop-in call goes (per-piece micro-timings, 20000 repetitions each).

    python tools/host_path_profile.py
"""
import ctypes, os, sys, time
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import diffpose_nw_b200 as D
from diffpose_nw_b200 import _lib, sampler as S
from oracle import diffpose_oracle as O

dev = torch.device("cuda:0")
torch.manual_seed(0)
torch.set_grad_enabled(False)
model = D.FusedGCNdiff(D.adj_mx_from_edges(), O.default_config()).to(dev).eval()
betas = torch.from_numpy(O.beta_schedule("linear", 1e-4, 1e-3, 51)).float()
x = O.synthetic_poses(1024, seed=1).to(dev)
seq = range(0, 24, 12)
steps = D.ddim_steps(betas, seq, 0.0)
out = D.sample(model, x, None, seq, betas, steps=steps)
torch.cuda.synchronize()
lib = _lib.load()
N = 20000


def t(name, fn, n=N):
    for _ in range(100):
        fn()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    dt = (time.perf_counter() - t0) / n * 1e6
    print(f"{name:48s} {dt:7.2f} us")
    return dt


t("S._unwrap(model)", lambda: S._unwrap(model))
t("model._check_x(x, 5)", lambda: model._check_x(x, 5))
t("model._ensure_packed(dev)", lambda: model._ensure_packed(dev))
t("cached_ddim_steps(betas, seq, 0)", lambda: S.cached_ddim_steps(betas, seq, 0.0))
t("any(s.c1 != 0 for s in steps)", lambda: any(s.c1 != 0.0 for s in steps))
t("torch.empty(1024,17,5,device)", lambda: torch.empty(1024, 17, 5, device=dev, dtype=torch.float32))
t("torch.cuda.current_stream(dev).cuda_stream", lambda: torch.cuda.current_stream(dev).cuda_stream)
t("torch.cuda.current_device()", lambda: torch.cuda.current_device())
t("x.data_ptr()", lambda: x.data_ptr())
t("lib.dp_launch_count() (ctypes, no args)", lambda: lib.dp_launch_count())
t("lib.dp_get_engine(h) (ctypes, 1 arg)", lambda: lib.dp_get_engine(model._handle))
stream = torch.cuda.current_stream(dev).cuda_stream
xp, op = x.data_ptr(), out.data_ptr()


def raw():
    lib.dp_sample(model._handle, xp, 0, op, 1024, 1, steps, 2, None, None, None, 0, None, None, stream)


torch.cuda.synchronize()
d_raw = t("lib.dp_sample(...) raw ctypes call (GPU queue full)", raw, 3000)
torch.cuda.synchronize()
d_s = t("D.sample(model, x, None, seq, betas, steps=steps)", lambda: D.sample(model, x, None, seq, betas, steps=steps), 3000)
torch.cuda.synchronize()
d_g = t("D.generalized_steps(x, None, seq, model, betas)", lambda: D.generalized_steps(x, None, seq, model, betas, eta=0.0), 3000)
torch.cuda.synchronize()
# host-only cost of the raw call: launch into an empty queue a few at a time
ts = []
for _ in range(200):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    raw()
    ts.append(time.perf_counter() - t0)
ts.sort()
print(f"raw dp_sample into an idle queue: median {ts[100] * 1e6:.2f} us, p10 {ts[20] * 1e6:.2f} us")
ts = []
for _ in range(200):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    D.sample(model, x, None, seq, betas, steps=steps)
    ts.append(time.perf_counter() - t0)
ts.sort()
print(f"D.sample into an idle queue:      median {ts[100] * 1e6:.2f} us, p10 {ts[20] * 1e6:.2f} us")
