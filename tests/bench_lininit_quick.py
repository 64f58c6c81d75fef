"""Quick timing of vsom_linear_init (not a test, not the bench): 60 000 x 784 rows (config 1's data shape, 20 x 20 map) and
4 M x 256 rows (128 x 128 map), from pinned host memory, split into the co-moment pass (with the row copies), the eigen step and
the fill; the pass's achieved f64 FMA rate (n D (D + 1) / 2 multiply-adds over the pass time); numpy's time for the same work on
the host cores (f64 co-moments in slabs of 256 Ki rows through BLAS, then eigh).  Rows are low rank plus noise, MNIST-scaled.
For information: evaluate() on held-out rows after one online epoch at config 1's shape (20 x 20 x 784, Standard), once from
randomInitialize(42, 1.0) and once from linear_init.  usage: bench_lininit_quick.py [repeats]"""
import importlib
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
v = importlib.import_module("variational-self-organizing-maps_b200")
from oracle import pyoracle as po  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
F32 = np.float32

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {q.stdout.strip() or q.stderr.strip()}", flush=True)


def rows(n, D, seed):
    """offset 100 + rank-20 signal (scales 60 * 0.8^k) + noise 5, generated on the device, returned pinned on the host"""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    basis = torch.linalg.qr(torch.randn((D, 20), device="cuda", generator=g, dtype=torch.float64))[0].T.float()
    scales = (60.0 * 0.8 ** torch.arange(20, device="cuda")).float()
    out = torch.empty((n, D), dtype=torch.float32, pin_memory=True)
    blk = 1 << 20
    for i in range(0, n, blk):
        k = min(blk, n - i)
        z = torch.randn((k, 20), device="cuda", generator=g) * scales
        out[i:i + k] = (100.0 + z @ basis + 5.0 * torch.randn((k, D), device="cuda", generator=g)).cpu()
    return out


def numpy_same_work(x):
    t0 = time.perf_counter()
    D = x.shape[1]
    x0 = x[0].astype(np.float64)
    s1, s2 = np.zeros(D), np.zeros((D, D))
    for i in range(0, x.shape[0], 1 << 18):
        d = x[i:i + (1 << 18)].astype(np.float64) - x0
        s1 += d.sum(0)
        s2 += d.T @ d
    n = x.shape[0]
    C = (s2 - np.outer(s1, s1) / n) / (n - 1)
    np.linalg.eigh(C)
    return time.perf_counter() - t0


for (n, D, W, H) in ((60000, 784, 20, 20), (1 << 22, 256, 128, 128)):
    x = rows(n, D, seed=D)
    ctx = v.VsomContext(W, H, D, v.STANDARD, v.ORDER_REFERENCE)
    ctx.linear_init_host_ptr(x.data_ptr(), n)  # warm-up
    best, ph = 1e9, None
    for _ in range(reps):
        t0 = time.perf_counter()
        ctx.linear_init_host_ptr(x.data_ptr(), n)
        t = time.perf_counter() - t0
        if t < best:
            best, ph = t, ctx.linear_init_phases()
    fma = n * D * (D + 1) / 2
    tn = numpy_same_work(x.numpy())
    print(f"{n} x {D} ({W}x{H} map): call {best * 1e3:8.2f} ms = pass {ph['pass_ms']:8.2f} + eigen {ph['eigen_ms']:6.2f} "
          f"({ph['iterations']} iterations) + fill {ph['fill_ms']:5.2f} ms;  pass {fma / (ph['pass_ms'] * 1e-3) / 1e12:6.2f} T f64 FMA/s "
          f"(rows {n * D * 4 / (ph['pass_ms'] * 1e-3) / 1e9:5.1f} GB/s from pinned memory);  numpy {tn * 1e3:9.1f} ms on {os.cpu_count()} cores",
          flush=True)
    ctx.close()
    del x

# evaluate() after one online epoch from either start (information only)
W, H, D = 20, 20, 784
x = rows(70000, D, seed=1).numpy()
train, held = x[:60000], x[60000:]
for start in ("randomInitialize(42, 1.0)", "linear_init"):
    ctx = v.VsomContext(W, H, D, v.STANDARD, v.ORDER_REFERENCE)
    if start == "linear_init":
        ctx.linear_init(train)
    else:
        o = po.Oracle(W, H, D, po.STANDARD)
        o.random_initialize(42, 1.0)
        ctx.upload_state(**o.get_state())
    before = ctx.evaluate(held)
    t0 = time.perf_counter()
    for i, c in enumerate(range(0, 60000, 6000)):  # ten chunks, sigma 10 -> 1.3, eta 0.1 -> 0.013 (exponential schedule)
        ctx.train_chunk(train[c:c + 6000], 0.1 * 0.8 ** i, 10.0 * 0.8 ** i, v.EXPONENTIAL)
    ctx.synchronize()
    print(f"config 1 shape, start {start:26s}: evaluate() on 10 000 held-out rows {before:12.2f} before, {ctx.evaluate(held):12.2f} after one "
          f"online epoch ({time.perf_counter() - t0:.2f} s)", flush=True)
    ctx.close()
