"""Quick timing of vsom_predict_columns (not a test, not the bench).

On bench's trained 128 x 128 x 256 scoring map, 4 M rows from device memory and 4 M from pinned host memory, |S| in {256, 192, 128}
scattered columns, rows/s of:
- predict_columns[_device] on the map (the gathers, the search over S and the fill of the other columns);
- find_bmu[_device] on the full map (all 256 columns);
- find_bmu[_device] on a context whose plane is the columns S, with the rows already compacted (the search alone).
For device rows, the first minus the third is the cost of the gathers and the fill.  For host rows the first is compared with
the second: both copy the full-width rows in, and the prediction call also copies 8 q bytes per row of predictions back out.
The variants alternate within each round; every shape is warmed up first; the best of `repeats` rounds is printed with the median.  Then a MNIST-shaped map (20 x 20 x 794, ten label
columns behind 784 'pixels'): rows/s of predicting the labels from the pixels, and the label accuracy.
usage: bench_predict_quick.py [repeats]"""
import ctypes as C
import importlib
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
v = importlib.import_module("variational-self-organizing-maps_b200")
binding = importlib.import_module("variational-self-organizing-maps_b200.binding")
from test_gpu_benchmark_shapes import _row_count_map  # noqa: E402  (bench's trained scoring map)
from test_gpu_predict_columns import mnist_rows  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
N_ROWS = 4 << 20
f32p, u32p, u8p = C.POINTER(C.c_float), C.POINTER(C.c_uint32), C.POINTER(C.c_uint8)

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {q.stdout.strip() or q.stderr.strip()}", flush=True)


def rows_like_bench(n, D, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    centres = torch.randn((64, D), device="cuda", generator=g) * 3
    return (torch.randn((n, D), device="cuda", generator=g) + centres[torch.randint(0, 64, (n,), device="cuda", generator=g)]).contiguous()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


W, H, D, mean, _ = _row_count_map(v, "trained")
full = v.VsomContext(W, H, D, v.STANDARD, v.ORDER_EIGEN_SSE)
full.upload_state(mean=mean)
x_dev = rows_like_bench(N_ROWS, D, 5)
x_host = x_dev.cpu().pin_memory()
n = N_ROWS
bmu_dev = torch.empty(n, dtype=torch.int32, device="cuda")
dist_dev = torch.empty(n, dtype=torch.float32, device="cuda")
bmu_h = torch.empty(n, dtype=torch.int32).pin_memory()
dist_h = torch.empty(n, dtype=torch.float32).pin_memory()
L = binding.lib()

for m in (256, 192, 128):
    S = np.sort(np.random.default_rng(m).choice(D, m, replace=False))
    match = np.zeros(D, np.uint8)
    match[S] = 1
    nq = D - m
    mean_dev = torch.empty(max(n * nq, 1), dtype=torch.float32, device="cuda")
    sigma_dev = torch.empty_like(mean_dev)
    mean_h = torch.empty(max(n * nq, 1), dtype=torch.float32).pin_memory()
    sigma_h = torch.empty_like(mean_h).pin_memory()
    comp = v.VsomContext(W, H, m, v.STANDARD, v.ORDER_EIGEN_SSE)
    comp.upload_state(mean=np.ascontiguousarray(mean[:, S]))
    xc_dev = x_dev[:, torch.from_numpy(S).cuda()].contiguous()
    xc_host = xc_dev.cpu().pin_memory()
    mp = match.ctypes.data_as(u8p)

    def predict_device():
        full.predict_columns_device(x_dev, n, match, bmu_dev, dist_dev, mean_dev, sigma_dev)

    def predict_host():
        full._check(L.vsom_predict_columns(full._h, C.cast(x_host.data_ptr(), f32p), n, mp, 0, C.cast(bmu_h.data_ptr(), u32p), C.cast(dist_h.data_ptr(), f32p),
                                           C.cast(mean_h.data_ptr(), f32p), C.cast(sigma_h.data_ptr(), f32p)))

    variants = {
        "predict_columns_device": (predict_device, lambda: full.last_score_tc),
        "find_bmu_device full": (lambda: full.find_bmu_device(x_dev, n, bmu_dev, dist_dev), lambda: full.last_score_tc),
        "find_bmu_device compact": (lambda: comp.find_bmu_device(xc_dev, n, bmu_dev, dist_dev), lambda: comp.last_score_tc),
        "predict_columns host": (predict_host, lambda: full.last_score_tc),
        "find_bmu host full": (lambda: full.find_bmu_host_ptr(x_host.data_ptr(), n, bmu_h.data_ptr(), dist_h.data_ptr()), lambda: full.last_score_tc),
        "find_bmu host compact": (lambda: comp.find_bmu_host_ptr(xc_host.data_ptr(), n, bmu_h.data_ptr(), dist_h.data_ptr()), lambda: comp.last_score_tc),
    }
    times = {k: [] for k in variants}
    tiers = {}
    for k, (fn, tier) in variants.items():  # warm-up of every shape
        fn()
        tiers[k] = tier()
    for _ in range(reps):
        for k, (fn, _) in variants.items():
            times[k].append(timed(fn))
    for k, ts in times.items():
        best, med = min(ts), float(np.median(ts))
        print(f"|S| {m:3d} of {D}, {n} rows, {k:24s}: best {best * 1e3:8.2f} ms = {n / best / 1e6:7.2f} M rows/s, median {n / med / 1e6:7.2f} M rows/s "
              f"(tier {tiers[k]})", flush=True)
    # device rows: predict against the search on pre-compacted rows = the gathers and the fill.  Host rows: predict against find_bmu
    # on the same full-width rows (both copy 4 d_in bytes per row in), so the difference is the predictions coming back (8 q bytes per
    # row) plus the gathers and the fill
    for label, a, b in (("device: predict over the compacted search (gathers + fill)", "predict_columns_device", "find_bmu_device compact"),
                        ("host: predict over full-width find_bmu (predictions out + gathers + fill)", "predict_columns host", "find_bmu host full")):
        ta, tb = min(times[a]), min(times[b])
        print(f"|S| {m:3d}: {label}: {(ta - tb) * 1e3:+7.2f} ms = {(ta - tb) / n * 1e9:+6.2f} ns per row ({(ta / tb - 1) * 100:+5.1f} %)", flush=True)
    comp.close()
    del mean_dev, sigma_dev, mean_h, sigma_h, xc_dev, xc_host
full.close()
del x_dev, x_host

# ---- MNIST-shaped map: predict the ten label columns from the 784 pixels
x, cls = mnist_rows(70000, 11)
ctx = v.VsomContext(20, 20, 794, v.STANDARD, v.ORDER_EIGEN_SSE)
ctx.upload_state(mean=np.random.default_rng(3).random((400, 794)).astype(np.float32))
for i, (sg, eta) in enumerate(((10.0, 0.5), (5.0, 0.3), (2.0, 0.1))):
    ctx.train_chunk(x[1000 * i:1000 * (i + 1)], eta, sg, v.EXPONENTIAL)
test, tcls = x[10000:], cls[10000:]
match = np.zeros(794, np.uint8)
match[:784] = 1
ctx.predict_columns(test, match)
ts = []
for _ in range(reps):
    t0 = time.perf_counter()
    _, _, pm, _ = ctx.predict_columns(test, match)
    ts.append(time.perf_counter() - t0)
acc = float(np.mean(np.argmax(pm, axis=1) == tcls))
td_ = test.shape[0]
xt = torch.from_numpy(test).cuda()
b = torch.empty(td_, dtype=torch.int32, device="cuda")
pm_d = torch.empty(td_ * 10, dtype=torch.float32, device="cuda")
ctx.predict_columns_device(xt, td_, match, b, None, pm_d, None)
tsd = [timed(lambda: ctx.predict_columns_device(xt, td_, match, b, None, pm_d, None)) for _ in range(reps)]
accd = float(np.mean(np.argmax(pm_d.view(td_, 10).cpu().numpy(), axis=1) == tcls))
print(f"MNIST-shaped 20x20x794, {td_} rows, 10 label columns from 784 (tier {ctx.last_score_tc}): host (pageable numpy) {td_ / min(ts) / 1e6:6.2f} M rows/s, "
      f"device {td_ / min(tsd) / 1e6:6.2f} M rows/s; label accuracy {acc:.4f} (device {accd:.4f})", flush=True)
ctx.close()
