"""Quick timing of the top-2 search (vsom_find_bmu2_device) against the single-BMU search (vsom_find_bmu_device) at the
config-4 scoring shape, 128 x 128 x 256 (not a test, not the bench): bench's trained scoring map (the recipe of
tests/test_gpu_benchmark_shapes._row_count_map("trained")) and the random-init map.  Rows are generated on the device around
bench's 64 cluster centres.  The two calls alternate after a warm-up; each line reports the best of the repeats, the tier
taken, the share of rows that went to the exact scan and the topographic error.  usage: bench_topo_quick.py [rows] [repeats]"""
import importlib
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
v = importlib.import_module("variational-self-organizing-maps_b200")

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 22
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
W, H, D = 128, 128, 256
F32 = np.float32

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {q.stdout.strip() or q.stderr.strip()}", flush=True)

# bench's generators (bench.py init_map / synth_chunk, as restated in tests/test_gpu_benchmark_shapes.py)
init = (np.random.default_rng(43).integers(-1000, 1000, (W * H, D), dtype=np.int16).astype(F32) / F32(1000.0)).astype(F32)
centres = (np.random.default_rng(1234 + 4).standard_normal((64, D)) * 3).astype(F32)
rng = np.random.default_rng(1234 + 40)
warm = (rng.standard_normal((20000, D), dtype=F32) + centres[rng.integers(0, 64, 20000)]).astype(F32)

gen = torch.Generator(device="cuda")
gen.manual_seed(7)
cd = torch.from_numpy(centres).cuda()
x = torch.empty((n, D), dtype=torch.float32, device="cuda")
blk = 1 << 20
for i in range(0, n, blk):
    k = min(blk, n - i)
    lab = torch.randint(0, 64, (k,), device="cuda", generator=gen)
    x[i:i + k] = torch.randn((k, D), device="cuda", generator=gen) + cd[lab]
b1 = torch.empty(n, dtype=torch.int32, device="cuda")
d1 = torch.empty(n, dtype=torch.float32, device="cuda")
b2 = torch.empty_like(b1)
d2 = torch.empty_like(d1)
print(f"{n} rows, {reps} repeats per path, alternating", flush=True)

for name in ("trained, sigma 32 -> 2", "random init"):
    ctx = v.VsomContext(W, H, D, v.STANDARD, v.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=init)
    if name.startswith("trained"):
        for i, (sg, eta) in enumerate(((32.0, 0.5), (16.0, 0.3), (8.0, 0.2), (4.0, 0.1), (2.0, 0.05))):
            ctx.train_chunk(warm[4000 * i:4000 * (i + 1)], eta, sg, v.EXPONENTIAL)
    runs = {
        "top-1": lambda: ctx.find_bmu_batch_device(x, n, b1, d1),
        "top-2": lambda: ctx.find_bmu2_device(x, n, b1, d1, b2, d2),
    }
    best = {k: 1e9 for k in runs}
    info = {}
    for k, f in runs.items():  # warm-up
        f()
        ctx.synchronize()
    for _ in range(reps):
        for k, f in runs.items():
            before = ctx.tc_stats()
            t0 = time.perf_counter()
            fb = f()
            ctx.synchronize()
            best[k] = min(best[k], time.perf_counter() - t0)
            after = ctx.tc_stats()
            info[k] = (ctx.last_score_tc, fb, {c: after[c] - before[c] for c in after})
    # the top-2 call ran last: b1 / b2 hold its results
    bx, by, sx, sy = b1 % W, b1 // W, b2 % W, b2 // W
    has = b2 != -1
    cheb = torch.maximum((bx - sx).abs(), (by - sy).abs())
    te = float(((cheb != 1) & has).sum().item()) / n
    for k in runs:
        tier, fb, causes = info[k]
        print(f"{name:24s} {k}: {n / best[k] / 1e6:8.2f} M rows/s  {best[k] * 1e3:8.2f} ms  tier {tier}  fallback {fb} ({100.0 * fb / n:.3f} %)  "
              f"causes {causes}", flush=True)
    print(f"{name:24s} top-2 / top-1 time {best['top-2'] / best['top-1']:.3f};  topographic error {te:.6f};  distinct BMUs {len(torch.unique(b1))}", flush=True)
    ctx.close()
