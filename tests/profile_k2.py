"""Small driver for ncu captures of the tensor-core scoring kernel (not a test): scores n rows twice against a 128x128x256
map (random init, or trained with a decaying sigma when the second argument is "trained").
Usage: [VSOM_TC_TIER=1|2] [VSOM_TC_PAIR=0|1] python tests/profile_k2.py [rows] [random|trained]"""
import importlib
import sys
import time

import numpy as np

sys.path.insert(0, ".")
v = importlib.import_module("variational-self-organizing-maps_b200")
import torch

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
kind = sys.argv[2] if len(sys.argv) > 2 else "random"
rng = np.random.default_rng(0)
W, H, D = 128, 128, 256
cent = (rng.standard_normal((64, D)) * 3).astype(np.float32)
data = lambda k: (rng.standard_normal((k, D), dtype=np.float32) + cent[rng.integers(0, 64, k)])
q = torch.from_numpy(data(n)).cuda()
ob = torch.empty(n, dtype=torch.int32, device="cuda")
od = torch.empty(n, dtype=torch.float32, device="cuda")
ctx = v.VsomContext(W, H, D, v.STANDARD, v.ORDER_EIGEN_SSE)
ctx.upload_state(mean=(rng.integers(-1000, 1000, (W * H, D)) / 1000).astype(np.float32))
if kind == "trained":
    for sg, eta in ((32, .5), (16, .3), (8, .2), (4, .1), (2, .05)):
        ctx.train_chunk(data(4000), eta, float(sg), v.EXPONENTIAL)
for _ in range(2):
    t0 = time.perf_counter()
    fb = ctx.find_bmu_batch_device(q, n, ob, od)
    ctx.synchronize()
    dt = time.perf_counter() - t0
print(f"profile_k2 {kind}: {n / dt / 1e6:.2f} M rows/s, tier {ctx.last_score_tc}, fallback {fb}")
