"""Quick timing of vsom_cluster_nodes (not a test, not the bench) on maps whose nodes fall into groups (rows around 2k random centres,
MNIST-scaled).  Per shape: the wall time of a full call (max_iter = 300, best of `repeats`) with its iterations, and the device time
of its phases from CUDA events inside the call (vsom_debug_cluster_phases): seeding, per assignment, per update, outputs.  Rates:
N k Dm terms per assignment (the exact scan, K3), and plane bytes per seeding pick (the seeding time, one plane check included,
over k) against the HBM data-sheet peak (7.7 TB/s).  For comparison, one host Lloyd iteration in numpy, best of `repeats`: the
distances expanded into one f32 matrix product on all host cores, the update as a sort by label plus np.add.reduceat.
usage: bench_cluster_quick.py [repeats]"""
import importlib
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
v = importlib.import_module("variational-self-organizing-maps_b200")

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
HBM_PEAK = 7.7e12

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {q.stdout.strip() or q.stderr.strip()}", flush=True)


def plane(N, Dm, centres, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    c = torch.randn((centres, Dm), device="cuda", generator=g) * 60.0 + 100.0
    idx = torch.randint(0, centres, (N,), device="cuda", generator=g)
    return (c[idx] + 10.0 * torch.randn((N, Dm), device="cuda", generator=g)).contiguous()


def numpy_lloyd_iteration(m, cent):
    def once():
        t0 = time.perf_counter()
        mn = np.einsum("ij,ij->i", m, m)
        cn = np.einsum("ij,ij->i", cent, cent)
        d = mn[:, None] - 2.0 * (m @ cent.T) + cn[None, :]
        lab = np.argmin(d, axis=1)
        order = np.argsort(lab, kind="stable")
        labs = lab[order]
        starts = np.flatnonzero(np.r_[True, labs[1:] != labs[:-1]])
        sums = np.add.reduceat(m[order].astype(np.float64), starts, axis=0)
        cnt = np.diff(np.r_[starts, len(labs)])
        _ = sums / cnt[:, None]
        return time.perf_counter() - t0
    return min(once() for _ in range(reps))


for (W, H, Dm, k) in ((64, 64, 128, 16), (128, 128, 256, 64), (512, 512, 784, 64), (512, 512, 784, 256)):
    N = W * H
    m_dev = plane(N, Dm, 2 * k, seed=k + Dm)
    m = m_dev.cpu().numpy()
    ctx = v.VsomContext(W, H, Dm, v.STANDARD, v.ORDER_REFERENCE)
    ctx.upload_state(mean=m)
    ctx.cluster_nodes(k, 1, v.CLUSTER_UNIFORM, 300)  # warm-up
    best, ph = 1e30, None
    for _ in range(reps):
        t0 = time.perf_counter()
        full = ctx.cluster_nodes(k, 1, v.CLUSTER_UNIFORM, 300)
        t = time.perf_counter() - t0
        if t < best:
            best, ph = t, ctx.cluster_phases()
    a = ph["assignments"]
    assign = ph["assign_ms"] / a
    update = ph["update_ms"] / (a - 1) if a > 1 else float("nan")
    pick = ph["seeding_ms"] * 1e-3 / k
    terms = N * k * Dm
    plane_bytes = N * Dm * 4
    tn = numpy_lloyd_iteration(m, full[1].astype(np.float32))
    print(f"{W}x{H}x{Dm} k={k}: full call {best * 1e3:8.2f} ms, {a} assignments (converged {full[5]}); device: seeding {ph['seeding_ms']:8.2f} ms "
          f"({pick * 1e6:6.1f} us per pick = {plane_bytes / pick / 1e9:7.1f} GB/s of plane, {plane_bytes / pick / HBM_PEAK * 100:5.1f} % of 7.7 TB/s), "
          f"assignment {assign:7.3f} ms each ({terms / (assign * 1e-3) / 1e12:5.2f} T terms/s, {terms / 1e9:.1f} G terms), update {update:7.3f} ms each, "
          f"outputs {ph['outputs_ms']:6.3f} ms; numpy Lloyd iteration {tn * 1e3:8.1f} ms on {os.cpu_count()} cores", flush=True)
    ctx.close()
    del m_dev
