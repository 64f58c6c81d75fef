#!/usr/bin/env python
"""bench.py — measures the VSOM hot path on B200 (contract: see DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload = BASELINE.json configs[1]: VSOM 64x64 grid, median-estimator transformation, synthetic 128-dim data,
1M samples per step (one step = one pass of the online training hot path over one 1M-sample chunk at the
epoch-0 schedule point eta=0.05, sigma=32).  `value` = training samples/s with the chunk already resident in HBM
(CUDA events on the library's stream); `e2e` = the same through the host-buffer C-ABI call
(vsom_train_chunk: H2D of the chunk + kernel + D2H of per-sample BMU / distance inside the timed region).
A second object, `scoring`, reports batch BMU scoring rows/s on the config-4 shape (128x128 map, D=256).

N > 1: the online step at this map size does not shard (per-sample dependency; DESIGN.md §Multi-GPU), so each
rank trains an independent replica on its own stream of samples ("replicas only", weak scaling); scoring shards
by rows with no communication.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

# ---- workload: BASELINE.json configs[1]
W_, H_, D_ = 64, 64, 128
ROWS_PER_STEP = 1_000_000
ETA, SIGMA = 0.05, 32.0
WORKLOAD = "VSOM 64x64 grid, median-estimator transformation, synthetic 128-dim data, 1M samples per step (BASELINE configs[1])"
# ---- scoring side workload: BASELINE.json configs[3]: 100M synthetic 256-dim rows against a 128x128 map,
#      data-sharded over the ranks (each rank generates its share on the device)
SW_, SH_, SD_ = 128, 128, 256
SCORE_ROWS = 100_000_000
SCORE_E2E_ROWS = 1 << 22      # host-buffer leg: 4 GiB of pinned rows per pass
AGREE_ROWS = 2048             # rows of the scoring workload the CPU reference scores as well, inside the run


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


def peaks_burst():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("bf16_tflops", 1676.6)
    return 1676.6


def measured_traffic(kernel, units):
    """DRAM bytes of one launch processing `units`, scaled from the committed ncu captures (profiles/r02_traffic.json)."""
    p = os.path.join(REPO, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        return None
    k = json.load(open(p)).get(kernel)
    if not k:
        return None
    return (k["dram_bytes_read"] + k["dram_bytes_write"]) / k["units"] * units


def synth_chunk(n, d, seed):
    """Config 2 data: x ~ N(mu_c, 1) from 64 cluster centres (SURVEY.md §8d)."""
    rng = np.random.default_rng(seed)
    centres = (rng.standard_normal((64, d)) * 3).astype(np.float32)
    lab = rng.integers(0, 64, n)
    x = rng.standard_normal((n, d), dtype=np.float32)
    x += centres[lab]
    return x


def init_map(n_nodes, dm, seed):
    """Same distribution as Som::randomInitialize(seed, 1.0f) (src/Som.cpp:977-997): multiples of 1/1000 in [-1, 1)."""
    rng = np.random.default_rng(seed)
    return (rng.integers(-1000, 1000, (n_nodes, dm), dtype=np.int16).astype(np.float32) / np.float32(1000.0)).astype(np.float32)


def window_nodes(w, h, sigma):
    """Mean update-window size over BMU positions is data dependent; at sigma=32 on 64x64 the window is the whole map."""
    r = 2.5 * sigma
    if r >= max(w, h):
        return w * h
    side = int(np.ceil(r)) + int(np.floor(r))
    return min(side, w) * min(side, h)


def algorithmic_bytes_per_sample(n_nodes, dm, d_in, k):
    """SURVEY.md §8(d): 4*N*Dm (scan) + 20*K*Dm (window: read m,S; write m,S,sigma) + 4*D_in + 8*K."""
    return 4 * n_nodes * dm + 20 * k * dm + 4 * d_in + 8 * k


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [t.strip() for t in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        self.f.close()
        os.unlink(self.f.name)
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the same step, on the box's host cores.
    Online training is single-threaded by construction (sample t+1 depends on sample t, src/Som.cpp:1161-1171),
    so `cores` is 1.  Each step is a bounded sample of the 1M-sample chunk."""
    if rank != 0:
        return
    from oracle import pyoracle as po

    cls, kind = po.best_cpu_checker(po.ORDER_EIGEN_SSE if args.order == "eigen_sse" else po.ORDER_SEQUENTIAL)
    eigen_kind = (po.ReferenceSse if args.order == "eigen_sse" else po.Reference).eigen_kind() if kind == "reference" else "plain C restatement"
    sample = 400
    x = synth_chunk(sample * (args.steps + args.warmup), D_, 1234 + 2)
    r = cls(W_, H_, D_, po.MEDIAN)
    r.set_state(mean=init_map(W_ * H_, D_, 42))
    for i in range(args.warmup):
        r.train_rows(x[i * sample:(i + 1) * sample], ETA, SIGMA, po.EXPONENTIAL)
    t0 = time.perf_counter()
    for i in range(args.warmup, args.warmup + args.steps):
        r.train_rows(x[i * sample:(i + 1) * sample], ETA, SIGMA, po.EXPONENTIAL)
    dt = time.perf_counter() - t0
    v = sample * args.steps / dt
    sample_txt = f"{sample} samples per step of the 1M-sample chunk, 1 thread ({'reference TUs compiled unmodified; Eigen: ' + eigen_kind if kind == 'reference' else 'C port'})"
    print(json.dumps({
        "impl": "reference", "metric": "train_samples_per_s", "value": v, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD, "eta": ETA, "sigma": SIGMA, "decay": "Exponential", "reduction_order": args.order},
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": 1, "kind": kind, "sample": sample_txt, "ref_eigen_kind": eigen_kind},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def score_map_state(vsom, device, order):
    """The scoring map: random init like Som::randomInitialize, then a brief online training on the scoring distribution
    (SURVEY.md 8d-4: "trained briefly": 20000 samples, sigma 32 -> 2) so that neighbouring nodes resemble each other like on a
    real map — the case that matters: on such a map a single fp16 pass cannot separate the BMU from its neighbours and the
    library's probe switches to the hi / lo tier.  Deterministic
    (fixed seeds, bit-exact kernels): every rank builds the same replica."""
    ctx = vsom.VsomContext(SW_, SH_, SD_, vsom.STANDARD, order, device=device)
    ctx.upload_state(mean=init_map(SW_ * SH_, SD_, 43))
    # the SAME distribution the scored rows come from (same 64 cluster centres: first draw of seed 1234 + 4), other rows
    centres = (np.random.default_rng(1234 + 4).standard_normal((64, SD_)) * 3).astype(np.float32)
    rng = np.random.default_rng(1234 + 40)
    warm = (rng.standard_normal((20000, SD_), dtype=np.float32) + centres[rng.integers(0, 64, 20000)]).astype(np.float32)
    for i, (sg, eta) in enumerate(((32.0, 0.5), (16.0, 0.3), (8.0, 0.2), (4.0, 0.1), (2.0, 0.05))):  # sigma decays like a real schedule
        ctx.train_chunk(warm[4000 * i:4000 * (i + 1)], eta, sg, vsom.EXPONENTIAL)
    return ctx


def cpu_baseline_leg(train_gpu, score_state, score_rows_host, score_gpu, order_name):
    """The reference's own code (oracle/_ref) on one host core, bounded samples; and, from the same outputs, the measured
    BMU / distance agreement of the GPU path on identical inputs, state and order (north_star: "agreement rate reported").
    train_gpu(x, init) -> (bmu, dist) of the GPU online step; score_gpu = (bmu, dist) of the GPU scoring call."""
    from oracle import pyoracle as po

    sse = order_name == "eigen_sse"
    cls, kind = po.best_cpu_checker(po.ORDER_EIGEN_SSE if sse else po.ORDER_SEQUENTIAL)
    eigen_kind = (po.ReferenceSse if sse else po.Reference).eigen_kind() if kind == "reference" else "plain C restatement (" + order_name + " dot)"
    sample = 1500
    x = synth_chunk(sample + 100, D_, 1234 + 2)
    init = init_map(W_ * H_, D_, 42)
    r = cls(W_, H_, D_, po.MEDIAN)
    r.set_state(mean=init)
    b0, d0, _, _ = r.train_rows(x[:100], ETA, SIGMA, po.EXPONENTIAL)
    t0 = time.perf_counter()
    b1, d1, _, _ = r.train_rows(x[100:], ETA, SIGMA, po.EXPONENTIAL)
    dt = time.perf_counter() - t0
    out = {"value": sample / dt, "unit": "samples/s", "cores": 1, "kind": kind, "ref_eigen_kind": eigen_kind,
           "sample": f"first {sample} samples of the step's chunk after 100 warm-up samples, 1 thread (the path is sequential by construction)"}
    gb, gd = train_gpu(x, init)
    rb, rd = np.concatenate([b0, b1]), np.concatenate([d0, d1])
    out["train_agreement"] = {"samples": int(len(rb)), "bmu_equal": float(np.mean(gb == rb)), "dist_bits_equal": float(np.mean(gd.view(np.uint32) == rd.view(np.uint32))),
                              "what": "BMU sequence and distance-to-updated-BMU of the GPU online step vs the CPU reference, same init, same samples, same order"}
    # scoring side: Som::findBmu per row on the config-4 shape and map, 1 thread, bounded
    rs = cls(SW_, SH_, SD_, po.STANDARD)
    rs.set_state(**score_state)
    t0 = time.perf_counter()
    sb, sd = rs.find_bmu(score_rows_host)
    dt = time.perf_counter() - t0
    out["scoring"] = {"value": len(sb) / dt, "unit": "rows/s", "cores": 1, "sample": f"first {len(sb)} rows of the scoring workload, 128x128 map, D=256, 1 thread"}
    out["scoring_agreement"] = {"rows": int(len(sb)), "bmu_equal": float(np.mean(score_gpu[0] == sb)),
                                "dist_bits_equal": float(np.mean(score_gpu[1].view(np.uint32) == sd.view(np.uint32))),
                                "what": "BMU ids and f32 distances of the GPU scoring call (tensor-core search + exact rescore) vs the CPU reference on the same rows and map"}
    return out


DUMP_ROWS = 1 << 21  # per-sample outputs of up to this many rows are dumped whole, larger chunks as a fixed sample (dump < 64 MB)


def dump_outputs(out_dir, ctx, bmu_dev, dist_dev, n):
    """--dump-outputs: what the last timed step hands its caller, as <name>.npy: the per-sample BMU ids and distances it wrote
    into the caller's buffers, and the map it leaves behind (mean, S, sigma, weight, hits).  Integers are written as float64,
    which holds them exactly.  Above DUMP_ROWS samples, bmu / dist are taken at a fixed seeded set of rows, stored as row.npy."""
    os.makedirs(out_dir, exist_ok=True)
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    out = {"bmu": bmu_dev.cpu().numpy()[rows].astype(np.float64), "dist": dist_dev.cpu().numpy()[rows]}
    if n > DUMP_ROWS:
        out["row"] = rows.astype(np.float64)
    st = ctx.download_state()
    out.update(mean=st["mean"], S=st["S"], sigma=st["sigma"], weight=st["weight"], hits=st["hits"].astype(np.float64))
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def _claim_stdout():
    """Libraries under us (NCCL's version banner) write to the C-level stdout; the contract is ONE JSON line there.  Point fd 1 at
    stderr for the run and keep the real stdout for the result line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    sys.stdout = _claim_stdout()  # Python-level prints (the result line) keep going to the real stdout
    global SCORE_ROWS
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--order", default="eigen_sse", choices=["eigen_sse", "reference", "lanes"],
                    help="summation order of every distance: eigen_sse = dot() as real Eigen compiles it under the reference's -msse2 release flags "
                         "(what a user who installed libeigen3-dev runs); reference = sequential (the stand-in Eigen header); lanes = 32 partial sums (K1 only)")
    ap.add_argument("--rows", type=int, default=ROWS_PER_STEP)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--score-rows", type=int, default=SCORE_ROWS)
    ap.add_argument("--no-large-map", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--large-rows", type=int, default=1024)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (rank 0); the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    SCORE_ROWS = args.score_rows

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    vsom = importlib.import_module("variational-self-organizing-maps_b200")
    sharding = importlib.import_module("variational-self-organizing-maps_b200.sharding")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this framework has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n = args.rows
    order = {"reference": vsom.ORDER_REFERENCE, "lanes": vsom.ORDER_LANES, "eigen_sse": vsom.ORDER_EIGEN_SSE}[args.order]
    ctx = vsom.VsomContext(W_, H_, D_, vsom.MEDIAN, order, device=local_rank)
    ctx.upload_state(mean=init_map(W_ * H_, D_, 42 + rank))
    stream = torch.cuda.ExternalStream(ctx.stream, device=local_rank)

    x_host = torch.from_numpy(synth_chunk(n, D_, 1234 + 2 + rank)).pin_memory()
    x_dev = x_host.to(f"cuda:{local_rank}", non_blocking=False)
    out_bmu = torch.empty(n, dtype=torch.int32, device=x_dev.device)
    out_dist = torch.empty(n, dtype=torch.float32, device=x_dev.device)

    # ---------------- value: chunk resident in HBM, CUDA events on the launching stream
    for _ in range(args.warmup):
        ctx.train_chunk_device(x_dev, n, ETA, SIGMA, vsom.EXPONENTIAL, out_bmu, out_dist)
    ctx.synchronize()
    barrier()
    launches0 = ctx.launch_count
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    with torch.cuda.stream(stream):
        ev[0].record(stream)
        for i in range(args.steps):
            ctx.train_chunk_device(x_dev, n, ETA, SIGMA, vsom.EXPONENTIAL, out_bmu, out_dist)
            ev[i + 1].record(stream)
    ctx.synchronize()
    barrier()
    clocks = sampler.stop() if sampler else None
    launches = ctx.launch_count - launches0
    if args.dump_outputs and rank == 0:  # before the legs below reuse out_bmu / out_dist and train this map further
        dump_outputs(args.dump_outputs, ctx, out_bmu, out_dist, n)
    k1_name = "online_step_fast_kernel" if ctx.last_train_fast else "online_step_kernel"
    total_ms = ev[0].elapsed_time(ev[-1])
    kernel_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    t = torch.tensor([total_ms], dtype=torch.float64, device=x_dev.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = world * n * args.steps / (total_ms / 1e3)

    # ---------------- diagnostics (untimed): per-phase cycles of the persistent kernel on a 100k-sample chunk
    ctx.debug_profile(True)
    ctx.train_chunk_device(x_dev, min(n, 100_000), ETA, SIGMA, vsom.EXPONENTIAL, out_bmu, out_dist)
    ctx.synchronize()
    phases = ctx.debug_phase_cycles()
    phases_raw = ctx.debug_phase_cycles_raw()
    die_aware = ctx.die_aware
    ctx.debug_profile(False)
    onchip = ctx.measure_peaks()  # shared-memory and L2 read bandwidth of THIS device, measured now (csrc/peaks.cu)

    # ---------------- e2e: host buffers through the reference-facing C-ABI call, copies inside the timed region
    x_np = x_host.numpy()
    e2e_steps = max(1, min(args.steps, 3))
    ctx.train_chunk(x_np, ETA, SIGMA, vsom.EXPONENTIAL)  # warm-up at the timed size: the library sizes its staging buffers on first use
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        bmu, d, r2, last = ctx.train_chunk(x_np, ETA, SIGMA, vsom.EXPONENTIAL)
        mse = float(np.float32(r2.sum(dtype=np.float64) / n))  # the step's result (per-epoch MSE term), read on the host
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=x_dev.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * n * e2e_steps / float(t.item())

    # ---------------- scoring side (BASELINE configs[3]): SCORE_ROWS rows against a 128x128 map, D=256, data-sharded over the
    #   ranks, rows generated on the device and resident in HBM before the timed region.  The call is the reference-facing
    #   vsom_find_bmu_device (what Som::evaluate / measureSimilarity / mapDataSet reach): K2 tcgen05 candidate search +
    #   exact f32 rescore + certificate (+ exact scan of the rows it rejects).
    dev = x_dev.device
    del x_dev, out_bmu, out_dist
    torch.cuda.empty_cache()
    sctx = score_map_state(vsom, local_rank, vsom.ORDER_EIGEN_SSE if args.order == "eigen_sse" else vsom.ORDER_REFERENCE)
    score_state = sctx.download_state() if rank == 0 else None
    sstream = torch.cuda.ExternalStream(sctx.stream, device=local_rank)
    rows_rank = SCORE_ROWS // world
    free_b, _ = torch.cuda.mem_get_info()
    fit = int((free_b - (14 << 30)) // (SD_ * 4 + 8))  # leave room for the bf16 slab, scratch and the later legs
    score_note = None
    if rows_rank > fit:
        score_note = f"{rows_rank} rows per GPU do not fit next to the scratch buffers; ran {fit}"
        rows_rank = fit
    q_dev = torch.empty((rows_rank, SD_), dtype=torch.float32, device=dev)
    centres_d = torch.from_numpy((np.random.default_rng(1234 + 4).standard_normal((64, SD_)) * 3).astype(np.float32)).to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + 4 + rank)
    blk = 1 << 21
    for i0 in range(0, rows_rank, blk):  # x ~ N(mu_c, 1) from 64 cluster centres, like synth_chunk, generated on the device
        i1 = min(rows_rank, i0 + blk)
        torch.randn((i1 - i0, SD_), generator=gen, out=q_dev[i0:i1])
        q_dev[i0:i1] += centres_d[torch.randint(0, 64, (i1 - i0,), generator=gen, device=dev)]
    agree_rows = min(AGREE_ROWS, rows_rank)
    agree_host = synth_chunk(agree_rows, SD_, 1234 + 4)  # the parity subset is produced on the host: the same rows for the CPU reference
    q_dev[:agree_rows] = torch.from_numpy(agree_host).to(dev)
    s_bmu = torch.empty(rows_rank, dtype=torch.int32, device=dev)
    s_dist = torch.empty(rows_rank, dtype=torch.float32, device=dev)
    torch.cuda.synchronize()

    def timed(fn, warm=True):
        if warm:
            fn()  # warm-up (also sizes the staging buffers)
        sctx.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(sstream):
            e0.record(sstream)
            out = fn()
            e1.record(sstream)
        sctx.synchronize()
        barrier()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item()), out

    # warm-up on 2M rows; it also bounds the leg: if this map makes the run far slower than planned (rows ending in the
    # exact scan), fewer rows are timed and the line says so
    t0 = time.perf_counter()
    sctx.find_bmu_batch_device(q_dev, min(rows_rank, 1 << 21), s_bmu, s_dist)
    sctx.synchronize()
    warm_rate = min(rows_rank, 1 << 21) / (time.perf_counter() - t0)
    if rows_rank / warm_rate > 40.0:
        score_note = (score_note + "; " if score_note else "") + f"warm-up ran at {warm_rate / 1e6:.2f} M rows/s: timed {int(warm_rate * 30)} rows instead of {rows_rank} to stay within the time budget"
        rows_rank = int(warm_rate * 30) // 128 * 128
    ssampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = sctx.launch_count
    score_ms, fallback_rows = timed(lambda: sctx.find_bmu_batch_device(q_dev, rows_rank, s_bmu, s_dist), warm=False)
    score_launches = sctx.launch_count - l0
    score_clocks = ssampler.stop() if ssampler else None
    assert sctx.last_score_tc
    score_tier = sctx.last_score_tc
    # the same rows against the map BEFORE training (random init, Som::randomInitialize's distribution): the single-pass tier
    rctx = vsom.VsomContext(SW_, SH_, SD_, vsom.STANDARD, sctx.order, device=local_rank)
    rctx.upload_state(mean=init_map(SW_ * SH_, SD_, 43))
    rrows = min(rows_rank, 1 << 23)
    rctx.find_bmu_batch_device(q_dev, min(rrows, 1 << 21), s_bmu, s_dist)
    rctx.synchronize()
    barrier()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rs = torch.cuda.ExternalStream(rctx.stream, device=local_rank)
    with torch.cuda.stream(rs):
        r0.record(rs)
        rfb = rctx.find_bmu_batch_device(q_dev, rrows, s_bmu, s_dist)
        r1.record(rs)
    rctx.synchronize()
    rt = torch.tensor([r0.elapsed_time(r1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(rt, op=dist.ReduceOp.MAX)
    random_map = {"value": world * rrows / (float(rt.item()) / 1e3), "unit": "rows/s", "rows": rrows * world, "tier": rctx.last_score_tc, "fallback_rows": rfb,
                  "frac_of_sustained_peak": world * rrows / (float(rt.item()) / 1e3) / world * 2 * SW_ * SH_ * SD_ / 1e12 / peaks()[1],
                  "what": "same rows, same shape, map as Som::randomInitialize leaves it (no training): nodes far apart, one fp16 pass certifies every row"}
    rctx.close()
    sctx.find_bmu_batch_device(q_dev, min(rows_rank, agree_rows), s_bmu, s_dist)  # the parity rows again (s_bmu was reused above)
    score_rows_s = world * rows_rank / (score_ms / 1e3)
    score_gpu = (s_bmu[:agree_rows].cpu().numpy().view(np.uint32), s_dist[:agree_rows].cpu().numpy())
    exact_rows = 1 << 18
    exact_ms, _ = timed(lambda: sctx.find_bmu_exact_device(q_dev, exact_rows, s_bmu, s_dist))
    exact_rows_s = world * exact_rows / (exact_ms / 1e3)
    # ---- K5, SomIndex build on the scoring result: histogram of the BMU ids + rows grouped by BMU (stable radix sort)
    idx_rows = min(rows_rank, 1 << 24)
    i_counts = torch.empty(SW_ * SH_, dtype=torch.int64, device=dev)
    i_offsets = torch.empty(SW_ * SH_ + 1, dtype=torch.int64, device=dev)
    i_rows = torch.empty(idx_rows, dtype=torch.int32, device=dev)
    sctx.find_bmu_batch_device(q_dev, idx_rows, s_bmu, s_dist)  # the exact-scan timing above overwrote the first rows (same values; keep it simple)
    idx_ms, _ = timed(lambda: sctx.build_index_device(s_bmu, idx_rows, i_counts, i_offsets, i_rows))
    idx_passes = (int(np.ceil(np.log2(SW_ * SH_))) + 7) // 8
    idx_bytes = idx_rows * (4 + 16 * idx_passes)  # histogram reads the ids once; every radix pass reads and writes (key, row id)
    idx_ok = bool((i_counts.sum().item() == idx_rows) and (i_offsets[-1].item() == idx_rows))
    index_leg = {"kernel": "K5 index_hist + radix sort (som_index.cu)", "rows": idx_rows * world, "ms": idx_ms, "value": world * idx_rows / (idx_ms / 1e3), "unit": "rows/s",
                 "algorithmic_bytes": idx_bytes, "achieved_gbs_per_gpu": idx_bytes / (idx_ms / 1e3) / 1e9, "frac_of_hbm_peak": idx_bytes / (idx_ms / 1e3) / 1e9 / peaks()[0],
                 "radix_passes": idx_passes, "counts_sum_to_rows": idx_ok}
    del i_rows

    # ---- scoring end to end: pinned HOST rows through vsom_find_bmu (the C-ABI call behind Som::evaluate): H2D of slab
    #   i + 1, search + re-scoring of slab i and D2H of slab i - 1 overlap inside the call.  The PCIe ceiling is measured
    #   beside it: a plain pinned H2D copy of the same buffer.
    e2e_rows = min(SCORE_E2E_ROWS, rows_rank)
    q_pin = torch.empty((e2e_rows, SD_), dtype=torch.float32, pin_memory=True)
    q_pin.copy_(q_dev[:e2e_rows])
    b_pin = torch.empty(e2e_rows, dtype=torch.int32, pin_memory=True)
    d_pin = torch.empty(e2e_rows, dtype=torch.float32, pin_memory=True)
    sctx.find_bmu_host_ptr(q_pin.data_ptr(), min(e2e_rows, 1 << 20), b_pin.data_ptr(), d_pin.data_ptr())  # sizes the staging buffers
    barrier()
    se2e_calls = 2
    t0 = time.perf_counter()
    for _ in range(se2e_calls):  # each call returns with the per-row BMU ids and distances in the caller's (pinned) host arrays
        sctx.find_bmu_host_ptr(q_pin.data_ptr(), e2e_rows, b_pin.data_ptr(), d_pin.data_ptr())
    se2e_s = (time.perf_counter() - t0) / se2e_calls
    score_err = float(d_pin.double().mean())  # Som::evaluate's mean BMU distance from the returned host array (outside the timed region)
    # anomaly scoring end to end (the per-row pass of Som::measureSimilarity): BMU + largest normalised deviation per row, same rows
    r_pin = torch.empty(e2e_rows, dtype=torch.float32, pin_memory=True)
    sctx.measure_similarity_host_ptr(q_pin.data_ptr(), min(e2e_rows, 1 << 20), 3, b_pin.data_ptr(), r_pin.data_ptr())
    barrier()
    t0 = time.perf_counter()
    sctx.measure_similarity_host_ptr(q_pin.data_ptr(), e2e_rows, 3, b_pin.data_ptr(), r_pin.data_ptr())
    sim_s = time.perf_counter() - t0
    tsim = torch.tensor([sim_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tsim, op=dist.ReduceOp.MAX)
    sim_e2e = world * e2e_rows / float(tsim.item())
    sim_finite = float(torch.isfinite(r_pin).float().mean())
    tt = torch.tensor([se2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    score_e2e = world * e2e_rows / float(tt.item())
    e2e_matches = bool(np.array_equal(b_pin[:agree_rows].numpy().view(np.uint32), score_gpu[0]) and
                       np.array_equal(d_pin[:agree_rows].numpy().view(np.uint32), score_gpu[1].view(np.uint32)))
    tmp_dev = torch.empty((e2e_rows, SD_), dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    tmp_dev.copy_(q_pin, non_blocking=True)
    torch.cuda.synchronize()
    h2d_gbs = q_pin.numel() * 4 / (time.perf_counter() - t0) / 1e9
    del tmp_dev, q_pin, q_dev
    torch.cuda.empty_cache()

    # ---------------- large map (BASELINE configs[4] shape): 512x512 grid x 784-dim, online training with the grid rows
    #   node-sharded over the `world` GPUs (in-kernel NVLink min-loc exchange per sample); at N=1 the same map on one GPU,
    #   plus the full U-matrix.  Reported honestly either way.
    large = None
    if not args.no_large_map:
        LW, LH, LD, LROWS, LSIG = 512, 512, 784, args.large_rows, 16.0
        lctx = vsom.VsomContext(LW, LH, LD, vsom.STANDARD, order, device=local_rank, rank=rank, world=world)
        if world > 1:
            handles = [None] * world
            dist.all_gather_object(handles, lctx.peer_export())
            for r, hdl in enumerate(handles):
                lctx.peer_import(r, hdl)
        # the SAME initial map whatever the number of ranks (every rank draws the full map and uploads its share), so that
        # the BMU sequence can be compared across N: bmu_crc32 / dist_crc32 below must not depend on --gpus
        full = init_map(LW * LH, LD, 4242)
        lctx.upload_state(mean=full)
        del full
        lx = torch.from_numpy(synth_chunk(LROWS, LD, 777)).to(dev)  # the same samples on every rank
        lb = torch.empty(LROWS, dtype=torch.int32, device=dev)
        ld_ = torch.empty(LROWS, dtype=torch.float32, device=dev)
        lstream = torch.cuda.ExternalStream(lctx.stream, device=local_rank)
        lctx.train_chunk_device(lx, min(LROWS, 64), 0.05, LSIG, vsom.EXPONENTIAL, lb, ld_)
        lctx.synchronize()
        ld_.view(torch.int32).fill_(-1)  # sharded: only the owner of a sample's BMU writes its distance
        torch.cuda.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(lstream):
            e0.record(lstream)
            lctx.train_chunk_device(lx, LROWS, 0.05, LSIG, vsom.EXPONENTIAL, lb, ld_)
            e1.record(lstream)
        lctx.synchronize()
        barrier()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        lms = float(tt.item())
        # per-sample BMU (known to every rank) and distance to the updated BMU (reported by the rank that owns it; the others
        # hold 0xffffffff = -1 as int32, so an integer max over ranks keeps the owner's bits)
        lbits = ld_.view(torch.int32).clone()
        if world > 1:
            dist.all_reduce(lbits, op=dist.ReduceOp.MAX)
        bmu_crc = zlib.crc32(lb.cpu().numpy().tobytes())
        dist_crc = zlib.crc32(lbits.cpu().numpy().tobytes())
        kwin = min(int(np.ceil(2.5 * LSIG)) + int(np.floor(2.5 * LSIG)), LW) ** 2
        lbytes = algorithmic_bytes_per_sample(LW * LH, LD, LD, kwin)
        large = {"workload": "512x512 grid x 784-dim online training (BASELINE configs[4] shape), sigma=16, Standard, Exponential",
                 "layout": "single GPU" if world == 1 else f"grid rows dealt to {world} GPUs round-robin in blocks of {lctx.shard_rows()[0]} rows, per-sample 8-byte min-loc exchange inside the persistent kernel over NVLink peer memory",
                 "samples": LROWS, "bmu_crc32": bmu_crc, "dist_crc32": dist_crc,
                 "crc_note": "CRC-32 of the timed chunk's per-sample BMU ids / distance bits: equal for every --gpus N (same map, same samples, bit-exact kernels)",
                 "ms": lms, "value": LROWS / (lms / 1e3), "unit": "samples/s", "us_per_sample": 1e3 * lms / LROWS,
                 "roofline": {"bound": "hbm", "algorithmic_bytes_per_sample": lbytes, "achieved": lbytes * LROWS / (lms / 1e3) / 1e9 / world,
                              "unit": "GB/s per GPU", "window_nodes": kwin},
                 "planes_resident_in_smem": lctx.planes_resident, "reduction_order": args.order}
        if world == 1:
            large["roofline"]["traffic"] = measured_traffic("online_step_kernel_large_map", LROWS)
            large["roofline"]["traffic_source"] = "profiles/r02_traffic.json (ncu --set full of the streamed-scan kernel, scaled per sample)"
        # full U-matrix of the large map (config 5: "plus full UMatrix"): every rank computes its own grid rows; on sharded
        # contexts the border rows of means are read from the neighbours' planes over NVLink first (inside the timed call)
        barrier()
        um_host = lctx.update_umatrix()  # warm-up + the values
        barrier()
        with torch.cuda.stream(lstream):
            e0.record(lstream)
            lib_rc = vsom.lib().vsom_update_umatrix(lctx._h, None)
            e1.record(lstream)
        lctx.synchronize()
        barrier()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        umt = torch.from_numpy(um_host.view(np.int64).copy()).to(dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(umt)  # the rows of other ranks are zero
        ums = float(tt.item())
        ubytes = 8 * LW * LH * LD + 8 * LW * LH
        halo = len(sharding.halo_rows(LH, rank, world)) if world > 1 else 0
        large["umatrix"] = {"ms": ums, "algorithmic_bytes": ubytes, "achieved_gbs_per_gpu": ubytes / world / (ums / 1e3) / 1e9, "frac_of_hbm_peak": ubytes / world / (ums / 1e3) / 1e9 / peaks()[0],
                            "halo_rows_per_gpu": halo, "halo_bytes_per_gpu": halo * LW * LD * 4, "crc32": zlib.crc32(umt.cpu().numpy().tobytes()),
                            "layout": "single GPU" if world == 1 else f"grid rows in blocks of {lctx.shard_rows()[0]} dealt round-robin to {world} GPUs, halo rows over NVLink peer memory"}
        lctx.close()
        del lx

    # ---------------- the other named training shapes, short runs (resident chunk, CUDA events): BASELINE configs[0]
    #   (20x20, Standard, 784-dim — K1F) and configs[2] (50x50, combinatorial linear regression at J = 32 — generic K1)
    others = []
    if not args.no_other_configs:
        def clr_chunk(n, j, seed):
            rng = np.random.default_rng(seed)
            z = rng.standard_normal((n, 1)).astype(np.float32)
            a = rng.uniform(0.5, 1.5, (1, j)).astype(np.float32)
            bb = rng.uniform(-1, 1, (1, j)).astype(np.float32)
            return (a * z + bb + 0.1 * rng.standard_normal((n, j))).astype(np.float32)

        for name, (ow, oh, od, otr, oeta, osig, orows) in (("configs[0]: 20x20 grid, Standard, 784-dim", (20, 20, 784, vsom.STANDARD, 0.1, 10.0, 60000)),
                                                            ("configs[2]: 50x50 grid, combinatorial linear regression J=32 (992 parameters / node)", (50, 50, 32, vsom.CLR, 0.001, 25.0, 60000))):
            octx = vsom.VsomContext(ow, oh, od, otr, order, device=local_rank)
            odm = vsom.model_length(od, otr)
            octx.upload_state(mean=init_map(ow * oh, odm, 99 + rank))
            ox_np = clr_chunk(orows, od, 31 + rank) if otr == vsom.CLR else np.floor(256 * np.random.default_rng(5 + rank).random((orows, od), dtype=np.float32) ** 2).astype(np.float32)
            ox = torch.from_numpy(ox_np).to(dev)
            ob_ = torch.empty(orows, dtype=torch.int32, device=dev)
            od_ = torch.empty(orows, dtype=torch.float32, device=dev)
            ostream = torch.cuda.ExternalStream(octx.stream, device=local_rank)
            octx.train_chunk_device(ox, orows // 10, oeta, osig, vsom.EXPONENTIAL, ob_, od_)
            octx.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(ostream):
                e0.record(ostream)
                octx.train_chunk_device(ox, orows, oeta, osig, vsom.EXPONENTIAL, ob_, od_)
                e1.record(ostream)
            octx.synchronize()
            oms = e0.elapsed_time(e1)
            octx.debug_profile(True)
            octx.train_chunk_device(ox, min(orows, 20000), oeta, osig, vsom.EXPONENTIAL, ob_, od_)
            octx.synchronize()
            ophases = octx.debug_phase_cycles_raw()
            octx.debug_profile(False)
            kw = window_nodes(ow, oh, osig)
            obytes = algorithmic_bytes_per_sample(ow * oh, odm, od, kw)
            others.append({"workload": name, "samples": orows, "ms": oms, "value": orows / (oms / 1e3), "unit": "samples/s (per GPU)",
                           "kernel": "online_step_fast_kernel" if octx.last_train_fast else "online_step_kernel", "eta": oeta, "sigma": osig,
                           "algorithmic_bytes_per_sample": obytes, "achieved_gbs": obytes * orows / (oms / 1e3) / 1e9,
                           "roofline": {"bound": "smem", "achieved": obytes * orows / (oms / 1e3) / 1e9, "peak": onchip["smem_gbs"], "unit": "GB/s",
                                        "frac": obytes * orows / (oms / 1e3) / 1e9 / onchip["smem_gbs"]},
                           "phase_cycles_per_sample": ophases, "cycles_per_sample": sum(ophases.values())})
            octx.close()

    # ---------------- K6, batch-map trainer: one chunk-epoch (BMU of every row, then every neuron re-estimated from all rows in
    #   row order) on the configs[0] shape, through the host-buffer C-ABI call (vsom_batch_epoch: H2D inside)
    batch_leg = None
    if not args.no_other_configs:
        bw, bh, bd, brows = 20, 20, 784, 60000
        bctx = vsom.VsomContext(bw, bh, bd, vsom.STANDARD, vsom.ORDER_EIGEN_SSE if args.order == "eigen_sse" else vsom.ORDER_REFERENCE, device=local_rank)
        bctx.upload_state(mean=init_map(bw * bh, bd, 99 + rank))
        bx = np.floor(256 * np.random.default_rng(5 + rank).random((brows, bd), dtype=np.float32) ** 2).astype(np.float32)
        bx_pinned = torch.from_numpy(bx).pin_memory()  # the caller's chunk in page-locked memory, like the e2e legs
        bx = bx_pinned.numpy()
        bctx.batch_epoch(bx, 5.0, True)  # warm-up at the timed size (staging buffers are allocated on first use); this is epoch 1, the global search
        barrier()
        t0 = time.perf_counter()
        b_mse, _ = bctx.batch_epoch(bx, 5.0, False)  # a steady-state epoch: local walks from the previous BMUs, then the re-estimation
        b_s = time.perf_counter() - t0
        tt = torch.tensor([b_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        b_s = float(tt.item())
        updates = bw * bh * bd * brows  # (neuron, component, row) steps of the sequential West / Finch chains
        batch_leg = {"kernel": "K6 local_bmu_rows_kernel + batch_update_kernel", "workload": "20x20 grid, Standard, 784-dim, one steady-state chunk-epoch (the second) over 60000 rows, sigma = 5 (per GPU)",
                     "ms": b_s * 1e3, "value": world * brows / b_s, "unit": "row-epochs/s", "chain_steps_per_s_per_gpu": updates / b_s,
                     "bound": "fp32 issue (each chain step is 6 dependent f32 operations; 148 SMs x 128 lanes)",
                     "frac_of_fp32_issue_peak": updates * 6 / b_s / (148 * 128 * 1.9e9), "mse": b_mse, "includes": "H2D of the chunk (188 MB, pinned) and D2H of per-row BMU / residual"}
        bctx.close()

    if rank == 0:
        hbm_gbs, bf16_tf, peak_src = peaks()
        bf16_burst = peaks_burst()
        k = window_nodes(W_, H_, SIGMA)
        bps = algorithmic_bytes_per_sample(W_ * H_, D_, D_, k)
        kern_s = statistics.mean(kernel_ms) / 1e3
        achieved = bps * n / kern_s / 1e9
        resident = bool(ctx.planes_resident)
        line = {
            "metric": "train_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "eta": ETA, "sigma": SIGMA, "decay": "Exponential", "rows_per_step": n,
                       "reduction_order": args.order, "parity": "measured in this run: cpu_baseline.train_agreement / scoring_agreement",
                       "planes_resident_in_smem": ctx.planes_resident,
                       "parallelism": "1 persistent kernel / chunk" if world == 1 else f"{world} independent replicas (online step does not shard at this map size)",
                       "l2": "input chunk 512 MB > 126 MB L2; no flush needed"},
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": n * D_ * 4, "d2h_bytes_per_step": n * 12, "steps": e2e_steps,
                    "result_read": "per-sample BMU, distance, residual^2 + MSE on host", "mse": mse},
            "gpu_launches": launches,
            "k1_phase_cycles_per_sample": phases, "k1_phase_cycles_raw": phases_raw, "k1_exchange_rows_by_l2_die": die_aware,
            "clocks": clocks,
            "roofline": {"bound": "smem" if resident else "hbm", "achieved": achieved, "peak": onchip["smem_gbs"] if resident else hbm_gbs, "unit": "GB/s",
                         "frac": achieved / (onchip["smem_gbs"] if resident else hbm_gbs), "traffic": measured_traffic(k1_name, n),
                         "traffic_source": "profiles/r02_traffic.json (ncu --set full, scaled per sample): DRAM bytes, a tiny fraction of the algorithmic bytes because the map stays on chip",
                         "peak_source": "measured in this run (vsom_debug_measure_peaks, csrc/peaks.cu): aggregate conflict-free LDS.128 read bandwidth of the 148 SMs" if resident else peak_src,
                         "algorithmic_bytes_per_sample": bps, "window_nodes": k, "kernel": k1_name, "kernel_ms_per_launch": kern_s * 1e3,
                         "measured_peaks_gbs": {"smem_all_sms": onchip["smem_gbs"], "smem_per_sm": onchip["smem_gbs_per_sm"], "l2_read": onchip["l2_gbs"], "l2_set_mib": onchip["l2_set_mib"], "hbm_copy": hbm_gbs},
                         "frac_of_l2_peak": achieved / onchip["l2_gbs"], "frac_of_hbm_peak": achieved / hbm_gbs,
                         "latency_note": "the step is latency-bound by the strict sample-to-sample dependency: see k1_phase_cycles_raw (cycles per sample and phase); "
                                         "the bandwidth fraction is reported because the contract asks for it, the phase table is what explains the kernel"},
            "scoring": {"metric": "bmu_scoring_rows_per_s", "value": score_rows_s, "unit": "rows/s", "rows": rows_rank * world, "rows_per_gpu": rows_rank, "ms": score_ms,
                        "workload": "BASELINE configs[3]: 100M synthetic 256-dim rows against a 128x128 map (random init + 20000 online steps on the same distribution, sigma 32 -> 2), rows generated on the device, "
                                    "resident in HBM, data-sharded over the ranks",
                        "note": score_note,
                        "call": "vsom_find_bmu_device (the reference-facing scoring call: Som::evaluate / measureSimilarity / mapDataSet dispatch to it)",
                        "kernel": "K2 score_tc_kernel (tcgen05 fp16 candidate search, margin lists of <= 48 nodes) + exact f32 rescore + certificate + exact scan of rejected rows",
                        "tier": score_tier, "tier_note": "1 = one fp16 value per operand element (2 N D tensor flops per row); 2 = hi / lo pairs (6 N D), chosen by the library's probe "
                                                         "when the map's neighbouring nodes are closer than a single pass can resolve; frac is always against 2 N D",
                        "tensor_flops_issued_frac_of_peak": score_rows_s / world * 2 * SW_ * SH_ * SD_ * (3 if score_tier == 2 else 1) / 1e12 / bf16_tf,
                        "random_init_map": random_map,
                        "parity": "see cpu_baseline.scoring_agreement (measured in this run) and tests/test_gpu_parity.py",
                        "fallback_rows": fallback_rows, "fallback_frac": fallback_rows / rows_rank, "gpu_launches": score_launches, "clocks": score_clocks,
                        "roofline": {"bound": "tensor", "achieved": score_rows_s / world * 2 * SW_ * SH_ * SD_ / 1e12, "peak": bf16_tf, "unit": "TFLOP/s",
                                     "frac": score_rows_s / world * 2 * SW_ * SH_ * SD_ / 1e12 / bf16_tf, "traffic": measured_traffic(f"score_tc_kernel_tier{score_tier}", rows_rank),
                                     "flops_per_row": 2 * SW_ * SH_ * SD_, "peak_source": peak_src + " (sustained bf16; the timed region is > 1 s per GPU at N=1)",
                                     "frac_of_burst_peak": score_rows_s / world * 2 * SW_ * SH_ * SD_ / 1e12 / bf16_burst},
                        "e2e": {"value": score_e2e, "unit": "rows/s", "rows": e2e_rows * world, "h2d_bytes_per_step": e2e_rows * SD_ * 4, "d2h_bytes_per_step": e2e_rows * 8,
                                "call": "vsom_find_bmu with pinned host rows (H2D of slab i+1 / search of slab i / D2H of slab i-1 overlap)", "mean_bmu_distance": score_err,
                                "matches_device_run": e2e_matches,
                                "measure_similarity": {"value": sim_e2e, "unit": "rows/s", "call": "vsom_measure_similarity (what Som::measureSimilarity makes: restricted BMU + the row's largest ((x - m) / sM) / numOfSigmas, one trip over PCIe)", "finite_share": sim_finite}, "pcie_h2d_gbs_measured": h2d_gbs, "pcie_ceiling_rows_per_s": world * h2d_gbs * 1e9 / (SD_ * 4),
                                "frac_of_pcie_ceiling": score_e2e / (world * h2d_gbs * 1e9 / (SD_ * 4))},
                        "exact_scan_rows_per_s": exact_rows_s, "exact_scan_rows": exact_rows * world,
                        "scaling": "row-sharded, no communication"},
        }
        line["index_build"] = index_leg
        if batch_leg:
            line["batch_map"] = batch_leg
        if others:
            line["other_training_shapes"] = others
        if large is not None:
            large["roofline"]["peak"] = hbm_gbs
            large["roofline"]["frac"] = large["roofline"]["achieved"] / hbm_gbs
            line["large_map"] = large
        if world == 1 and not args.no_cpu_baseline:
            def train_gpu(xs, init):
                tctx = vsom.VsomContext(W_, H_, D_, vsom.MEDIAN, order, device=local_rank)
                tctx.upload_state(mean=init)
                gb, gd, _, _ = tctx.train_chunk(xs, ETA, SIGMA, vsom.EXPONENTIAL)
                tctx.close()
                return gb, gd

            line["cpu_baseline"] = cpu_baseline_leg(train_gpu, score_state, agree_host, score_gpu, args.order)
        print(json.dumps(line), flush=True)
    ctx.close()
    sctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
