"""Worker of tests/test_gpu_sharded.py — run under torchrun with one rank per GPU:
node-sharded online training (in-kernel NVLink exchange) must reproduce the CPU oracle bit for bit."""
import importlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def same(got, want):
    """NaN pattern identical, every other value bit for bit (NaN payload and sign are not part of the contract)."""
    nan = np.isnan(want)
    return np.array_equal(np.isnan(got), nan) and np.array_equal(got[~nan].view(np.uint32 if got.dtype == np.float32 else np.uint64),
                                                                  want[~nan].view(np.uint32 if want.dtype == np.float32 else np.uint64))


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    vsom = importlib.import_module("variational-self-organizing-maps_b200")
    sh = importlib.import_module("variational-self-organizing-maps_b200.sharding")
    from oracle import pyoracle as po

    ok = True
    # (W, H, Din, transform, rows, eta, sigma, decay, special): resident and global-memory planes, all transformations; then a
    # NaN component in the first node of rank 1's share (an ordinary node: its NaN distance must never win) and in node 0
    # (which seeds findBmu: its NaN distance wins every sample)
    cases = [(24, 16, 20, 0, 200, 0.2, 4.0, 0, None), (31, 9, 7, 1, 150, 0.05, 2.5, 1, None), (12, 10, 6, 2, 80, 0.002, 3.0, 0, None),
             (160, 100, 784, 0, 6, 0.1, 6.0, 0, None), (24, 16, 20, 0, 100, 0.2, 4.0, 0, "nan_rank1_first"), (24, 16, 20, 1, 100, 0.2, 4.0, 0, "nan_node0")]
    for ci, (W, H, D, tr, n, eta, sigma, decay, special) in enumerate(cases):
        rng = np.random.default_rng(100 + ci)
        o = po.Oracle(W, H, D, tr)
        o.random_initialize(42, 1.0)
        init = o.get_state()
        if special is not None:
            init["mean"][sh.shard_block_rows(H, world) * W if special == "nan_rank1_first" else 0, 3] = np.nan
            o.set_state(**init)
        if tr == 2:
            z = rng.standard_normal((2 * n, 1)).astype(np.float32)
            x = (rng.uniform(0.5, 1.5, (1, D)).astype(np.float32) * z + 0.1 * rng.standard_normal((2 * n, D))).astype(np.float32)
        else:
            x = rng.standard_normal((2 * n, D)).astype(np.float32)
        ctx = vsom.VsomContext(W, H, D, tr, vsom.ORDER_REFERENCE, device=local, rank=rank, world=world)
        handles = [None] * world
        dist.all_gather_object(handles, ctx.peer_export())
        for r, h in enumerate(handles):
            ctx.peer_import(r, h)
        blk, rows = ctx.shard_rows()
        assert blk == sh.shard_block_rows(H, world) and np.array_equal(rows, sh.node_rows(H, rank, world))
        ctx.upload_state(init["mean"], init["S"], init["sigma"], init["weight"], init["hits"])
        dist.barrier()
        for seg, sg in ((x[:n], sigma), (x[n:], sigma * 0.7)):  # two chunks: the global step counter carries over
            gb, gd, _, _ = ctx.train_chunk(seg, eta, sg, decay)
            ob, od, _, _ = o.train_rows(seg, eta, sg, decay)
            dists = [None] * world
            dist.all_gather_object(dists, gd)
            md = sh.merge_owner_outputs(dists)
            # a NaN distance of the BMU looks like "not the owner" on every rank: distances are compared where the oracle's is a number
            real = ~np.isnan(od)
            if not (np.array_equal(gb, ob) and np.array_equal(md[real].view(np.uint32), od[real].view(np.uint32))):
                ok = False
                print(f"[rank {rank}] case {ci}: BMU / distance mismatch", flush=True)
        # each rank downloads only its band; the bands are summed into the full planes
        st = ctx.download_state_zero_filled()
        want = o.get_state()
        for k in ("mean", "S", "sigma", "weight"):
            t = torch.from_numpy(st[k].view(np.int32).astype(np.int64))
            dist.all_reduce(t)
            full = t.numpy().astype(np.int32).view(np.float32).reshape(want[k].shape)
            if not same(full, want[k]):
                ok = False
                print(f"[rank {rank}] case {ci}: plane {k} differs", flush=True)
        t = torch.from_numpy(st["hits"].astype(np.int64))
        dist.all_reduce(t)
        if not np.array_equal(t.numpy().astype(np.uint64), want["hits"]):
            ok = False
            print(f"[rank {rank}] case {ci}: hits differ", flush=True)
        # sharded U-matrix: every rank computes its own grid rows, border rows of means come from the neighbours over NVLink
        dist.barrier()  # every rank's training stream is idle (train_chunk is synchronous)
        um = ctx.update_umatrix()
        dist.barrier()
        t = torch.from_numpy(um.view(np.int64).copy())
        dist.all_reduce(t)  # rows of other ranks are zero
        with np.errstate(all="ignore"):
            want_um = o.update_umatrix()
        if H >= 2 and W >= 2 and not same(t.numpy().view(np.float64), want_um):
            ok = False
            print(f"[rank {rank}] case {ci}: sharded U-matrix differs", flush=True)
        if rank == 0:
            print(f"case {ci} {W}x{H}x{D} transform {tr}: {'ok' if ok else 'FAILED'} (resident={ctx.planes_resident}, block rows={blk})", flush=True)
        ctx.close()
        dist.barrier()
    flag = torch.tensor([0 if ok else 1])
    dist.all_reduce(flag)
    dist.destroy_process_group()
    if flag.item():
        sys.exit(1)
    if rank == 0:
        print("SHARDED_OK", flush=True)


if __name__ == "__main__":
    main()
