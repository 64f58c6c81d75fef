"""Node-sharded online training over 2+ GPUs (BASELINE config 5's layout): one process per GPU, the per-sample min-loc
exchange runs inside the persistent kernel over NVLink peer memory; results must equal the oracle bit for bit."""
import os
import subprocess
import sys

import pytest

from conftest import REPO


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_node_sharded_training_matches_oracle():
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs (one training process per GPU)")
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1", "--master-port",
           "29533", os.path.join(REPO, "tests", "sharded_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=800)
    print(out.stdout[-3000:], out.stderr[-3000:])
    assert out.returncode == 0 and "SHARDED_OK" in out.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("world,order", [(2, 0), (3, 2), (8, 0)])
def test_sharded_layout_and_umatrix_halo_in_one_process(vsom, po, world, order):
    """The block-cyclic row layout and the sharded U-matrix (own rows + one halo row of means per block border, read from
    the owner's plane) on ONE GPU: `world` contexts of the same process attach each other directly (vsom_peer_attach).
    State round-trips through the full-map arrays; the ranks' U-matrix rows together equal the oracle's matrix bit for
    bit.  (Sharded TRAINING needs one GPU per rank — co-resident persistent kernels — and runs in the torchrun test above.)"""
    import importlib

    from conftest import PKG_NAME, assert_bit_equal

    sh = importlib.import_module(PKG_NAME + ".sharding")
    import numpy as np

    rng = np.random.default_rng(world)
    W, H, D = 13, 37, 10
    o = po.Oracle(W, H, D, po.STANDARD, order)
    o.random_initialize(7, 1.0)
    st = o.get_state()
    st["sigma"] = np.abs(rng.standard_normal(st["sigma"].shape)).astype(np.float32)
    st["S"] = rng.standard_normal(st["S"].shape).astype(np.float32)
    st["weight"] = rng.random(W * H).astype(np.float32)
    st["hits"] = rng.integers(0, 9, W * H).astype(np.uint64)
    o.set_state(**st)
    ctxs = [vsom.VsomContext(W, H, D, vsom.STANDARD, order, device=0, rank=r, world=world) for r in range(world)]
    for a in ctxs:
        for r, b in enumerate(ctxs):
            a.peer_attach(r, b)
    total = {k: np.zeros_like(v) for k, v in st.items()}
    for r, c in enumerate(ctxs):
        blk, rows = c.shard_rows()
        assert blk == sh.shard_block_rows(H, world) and np.array_equal(rows, sh.node_rows(H, r, world))
        c.upload_state(st["mean"], st["S"], st["sigma"], st["weight"], st["hits"])
    for r, c in enumerate(ctxs):
        got = c.download_state_zero_filled()
        ids = sh.node_ids(W, H, r, world)
        for k in total:
            assert_bit_equal(got[k][ids], st[k][ids], f"rank {r} {k}")
            mask = np.ones(W * H, bool)
            mask[ids] = False
            assert not got[k][mask].any(), f"rank {r} wrote outside its rows ({k})"
    um = np.zeros(W * H, np.float64)
    for c in ctxs:
        um += c.update_umatrix()  # rows of other ranks stay zero
    assert_bit_equal(um, o.update_umatrix(), "sharded U-matrix")
    with pytest.raises(vsom.VsomError):
        ctxs[0].find_bmu(np.zeros((3, D), np.float32))  # scoring needs an unsharded context
    for c in ctxs:
        c.close()
