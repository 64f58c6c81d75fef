"""Which online-step kernel runs a chunk, and what the call reports about it.

launch_online_step (online_step.cu) runs a chunk on K1F (online_step_fast.cu) when the context has a K1F plan, else on the
generic kernel K1.  For one map of each kind this checks the kernel that ran, vsom_planes_resident, that the launch count
goes up by exactly one per chunk, and that outputs and state match the oracle bit for bit.  It also checks the order of the
refusals (sharded + sigma <= 1, then the decay, then n == 0, then missing peers), and the phase profile of both kernels:
raw slots and their fold into the five documented phases.

The size limits of K1F (a grid side of 4096 against 4097, 512 owned nodes per CTA against 513) are covered by
test_gpu_benchmark_shapes.py::test_fast_kernel_eligibility_edges."""
import ctypes

import numpy as np
import pytest

from conftest import assert_bit_equal

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

ERR_INVALID, ERR_UNSUPPORTED = -1, -3


def kernel_env(monkeypatch, kernel):
    if kernel == "generic":
        monkeypatch.setenv("VSOM_ONLINE_KERNEL", "generic")
    else:
        monkeypatch.delenv("VSOM_ONLINE_KERNEL", raising=False)


def make_pair(vsom, po, W, H, Din, tr, order, seed):
    o = po.Oracle(W, H, Din, tr, 0 if order == vsom.ORDER_LANES else order)
    o.random_initialize(seed, 1.0)
    st = o.get_state()
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    ctx.upload_state(st["mean"], st["S"], st["sigma"], st["weight"], st["hits"])
    return ctx, o


# (W, H, Din, transform, order, sigma, VSOM_ONLINE_KERNEL, K1F runs, planes resident).  The LANES map has two-element rows:
# a sum of two squares has the same bits in every order, so the oracle's sequential sums are exact for it too.  The
# 128 x 128 x 256 map does not fit in shared memory: K1 streams its rows from HBM, and K1F is not eligible.
CASES = {
    "fast": (24, 16, 20, 1, 0, 4.0, "fast", True, True),
    "generic": (24, 16, 20, 1, 0, 4.0, "generic", False, True),
    "lanes": (24, 16, 2, 0, 1, 4.0, "fast", False, True),
    "hbm_resident": (128, 128, 256, 0, 0, 6.0, "fast", False, False),
    "local_walk_fast": (24, 16, 20, 0, 0, 0.8, "fast", True, True),
    "local_walk_generic": (24, 16, 20, 0, 0, 0.8, "generic", False, True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_chunk_runs_on_the_chosen_kernel(vsom, po, monkeypatch, case):
    W, H, Din, tr, order, sigma, kernel, fast, resident = CASES[case]
    kernel_env(monkeypatch, kernel)
    ctx, o = make_pair(vsom, po, W, H, Din, tr, order, seed=11)
    assert ctx.planes_resident == resident
    rng = np.random.default_rng(5)
    last = np.zeros(96, np.uint64) if sigma <= 1.0 else None
    for chunk in range(2):
        x = rng.standard_normal((96, Din)).astype(np.float32)
        before = ctx.launch_count
        ob, od, orr, ol = o.train_rows(x, 0.1, sigma, vsom.EXPONENTIAL, last_bmu=None if last is None else last.copy())
        gb, gd, gr, gl = ctx.train_chunk(x, 0.1, sigma, vsom.EXPONENTIAL, last_bmu=None if last is None else last.copy())
        assert ctx.launch_count == before + 1, f"chunk {chunk}"
        assert ctx.last_train_fast == fast, f"chunk {chunk}"
        assert_bit_equal(gb, ob, f"chunk {chunk}: bmu")
        assert_bit_equal(gd, od, f"chunk {chunk}: dist")
        assert_bit_equal(gr, orr, f"chunk {chunk}: resid2")
        assert_bit_equal(gl, ol, f"chunk {chunk}: lastBMU")
        if last is not None:
            last = ol
    got, want = ctx.download_state(), o.get_state()
    for k in ("mean", "S", "sigma", "weight", "hits"):
        assert_bit_equal(got[k], want[k], k)
    ctx.close()


def train_device_raw(vsom, ctx, n, sigma, decay):
    """vsom_train_chunk_device with n rows of zeros (none at all when n == 0), unchecked: (return code, error text)."""
    import torch

    L = vsom.lib()
    x = torch.zeros((max(n, 1), ctx.Din), dtype=torch.float32, device="cuda")
    rc = L.vsom_train_chunk_device(ctx._h, x.data_ptr() if n else None, n, 0.1, sigma, decay, None, None)
    torch.cuda.synchronize()
    return rc, (L.vsom_last_error(ctx._h) or b"").decode()


def test_empty_chunk_launches_nothing(vsom, po, monkeypatch):
    kernel_env(monkeypatch, "fast")
    ctx, o = make_pair(vsom, po, 24, 16, 20, 1, 0, seed=3)
    ctx.train_chunk(np.random.default_rng(1).standard_normal((8, 20)).astype(np.float32), 0.1, 4.0)
    assert ctx.last_train_fast
    before, state = ctx.launch_count, ctx.download_state()
    for sigma in (4.0, 0.8):
        assert train_device_raw(vsom, ctx, 0, sigma, vsom.EXPONENTIAL)[0] == 0
    assert ctx.launch_count == before
    assert ctx.last_train_fast
    got = ctx.download_state()
    for k in state:
        assert_bit_equal(got[k], state[k], k)
    ctx.close()


DECAY_TEXT = "online step: decay must be Exponential or InverseProportional"
LOCAL_TEXT = "online step: the findLocalBmu regime (sigma <= 1) is not available on node-sharded contexts"
PEERS_TEXT = "online step: sharded context without vsom_peer_import for every rank"


def test_refusals_and_their_order(vsom):
    """The checks run in a fixed order, which decides the error when several apply: on a node-sharded context, sigma <= 1
    first, then the decay, then n == 0 (nothing to do), then the peers of the other ranks.  Nothing is launched."""
    ctx = vsom.VsomContext(24, 16, 20, vsom.STANDARD, vsom.ORDER_REFERENCE, device=0, rank=0, world=2)  # no peers attached
    bad = 7
    cases = [
        (5, 0.8, bad, ERR_UNSUPPORTED, LOCAL_TEXT),
        (0, 0.8, vsom.EXPONENTIAL, ERR_UNSUPPORTED, LOCAL_TEXT),
        (5, 4.0, bad, ERR_INVALID, DECAY_TEXT),
        (0, 4.0, bad, ERR_INVALID, DECAY_TEXT),
        (0, 4.0, vsom.EXPONENTIAL, 0, None),
        (5, 4.0, vsom.EXPONENTIAL, ERR_INVALID, PEERS_TEXT),
    ]
    for n, sigma, decay, rc_want, text in cases:
        rc, msg = train_device_raw(vsom, ctx, n, sigma, decay)
        assert rc == rc_want, (n, sigma, decay, msg)
        if text:
            assert msg == text, (n, sigma, decay)
    assert ctx.launch_count == 0
    ctx.close()


def test_bad_decay_on_one_gpu(vsom, po):
    ctx, _ = make_pair(vsom, po, 24, 16, 20, 0, 0, seed=2)
    for n in (0, 5):
        rc, msg = train_device_raw(vsom, ctx, n, 4.0, 2)
        assert (rc, msg) == (ERR_INVALID, DECAY_TEXT)
    assert ctx.launch_count == 0
    ctx.close()


def phase_cycles(vsom, ctx):
    """vsom_debug_phase_cycles_raw and vsom_debug_phase_cycles, unchecked: both return codes, all eight raw slots, the five phases."""
    raw, folded = np.zeros(8, np.float64), np.zeros(5, np.float64)
    f64p = ctypes.POINTER(ctypes.c_double)
    rc_raw = vsom.lib().vsom_debug_phase_cycles_raw(ctx._h, raw.ctypes.data_as(f64p))
    rc = vsom.lib().vsom_debug_phase_cycles(ctx._h, folded.ctypes.data_as(f64p))
    return rc_raw, rc, raw, folded


@pytest.mark.parametrize("kernel", ["fast", "generic"])
def test_phase_cycles_follow_the_kernel_that_ran(vsom, po, monkeypatch, kernel):
    """Before any chunk both calls refuse.  After a profiled chunk the raw slots are K1F's seven (chain, CTA min, exchange,
    coefficients, barrier, update, barrier; slot 7 zero) or K1's five (slots 5-7 zero), and the five phases are their stated
    sums: K1F (0, chain + CTA min, exchange, coefficients + barrier, update + barrier), K1 the first five slots."""
    kernel_env(monkeypatch, kernel)
    ctx, o = make_pair(vsom, po, 24, 16, 20, 1, 0, seed=4)
    rc_raw, rc, _, _ = phase_cycles(vsom, ctx)
    assert rc_raw == rc == ERR_INVALID
    ctx.debug_profile(True)
    rc_raw, rc, _, _ = phase_cycles(vsom, ctx)
    assert rc_raw == rc == ERR_INVALID
    x = np.random.default_rng(9).standard_normal((200, 20)).astype(np.float32)
    gb, gd, _, _ = ctx.train_chunk(x, 0.1, 4.0)
    ob, od, _, _ = o.train_rows(x, 0.1, 4.0, vsom.EXPONENTIAL)
    assert_bit_equal(gb, ob, "bmu")
    assert_bit_equal(gd, od, "dist")
    assert ctx.last_train_fast == (kernel == "fast")
    rc_raw, rc, raw, folded = phase_cycles(vsom, ctx)
    assert rc_raw == rc == 0
    assert raw[2] > 0, "exchange"
    if kernel == "fast":
        assert raw[7] == 0
        want = [0.0, raw[0] + raw[1], raw[2], raw[3] + raw[4], raw[5] + raw[6]]
    else:
        assert not raw[5:].any()
        want = raw[:5].tolist()
    assert folded.tolist() == want
    ctx.close()
