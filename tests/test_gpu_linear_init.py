"""Linear initialisation along the two leading principal components (vsom_linear_init, VsomContext.linear_init,
Som::linearInitialize).

The oracle is numpy in f64: x.mean(0), np.cov(x, rowvar=False) and np.linalg.eigh, with the header's sign rule.  Every case checks
mu, lambda and the axes against it, the mean plane bit for bit against the header's expression evaluated here from the call's own
outputs, the plane within 1e-6 (max|mu| + sqrt(lambda_1)) of the same expression built from numpy's mu, lambda and v, and that S,
sigma, weight and hits are zero."""
import importlib
import os
import struct
import subprocess

import numpy as np
import pytest

from conftest import PKG_NAME, REPO, assert_bit_equal

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

F32, F64 = np.float32, np.float64
SLAB_ROWS = 16384  # VSOM_LINEAR_INIT_SLAB_ROWS
LININIT_DRIVER = os.path.join(REPO, "tests", "cpp", "lininit_driver")


# ------------------------------------------------------------------------------------------------ numpy side of the contract
def orient(v):
    """The sign rule: the component of largest magnitude is positive (np.argmax takes the lowest index among equal magnitudes)."""
    return -v if v[np.argmax(np.abs(v))] < 0 else v


def numpy_fit(x):
    x64 = x.astype(F64)
    mu = x64.mean(0)
    D = x.shape[1]
    C = np.cov(x64, rowvar=False).reshape(D, D)
    w, V = np.linalg.eigh(C)
    lam = np.maximum(w[::-1][:2], 0.0) if D > 1 else np.array([max(w[0], 0.0), 0.0])
    v1 = orient(V[:, -1]) if D > 1 else np.ones(1)
    v2 = orient(V[:, -2]) if D > 1 else np.zeros(1)
    return mu, lam, np.stack([v1, v2]), C


def coords(L):
    return (2 * np.arange(L) - (L - 1)) / (L - 1) if L > 1 else np.zeros(1)


def plane(W, H, mu, lam, axes):
    """m[y*W + x] = f32((mu + (c_W(x) s_x) v_x) + (c_H(y) s_y) v_y), in f64 in exactly that order."""
    wide = W >= H
    vx, vy = (axes[0], axes[1]) if wide else (axes[1], axes[0])
    sx, sy = (np.sqrt(lam[0]), np.sqrt(lam[1])) if wide else (np.sqrt(lam[1]), np.sqrt(lam[0]))
    cx, cy = coords(W) * sx, coords(H) * sy
    m = (mu[None, None, :] + cx[None, :, None] * vx[None, None, :]) + cy[:, None, None] * vy[None, None, :]
    return m.reshape(W * H, -1).astype(F32)


def assert_zero_rest(st, what=""):
    for k in ("S", "sigma", "weight"):
        assert not st[k].view(np.uint32).any(), f"{what}: {k} is not +0"
    assert not st["hits"].any(), f"{what}: hits are not 0"


def check_outputs(W, H, x, mu, lam, axes, st, vectors=(0, 1)):
    """Tolerances against numpy, the plane bit for bit from the call's outputs, the rest of the state zero."""
    nmu, nlam, naxes, _ = numpy_fit(x)
    assert np.all(np.abs(mu - nmu) <= 1e-12 * max(np.abs(x).max(), 1e-300)), "mu"
    assert np.all(np.abs(lam - nlam) <= 1e-9 * nlam[0]), (lam, nlam)
    for i in vectors:
        if not naxes[i].any():
            assert not axes[i].any(), f"axis {i + 1} must be 0"
        else:
            assert naxes[i] @ axes[i] >= 1 - 1e-9, f"axis {i + 1}: <v, v_np> = {naxes[i] @ axes[i]}"
    assert_bit_equal(st["mean"], plane(W, H, mu, lam, axes), "mean plane vs the expression from the call's outputs")
    want = plane(W, H, nmu, nlam, naxes).astype(F64)
    if set(vectors) == {0, 1}:
        assert np.abs(st["mean"].astype(F64) - want).max() <= 1e-6 * (np.abs(nmu).max() + np.sqrt(nlam[0])), "mean plane vs numpy"
    assert_zero_rest(st)


def spectrum_data(n, D, scales, noise, offset, seed):
    """offset + low-rank signal along near-coordinate directions (each with a clear largest component) + isotropic noise"""
    rng = np.random.default_rng(seed)
    r = len(scales)
    B = np.zeros((D, r))
    B[np.arange(r) % D, np.arange(r)] = 1.0
    B += 0.25 * rng.standard_normal((D, r)) / np.sqrt(D)
    Q, _ = np.linalg.qr(B)
    z = rng.standard_normal((n, r)) * np.asarray(scales)
    return (offset + z @ Q.T + noise * rng.standard_normal((n, D))).astype(F32)


SHAPES = {
    # W, H, D, n, scales, noise, offset
    "20x20x784_mnist_scale": (20, 20, 784, 60000, 60.0 * 0.8 ** np.arange(20), 5.0, 100.0),
    "64x64x128": (64, 64, 128, 20000, [9.0, 6.0, 4.0, 2.0, 1.5], 0.3, -2.0),
    "13x37x10_swapped": (13, 37, 10, 3000, [5.0, 3.0, 1.5], 0.2, 1.0),
    "1x50x6": (1, 50, 6, 500, [4.0, 2.0, 1.0], 0.1, 0.5),
    "50x1x6": (50, 1, 6, 500, [4.0, 2.0, 1.0], 0.1, 0.5),
    "1x1x5": (1, 1, 5, 500, [4.0, 2.0, 1.0], 0.1, 0.5),
    "D1": (8, 6, 1, 1000, [3.0], 0.0, 2.0),
    "D2": (7, 9, 2, 1000, [3.0, 1.0], 0.0, -1.0),
    "n2": (5, 4, 2, 2, [3.0, 1.0], 0.0, 0.0),
    "n3": (5, 4, 3, 3, [3.0, 1.0], 0.0, 0.0),
}


@pytest.mark.parametrize("name", list(SHAPES))
def test_shapes_against_numpy(vsom, name):
    W, H, D, n, scales, noise, offset = SHAPES[name]
    x = spectrum_data(n, D, scales, noise, offset, seed=D + n)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    mu, lam, axes = ctx.linear_init(x)
    check_outputs(W, H, x, mu, lam, axes, ctx.download_state())
    ctx.close()


def test_state_reset_after_training(vsom):
    """S, sigma, weight and hits are zero again after a training chunk had made them non-zero."""
    W, H, D = 13, 37, 10
    x = spectrum_data(3000, D, [5.0, 3.0, 1.5], 0.2, 1.0, seed=5)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    ctx.linear_init(x)
    ctx.train_chunk(x[:500], 0.1, 4.0, vsom.EXPONENTIAL)
    st = ctx.download_state()
    assert st["S"].any() and st["weight"].any() and st["hits"].any()
    mu, lam, axes = ctx.linear_init(x)
    check_outputs(W, H, x, mu, lam, axes, ctx.download_state())
    ctx.close()


def test_invariance(vsom):
    """Bit-identical across Standard / Median, the three summation orders, two calls on one context and a fresh context."""
    W, H, D = 13, 37, 10
    x = spectrum_data(3000, D, [5.0, 3.0, 1.5], 0.2, 1.0, seed=11)
    runs = []
    for tr, order in ((vsom.STANDARD, vsom.ORDER_REFERENCE), (vsom.STANDARD, vsom.ORDER_LANES), (vsom.STANDARD, vsom.ORDER_EIGEN_SSE),
                      (vsom.MEDIAN, vsom.ORDER_REFERENCE)):
        ctx = vsom.VsomContext(W, H, D, tr, order)
        for _ in range(2):
            mu, lam, axes = ctx.linear_init(x)
            runs.append((mu, lam, axes, ctx.download_state()["mean"]))
        ctx.close()
    for i, r in enumerate(runs[1:], 1):
        for a, b, what in zip(runs[0], r, ("mean", "lambda", "axes", "plane")):
            assert_bit_equal(b, a, f"run {i}: {what}")


def test_slab_boundaries(vsom):
    """Rows crossing two host-slab boundaries and ending in a partial slab: same tolerances, repeatable bit for bit."""
    W, H, D = 8, 8, 6
    n = 2 * SLAB_ROWS + 12345
    x = spectrum_data(n, D, [4.0, 2.0, 1.0], 0.1, 3.0, seed=2)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    a = ctx.linear_init(x)
    st = ctx.download_state()
    check_outputs(W, H, x, *a, st)
    b = ctx.linear_init(x)
    for u, v, what in zip(a, b, ("mean", "lambda", "axes")):
        assert_bit_equal(v, u, what)
    assert_bit_equal(ctx.download_state()["mean"], st["mean"], "plane")
    ctx.close()


def _planted(rows_per_axis, weights):
    """Rows +-sqrt(w_k) e_k: mean 0 and a diagonal covariance proportional to w"""
    D = len(weights)
    e = np.sqrt(np.asarray(weights, F64))[:, None] * np.eye(D)
    return np.tile(np.concatenate([e, -e]), (rows_per_axis, 1)).astype(F32)


def test_degenerate_rank_one(vsom):
    rng = np.random.default_rng(3)
    D, n = 12, 1000
    u = rng.integers(-8, 9, D).astype(F64) / 8.0
    u[4] = 3.0
    x = (rng.integers(-50, 51, n)[:, None] * u[None, :] + np.arange(D)).astype(F32)  # exact in f32
    W, H = 9, 7
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    mu, lam, axes = ctx.linear_init(x)
    assert lam[1] <= 1e-12 * lam[0]
    check_outputs(W, H, x, mu, lam, axes, ctx.download_state(), vectors=(0,))
    assert abs(np.linalg.norm(axes[1]) - 1.0) <= 1e-12 and abs(axes[0] @ axes[1]) <= 1e-12
    ctx.close()


def test_degenerate_constant_rows(vsom):
    W, H, D = 6, 5, 7
    row = np.linspace(-3.0, 250.0, D).astype(F32)
    x = np.tile(row, (100, 1))
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    mu, lam, axes = ctx.linear_init(x)
    assert np.array_equal(lam, [0.0, 0.0])
    st = ctx.download_state()
    assert_bit_equal(st["mean"], np.tile(mu.astype(F32), (W * H, 1)), "every node is f32(mu)")
    assert_bit_equal(st["mean"], np.tile(row, (W * H, 1)), "f32(mu) is the row")
    assert_bit_equal(st["mean"], plane(W, H, mu, lam, axes), "plane from the call's outputs")
    assert_zero_rest(st)
    ctx.close()


@pytest.mark.parametrize("spread", [0.0, 1e-7])
def test_degenerate_isotropic(vsom, spread):
    """spread 0: C is a multiple of I (every vector is an eigenvector); 1e-7: 32 nearly equal eigenvalues, so the iteration cap
    ends the call, which still succeeds with its Ritz pairs."""
    D, W, H = 32, 10, 8
    x = _planted(40, 1.0 + spread * np.arange(D))
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    mu, lam, axes = ctx.linear_init(x)
    _, nlam, _, C = numpy_fit(x)
    assert np.abs(axes @ axes.T - np.eye(2)).max() <= 1e-12, "axes orthonormal"
    for i in range(2):
        assert abs(axes[i] @ C @ axes[i] - lam[i]) <= 1e-9 * nlam[0], f"Rayleigh quotient of axis {i + 1}"
    w = np.linalg.eigvalsh(C)
    assert np.all(lam >= w[0] - 1e-12 * w[-1]) and np.all(lam <= w[-1] * (1 + 1e-12)), "Ritz values lie in C's spectrum"
    st = ctx.download_state()
    assert_bit_equal(st["mean"], plane(W, H, mu, lam, axes), "plane from the call's outputs")
    assert_zero_rest(st)
    if spread:
        assert ctx.linear_init_phases()["iterations"] == 300
    ctx.close()


def test_refusals_leave_state(vsom):
    rng = np.random.default_rng(9)
    W, H, D = 8, 6, 5

    def seeded(ctx, N, Dm):
        ctx.upload_state(rng.standard_normal((N, Dm)).astype(F32), rng.standard_normal((N, Dm)).astype(F32),
                         rng.random((N, Dm)).astype(F32), rng.random(N).astype(F32), rng.integers(0, 9, N).astype(np.uint64))
        return ctx.download_state()

    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    before = seeded(ctx, W * H, D)
    x = rng.standard_normal((1000, D)).astype(F32)
    bad_nan, bad_inf = x.copy(), x.copy()
    bad_nan[-1, 3] = np.nan
    bad_inf[-1, 3] = np.inf
    for rows, what in ((x[:0], "n = 0"), (x[:1], "n = 1"), (bad_nan, "NaN"), (bad_inf, "+inf")):
        with pytest.raises(vsom.VsomError) as e:
            ctx.linear_init(rows)
        assert e.value.code == -1, what
        after = ctx.download_state()
        for k in before:
            assert_bit_equal(after[k], before[k], f"{what}: {k}")
    ctx.close()
    J = 4
    clr = vsom.VsomContext(W, H, J, vsom.CLR, vsom.ORDER_REFERENCE)
    before = seeded(clr, W * H, clr.Dm)
    with pytest.raises(vsom.VsomError) as e:
        clr.linear_init(rng.standard_normal((50, J)).astype(F32))
    assert e.value.code == -3
    after = clr.download_state()
    for k in before:
        assert_bit_equal(after[k], before[k], f"CLR: {k}")
    clr.close()


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_in_one_process(vsom, world):
    """Every rank writes exactly the unsharded context's rows for its own grid rows, and nothing else."""
    sh = importlib.import_module(PKG_NAME + ".sharding")
    W, H, D = 13, 37, 10
    x = spectrum_data(3000, D, [5.0, 3.0, 1.5], 0.2, 1.0, seed=world)
    ref = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    ref.linear_init(x)
    want = ref.download_state()
    ref.close()
    ctxs = [vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE, device=0, rank=r, world=world) for r in range(world)]
    for a in ctxs:
        for r, b in enumerate(ctxs):
            a.peer_attach(r, b)
    for r, c in enumerate(ctxs):
        c.linear_init(x)
        got = c.download_state_zero_filled()
        ids = sh.node_ids(W, H, r, world)
        mask = np.ones(W * H, bool)
        mask[ids] = False
        for k in want:
            assert_bit_equal(got[k][ids], want[k][ids], f"rank {r} {k}")
            assert not got[k][mask].any(), f"rank {r} wrote outside its rows ({k})"
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("kernel", ["fast", "generic"])
def test_training_from_initialised_map(vsom, po, monkeypatch, kernel):
    """train_chunk after linear_init matches the CPU oracle started from the downloaded state, bit for bit (K1F on 20 x 20 x 784,
    the generic online-step kernel on 24 x 16 x 20)."""
    if kernel == "generic":
        monkeypatch.setenv("VSOM_ONLINE_KERNEL", "generic")
        W, H, D = 24, 16, 20
    else:
        monkeypatch.delenv("VSOM_ONLINE_KERNEL", raising=False)
        W, H, D = 20, 20, 784
    x = spectrum_data(4000, D, 20.0 * 0.8 ** np.arange(8), 2.0, 50.0, seed=D)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    ctx.linear_init(x)
    o = po.Oracle(W, H, D, po.STANDARD, 0)
    o.set_state(**ctx.download_state())
    gb, gd, _, _ = ctx.train_chunk(x[:400], 0.1, 5.0, vsom.EXPONENTIAL)
    assert ctx.last_train_fast == (kernel == "fast")
    ob, od, _, _ = o.train_rows(x[:400], 0.1, 5.0, po.EXPONENTIAL)
    assert_bit_equal(gb, ob, "BMUs")
    assert_bit_equal(gd, od, "distances")
    got, want = ctx.download_state(), o.get_state()
    for k in want:
        assert_bit_equal(got[k], want[k], k)
    ctx.close()


def _run_driver(tmp_path, W, H, D, transform, x, chunk, sched):
    case, out = tmp_path / "case.bin", tmp_path / "out.bin"
    with open(case, "wb") as f:
        f.write(struct.pack("<6i", W, H, D, transform, x.shape[0], chunk))
        f.write(struct.pack("<4d", *sched))
        f.write(np.ascontiguousarray(x, F32).tobytes())
    r = subprocess.run([LININIT_DRIVER, str(case), str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    return out.read_bytes()


def test_host_api(vsom, po, tmp_path):
    """Som::linearInitialize + one epoch of Som::train (tests/cpp/lininit_driver) against the binding's linear_init followed by the
    oracle's training; a CLR Som throws."""
    W, H, D, n, chunk = 12, 9, 16, 400, 100
    sched = (0.1, 0.05, 3.0, 0.1)
    x = spectrum_data(n, D, [5.0, 3.0, 1.5], 0.2, 1.0, seed=8)
    raw = _run_driver(tmp_path, W, H, D, 0, x, chunk, sched)
    N = W * H
    pos = 0

    def take(dtype, count):
        nonlocal pos
        a = np.frombuffer(raw, dtype, count, pos)
        pos += a.nbytes
        return a

    assert take(np.int32, 1)[0] == 0
    init = dict(mean=take(F32, N * D).reshape(N, D), sigma=take(F32, N * D).reshape(N, D), weight=take(F32, N), hits=take(np.uint64, N))
    umatrix, metrics_len = take(F64, N), take(np.uint64, 1)[0]
    mse = take(F32, 1)
    trained = dict(mean=take(F32, N * D).reshape(N, D), sigma=take(F32, N * D).reshape(N, D), weight=take(F32, N), hits=take(np.uint64, N))
    assert pos == len(raw)

    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    ctx.linear_init(x)
    st = ctx.download_state()
    ctx.close()
    for k in init:
        assert_bit_equal(init[k], st[k], f"after linearInitialize: {k}")
    assert not umatrix.any() and metrics_len == D
    o = po.Oracle(W, H, D, po.STANDARD, 0)
    o.set_state(**st)
    want_mse = o.train(x, chunk, 1, *sched, po.EXPONENTIAL)
    assert_bit_equal(mse, want_mse, "epoch MSE")
    want = o.get_state()
    for k in trained:
        assert_bit_equal(trained[k], want[k], f"after one epoch: {k}")

    raw = _run_driver(tmp_path, W, H, 4, 2, x[:, :4], chunk, sched)
    assert np.frombuffer(raw, np.int32, 1)[0] == 1 and len(raw) == 4, "a CLR Som must throw"
