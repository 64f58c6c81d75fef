"""The smaller entry points of the C-ABI against the CPU oracle, at the launch shapes where they can go wrong: soft assignment
(vsom_soft_assign), the U-matrix (vsom_update_umatrix), the device form of the index build (vsom_build_index_device), the node
read-back (vsom_get_node), and every path of a VSOM_ORDER_LANES context other than training.

Tolerances: 0 ulp everywhere except soft-assign probabilities, which carry the device's f64 exp(): rtol 1e-13 there, with an
identical zero pattern and an identical NaN pattern (include/vsom_b200.h)."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_bit_equal

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

VSOM_ERR_INVALID, VSOM_ERR_UNSUPPORTED = -1, -3
_f32p, _f64p, _u32p, _u64p = C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)


def _ptr(a, t):
    return a.ctypes.data_as(t)


def synth(rng, n, Din, tr, scale=1.0):
    if tr == 2:  # CLR: rows along a line, so that the pair regressions are well conditioned
        z = rng.standard_normal((n, 1)).astype(np.float32)
        a = rng.uniform(0.5, 1.5, (1, Din)).astype(np.float32)
        return (scale * (a * z + 0.1 * rng.standard_normal((n, Din)))).astype(np.float32)
    return (scale * rng.standard_normal((n, Din))).astype(np.float32)


def raises_code(vsom, code, fn, *args):
    with pytest.raises(vsom.VsomError) as e:
        fn(*args)
    assert e.value.code == code, str(e.value)


# ------------------------------------------------------------------------------------------------ soft assignment
def soft_assign_map(vsom, po, W, H, Din, tr=0, order=0, seed=0):
    """A map close to the origin (nodes in [-0.2, 0.2]) with hit counts 0..3, on the oracle and on the device."""
    rng = np.random.default_rng(seed)
    o = po.Oracle(W, H, Din, tr, order)
    o.random_initialize(seed + 3, 0.2)
    st = o.get_state()
    st["hits"] = rng.integers(0, 4, W * H).astype(np.uint64)
    o.set_state(**st)
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    ctx.upload_state(**st)
    return rng, o, ctx


def assert_soft_assign_rows(got, o, x, min_hits, what):
    """got[r] against Oracle.find_restricted_bmd(x[r]) — C summed in node order like the reference (np.sum is pairwise, so it
    is no reference for C) — in blocks of rows, so that the oracle never holds a second copy of a large output."""
    n, N = got.shape
    block = max(1, (1 << 22) // N)
    for r0 in range(0, n, block):
        want = np.stack([o.find_restricted_bmd(x[r], min_hits) for r in range(r0, min(n, r0 + block))])
        g = got[r0:r0 + len(want)]
        assert np.array_equal(np.isnan(g), np.isnan(want)), f"{what}: NaN pattern (rows {r0}..)"
        assert np.array_equal(g == 0, want == 0), f"{what}: zero pattern (rows {r0}..)"
        ok = ~np.isnan(want)
        np.testing.assert_allclose(g[ok], want[ok], rtol=1e-13, atol=0, err_msg=f"{what} (rows {r0}..)")


@pytest.mark.parametrize("W,H,n", [(9, 7, 65535), (9, 7, 65536), (9, 7, 70001), (32, 16, 65536)])
def test_soft_assign_past_the_grid_limit(vsom, po, W, H, n):
    """The terms kernel puts one data row on each grid row, and gridDim.y stops at 65 535: a batch of more rows (every batch of
    65 536 rows or more on a map of up to 512 nodes, whose 256 MiB batch is at least 65 536 rows) takes several launches."""
    rng, o, ctx = soft_assign_map(vsom, po, W, H, 4, seed=n + W)
    x = synth(rng, n, 4, 0, 0.2)
    for min_hits in (0, 2):
        got = ctx.soft_assign(x, min_hits)
        assert_soft_assign_rows(got, o, x, min_hits, f"{W}x{H}, {n} rows, min_hits={min_hits}")
        assert np.all(np.abs(got.sum(axis=1) - 1.0) < 1e-12)
    ctx.close()


def test_soft_assign_in_several_batches(vsom, po):
    """A map of 32 768 nodes: batches of 2^28 / (8 N) = 1 024 rows, so 2 049 rows take three batches, the last one a single
    row.  About 0.5 GB of f64 probabilities (what crossing a 256 MiB batch takes), compared against the oracle in blocks."""
    W, H, Din, n = 256, 128, 3, 2049
    rng, o, ctx = soft_assign_map(vsom, po, W, H, Din, seed=5)
    x = synth(rng, n, Din, 0, 0.2)
    got = ctx.soft_assign(x, 1)
    assert_soft_assign_rows(got, o, x, 1, "three batches")
    ctx.close()


@pytest.mark.parametrize("tr,Din,order", [(2, 6, 0), (0, 5, 2), (1, 7, 2)], ids=["clr_j6-seq", "std-eigen_sse", "med-eigen_sse"])
def test_soft_assign_node_count_not_a_multiple_of_128(vsom, po, tr, Din, order):
    """40 x 30 = 1 200 nodes: ten x-blocks of the terms kernel, the last one partly empty; CLR (Dm = 30, 15 pairs) and the Eigen
    order, whose distances are chains the sequential path never runs."""
    rng, o, ctx = soft_assign_map(vsom, po, 40, 30, Din, tr, order, seed=Din)
    x = synth(rng, 300, Din, tr, 0.2)
    for min_hits in (0, 3):
        assert_soft_assign_rows(ctx.soft_assign(x, min_hits), o, x, min_hits, f"min_hits={min_hits}")
    ctx.close()


def test_soft_assign_with_a_zero_sum_is_nan_like_the_reference(vsom, po):
    """C = 0: rows so far from the map that every term underflows, and a min_hits above every node's hits.  The reference divides
    0 by 0 without a guard, so the whole row is NaN; rows of the same batch that are close to the map are not affected."""
    rng, o, ctx = soft_assign_map(vsom, po, 9, 7, 4, seed=11)
    x = synth(rng, 40, 4, 0, 0.2)
    x[::3] = np.float32(1e4) * np.sign(x[::3])  # squared distance ~ 4e8: exp(-d^2 / 2) is 0 for every node
    got = ctx.soft_assign(x, 0)
    assert np.isnan(got[::3]).all() and not np.isnan(np.delete(got, np.s_[::3], axis=0)).any()
    assert_soft_assign_rows(got, o, x, 0, "far rows")
    got = ctx.soft_assign(x, 4)  # hits are 0..3
    assert np.isnan(got).all()
    assert_soft_assign_rows(got, o, x, 4, "min_hits above every node")
    ctx.close()


def test_soft_assign_of_no_rows_launches_nothing(vsom, po):
    _, _, ctx = soft_assign_map(vsom, po, 9, 7, 4)
    before = ctx.launch_count
    assert vsom.lib().vsom_soft_assign(ctx._h, None, 0, 0, None) == 0
    assert ctx.soft_assign(np.zeros((0, 4), np.float32)).shape == (0, 63)
    assert ctx.launch_count == before
    ctx.close()


# ------------------------------------------------------------------------------------------------ U-matrix
def umatrix_state(rng, N, Dm):
    mean = rng.standard_normal((N, Dm)).astype(np.float32)
    sigma = np.abs(rng.standard_normal((N, Dm))).astype(np.float32)
    sigma[rng.random((N, Dm)) < 0.15] = 0.0  # exact zeros: the reference clamps them to 1e-5
    return mean, sigma


def assert_umatrix_matches(ctx, o, mean, sigma, what):
    o.set_state(mean=mean, sigma=sigma)
    ctx.upload_state(mean=mean, sigma=sigma)
    assert_bit_equal(ctx.update_umatrix(), o.update_umatrix(), what)


@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
@pytest.mark.parametrize("W,H", [(2, 2), (2, 3), (3, 2), (2, 9), (9, 2), (16, 4), (17, 5), (15, 8), (33, 9)])
def test_umatrix_grid_shapes(vsom, po, W, H, order):
    """Grids around the 16 x 4 tile and the one-node border (every node an edge or a corner on the thin ones), both kernels.
    Two states through one context with an upload between them: the row and tile tables are built once and cached, and the
    second matrix must be the new state's."""
    Din = 37
    rng = np.random.default_rng(W * 100 + H)
    o = po.Oracle(W, H, Din, 0, order)
    ctx = vsom.VsomContext(W, H, Din, 0, order)
    assert_umatrix_matches(ctx, o, *umatrix_state(rng, W * H, Din), "first state")
    assert_umatrix_matches(ctx, o, *umatrix_state(rng, W * H, Din), "second state")
    ctx.close()


@pytest.mark.parametrize("W,H", [(1, 5), (5, 1)])
def test_umatrix_refuses_one_row_and_one_column_maps(vsom, W, H):
    ctx = vsom.VsomContext(W, H, 3)
    raises_code(vsom, VSOM_ERR_INVALID, ctx.update_umatrix)
    ctx.close()


@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
@pytest.mark.parametrize("tr", [1, 2], ids=["median", "clr"])
@pytest.mark.parametrize("J", [3, 9, 12])
def test_umatrix_model_length_differs_from_the_rows(vsom, po, tr, J, order):
    """The U-matrix runs over the model vector (Dm), not the rows (Din): Median has Dm = J, CLR Dm = J (J - 1) = 6, 72, 132."""
    W, H = 17, 6
    rng = np.random.default_rng(J * 10 + tr)
    o = po.Oracle(W, H, J, tr, order)
    ctx = vsom.VsomContext(W, H, J, tr, order)
    assert ctx.Dm == o.Dm == (J * (J - 1) if tr == 2 else J)
    assert_umatrix_matches(ctx, o, *umatrix_state(rng, W * H, ctx.Dm), f"J={J}")
    ctx.close()


@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
def test_umatrix_taller_than_the_grid_limit(vsom, po, order):
    """2 x 262 148 nodes: ceil(H / 4) = 65 537 tiles, one more than gridDim.y allows in one launch."""
    W, H = 2, 262148
    rng = np.random.default_rng(order)
    o = po.Oracle(W, H, 1, 0, order)
    ctx = vsom.VsomContext(W, H, 1, 0, order)
    assert_umatrix_matches(ctx, o, *umatrix_state(rng, W * H, 1), "tall map")
    ctx.close()


# ------------------------------------------------------------------------------------------------ index build, device form
def index_map(vsom, N):
    W = next(w for w in range(int(np.sqrt(N)), 0, -1) if N % w == 0)
    if W == 1:
        W = N  # a prime node count: one row
    return vsom.VsomContext(W, N // W, 2)


def index_bmu(rng, n, N):
    bmu = np.where(rng.random(n) < 0.5, rng.integers(0, N, n), rng.zipf(1.3, n) % N).astype(np.uint32)
    if n:
        bmu[-1] = N - 1
    return bmu


def build_index_on_device(ctx, bmu):
    import torch

    n = len(bmu)
    bmu_d = torch.from_numpy(bmu.view(np.int32)).cuda()
    counts = torch.full((ctx.N,), -1, dtype=torch.int64, device="cuda")
    offsets = torch.full((ctx.N + 1,), -1, dtype=torch.int64, device="cuda")
    rows = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()  # the inputs are written on torch's stream; the call enqueues on the context's
    ctx.build_index_device(bmu_d, n, counts, offsets, rows)
    ctx.synchronize()
    return counts.cpu().numpy().view(np.uint64), offsets.cpu().numpy().view(np.uint64), rows.cpu().numpy().view(np.uint32)


@pytest.mark.parametrize("n,N", [(0, 12), (1, 12), (2049, 100), (65536, 24576), (65536, 24577), (70001, 65537), (3000, 1)],
                         ids=["empty", "one_row", "two_sort_ctas", "smem_hist", "global_hist", "three_radix_passes", "one_node"])
def test_build_index_device_form(vsom, po, n, N):
    """vsom_build_index_device on torch device tensors equals the host form and the oracle: the shared-memory histogram (maps of
    up to 24 576 nodes, 65 536 rows or more) and the global one, one to three radix passes, two sort CTAs, a 1 x 1 map.  The host
    form with NULL row ids skips the sort; its counts and offsets must be the same."""
    rng = np.random.default_rng(n + N)
    ctx = index_map(vsom, N)
    assert ctx.N == N
    bmu = index_bmu(rng, n, N)
    oc, oo, orows = po.Oracle.build_index(bmu, N)
    dc, do, drows = build_index_on_device(ctx, bmu)
    hc, ho, hrows = ctx.build_index(bmu)
    for what, (d, h, want) in {"counts": (dc, hc, oc), "offsets": (do, ho, oo), "row ids": (drows, hrows, orows)}.items():
        assert_bit_equal(d, want, f"device form: {what}")
        assert_bit_equal(h, want, f"host form: {what}")
    counts, offsets = np.empty(N, np.uint64), np.empty(N + 1, np.uint64)
    assert vsom.lib().vsom_build_index(ctx._h, _ptr(bmu, _u32p), n, _ptr(counts, _u64p), _ptr(offsets, _u64p), None) == 0
    assert_bit_equal(counts, oc, "counts without row ids")
    assert_bit_equal(offsets, oo, "offsets without row ids")
    ctx.close()


def test_build_index_device_out_of_range_id_leaves_the_context_usable(vsom, po):
    """The device form does not report an out-of-range BMU id (only the host form does), so the call succeeds.  The error flag it
    raises is cleared by each of its users: the next host-form index build, scoring and training on the same context succeed
    and still match the oracle."""
    import torch

    W, H, Din = 12, 10, 6
    N = W * H
    rng = np.random.default_rng(3)
    o = po.Oracle(W, H, Din)
    o.random_initialize(8, 1.0)
    ctx = vsom.VsomContext(W, H, Din)
    ctx.upload_state(**o.get_state())
    bad = rng.integers(0, N, 5000).astype(np.uint32)
    bad[[17, 4000]] = [N, 0xFFFFFFFF]
    bad_d = torch.from_numpy(bad.view(np.int32)).cuda()
    counts = torch.empty(N, dtype=torch.int64, device="cuda")
    offsets = torch.empty(N + 1, dtype=torch.int64, device="cuda")
    rows = torch.empty(len(bad), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.build_index_device(bad_d, len(bad), counts, offsets, rows)
    ctx.synchronize()

    good = index_bmu(rng, 3000, N)
    hc, ho, hrows = ctx.build_index(good)
    oc, oo, orows = po.Oracle.build_index(good, N)
    assert_bit_equal(hc, oc, "counts")
    assert_bit_equal(ho, oo, "offsets")
    assert_bit_equal(hrows, orows, "row ids")
    x = synth(rng, 1100, Din, 0)  # enough rows for K2, which reads the flag back
    gb, gd = ctx.find_bmu(x)
    assert ctx.last_score_tc >= 1
    ob, od = o.find_bmu(x)
    assert_bit_equal(gb, ob, "bmu")
    assert_bit_equal(gd, od, "dist")
    gb, gd, gr, _ = ctx.train_chunk(x, 0.1, 3.0, vsom.EXPONENTIAL)
    ob, od, orr, _ = o.train_rows(x, 0.1, 3.0, 0)
    assert_bit_equal(gb, ob, "trained bmu")
    assert_bit_equal(gd, od, "trained dist")
    got, want = ctx.download_state(), o.get_state()
    for k in ("mean", "S", "sigma", "weight", "hits"):
        assert_bit_equal(got[k], want[k], f"trained {k}")
    ctx.close()


# ------------------------------------------------------------------------------------------------ node read-back
@pytest.mark.parametrize("Din", [4, 5, 6, 7])
def test_get_node_reads_the_node_row(vsom, po, Din):
    """vsom_get_node (Som::getNeuron / getSigmaNeuron, what Som::trainSingle reads back): the device rows are padded to a multiple
    of four floats, so the read-back must start at node * rowStride, not node * Dm."""
    W, H = 9, 7
    N = W * H
    rng = np.random.default_rng(Din)
    mean = rng.standard_normal((N, Din)).astype(np.float32)
    sigma = np.abs(rng.standard_normal((N, Din))).astype(np.float32)
    ctx = vsom.VsomContext(W, H, Din)
    ctx.upload_state(mean=mean, sigma=sigma)
    nodes = (0, N // 2, N - 1)
    for p in nodes:
        m, s = ctx.get_node(p)
        assert_bit_equal(m, mean[p], f"mean of node {p}")
        assert_bit_equal(s, sigma[p], f"sigma of node {p}")
    ctx.train_chunk(synth(rng, 64, Din, 0), 0.2, 2.5, vsom.EXPONENTIAL)
    st = ctx.download_state()
    for p in nodes:
        m, s = ctx.get_node(p)
        assert_bit_equal(m, st["mean"][p], f"trained mean of node {p}")
        assert_bit_equal(s, st["sigma"][p], f"trained sigma of node {p}")
    # either output may be NULL
    L = vsom.lib()
    m = np.full(Din, np.nan, np.float32)
    s = np.full(Din, np.nan, np.float32)
    assert L.vsom_get_node(ctx._h, N - 1, None, _ptr(s, _f32p)) == 0
    assert_bit_equal(s, st["sigma"][N - 1], "sigma only")
    assert L.vsom_get_node(ctx._h, N - 1, _ptr(m, _f32p), None) == 0
    assert_bit_equal(m, st["mean"][N - 1], "mean only")
    assert L.vsom_get_node(ctx._h, 0, None, None) == 0
    raises_code(vsom, VSOM_ERR_INVALID, ctx.get_node, N)
    ctx.close()


def test_get_node_on_a_sharded_context_is_unsupported(vsom):
    ctxs = [vsom.VsomContext(13, 37, 10, vsom.STANDARD, vsom.ORDER_REFERENCE, device=0, rank=r, world=2) for r in range(2)]
    for c in ctxs:
        raises_code(vsom, VSOM_ERR_UNSUPPORTED, c.get_node, 0)
    for c in ctxs:
        c.close()


# ------------------------------------------------------------------------------------------------ ORDER_LANES outside training
@pytest.mark.parametrize("tr,Din", [(0, 37), (1, 20), (2, 6)], ids=["standard", "median", "clr"])
def test_lanes_context_outside_training_sums_in_the_reference_order(vsom, po, tr, Din):
    """Only the online step sums in the lanes order.  On a VSOM_ORDER_LANES context the exact scan, K2 and its rescore, all_dists,
    soft assignment, the U-matrix and the batch-map trainer must return the sequential-order oracle's bits."""
    W, H = 24, 20
    N = W * H
    rng = np.random.default_rng(Din)
    o = po.Oracle(W, H, Din, tr, po.ORDER_SEQUENTIAL)
    st = o.get_state()
    st["mean"] = (0.1 * rng.standard_normal(st["mean"].shape)).astype(np.float32)  # small distances: no term of the soft assignment underflows
    st["sigma"] = np.abs(rng.standard_normal(st["sigma"].shape)).astype(np.float32)
    st["hits"] = rng.integers(0, 4, N).astype(np.uint64)
    o.set_state(**st)
    ctx = vsom.VsomContext(W, H, Din, tr, vsom.ORDER_LANES)
    ctx.upload_state(**st)
    x = synth(rng, 1500, Din, tr, 0.1)

    ob, od = o.find_bmu(x)
    eb, ed = ctx.find_bmu_exact(x)
    assert_bit_equal(eb, ob, "exact scan bmu")
    assert_bit_equal(ed, od, "exact scan dist")
    assert_bit_equal(ctx.find_bmu_exact(x, min_hits=2)[0], o.find_restricted_bmu(x, 2), "restricted exact scan")
    tb, td = ctx.find_bmu(x)
    assert ctx.last_score_tc >= 1 if tr != 2 else ctx.last_score_tc == 0  # K2 covers Standard / Median only
    assert_bit_equal(tb, ob, "dispatched bmu")
    assert_bit_equal(td, od, "dispatched dist")
    assert_bit_equal(ctx.all_dists(x[7]), o.all_dists(x[7]), "all dists")
    assert_soft_assign_rows(ctx.soft_assign(x[:64], 1), o, x[:64], 1, "soft assignment")
    assert_bit_equal(ctx.update_umatrix(), o.update_umatrix(), "umatrix")

    last = None
    for epoch, sigma in enumerate((3.0, 1.5)):
        om, ol = o.batch_epoch(x, sigma, epoch == 0, last)
        gm, gl = ctx.batch_epoch(x, sigma, epoch == 0, last)
        assert np.float32(gm).view(np.uint32) == np.float32(om).view(np.uint32), f"mse, epoch {epoch}"
        assert np.array_equal(gl, ol), f"lastBMU, epoch {epoch}"
        got, want = ctx.download_state(), o.get_state()
        for k in ("mean", "S", "sigma", "weight"):
            # a neuron without weight divides 0 by 0 in the reference too; NaN payloads are not part of the contract
            g, w = got[k].copy(), want[k].copy()
            assert np.array_equal(np.isnan(g), np.isnan(w)), f"epoch {epoch}: {k} NaN pattern"
            g[np.isnan(g)] = 0
            w[np.isnan(w)] = 0
            assert_bit_equal(g, w, f"epoch {epoch}: {k}")
        assert_bit_equal(got["hits"], want["hits"], f"epoch {epoch}: hits")
        last = ol
    ctx.close()
