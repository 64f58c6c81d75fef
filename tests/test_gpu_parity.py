"""GPU parity tests proper: libvsom_b200.so (through its C-ABI) against the CPU oracle and against the committed
fixtures generated from the reference's own code.  Bit-exact everywhere the reduction order is the reference's
(VSOM_ORDER_REFERENCE, all scoring, U-matrix, index); near-tie rule for VSOM_ORDER_LANES.

Tolerances (stated here as the north-star asks):
  * ORDER_REFERENCE: 0 ulp on BMU ids, distances, mean / S / sigma / weight planes, hits, U-matrix, evaluate().
  * ORDER_LANES: BMU ids equal except documented near-ties: the two candidates' distances, re-evaluated in f64
    from the same f32 state, differ by at most EPS_REL = 2*Dm*2^-24 relative; distances within 1e-5 relative."""
import numpy as np
import pytest

from conftest import assert_bit_equal, load_golden

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

CASES = ["std_exp", "std_inv", "med_exp", "med_inv", "clr_exp", "clr_inv"]


def upload_like(ctx, st):
    ctx.upload_state(st["mean"], st["S"], st["sigma"], st["weight"], st["hits"])


def assert_state_equal(ctx, ref_state, what):
    got = ctx.download_state()
    for k in ("mean", "S", "sigma", "weight", "hits"):
        assert_bit_equal(got[k], ref_state[k], f"{what}: {k}")


@pytest.fixture(params=["fast", "generic"])
def online_kernel(request, monkeypatch):
    """Both online-step kernels must reproduce the reference: K1F (online_step_fast.cu) where it is eligible, and the
    generic kernel forced through VSOM_ONLINE_KERNEL=generic (read by vsom_create)."""
    if request.param == "generic":
        monkeypatch.setenv("VSOM_ONLINE_KERNEL", "generic")
    else:
        monkeypatch.delenv("VSOM_ONLINE_KERNEL", raising=False)
    return request.param


@pytest.mark.parametrize("name", CASES)
def test_online_step_matches_reference_fixture(vsom, name, online_kernel):
    """K1 (reference order) replays the fixture the reference's own code produced, bit for bit."""
    g = load_golden(f"ref_{name}.npz")
    W, H, Din, tr, dec = int(g["W"]), int(g["H"]), int(g["Din"]), int(g["transform"]), int(g["decay"])
    ctx = vsom.VsomContext(W, H, Din, tr, vsom.ORDER_REFERENCE)
    ctx.upload_state(mean=g["init_mean"])
    rows = int(g["rows"])
    for si, sg in enumerate(g["sigmas"]):
        seg = g["x"][si * rows:(si + 1) * rows]
        bmu, dist, resid2, last = ctx.train_chunk(seg, float(g["eta"]), float(sg), dec)
        assert ctx.last_train_fast == (online_kernel == "fast")  # K1F serves sigma > 1 and the local-walk regime alike
        assert_bit_equal(bmu, g[f"bmu{si}"], f"bmu seg {si}")
        assert_bit_equal(dist, g[f"dist{si}"], f"dist seg {si}")
        assert_bit_equal(resid2, g[f"resid2{si}"], f"resid2 seg {si}")
        assert_bit_equal(last, g[f"last{si}"], f"lastBMU seg {si}")
        assert_state_equal(ctx, {k: g[f"{k}{si}"] for k in ("mean", "S", "sigma", "weight", "hits")}, f"seg {si}")
    ctx.close()


@pytest.mark.parametrize("name", CASES)
def test_scoring_umatrix_match_reference_fixture(vsom, name):
    """K3 / K4 on the fixture's final state."""
    g = load_golden(f"ref_{name}.npz")
    W, H, Din, tr = int(g["W"]), int(g["H"]), int(g["Din"]), int(g["transform"])
    last = len(g["sigmas"]) - 1
    ctx = vsom.VsomContext(W, H, Din, tr)
    upload_like(ctx, {k: g[f"{k}{last}"] for k in ("mean", "S", "sigma", "weight", "hits")})
    assert_bit_equal(ctx.update_umatrix(), g["umatrix"], "umatrix")
    q = g["x"][:64]
    b, d = ctx.find_bmu(q)
    assert_bit_equal(b, g["score_bmu"], "bmu")
    assert_bit_equal(d, g["score_dist"], "dist")
    assert_bit_equal(ctx.find_bmu(q, min_hits=2)[0], g["restricted_bmu"], "restricted bmu")
    assert_bit_equal(ctx.all_dists(q[0]), g["all_dists_row0"], "all dists")
    if "evaluate" in g.files:
        assert ctx.evaluate(q) == float(g["evaluate"])
    ctx.close()


# (W, H, Din, transform, rows, eta, sigma) — covers: fewer nodes than SMs, several nodes per CTA, planes resident
# in shared memory and planes left in global memory (100x100x784 does not fit), CLR at J=32 (992 params / node).
SHAPES = [
    (4, 3, 3, 0, 64, 0.5, 1.5),
    (20, 20, 784, 0, 48, 0.1, 5.0),
    (64, 64, 128, 1, 96, 0.05, 16.0),
    (64, 64, 784, 0, 24, 0.1, 3.0),
    (100, 100, 784, 0, 12, 0.1, 4.0),
    (50, 50, 32, 2, 32, 0.001, 12.0),
    (33, 7, 20, 2, 64, 0.002, 2.0),
    # K1F corner cases: more than 32 nodes per CTA (several scan warps), sample length not a multiple of 4 (4-byte
    # cp.async path, padded rows), one-row / one-column maps, a window that never covers the whole map
    (128, 128, 16, 1, 64, 0.05, 20.0),
    (150, 90, 8, 0, 48, 0.1, 6.0),
    (37, 29, 33, 0, 64, 0.1, 4.0),
    (31, 1, 5, 1, 40, 0.2, 2.0),
    (1, 200, 130, 0, 40, 0.2, 3.0),
    (40, 40, 64, 1, 48, 0.1, 6.0),     # 11 nodes per CTA: two register-resident items per warp
    # generic kernel with many owned nodes per CTA: window-cell enumeration instead of a test of every owned node, on an
    # HBM-resident map (warp-tiled scan) and on a shared-memory-resident CLR map
    (150, 150, 784, 0, 10, 0.1, 6.0),
    (130, 130, 8, 2, 24, 0.001, 5.0),
]


def synth(rng, n, Din, tr):
    if tr == 2:
        z = rng.standard_normal((n, 1)).astype(np.float32)
        a = rng.uniform(0.5, 1.5, (1, Din)).astype(np.float32)
        return (a * z + 0.1 * rng.standard_normal((n, Din))).astype(np.float32)
    return rng.standard_normal((n, Din)).astype(np.float32)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("decay,order", [(0, 0), (1, 0), (0, 2), (1, 2)], ids=["exp-seq", "inv-seq", "exp-eigen_sse", "inv-eigen_sse"])
def test_online_step_matches_oracle_bit_exact(vsom, po, shape, decay, order, online_kernel):
    """order 0 = VSOM_ORDER_REFERENCE (sequential dot, the reference built against the stand-in Eigen header), order 2 =
    VSOM_ORDER_EIGEN_SSE (the reference built against real Eigen under -msse2: Packet4f redux order); the oracle runs the
    same order and the whole trajectory must be bit-identical either way."""
    W, H, Din, tr, n, eta, sigma = shape
    if online_kernel == "generic" and (W, H, Din) in ((100, 100, 784), (64, 64, 784), (150, 150, 784)):
        pytest.skip("the generic kernel is what runs these shapes in the fast variant too (K1F does not fit)")
    if order == 2 and decay == 1 and (W * H > 5000 or Din > 200):
        pytest.skip("the decay mode does not interact with the summation order: the large shapes run Exponential only in the Eigen order")
    rng = np.random.default_rng(hash((W, H, Din, tr, decay)) % (2 ** 32))
    o = po.Oracle(W, H, Din, tr, order)
    o.random_initialize(42, 1.0)
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    upload_like(ctx, o.get_state())
    x = synth(rng, 2 * n, Din, tr)
    # second chunk: smaller window, carried state; third and fourth: the findLocalBmu regime (sigma <= 1), once from node
    # 0 like DataSet gives it, once from arbitrary start nodes
    m = max(8, n // 3)
    starts = rng.integers(0, W * H, m).astype(np.uint64)
    for seg, sg, last in ((x[:n], sigma, None), (x[n:], max(1.0001, sigma * 0.6), None), (x[:m], 1.0, None), (x[m:2 * m], 0.75, starts)):
        ob, od, orr, ol = o.train_rows(seg, eta, sg, decay, last_bmu=None if last is None else last.copy())
        gb, gd, gr, gl = ctx.train_chunk(seg, eta, sg, decay, last_bmu=None if last is None else last.copy())
        assert_bit_equal(gb, ob, f"bmu sigma={sg}")
        assert_bit_equal(gd, od, f"dist sigma={sg}")
        assert_bit_equal(gr, orr, f"resid2 sigma={sg}")
        assert np.array_equal(gl, ol)
        assert_state_equal(ctx, o.get_state(), f"sigma={sg}")
    # scoring / U-matrix on the trained state
    q = x[:40]
    ob, od = o.find_bmu(q)
    gb, gd = ctx.find_bmu(q)
    assert_bit_equal(gb, ob, "score bmu")
    assert_bit_equal(gd, od, "score dist")
    assert_bit_equal(ctx.find_bmu(q, min_hits=1)[0], o.find_restricted_bmu(q, 1), "restricted")
    assert_bit_equal(ctx.all_dists(q[3]), o.all_dists(q[3]), "all dists")
    if W >= 2 and H >= 2:  # the reference's updateUMatrix indexes out of bounds on one-row / one-column maps
        assert_bit_equal(ctx.update_umatrix(), o.update_umatrix(), "umatrix")
    if tr != 2:
        assert ctx.evaluate(q) == o.evaluate(q)
    ctx.close()


def test_resident_and_global_plane_modes_are_both_exercised(vsom):
    a = vsom.VsomContext(64, 64, 128, vsom.MEDIAN)
    b = vsom.VsomContext(100, 100, 784, vsom.STANDARD)
    c = vsom.VsomContext(50, 50, 32, vsom.CLR)
    assert a.planes_resident and c.planes_resident and not b.planes_resident
    for k in (a, b, c):
        k.close()


@pytest.mark.parametrize("shape", [(20, 20, 784, 0, 400, 0.1, 5.0), (64, 64, 128, 1, 600, 0.05, 16.0), (50, 50, 32, 2, 60, 0.001, 12.0)])
def test_online_step_lanes_order_near_tie_rule(vsom, po, shape):
    """ORDER_LANES: same update arithmetic, different summation order of the distance.  Any BMU that differs
    from the oracle's must be a near-tie at the first point of divergence."""
    W, H, Din, tr, n, eta, sigma = shape
    rng = np.random.default_rng(7)
    o = po.Oracle(W, H, Din, tr)
    o.random_initialize(42, 1.0)
    init = o.get_state()
    x = synth(rng, n, Din, tr)
    ctx = vsom.VsomContext(W, H, Din, tr, vsom.ORDER_LANES)
    upload_like(ctx, init)
    gb, gd, _, _ = ctx.train_chunk(x, eta, sigma, 0)
    ob, od, _, _ = o.train_rows(x, eta, sigma, 0)
    Dm = ctx.Dm
    eps_rel = 2 * Dm * 2.0 ** -24
    diff = np.nonzero(gb != ob)[0]
    agree = 1.0 - len(diff) / n
    print(f"lanes-order BMU agreement {agree:.6f} ({len(diff)} of {n} differ), eps_rel={eps_rel:.3e}")
    if len(diff) == 0:
        assert_state_equal(ctx, o.get_state(), "lanes order, all BMUs equal")
        np.testing.assert_allclose(gd, od, rtol=1e-5, atol=1e-30)
    else:
        i = int(diff[0])  # first divergence: states were identical up to here
        o2 = po.Oracle(W, H, Din, tr)
        o2.set_state(**init)
        if i:
            o2.train_rows(x[:i], eta, sigma, 0)
            np.testing.assert_allclose(gd[:i], od[:i], rtol=1e-5, atol=1e-30)
        d64 = o2.all_dists_f64(x[i])
        a, b = d64[gb[i]], d64[ob[i]]
        assert abs(a - b) <= eps_rel * max(a, b), f"row {i}: BMU {gb[i]} vs {ob[i]} is not a near-tie: {a} vs {b}"
    ctx.close()


@pytest.mark.parametrize("n,N", [(0, 12), (1, 12), (2047, 100), (2048, 400), (2049, 4096), (100000, 16384), (300000, 24576), (70001, 70000)])
def test_build_index(vsom, po, n, N):
    W = N // 4 if N % 4 == 0 else N
    H = N // W
    ctx = vsom.VsomContext(W, H, 2)
    rng = np.random.default_rng(n + N)
    bmu = (rng.zipf(1.3, n) % N).astype(np.uint32) if n else np.zeros(0, np.uint32)
    counts, offsets, rows = ctx.build_index(bmu)
    oc, oo, orows = po.Oracle.build_index(bmu, N)
    assert_bit_equal(counts, oc, "counts")
    assert_bit_equal(offsets, oo, "offsets")
    assert_bit_equal(rows, orows, "row ids")
    if n:
        with pytest.raises(vsom.VsomError):
            ctx.build_index(np.array([N], np.uint32))
    ctx.close()


def test_full_size_properties_config2(vsom):
    """BASELINE config 2 shape (64x64, median, D=128) at a size the oracle cannot replay in seconds: properties."""
    rng = np.random.default_rng(5)
    n, W, H, D = 60000, 64, 64, 128
    centres = rng.standard_normal((64, D)).astype(np.float32) * 3
    x = (centres[rng.integers(0, 64, n)] + rng.standard_normal((n, D))).astype(np.float32)
    ctx = vsom.VsomContext(W, H, D, vsom.MEDIAN)
    init = (rng.integers(-1000, 1000, (W * H, D)) / 1000).astype(np.float32)
    ctx.upload_state(mean=init)
    bmu, dist, resid2, last = ctx.train_chunk(x, 0.05, 32.0, vsom.EXPONENTIAL)
    st = ctx.download_state()
    assert bmu.max() < W * H
    assert_bit_equal(dist, resid2, "dist == resid2")
    assert int(st["hits"].sum()) == n and np.array_equal(st["hits"], np.bincount(bmu, minlength=W * H).astype(np.uint64))
    assert np.isfinite(st["mean"]).all() and np.isfinite(st["sigma"]).all() and (st["sigma"] >= 0).all()
    assert (st["weight"] > 0).all()
    # sigma is always sqrt(|S / W|) of the same node (src/Som.cpp:939-942)
    np.testing.assert_array_equal(st["sigma"], np.sqrt(np.abs(st["S"] / st["weight"][:, None])).astype(np.float32))
    # idempotence of scoring: the BMU distance is the minimum of the row's distances, lowest index on ties
    b2, d2 = ctx.find_bmu(x[:512])
    for r in (0, 17, 511):
        d = ctx.all_dists(x[r])
        assert int(np.argmin(d)) == int(b2[r]) and np.float32(d.min()) == d2[r]
    # determinism: the same chunk from the same state gives the same bits
    ctx.upload_state(mean=init, S=np.zeros_like(init), sigma=np.zeros_like(init), weight=np.zeros(W * H, np.float32), hits=np.zeros(W * H, np.uint64))
    bmu2, dist2, _, _ = ctx.train_chunk(x, 0.05, 32.0, vsom.EXPONENTIAL)
    assert_bit_equal(bmu2, bmu, "rerun bmu")
    assert_bit_equal(dist2, dist, "rerun dist")
    c, o, rows = ctx.build_index(bmu)
    assert np.array_equal(c, st["hits"]) and np.all(np.diff(bmu[rows].astype(np.int64)) >= 0)
    ctx.close()


# ------------------------------------------------------------------------------------------------ K2 (tensor cores)
def _tc_case(rng, W, H, D, n, near_nodes):
    m = rng.standard_normal((W * H, D)).astype(np.float32)
    if near_nodes:  # rows close to (several) nodes: small gaps between candidates, exercises the guard / fallback
        x = (m[rng.integers(0, W * H, n)] * 0.5 + m[rng.integers(0, W * H, n)] * 0.5 + 0.05 * rng.standard_normal((n, D))).astype(np.float32)
    else:
        x = rng.standard_normal((n, D)).astype(np.float32)
    return m, x


@pytest.mark.parametrize("shape", [(64, 64, 128, 5000, False), (128, 128, 256, 3001, False), (30, 21, 100, 4097, True), (128, 128, 256, 2048, True),
                                   (16, 16, 7, 1500, False)])
def test_tensor_core_scoring_equals_exact_scan(vsom, shape):
    """K2 (tcgen05 candidate search + exact rescore + guarded fallback) must return exactly what K3 returns:
    same BMU ids (bit-exact) and same f32 distances (bit-exact) — the tensor cores only select candidates."""
    W, H, D, n, near = shape
    rng = np.random.default_rng(W * H + D + n)
    m, x = _tc_case(rng, W, H, D, n, near)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD)
    hits = rng.integers(0, 4, W * H).astype(np.uint64)
    ctx.upload_state(mean=m, hits=hits)
    eb, ed = ctx.find_bmu_exact(x)
    assert not ctx.last_score_tc
    tb, td, fb = ctx.find_bmu_batch(x)
    assert ctx.last_score_tc
    print(f"K2 {W}x{H}x{D}, {n} rows, near={near}: {fb} rows ({100.0 * fb / n:.2f}%) took the exact-scan fallback")
    assert_bit_equal(tb, eb, "bmu")
    assert_bit_equal(td, ed, "dist")
    assert fb < n  # the tensor-core path did the selection for at least some rows
    # the reference-facing calls (vsom_find_bmu / vsom_evaluate: what Som::evaluate, measureSimilarity and mapDataSet use)
    # dispatch to the same tensor-core path for batches like this one
    db, dd = ctx.find_bmu(x)
    assert ctx.last_score_tc
    assert_bit_equal(db, eb, "dispatched bmu")
    assert_bit_equal(dd, ed, "dispatched dist")
    err = 0.0
    for i, d in enumerate(ed):  # src/Som.cpp:519
        err += 1.0 / (i + 1.0) * (float(d) - err)
    assert ctx.evaluate(x) == err and ctx.last_score_tc
    eb2, _ = ctx.find_bmu_exact(x[:2000], min_hits=2)
    tb2, _, _ = ctx.find_bmu_batch(x[:2000], min_hits=2)
    assert_bit_equal(tb2, eb2, "restricted bmu")
    ctx.close()


def test_tensor_core_scoring_unsupported_shapes_use_exact(vsom):
    ctx = vsom.VsomContext(12, 12, 9, vsom.CLR)  # CLR residuals are not a plain |m - x|^2: exact scan
    rng = np.random.default_rng(1)
    ctx.upload_state(mean=rng.standard_normal((144, 72)).astype(np.float32))
    x = rng.standard_normal((1500, 9)).astype(np.float32)
    eb, ed = ctx.find_bmu_exact(x)
    tb, td, fb = ctx.find_bmu_batch(x)
    assert fb == 1500 and not ctx.last_score_tc
    assert_bit_equal(tb, eb, "bmu")
    assert_bit_equal(td, ed, "dist")
    ctx.close()


@pytest.mark.parametrize("tier", ["1", "2"])
@pytest.mark.parametrize("shape", [(64, 64, 128, 3000 + 77), (40, 25, 300, 1300)])
def test_tensor_core_single_cta_variant_equals_the_pair_kernel(vsom, monkeypatch, shape, tier):
    """score_tc_kernel<PAIR=false> (VSOM_TC_PAIR=0: one CTA per 128 rows, whole B tile per SM) is kept beside the default CTA-pair
    kernel; both must return the exact scan's results on a trained map, resident and streamed A alike, with an odd number of
    row tiles (the pair's last unit is half empty)."""
    monkeypatch.setenv("VSOM_TC_TIER", tier)
    W, H, D, n = shape
    rng = np.random.default_rng(W + D)
    centres = (rng.standard_normal((12, D)) * 2).astype(np.float32)
    data = lambda k: (centres[rng.integers(0, 12, k)] + 0.4 * rng.standard_normal((k, D))).astype(np.float32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=(rng.integers(-1000, 1000, (W * H, D)) / 1000).astype(np.float32))
    for sg, eta in ((W / 3.0, 0.4), (W / 8.0, 0.2), (2.0, 0.1)):
        ctx.train_chunk(data(1500), eta, sg, vsom.EXPONENTIAL)
    q = data(n)
    eb, ed = ctx.find_bmu_exact(q)
    for pair in ("1", "0"):
        monkeypatch.setenv("VSOM_TC_PAIR", pair)
        tb, td, fb = ctx.find_bmu_batch(q)
        assert ctx.last_score_tc == int(tier) and ctx.last_score_pair == int(pair)  # a whole B200 schedules clusters of two
        assert_bit_equal(tb, eb, f"bmu, pair={pair}")
        assert_bit_equal(td, ed, f"dist, pair={pair}")
    ctx.close()


@pytest.mark.parametrize("tier", ["1", "2", "auto"])
@pytest.mark.parametrize("shape", [(20, 20, 784, 1500), (64, 64, 128, 3000), (128, 128, 256, 2500), (40, 25, 300, 1300), (9, 9, 5, 1100)])
def test_tensor_core_tiers_and_long_rows(vsom, po, monkeypatch, shape, tier):
    """Both precision tiers of K2 (one fp16 value per operand element / hi-lo pairs) and rows longer than the resident A area
    (A k-blocks streamed with B: BASELINE configs 1 and 5 have 784-dim rows) against the ORACLE, on a clustered map."""
    if tier != "auto":
        monkeypatch.setenv("VSOM_TC_TIER", tier)
    else:
        monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    W, H, D, n = shape
    rng = np.random.default_rng(W * D)
    centres = (rng.standard_normal((12, D)) * 2).astype(np.float32)
    data = lambda k: (centres[rng.integers(0, 12, k)] + 0.4 * rng.standard_normal((k, D))).astype(np.float32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=(rng.integers(-1000, 1000, (W * H, D)) / 1000).astype(np.float32))
    for sg, eta in ((W / 3.0, 0.4), (W / 8.0, 0.2), (2.0, 0.1)):
        ctx.train_chunk(data(1500), eta, sg, vsom.EXPONENTIAL)
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.set_state(**ctx.download_state())
    q = data(n)
    ob, od = o.find_bmu(q[:1024] if W * H * D > 2_000_000 else q)
    tb, td, fb = ctx.find_bmu_batch(q)
    print(f"{W}x{H}x{D} tier {tier}: ran tier {ctx.last_score_tc}, {fb} of {n} rows took the exact scan")
    assert ctx.last_score_tc == (int(tier) if tier != "auto" else ctx.last_score_tc) and ctx.last_score_tc in (1, 2)
    assert_bit_equal(tb[:len(ob)], ob, "bmu vs oracle")
    assert_bit_equal(td[:len(od)], od, "dist vs oracle")
    if len(ob) < n:
        eb, ed = ctx.find_bmu_exact(q)
        assert_bit_equal(tb, eb, "bmu vs exact scan")
        assert_bit_equal(td, ed, "dist vs exact scan")
    ctx.close()


def test_tensor_core_scoring_ties_and_overflow_take_the_exact_scan(vsom):
    """A map made of 40 distinct rows repeated many times: every row has dozens of EXACT ties at its best distance.
    The candidate lists overflow, those rows go through the exact scan, and the reference's lowest-index rule must
    hold (the BMU is the first copy)."""
    rng = np.random.default_rng(9)
    W, H, D, n = 48, 48, 64, 3000
    base = rng.standard_normal((40, D)).astype(np.float32)
    m = base[np.arange(W * H) % 40]
    x = (base[rng.integers(0, 40, n)] + 0.01 * rng.standard_normal((n, D))).astype(np.float32)
    ctx = vsom.VsomContext(W, H, D, vsom.MEDIAN)
    ctx.upload_state(mean=m)
    eb, ed = ctx.find_bmu_exact(x)
    tb, td, fb = ctx.find_bmu_batch(x)
    assert eb.max() < 40  # lowest index among the copies
    assert_bit_equal(tb, eb, "bmu")
    assert_bit_equal(td, ed, "dist")
    assert fb > 0
    ctx.close()


def test_tensor_core_probes_hand_hopeless_batches_to_the_exact_scan(vsom):
    """A map whose nodes nearly coincide (what a batch-map epoch with a wide neighbourhood leaves): every node is inside every
    row's margin, no candidate list can be certified at either precision.  The tier-1 and tier-2 probes (8192 rows each, results
    kept) must notice and send the remainder to the exact scan; results stay bit-exact, through the device call and the
    host-buffer call."""
    rng = np.random.default_rng(77)
    W, H, D, n = 20, 20, 96, 3 * 8192 + 1234
    base = rng.standard_normal(D).astype(np.float32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=(base[None, :] + 1e-4 * rng.standard_normal((W * H, D))).astype(np.float32))
    x = (base[None, :] + rng.standard_normal((n, D))).astype(np.float32)
    eb, ed = ctx.find_bmu_exact(x)
    tb, td, fb = ctx.find_bmu_batch(x)
    print(f"probes: tier {ctx.last_score_tc}, {fb} of {n} rows took the exact scan")
    assert ctx.last_score_tc == 3 and fb >= n - 2 * 8192
    assert_bit_equal(tb, eb, "bmu")
    assert_bit_equal(td, ed, "dist")
    import torch
    xd = torch.from_numpy(x).cuda()
    ob = torch.empty(n, dtype=torch.int32, device="cuda")
    od = torch.empty(n, dtype=torch.float32, device="cuda")
    fbd = ctx.find_bmu_batch_device(xd, n, ob, od)
    ctx.synchronize()
    assert ctx.last_score_tc == 3 and fbd >= n - 2 * 8192
    assert_bit_equal(ob.cpu().numpy().astype(eb.dtype), eb, "device bmu")
    assert_bit_equal(od.cpu().numpy(), ed, "device dist")
    ctx.close()


@pytest.mark.parametrize("n, slab_log2", [(300, None), (3 * 8192 + 777, "12"), (20000, None)])
def test_measure_similarity_row_pass_matches_the_reference_formula(vsom, monkeypatch, n, slab_log2):
    """vsom_measure_similarity (the per-row pass of Som::measureSimilarity, src/Som.cpp:631-714): restricted BMU + the row's largest
    ((x - m_bmu) / sM) / numOfSigmas, on the exact-scan path (300 rows), through the tensor-core pipeline with many small slabs and
    both probes, and in one slab — against the same three f32 operations in numpy on the exact scan's BMUs."""
    if slab_log2:
        monkeypatch.setenv("VSOM_TC_HOST_SLAB_LOG2", slab_log2)
    if n < 1024:
        monkeypatch.setenv("VSOM_EXACT_HOST_SLAB_LOG2", "7")  # the exact host path in three slabs of 128 rows
    rng = np.random.default_rng(n)
    W, H, D = 24, 20, 48
    centres = (rng.standard_normal((10, D)) * 2).astype(np.float32)
    data = lambda k: (centres[rng.integers(0, 10, k)] + 0.4 * rng.standard_normal((k, D))).astype(np.float32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=(rng.integers(-1000, 1000, (W * H, D)) / 1000).astype(np.float32))
    for sg, eta in ((8.0, 0.4), (3.0, 0.2), (1.5, 0.1)):
        ctx.train_chunk(data(1500), eta, sg, vsom.EXPONENTIAL)
    st = ctx.download_state()
    sigma = st["sigma"].copy()
    sigma[::7] *= np.float32(1e-6)  # some sigmas below the reference's cap of 1e-5 (src/Som.cpp:648 caps, it does not floor)
    ctx.upload_state(mean=st["mean"], sigma=sigma)
    x = data(n)
    x[5, 3] = np.nan
    min_hits = 1
    eb, _ = ctx.find_bmu_exact(x, min_hits)
    bmu, row_max = ctx.measure_similarity(x, 3, min_hits)
    assert_bit_equal(bmu, eb, "bmu")
    m, s = st["mean"][eb], sigma[eb]
    sM = np.where(s > np.float32(0.00001), np.float32(0.00001), s).astype(np.float32)
    with np.errstate(all="ignore"):
        delta = (((x - m).astype(np.float32) / sM).astype(np.float32) / np.float32(3)).astype(np.float32)
    want = np.where(np.isnan(delta), -np.inf, delta).max(axis=1).astype(np.float32)
    assert_bit_equal(row_max, want, "row maxima")
    ctx.close()


def test_tc_scoring_pipelines_slabs(vsom, monkeypatch):
    monkeypatch.setenv("VSOM_TC_SLAB_LOG2", "20")  # 1M-row slabs instead of 4M, so that three of them fit a test
    _tc_scoring_pipelines_slabs(vsom)


def _tc_scoring_pipelines_slabs(vsom):
    """More than two 1M-row slabs: the search of slab i+1 overlaps the re-scoring of slab i on a second stream and the
    candidate scratch is reused by parity — results must still equal the exact scan row for row (some duplicated nodes so
    that every slab also has rows for the exact-scan fallback)."""
    rng = np.random.default_rng(11)
    W, H, D, n = 16, 16, 32, (1 << 21) + 300_001
    m = rng.standard_normal((W * H, D)).astype(np.float32)
    m[216:] = m[0]  # 41 copies of node 0: more exact ties than the candidate list holds
    x = rng.standard_normal((n, D)).astype(np.float32)
    hot = rng.integers(0, n, 3000)
    x[hot] = m[0] + 0.001 * rng.standard_normal((3000, D)).astype(np.float32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD)
    ctx.upload_state(mean=m)
    eb, ed = ctx.find_bmu_exact(x)
    tb, td, fb = ctx.find_bmu_batch(x)
    assert_bit_equal(tb, eb, "bmu")
    assert_bit_equal(td, ed, "dist")
    assert fb > 0
    # host-buffer path: the rows cross PCIe in slabs behind the search of the previous slab (several slabs here)
    hb, hd = ctx.find_bmu(x)
    assert_bit_equal(hb, eb, "pipelined host bmu")
    assert_bit_equal(hd, ed, "pipelined host dist")
    ctx.close()


def test_tensor_core_scoring_adversarial_bf16_rounding(vsom):
    """Worst case for the bf16 operands: every component of every row and node sits next to a bf16 rounding midpoint
    (1 + 2^-8 -+ 2^-20, scaled), so x^ . m^ is off by almost the full 2 (2u + u^2) |x| |m| bound, in both directions, on maps
    with few dimensions where nothing averages out; many nodes are exact or near ties in the true distance.  Whatever the
    tensor cores select, the certificate must send every row it cannot prove to the exact scan: results equal K3's."""
    rng = np.random.default_rng(2024)
    for D, W, H in ((2, 32, 32), (3, 40, 30), (8, 64, 32), (16, 48, 48)):
        N, n = W * H, 4096
        def midpoints(shape):
            sign = rng.choice(np.float32([-1.0, 1.0]), shape)
            eps = rng.choice(np.float32([-2.0 ** -20, 2.0 ** -20]), shape)
            scale = np.float32(2.0) ** rng.integers(-1, 2, shape).astype(np.float32)
            return (sign * scale * (np.float32(1.0) + np.float32(2.0 ** -8) + eps)).astype(np.float32)
        m = midpoints((N, D))
        m[N // 2:] = m[: N - N // 2] * np.float32(1.0)  # duplicated nodes: exact ties, the lowest index must win
        m[N // 2:, 0] += rng.choice(np.float32([0.0, 2.0 ** -18]), N - N // 2)
        x = midpoints((n, D))
        ctx = vsom.VsomContext(W, H, D, vsom.STANDARD)
        ctx.upload_state(mean=m)
        eb, ed = ctx.find_bmu_exact(x)
        tb, td, fb = ctx.find_bmu_batch(x)
        assert ctx.last_score_tc
        print(f"adversarial D={D}: {fb} of {n} rows took the exact scan")
        assert_bit_equal(tb, eb, f"bmu D={D}")
        assert_bit_equal(td, ed, f"dist D={D}")
        ctx.close()


@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
@pytest.mark.parametrize("shape", [(64, 64, 128, 1, 3000, 1536), (128, 128, 256, 0, 1500, 1100), (40, 30, 77, 0, 800, 1300)])
def test_scoring_on_a_trained_map_matches_the_oracle(vsom, po, shape, order):
    """K2 and K3 against the ORACLE (not against each other) on a map the online step has clustered: neighbouring nodes
    are close to each other there, so near-candidates crowd the lists.  Includes 128x128x256 (BASELINE configs[3])."""
    W, H, D, tr, ntrain, n = shape
    rng = np.random.default_rng(W + D)
    centres = (rng.standard_normal((16, D)) * 2).astype(np.float32)
    data = lambda k: (centres[rng.integers(0, 16, k)] + 0.3 * rng.standard_normal((k, D))).astype(np.float32)
    ctx = vsom.VsomContext(W, H, D, tr, order)
    ctx.upload_state(mean=(rng.integers(-1000, 1000, (W * H, D)) / 1000).astype(np.float32))
    ctx.train_chunk(data(ntrain), 0.2, W / 6.0, vsom.EXPONENTIAL)
    ctx.train_chunk(data(ntrain), 0.1, W / 16.0, vsom.EXPONENTIAL)
    st = ctx.download_state()
    o = po.Oracle(W, H, D, tr, order)
    o.set_state(**st)
    q = data(n)
    ob, od = o.find_bmu(q)
    tb, td, fb = ctx.find_bmu_batch(q)
    assert ctx.last_score_tc
    print(f"trained {W}x{H}x{D}: {fb} of {n} rows took the exact scan; {len(np.unique(ob))} distinct BMUs")
    assert_bit_equal(tb, ob, "K2 bmu vs oracle")
    assert_bit_equal(td, od, "K2 dist vs oracle")
    eb, ed = ctx.find_bmu_exact(q[:512])
    assert_bit_equal(eb, ob[:512], "K3 bmu vs oracle")
    assert_bit_equal(ed, od[:512], "K3 dist vs oracle")
    assert ctx.evaluate(q) == o.evaluate(q)
    rb, _, _ = ctx.find_bmu_batch(q, min_hits=3)
    assert_bit_equal(rb, o.find_restricted_bmu(q, 3), "restricted K2 bmu vs oracle")
    ctx.close()


# ------------------------------------------------------------------------------------------------ K6 (batch-map trainer)
@pytest.mark.parametrize("shape", [(6, 6, 11, 0, 90), (7, 4, 11, 1, 90), (4, 9, 5, 2, 70), (20, 20, 784, 0, 60), (33, 17, 100, 1, 300),
                                   (12, 12, 32, 2, 150), (64, 64, 128, 0, 1500)])
@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
def test_batch_map_epochs_match_oracle_bit_exact(vsom, po, shape, order):
    """Som::trainBatchSom's loop over chunk-epochs (global BMU on the first epoch, local walks from node 0 afterwards,
    every neuron re-estimated from all rows) — bit-exact planes, hits, MSE and lastBMU against the oracle."""
    W, H, Din, tr, n = shape
    rng = np.random.default_rng(W * H + Din)
    o = po.Oracle(W, H, Din, tr, order)
    o.random_initialize(3, 1.0)
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    upload_like(ctx, o.get_state())
    x = synth(rng, n, Din, tr)
    chunk = n // 2 + 3
    for epoch, sigma in enumerate((3.0, 2.0, 1.2, 1.0)):
        for lo in range(0, n, chunk):
            seg = x[lo:lo + chunk]
            om, ol = o.batch_epoch(seg, sigma, epoch == 0)   # lastBMU zeroed per chunk load, like DataSet
            gm, gl = ctx.batch_epoch(seg, sigma, epoch == 0)
            # the MSE sums over every row's BMU residual: once a NaN neuron exists (sigma == 1, below) it is NaN on both sides
            assert (np.isnan(gm) and np.isnan(om)) or np.float32(gm).view(np.uint32) == np.float32(om).view(np.uint32), f"mse epoch {epoch}"
            assert np.array_equal(gl, ol), f"lastBMU epoch {epoch}"
            # at sigma == 1.0 the neighbourhood is a delta: a neuron that is nobody's BMU divides 0 by 0 and becomes NaN in
            # the reference too; NaN payload / sign bits are not part of the contract (x86 gives 0xFFC00000, the GPU
            # 0x7FFFFFFF), every other value must match bit for bit
            got, want = ctx.download_state(), o.get_state()
            for k in ("mean", "S", "sigma", "weight"):
                g, w = got[k].copy(), want[k].copy()
                assert np.array_equal(np.isnan(g), np.isnan(w)), f"{k}: NaN pattern differs (epoch {epoch})"
                g[np.isnan(g)] = 0
                w[np.isnan(w)] = 0
                assert_bit_equal(g, w, f"epoch {epoch} sigma {sigma}: {k}")
            assert_bit_equal(got["hits"], want["hits"], "hits")
    ctx.close()


# ------------------------------------------------------------------------------------------------ K3 / K4 corner cases
@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
@pytest.mark.parametrize("tr,Din", [(0, 1), (0, 3), (0, 4), (0, 7), (0, 8), (0, 13), (0, 37), (0, 64), (2, 2), (2, 4), (2, 5), (2, 9)])
def test_exact_scan_every_residue_of_the_vector_length(vsom, po, tr, Din, order):
    """K3 (both orders) on vector lengths that hit every branch of the reductions: fewer than 4 terms, 4..7, multiples of
    8, an extra packet, a scalar tail; CLR pair counts likewise.  Ragged row / node counts (partial tiles)."""
    rng = np.random.default_rng(Din * 7 + tr)
    W, H, n = 11, 7, 131
    o = po.Oracle(W, H, Din, tr, order)
    o.random_initialize(5, 1.0)
    st = o.get_state()
    st["hits"] = rng.integers(0, 3, W * H).astype(np.uint64)
    o.set_state(**st)
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    upload_like(ctx, st)
    x = synth(rng, n, Din, tr)
    ob, od = o.find_bmu(x)
    gb, gd = ctx.find_bmu_exact(x)
    assert_bit_equal(gb, ob, "bmu")
    assert_bit_equal(gd, od, "dist")
    assert_bit_equal(ctx.find_bmu_exact(x, min_hits=2)[0], o.find_restricted_bmu(x, 2), "restricted")
    assert_bit_equal(ctx.all_dists(x[0]), o.all_dists(x[0]), "all dists")
    ctx.close()


@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
@pytest.mark.parametrize("Dm", [1, 5, 7, 8, 9, 12, 31, 32, 33, 63, 64, 65, 72, 100, 127, 129])
def test_umatrix_division_corner_cases(vsom, po, Dm, order):
    """K4 replaces the reference's IEEE division by a shared reciprocal + one correction step; every term must still be
    the reference's bits.  Sigmas: zero (clamped to 1e-5), tiny, ordinary, huge, 2^100 and beyond, infinite; differences:
    exact zeros, denormals, tiny, ordinary, huge (the quotient or its square overflows), infinite.
    Model lengths around the kernels' slices (32 elements in the sequential kernel, 64 in the Eigen one), the block of
    eight and the padded rows (Dm % 4 != 0); at Dm = 65 the Eigen kernel's last slice holds only the rest block."""
    rng = np.random.default_rng(Dm)
    W, H = 19, 6
    N = W * H
    mags = np.float32([0.0, 1e-42, 1e-38, 3e-33, 1e-30, 1e-20, 1e-6, 1.0, 3.7, 1e6, 1e20, 1.3e30])
    mean = (rng.choice(mags, (N, Dm)) * rng.choice(np.float32([-1, 1]), (N, Dm)) + rng.standard_normal((N, Dm)).astype(np.float32) *
            rng.choice(np.float32([0, 0, 1e-3, 1]), (N, Dm))).astype(np.float32)
    mean[::5] = mean[1::5][: len(mean[::5])]  # exact zeros in many differences
    sig_mags = np.float32([0.0, 1e-7, 1e-5, 1.0000001e-5, 1e-3, 0.5, 1.0, 3.0, 1e10, 1.2e30, 1.3e30, 1e38])
    sigma = rng.choice(sig_mags, (N, Dm)).astype(np.float32)
    # a few cells that turn whole nodes into NaN / inf (inf - inf, inf / inf): present, but not everywhere
    for cell in rng.integers(0, N * Dm, 6):
        mean.flat[cell] = rng.choice(np.float32([1e35, np.inf, -np.inf]))
        sigma.flat[(cell * 7) % (N * Dm)] = np.inf
    o = po.Oracle(W, H, Dm, 0, order)
    o.set_state(mean=mean, sigma=sigma)
    ctx = vsom.VsomContext(W, H, Dm, 0, order)
    ctx.upload_state(mean=mean, sigma=sigma)
    with np.errstate(all="ignore"):
        want = o.update_umatrix()
    got = ctx.update_umatrix()
    assert np.array_equal(np.isnan(got), np.isnan(want)), "NaN pattern"
    ok = ~np.isnan(want)
    assert_bit_equal(got[ok], want[ok], "umatrix")
    assert ok.sum() > 0
    # and an ordinary map next to it (no special values at all)
    mean2 = rng.standard_normal((N, Dm)).astype(np.float32)
    sigma2 = np.abs(rng.standard_normal((N, Dm))).astype(np.float32)
    o.set_state(mean=mean2, sigma=sigma2)
    ctx.upload_state(mean=mean2, sigma=sigma2)
    assert_bit_equal(ctx.update_umatrix(), o.update_umatrix(), "umatrix (ordinary values)")
    ctx.close()


# ------------------------------------------------------------------------------------------------ soft assignment (f3)
@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
@pytest.mark.parametrize("tr,Din", [(0, 12), (1, 33), (2, 6)])
def test_soft_assign_matches_find_restricted_bmd(vsom, po, tr, Din, order):
    """vsom_soft_assign = Som::findRestrictedBmd (src/Som.cpp:457-487) per row: exp(-d^2 / 2) of the (already squared) distance for
    nodes with enough hits, normalised.  Distances are the reference's bits; exp() is the device's f64 exp, so the tolerance is
    1e-13 relative (stated in include/vsom_b200.h); the zero pattern (nodes below min_hits) must be identical."""
    rng = np.random.default_rng(Din)
    W, H = 9, 7
    o = po.Oracle(W, H, Din, tr, order)
    o.random_initialize(3, 0.2)
    st = o.get_state()
    st["hits"] = rng.integers(0, 4, W * H).astype(np.uint64)
    o.set_state(**st)
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    upload_like(ctx, st)
    x = (0.2 * synth(rng, 7, Din, tr)).astype(np.float32)  # close to the map: probabilities that do not underflow
    for min_hits in (0, 2):
        got = ctx.soft_assign(x, min_hits)
        for r in range(len(x)):
            want = o.find_restricted_bmd(x[r], min_hits)
            assert np.array_equal(got[r] == 0, want == 0), "zero pattern"
            np.testing.assert_allclose(got[r], want, rtol=1e-13, atol=0)
            assert abs(got[r].sum() - 1.0) < 1e-12
    ctx.close()
