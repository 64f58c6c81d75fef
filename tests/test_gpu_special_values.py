"""Special values against the CPU oracle: NaN, +-inf, overflowing distances, fp32 subnormals and magnitudes far from 1, in
the maps and in the rows, through scoring (K2 / K3, host and device forms), measure_similarity, soft_assign, online training
(K1F and the generic kernel) and the batch-map trainer (K6).

Contract (DESIGN.md section 2): NaN positions identical, every non-NaN value bit-identical, BMU ids exact.  NaN payload and
sign are not part of it (x86 gives 0xFFC00000, the GPU 0x7FFFFFFF).  The reference seeds findBmu / findRestrictedBmu /
findLocalBmu with the distance of the first node it measures and updates on a strict '<' in double, so a NaN distance never
wins unless it sits at that seed node — node 0 for the global searches."""
import functools
import zlib

import numpy as np
import pytest

from conftest import assert_bit_equal

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

F32 = np.float32


def assert_same(got, want, what):
    """NaN pattern identical, every other value bit for bit (sign of zero and of infinity included)."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    assert got.dtype == want.dtype, f"{what}: dtype {got.dtype} vs {want.dtype}"
    if got.dtype.kind == "f":
        gn, wn = np.isnan(got), np.isnan(want)
        if not np.array_equal(gn, wn):
            i = tuple(np.argwhere(gn != wn)[0])
            raise AssertionError(f"{what}: NaN pattern differs ({int((gn != wn).sum())} entries); first at {i}: {got[i]!r} vs {want[i]!r}")
        got, want = np.where(gn, 0, got).astype(got.dtype), np.where(wn, 0, want).astype(want.dtype)
    assert_bit_equal(got, want, what)


def assert_same_scalar(got, want, what):
    assert_same(np.float64([got]), np.float64([want]), what)


# ------------------------------------------------------------------------------------------------ scoring
MAP_CASES = ["nan_node0", "nan_nodes", "inf_node0", "inf_middle", "outlier", "tiny", "huge", "min_hits_above_all"]
HUGE = F32(2.0 ** 85)   # map magnitude where s_m^2 underflows in f32 (s_m = 2^-76)
HUGE_STEP = F32(2.0 ** 62)  # one ulp above 2^85: node / row differences that keep |m - x|^2 below FLT_MAX
TINY = F32(2.0 ** -60)  # map magnitude where s_m^2 overflows in f32


def _huge_vectors(rng, n, D):
    """2^85 everywhere, plus 2^62 in three random components: at most six differing components, so every squared
    distance is at most 6 * 2^124 < FLT_MAX."""
    v = np.full((n, D), HUGE, F32)
    for i in range(n):
        v[i, rng.choice(D, 3, replace=False)] += HUGE_STEP
    return v


def special_map(case, rng, N, D):
    """(mean, hits, min_hits, row scale) of one map case.  The base map is clustered like a trained one."""
    centres = (rng.standard_normal((12, D)) * 2).astype(F32)
    m = (centres[rng.integers(0, 12, N)] + 0.3 * rng.standard_normal((N, D))).astype(F32)
    hits = rng.integers(0, 4, N).astype(np.uint64)
    min_hits, scale = 2, None
    if case == "nan_node0":
        m[0, D // 2] = np.nan
    elif case == "nan_nodes":
        for p in (1, 5, N // 2, N - 1):
            m[p, (p * 7) % D] = np.nan
    elif case == "inf_node0":
        m[0, 1] = np.inf
        m[0, D - 1] = -np.inf
    elif case == "inf_middle":
        m[N // 2, 0] = -np.inf
    elif case == "outlier":
        m[N // 3, 0] = F32(1e20)
        m[(2 * N) // 3] = F32(1e30)
    elif case == "tiny":  # max |m| < 2^-54, and every seventh node in fp32 subnormals
        m = (m * TINY).astype(F32)
        m[::7] = (m[::7] * F32(2.0 ** -80)).astype(F32)
        scale = TINY
    elif case == "huge":
        m = _huge_vectors(rng, N, D)
        scale = HUGE
    elif case == "min_hits_above_all":  # the reference answers node 0 for every row: it seeds with node 0 whatever its hits
        min_hits = 10
    return m, hits, min_hits, centres, scale


def special_rows(rng, x, m):
    """Special rows mixed through an ordinary batch, in the first probe, the second one and the remainder where the batch is
    long enough.  Returns the row ids of each kind."""
    n, D = x.shape
    kinds = {
        "nan": lambda r: r.__setitem__(D // 3, np.nan),
        "+inf": lambda r: r.__setitem__(1, np.inf),
        "-inf": lambda r: r.__setitem__(D - 1, -np.inf),
        "overflow": lambda r: r.__setitem__(0, F32(1e20)),   # every distance overflows: BMU 0, distance inf
        "ties": lambda r: r.__setitem__(D // 2, F32(1e15)),  # finite distances, massive exact ties
        "zero": lambda r: r.__setitem__(slice(None), 0.0),
        "subnormal": lambda r: r.__setitem__(slice(None), (rng.standard_normal(D) * 1e-40).astype(F32)),
        "node0": lambda r: r.__setitem__(slice(None), m[0]),  # distance +0 (or NaN where node 0 has one)
        "nodeN/2": lambda r: r.__setitem__(slice(None), m[len(m) // 2]),
    }
    where = {}
    for j, (name, put) in enumerate(kinds.items()):
        ids = [i for i in (3 + 11 * j, 700 + j, 8192 + 5 + j, 2 * 8192 + 17 + j, n - 1 - j) if i < n]
        for i in ids:
            put(x[i])
        where[name] = ids
    return where


SCORE_SHAPES = [(24, 20, 48, 0, 2 * 8192 + 333), (64, 64, 128, 1, 1100), (20, 20, 784, 0, 1100)]  # (W, H, D, transform, rows); 784: A streamed with B


@functools.lru_cache(maxsize=None)
def _scoring_case(po, shape, order, case):
    """Map, rows and the oracle's answers of one case (shared by the three tiers)."""
    W, H, D, tr, n = shape
    N = W * H
    rng = np.random.default_rng(zlib.crc32(repr((shape, case)).encode()))
    m, hits, min_hits, centres, scale = special_map(case, rng, N, D)
    if case == "huge":
        x = _huge_vectors(rng, n, D)
    else:
        x = (centres[rng.integers(0, 12, n)] + 0.4 * rng.standard_normal((n, D))).astype(F32)
        if scale is not None:
            x = (x * scale).astype(F32)
    where = special_rows(rng, x, m)
    o = po.Oracle(W, H, D, tr, order)
    o.set_state(mean=m, hits=hits)
    with np.errstate(all="ignore"):
        ob, od = o.find_bmu(x)
        orb = o.find_restricted_bmu(x, min_hits)
        clean = ~np.isin(np.arange(n), [i for k in ("nan", "+inf", "-inf", "overflow") for i in where[k]])
        oe = (o.evaluate(x), o.evaluate(x[clean]))
        probe = sorted({i for ids in where.values() for i in ids})
        alld = {i: o.all_dists(x[i]) for i in probe[:12]}
    return m, hits, min_hits, x, clean, ob, od, orb, oe, alld


@pytest.mark.parametrize("tier", ["1", "2", "auto"])
@pytest.mark.parametrize("case", MAP_CASES)
@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
@pytest.mark.parametrize("shape", SCORE_SHAPES, ids=lambda s: "x".join(map(str, s[:3])))
def test_scoring_special_values_match_oracle(vsom, po, monkeypatch, shape, order, case, tier):
    """vsom_find_bmu_batch / vsom_find_bmu / the device form (K2 for >= 1024 rows), vsom_find_bmu_exact (K3, also below 1024
    rows), the restricted search, vsom_evaluate (NaN / inf propagate through the running mean) and all_dists, against the
    oracle on maps and rows with special values."""
    import torch

    if tier == "auto":
        monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    else:
        monkeypatch.setenv("VSOM_TC_TIER", tier)
    if shape[4] > 2 * 8192:
        monkeypatch.setenv("VSOM_TC_HOST_SLAB_LOG2", "12")  # several slabs of the host-buffer pipeline
    W, H, D, tr, n = shape
    m, hits, min_hits, x, clean, ob, od, orb, oe, alld = _scoring_case(po, shape, order, case)
    nan_rows = int(np.isnan(x).any(axis=1).sum())
    ctx = vsom.VsomContext(W, H, D, tr, order)
    ctx.upload_state(mean=m, hits=hits)

    s0 = ctx.tc_stats()
    tb, td, fb = ctx.find_bmu_batch(x)
    s1 = ctx.tc_stats()
    print(f"{case} {W}x{H}x{D} tier {tier}: ran tier {ctx.last_score_tc}, {fb} of {n} rows took the exact scan, "
          f"stats delta {({k: s1[k] - s0[k] for k in s1})}")
    assert_same(tb, ob, "find_bmu_batch bmu")
    assert_same(td, od, "find_bmu_batch dist")
    assert fb >= nan_rows  # a row with a NaN element has no finite approximate score: it always takes the exact scan

    db, dd = ctx.find_bmu(x)
    assert n < 1024 or ctx.last_score_tc or fb == n  # the dispatch reached K2 (or K2 declined the whole call)
    assert_same(db, ob, "find_bmu bmu")
    assert_same(dd, od, "find_bmu dist")

    xd = torch.from_numpy(x).cuda()
    gb = torch.empty(n, dtype=torch.int32, device="cuda")
    gd = torch.empty(n, dtype=torch.float32, device="cuda")
    ctx.find_bmu_batch_device(xd, n, gb, gd)
    ctx.synchronize()
    assert_same(gb.cpu().numpy().astype(np.uint32), ob, "device bmu")
    assert_same(gd.cpu().numpy(), od, "device dist")

    eb, ed = ctx.find_bmu_exact(x)
    assert not ctx.last_score_tc
    assert_same(eb, ob, "exact bmu")
    assert_same(ed, od, "exact dist")
    eb, ed = ctx.find_bmu_exact(x[:300])
    assert_same(eb, ob[:300], "exact bmu, 300 rows")
    assert_same(ed, od[:300], "exact dist, 300 rows")

    rb, _ = ctx.find_bmu(x, min_hits=min_hits)
    assert_same(rb, orb, f"find_bmu(min_hits={min_hits})")
    rb, _, _ = ctx.find_bmu_batch(x, min_hits=min_hits)
    assert_same(rb, orb, f"find_bmu_batch(min_hits={min_hits})")

    assert_same_scalar(ctx.evaluate(x), oe[0], "evaluate")
    assert_same_scalar(ctx.evaluate(x[clean]), oe[1], "evaluate without NaN / inf / overflowing rows")
    for i, want in alld.items():
        assert_same(ctx.all_dists(x[i]), want, f"all_dists of row {i}")
    ctx.close()


# ------------------------------------------------------------------------------------------------ measure_similarity / soft_assign
def _nan_neuron_map(rng, W, H, D):
    centres = (rng.standard_normal((10, D)) * 2).astype(F32)
    m = (centres[rng.integers(0, 10, W * H)] + 0.3 * rng.standard_normal((W * H, D))).astype(F32)
    sigma = np.abs(rng.standard_normal((W * H, D))).astype(F32)
    for p in (3, 17, W * H // 2):  # NaN neurons (what a batch-map epoch at sigma = 1 leaves), node 0 finite
        m[p] = np.nan
        sigma[p] = np.nan
    hits = rng.integers(0, 4, W * H).astype(np.uint64)
    return centres, m, sigma, hits


@pytest.mark.parametrize("n", [300, 3 * 8192 + 777])
def test_measure_similarity_special_values(vsom, po, monkeypatch, n):
    """The per-row pass of Som::measureSimilarity on a map with NaN neurons and NaN / inf rows (exact path and the K2 pipeline
    with many slabs), against the oracle's restricted BMUs and the same three f32 operations in numpy."""
    monkeypatch.setenv("VSOM_TC_HOST_SLAB_LOG2", "12")
    rng = np.random.default_rng(n)
    W, H, D = 24, 20, 48
    centres, m, sigma, hits = _nan_neuron_map(rng, W, H, D)
    x = (centres[rng.integers(0, 10, n)] + 0.4 * rng.standard_normal((n, D))).astype(F32)
    for i in range(5, n, 997):
        x[i, i % D] = (np.nan, np.inf, -np.inf, F32(1e20))[(i // 997) % 4]
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=m, sigma=sigma, hits=hits)
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.set_state(mean=m, sigma=sigma, hits=hits)
    min_hits = 1
    ob = o.find_restricted_bmu(x, min_hits)
    bmu, row_max = ctx.measure_similarity(x, 3, min_hits)
    assert_same(bmu, ob, "bmu")
    s = sigma[ob]
    sM = np.where(s > F32(0.00001), F32(0.00001), s).astype(F32)
    with np.errstate(all="ignore"):
        delta = (((x - m[ob]).astype(F32) / sM).astype(F32) / F32(3)).astype(F32)
    want = np.where(np.isnan(delta), -np.inf, delta).max(axis=1).astype(F32)
    assert_same(row_max, want, "row maxima")
    ctx.close()


@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
def test_soft_assign_special_values(vsom, po, order):
    """vsom_soft_assign on a map with NaN neurons, for ordinary, NaN and inf rows: zero and NaN patterns identical to
    Som::findRestrictedBmd, values within the 1e-13 relative tolerance of include/vsom_b200.h."""
    rng = np.random.default_rng(31 + order)
    W, H, D = 9, 7, 12
    centres, m, sigma, hits = _nan_neuron_map(rng, W, H, D)
    m = (0.2 * m).astype(F32)
    o = po.Oracle(W, H, D, po.STANDARD, order)
    o.set_state(mean=m, sigma=sigma, hits=hits)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, order)
    ctx.upload_state(mean=m, sigma=sigma, hits=hits)
    x = (0.2 * centres[rng.integers(0, 10, 6)] + 0.05 * rng.standard_normal((6, D))).astype(F32)
    x[1, 2], x[2, 0], x[3, 5], x[4] = np.nan, np.inf, F32(1e20), m[0]
    for min_hits in (0, 2):
        got = ctx.soft_assign(x, min_hits)
        for r in range(len(x)):
            with np.errstate(all="ignore"):
                want = o.find_restricted_bmd(x[r], min_hits)
            assert np.array_equal(np.isnan(got[r]), np.isnan(want)), f"row {r}: NaN pattern"
            assert np.array_equal(got[r] == 0, want == 0), f"row {r}: zero pattern"
            ok = ~np.isnan(want)
            np.testing.assert_allclose(got[r][ok], want[ok], rtol=1e-13, atol=0)
    ctx.close()


# ------------------------------------------------------------------------------------------------ online training
# one shape whose planes K1F keeps in shared memory, one whose planes stay in HBM (generic kernel), and CLR
ONLINE_SHAPES = [(40, 40, 64, 0), (40, 40, 64, 1), (100, 100, 784, 0), (100, 100, 784, 1), (50, 50, 32, 2)]
ONLINE_CASES = ["nan_row", "nan_node0", "nan_in_window", "inf_row", "overflow_row", "local_walk_nan_neighbours"]


def _online_rows(rng, n, Din, tr):
    if tr == 2:
        z = rng.standard_normal((n, 1)).astype(F32)
        a = rng.uniform(0.5, 1.5, (1, Din)).astype(F32)
        return (a * z + 0.1 * rng.standard_normal((n, Din))).astype(F32)
    return rng.standard_normal((n, Din)).astype(F32)


@pytest.fixture(params=["fast", "generic"])
def online_kernel(request, monkeypatch):
    if request.param == "generic":
        monkeypatch.setenv("VSOM_ONLINE_KERNEL", "generic")
    else:
        monkeypatch.delenv("VSOM_ONLINE_KERNEL", raising=False)
    return request.param


@pytest.mark.parametrize("case", ONLINE_CASES)
@pytest.mark.parametrize("shape", ONLINE_SHAPES, ids=lambda s: "x".join(map(str, s[:3])) + f"-tr{s[3]}")
def test_online_training_special_values_match_oracle(vsom, po, shape, case, online_kernel):
    """The online step (src/Som.cpp:885-950) on NaN / inf / overflowing rows and maps with NaN nodes: the whole trajectory
    (BMU, dist, resid2, lastBMU, the five planes, hits) against the oracle, NaN-aware.  After a NaN row the BMU's window
    is NaN, node 0 among it, and every later row must pin to node 0."""
    W, H, Din, tr = shape
    if online_kernel == "generic" and Din == 784:
        pytest.skip("the generic kernel is what runs this shape in the fast variant too")
    N = W * H
    rng = np.random.default_rng(zlib.crc32(repr((shape, case)).encode()))
    o = po.Oracle(W, H, Din, tr, po.ORDER_SEQUENTIAL)
    o.random_initialize(42, 1.0)
    st = o.get_state()
    n, eta, sigma = 24, 0.1, 4.0
    x = _online_rows(rng, 2 * n, Din, tr)
    mean = st["mean"]
    segs = [(x[:n], sigma, None), (x[n:], 0.6 * sigma, None)]
    if case == "nan_row":
        x[n // 2, Din // 2] = np.nan
    elif case == "nan_node0":
        mean[0, 1] = np.nan
    elif case == "nan_in_window":  # a NaN node next to where the rows land: updated every step, never the winner
        c = (H // 2) * W + W // 2
        mean[c, 0] = np.nan
        if tr != 2:
            x[:] = (mean[c + rng.choice([1, -1, W, -W], 2 * n)] + 0.01 * rng.standard_normal((2 * n, Din))).astype(F32)
            x[:, 0] = rng.standard_normal(2 * n).astype(F32)
    elif case == "inf_row":
        x[n // 3, 2] = np.inf
    elif case == "overflow_row":
        x[n // 3, 0] = F32(1e20)
    elif case == "local_walk_nan_neighbours":  # findLocalBmu (sigma <= 1) around NaN nodes, some walks starting on one
        bad = np.arange(7, N, 13)
        mean[bad, 0] = np.nan
        starts = rng.integers(0, N, n).astype(np.uint64)
        starts[::3] = bad[rng.integers(0, len(bad), len(starts[::3]))]
        segs = [(x[:n], 1.0, None), (x[n:], 0.75, starts)]
    st["mean"] = mean
    o.set_state(**st)
    ctx = vsom.VsomContext(W, H, Din, tr, vsom.ORDER_REFERENCE)
    ctx.upload_state(st["mean"], st["S"], st["sigma"], st["weight"], st["hits"])
    first = None
    for si, (seg, sg, last) in enumerate(segs):
        with np.errstate(all="ignore"):
            ob, od, orr, ol = o.train_rows(seg, eta, sg, 0, last_bmu=None if last is None else last.copy())
        gb, gd, gr, gl = ctx.train_chunk(seg, eta, sg, 0, last_bmu=None if last is None else last.copy())
        what = f"{case} chunk {si} (sigma {sg})"
        assert_same(gb, ob, f"{what}: bmu")
        assert_same(gd, od, f"{what}: dist")
        assert_same(gr, orr, f"{what}: resid2")
        assert_same(gl, ol, f"{what}: lastBMU")
        got, want = ctx.download_state(), o.get_state()
        for k in ("mean", "S", "sigma", "weight", "hits"):
            assert_same(got[k], want[k], f"{what}: {k}")
        first = first if first is not None else ob
    if case == "nan_row":  # the case is what it claims to be: the rows after the NaN row pin to node 0
        assert (first[n // 2:] == 0).all() and np.isnan(o.get_state()["mean"][0]).any()
    ctx.close()


# ------------------------------------------------------------------------------------------------ batch-map trainer
@pytest.mark.parametrize("schedule", ["wide_to_delta", "node0_far"])
@pytest.mark.parametrize("order", [0, 2], ids=["seq", "eigen_sse"])
@pytest.mark.parametrize("shape", [(24, 20, 48, 0, 1300), (12, 12, 32, 1, 1100)], ids=lambda s: "x".join(map(str, s[:3])))
def test_batch_map_into_nan_neurons_then_score(vsom, po, shape, order, schedule):
    """Som::trainBatchSom down to sigma = 1 leaves every neuron that is nobody's BMU NaN (0 / 0, in the reference too).  Then:
    one more local-walk epoch, one global epoch over >= 1024 rows (its BMU search goes through K2), and scoring / evaluate
    of the map that results.  'node0_far' starts node 0 far from all data, so that it is NaN when the K2 epoch runs: every
    row's BMU is node 0 there."""
    W, H, Din, tr, n = shape
    rng = np.random.default_rng(W * H + Din + order)
    o = po.Oracle(W, H, Din, tr, order)
    o.random_initialize(3, 1.0)
    st = o.get_state()
    x = _online_rows(rng, n, Din, tr)
    chunks = [x[:n // 2 + 3], x[n // 2 + 3:]]
    if schedule == "node0_far":  # node 0 is nobody's BMU in the first chunk: NaN when the global epoch over all rows runs on K2
        st["mean"][0] = F32(50.0)
        epochs = [(1.0, True, chunks[:1]), (1.0, True, [x]), (1.0, False, chunks)]
    else:
        epochs = [(sg, e == 0, chunks) for e, sg in enumerate((3.0, 2.0, 1.2, 1.0))] + [(1.0, False, chunks), (1.0, True, [x])]
    o.set_state(**st)
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    ctx.upload_state(st["mean"], st["S"], st["sigma"], st["weight"], st["hits"])
    for e, (sg, first, segs) in enumerate(epochs):
        if schedule == "node0_far" and len(segs[0]) == n:
            assert np.isnan(o.get_state()["mean"][0]).any()
        for seg in segs:
            with np.errstate(all="ignore"):
                om, ol = o.batch_epoch(seg, sg, first)
            gm, gl = ctx.batch_epoch(seg, sg, first)
            what = f"{schedule} epoch {e} (sigma {sg}, first={first}, {len(seg)} rows)"
            assert_same(F32(gm), F32(om), f"{what}: mse")
            assert_same(gl, ol, f"{what}: lastBMU")
            got, want = ctx.download_state(), o.get_state()
            for k in ("mean", "S", "sigma", "weight", "hits"):
                assert_same(got[k], want[k], f"{what}: {k}")
    mean = o.get_state()["mean"]
    print(f"{schedule}: {int(np.isnan(mean).any(axis=1).sum())} of {W * H} neurons NaN, node 0 NaN: {bool(np.isnan(mean[0]).any())}")
    q = _online_rows(rng, 1500, Din, tr)
    with np.errstate(all="ignore"):
        ob, od = o.find_bmu(q)
        oe = o.evaluate(q)
    tb, td, fb = ctx.find_bmu_batch(q)
    print(f"scoring: tier {ctx.last_score_tc}, {fb} of {len(q)} rows took the exact scan")
    assert_same(tb, ob, "bmu")
    assert_same(td, od, "dist")
    db, dd = ctx.find_bmu(q)
    assert_same(db, ob, "find_bmu bmu")
    assert_same(dd, od, "find_bmu dist")
    assert_same_scalar(ctx.evaluate(q), oe, "evaluate")
    ctx.close()
