"""Best and second-best matching node (vsom_find_bmu2 / _device / _exact) and the topographic error built on them.

Every case checks, bit for bit:
- bmu / dist of every row against vsom_find_bmu_exact (the single-BMU exact scan);
- bmu2 / dist2 of every row against vsom_find_bmu2_exact (the top-2 exact scan, K3);
- all four against the rule applied to the oracle's own distances (pyoracle Oracle.all_dists, whose f64 values are the f32
  bits) on a subset of rows: the first and last rows, the rows around the 8192-row probe boundaries, and the 256 rows whose
  relative gap (dist2 - dist) / dist2 is smallest, where K2's certificate is tightest.
The rule: eligible nodes are node 0 and the nodes with hits >= min_hits; bmu is findBmu's (a NaN distance at node 0 wins);
bmu2 is the eligible node other than bmu with the smallest (distance, index), NaN distances after every number; without one,
bmu2 = 0xFFFFFFFF and dist2 is NaN.

K2 (the tensor-core search, >= 1024 rows) runs in tiers 1, 2 and the probed choice, host and device forms, both summation orders,
on bench's trained 128 x 128 x 256 scoring map at 2^20 rows and at row counts either side of 1024 / 8192 / 16384, and on the
coincident map that sends the rest of a call to the exact scan (tier 3).  K3 (< 1024 rows, CLR) covers Standard, Median and
CLR.  Edge cases: duplicated nodes, min_hits with one eligible node and with 64-bit hit counts, 1 x 1 / 1 x 37 / 37 x 1 grids,
NaN and infinite values in rows and maps, and slab boundaries of the host form.  Som::topographicError / mapDataSetTopTwo
(tests/cpp/topo_driver) are checked against the topographic error computed here from the oracle's distances."""
import os
import subprocess

import numpy as np
import pytest

from conftest import REPO, assert_bit_equal
from test_gpu_benchmark_shapes import PROBE, TC_MIN_ROWS, _row_count_map, init_map, synth_chunk

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

F32 = np.float32
NONE = np.uint32(0xFFFFFFFF)
TOPO_DRIVER = os.path.join(REPO, "tests", "cpp", "topo_driver")


# ------------------------------------------------------------------------------------------------ the rule on the oracle's distances
def rule_top2(d, eligible):
    """(bmu, dist, bmu2, dist2) of one row from its N distances (f32 values) and the eligibility mask."""
    idx = np.flatnonzero(eligible)
    dd = d[idx].astype(F32)
    nan = np.isnan(dd)
    rank = np.where(nan, 1, 0)
    rank[(idx == 0) & nan] = -1  # findBmu seeds with node 0: a NaN there is never beaten
    order = np.lexsort((idx, np.where(nan, F32(0), dd), rank))
    canon = lambda v: F32(np.nan) if np.isnan(v) else F32(v)
    b, bd = np.uint32(idx[order[0]]), canon(dd[order[0]])
    if len(order) < 2:
        return b, bd, NONE, F32(np.nan)
    return b, bd, np.uint32(idx[order[1]]), canon(dd[order[1]])


def oracle_top2(po, W, H, D, order, mean, x, rows, transform=None, hits=None, min_hits=0):
    o = po.Oracle(W, H, D, po.STANDARD if transform is None else transform, order)
    o.set_state(mean=mean)
    N = W * H
    eligible = np.ones(N, bool)
    if min_hits:
        eligible = np.asarray(hits, np.uint64) >= np.uint64(min_hits)
        eligible[0] = True
    out = [rule_top2(o.all_dists(x[r]), eligible) for r in rows]
    return tuple(np.array([t[i] for t in out], dtype=(np.uint32 if i % 2 == 0 else F32)) for i in range(4))


def assert_same(got, want, what):
    """bmu / bmu2 bit for bit; distances bit for bit where the reference is a number, NaN where it is NaN."""
    for name, g, w in zip(("bmu", "dist", "bmu2", "dist2"), got, want):
        g, w = np.asarray(g), np.asarray(w)
        if g.dtype == F32:
            gn, wn = np.isnan(g), np.isnan(w)
            assert np.array_equal(gn, wn), f"{what}: {name} NaN at {np.flatnonzero(gn != wn)[:8]}"
            assert_bit_equal(g[~gn], w[~wn], f"{what}: {name}")
        else:
            assert_bit_equal(g, w, f"{what}: {name}")


def oracle_rows(n, dist, dist2, tight=256):
    """First and last rows, rows around the probe boundaries, and the rows with the smallest relative gap."""
    rows = [np.arange(min(n, 16)), np.arange(max(0, n - 16), n)]
    for b in (PROBE, 2 * PROBE):
        rows.append(np.arange(b - 3, b + 3))
    with np.errstate(invalid="ignore", divide="ignore"):
        gap = (dist2.astype(np.float64) - dist) / dist2
    gap = np.where(np.isfinite(gap), gap, np.inf)
    rows.append(np.argsort(gap, kind="stable")[:tight])
    r = np.unique(np.concatenate(rows))
    return r[(r >= 0) & (r < n)]


def check_against_exact(ctx, x, min_hits, what):
    """Exact scans (K3, top-1 and top-2) of the rows; asserts they agree on (bmu, dist).  Returns the top-2 scan's results."""
    eb, ed = ctx.find_bmu_exact(x, min_hits=min_hits)
    e = ctx.find_bmu2_exact(x, min_hits=min_hits)
    assert ctx.last_score_tc == 0
    assert_bit_equal(e[0], eb, f"{what}: top-2 exact bmu vs find_bmu_exact")
    assert_bit_equal(e[1], ed, f"{what}: top-2 exact dist vs find_bmu_exact")
    return e


def run_forms(vsom, ctx, x, min_hits, exact, what):
    """Host and device forms of vsom_find_bmu2 against the exact top-2 scan on every row; returns their tiers and fallbacks."""
    import torch

    n = len(x)
    b, d, b2, d2, fb = ctx.find_bmu2(x, min_hits=min_hits)
    tier = ctx.last_score_tc
    assert_same((b, d, b2, d2), exact, f"{what}: host form")
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    outs = [torch.full((n,), -1, dtype=torch.int32, device="cuda") for _ in range(4)]
    fbd = ctx.find_bmu2_device(xd, n, outs[0], outs[1].view(torch.float32), outs[2], outs[3].view(torch.float32), min_hits=min_hits)
    ctx.synchronize()
    tierd = ctx.last_score_tc
    got = (outs[0].cpu().numpy().view(np.uint32), outs[1].cpu().numpy().view(F32), outs[2].cpu().numpy().view(np.uint32),
           outs[3].cpu().numpy().view(F32))
    assert_same(got, exact, f"{what}: device form")
    assert fb <= n and fbd <= n
    return tier, tierd, fb, fbd


def _tier(monkeypatch, tier):
    if tier == "auto":
        monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    else:
        monkeypatch.setenv("VSOM_TC_TIER", tier)


# ------------------------------------------------------------------------------------------------ bench's trained scoring map
BIG_N = 1 << 20
_big = {}


def trained_case(vsom):
    if "x" not in _big:
        W, H, D, mean, _ = _row_count_map(vsom, "trained")
        _big.update(W=W, H=H, D=D, mean=mean, x=synth_chunk(BIG_N, D, 1234 + 5))
    return _big


def trained_exact(vsom, order):
    key = ("exact", order)
    if key not in _big:
        c = trained_case(vsom)
        ctx = vsom.VsomContext(c["W"], c["H"], c["D"], vsom.STANDARD, order)
        ctx.upload_state(mean=c["mean"])
        _big[key] = check_against_exact(ctx, c["x"], 0, f"trained map, order {order}")
        ctx.close()
    return _big[key]


@pytest.mark.parametrize("tier", ["1", "2", "auto"])
@pytest.mark.parametrize("order", [0, 2])
def test_top2_trained_map_tiers(vsom, po, monkeypatch, order, tier):
    """2^20 rows of bench's scoring data on bench's trained map through K2's top-2 mode, host and device forms."""
    c = trained_case(vsom)
    W, H, D, mean, x = c["W"], c["H"], c["D"], c["mean"], c["x"]
    exact = trained_exact(vsom, order)
    _tier(monkeypatch, tier)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, order)
    ctx.upload_state(mean=mean)
    before = ctx.tc_stats()
    t, td, fb, fbd = run_forms(vsom, ctx, x, 0, exact, f"trained, order {order}, tier {tier}")
    after = ctx.tc_stats()
    print(f"order {order} tier {tier}: ran {t} / {td}, fallback {fb} / {fbd} of {len(x)}; causes {after} (before {before})")
    assert t == td and t in (1, 2) and (tier == "auto" or t == int(tier))
    if tier != "1":
        assert fb < 0.25 * len(x) and fbd < 0.25 * len(x)
    rows = oracle_rows(len(x), exact[1], exact[3])
    want = oracle_top2(po, W, H, D, order, mean, x, rows)
    assert_same(tuple(a[rows] for a in exact), want, "exact top-2 vs oracle rule")
    ctx.close()


@pytest.mark.parametrize("n", [1023, 1024, PROBE + 1, 2 * PROBE + 1])
@pytest.mark.parametrize("kind", ["trained", "coincident"])
def test_top2_probe_row_counts(vsom, po, monkeypatch, kind, n):
    """Batch sizes either side of 1024 (K3 / K2) and of both probes; the coincident map sends the rest to the exact scan."""
    monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    W, H, D, mean, xall = _row_count_map(vsom, kind)
    x = xall[:n]
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean)
    exact = check_against_exact(ctx, x, 0, f"{kind}, {n} rows")
    t, td, fb, fbd = run_forms(vsom, ctx, x, 0, exact, f"{kind}, {n} rows")
    want = 0 if n < TC_MIN_ROWS else (2 if kind == "trained" else (3 if n > 2 * PROBE else 2))
    assert t == want and td == want, f"tier {t} / {td}, expected {want}"
    rows = oracle_rows(n, exact[1], exact[3], tight=64)
    assert_same(tuple(a[rows] for a in exact), oracle_top2(po, W, H, D, po.ORDER_EIGEN_SSE, mean, x, rows), "exact vs oracle")
    ctx.close()


# ------------------------------------------------------------------------------------------------ small maps: K3, CLR, edge cases
def _small(rng, W, H, Din, tr):
    D = Din * (Din - 1) if tr == 2 else Din
    mean = rng.standard_normal((W * H, D)).astype(F32)
    if tr == 2:
        z = rng.standard_normal((1, 1)).astype(F32)
        x = (rng.uniform(0.5, 1.5, (1, Din)) * z + 0.3 * rng.standard_normal((2048, Din))).astype(F32)
    else:
        x = rng.standard_normal((2048, Din)).astype(F32)
    return D, mean, x


# the tier only matters on K2: >= 1024 rows of Standard / Median
TR_CASES = [(tr, n, tier) for tr in (0, 1) for n, tier in ((300, "auto"), (2048, "1"), (2048, "2"), (2048, "auto"))] + [(2, 300, "auto"), (2, 2048, "auto")]


@pytest.mark.parametrize("order", [0, 2])
@pytest.mark.parametrize("tr, n, tier", TR_CASES)
def test_top2_transforms_orders(vsom, po, monkeypatch, tr, n, tier, order):
    """Standard, Median and CLR in both orders; below 1024 rows (K3) and above (K2 in each tier; CLR always K3)."""
    _tier(monkeypatch, tier)
    rng = np.random.default_rng(100 + 10 * tr + order)
    W, H, Din = 13, 11, (6 if tr == 2 else 40)
    D, mean, x = _small(rng, W, H, Din, tr)
    x = x[:n]
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    ctx.upload_state(mean=mean)
    exact = check_against_exact(ctx, x, 0, "small map")
    t, td, _, _ = run_forms(vsom, ctx, x, 0, exact, f"tr {tr} order {order} tier {tier} n {n}")
    want_k2 = tr != 2 and len(x) >= TC_MIN_ROWS
    assert (t > 0) == want_k2 and (td > 0) == want_k2
    rows = np.r_[0:len(x):7]
    assert_same(tuple(a[rows] for a in exact), oracle_top2(po, W, H, Din, order, mean, x, rows, transform=tr), "exact vs oracle")
    ctx.close()


@pytest.mark.parametrize("n", [300, 4096])
def test_top2_duplicated_nodes(vsom, po, n):
    """Every node appears twice or three times: dist == dist2 and the lower index is the BMU."""
    rng = np.random.default_rng(5)
    W, H, D = 16, 12, 24
    base = rng.standard_normal((W * H // 3 + 1, D)).astype(F32)
    mean = base[rng.permutation(np.arange(W * H) % len(base))]
    x = rng.standard_normal((n, D)).astype(F32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    ctx.upload_state(mean=mean)
    exact = check_against_exact(ctx, x, 0, "duplicates")
    run_forms(vsom, ctx, x, 0, exact, "duplicates")
    assert np.array_equal(exact[1].view(np.uint32), exact[3].view(np.uint32))
    assert (exact[0] < exact[2]).all()
    rows = np.r_[0:n:11]
    assert_same(tuple(a[rows] for a in exact), oracle_top2(po, W, H, D, 0, mean, x, rows), "exact vs oracle")
    ctx.close()


BIG = 1 << 32


@pytest.mark.parametrize("n", [300, 4096])
@pytest.mark.parametrize("case", ["node0_only", "two_eligible", "above_2^32"])
def test_top2_min_hits(vsom, po, case, n):
    """Restricted search: only node 0 eligible (no runner-up), node 0 and the last node, hit counts whose low words mislead."""
    rng = np.random.default_rng(9)
    W, H, D = 14, 10, 32
    N = W * H
    mean = rng.standard_normal((N, D)).astype(F32)
    x = rng.standard_normal((n, D)).astype(F32)
    if case == "node0_only":
        hits, mh = np.zeros(N, np.uint64), 1
    elif case == "two_eligible":
        hits, mh = np.zeros(N, np.uint64), 5
        hits[N - 1] = 5
    else:
        hits, mh = rng.choice(np.array([0, 1, BIG - 1, BIG, BIG + 1, 3 * BIG], np.uint64), N), BIG
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean, hits=hits)
    exact = check_against_exact(ctx, x, mh, case)
    run_forms(vsom, ctx, x, mh, exact, case)
    if case == "node0_only":
        assert (exact[0] == 0).all() and (exact[2] == NONE).all() and np.isnan(exact[3]).all()
    rows = np.r_[0:n:13]
    assert_same(tuple(a[rows] for a in exact), oracle_top2(po, W, H, D, 2, mean, x, rows, hits=hits, min_hits=mh), "exact vs oracle")
    ctx.close()


@pytest.mark.parametrize("n", [100, 2048])
@pytest.mark.parametrize("grid", [(1, 1), (1, 37), (37, 1)])
def test_top2_tiny_grids(vsom, po, grid, n):
    W, H = grid
    D = 20
    rng = np.random.default_rng(W * 100 + H)
    mean = rng.standard_normal((W * H, D)).astype(F32)
    x = rng.standard_normal((n, D)).astype(F32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_REFERENCE)
    ctx.upload_state(mean=mean)
    exact = check_against_exact(ctx, x, 0, f"grid {grid}")
    run_forms(vsom, ctx, x, 0, exact, f"grid {grid}")
    if W * H == 1:
        assert (exact[2] == NONE).all()
    rows = np.r_[0:n:9]
    assert_same(tuple(a[rows] for a in exact), oracle_top2(po, W, H, D, 0, mean, x, rows), "exact vs oracle")
    ctx.close()


@pytest.mark.parametrize("n", [500, 4096])
@pytest.mark.parametrize("order", [0, 2])
@pytest.mark.parametrize("case", ["rows", "nan_node0", "nan_nodes", "inf_map"])
def test_top2_special_values(vsom, po, monkeypatch, case, order, n):
    """NaN / +-inf row elements; a NaN component at node 0 (every row's BMU is node 0) and at other nodes; an infinite map value."""
    monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    rng = np.random.default_rng(31)
    W, H, D = 12, 12, 48
    mean = rng.standard_normal((W * H, D)).astype(F32)
    x = rng.standard_normal((n, D)).astype(F32)
    if case == "rows":
        for i in range(0, n, 37):
            x[i, i % D] = (np.nan, np.inf, -np.inf)[(i // 37) % 3]
    elif case == "nan_node0":
        mean[0, 5] = np.nan
    elif case == "nan_nodes":
        mean[[3, 4, 50, 143], 7] = np.nan
    else:
        mean[77, 2] = np.inf
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, order)
    ctx.upload_state(mean=mean)
    exact = check_against_exact(ctx, x, 0, case)
    run_forms(vsom, ctx, x, 0, exact, case)
    if case == "nan_node0":
        assert (exact[0] == 0).all() and np.isnan(exact[1]).all()
    rows = np.r_[0:n:17]
    assert_same(tuple(a[rows] for a in exact), oracle_top2(po, W, H, D, order, mean, x, rows), "exact vs oracle")
    ctx.close()


@pytest.mark.parametrize("tier", ["1", "2"])
def test_top2_host_slab_boundaries(vsom, monkeypatch, tier):
    """Host form in 1024-row slabs (VSOM_TC_HOST_SLAB_LOG2=10): 5000 rows cross four slab boundaries and three staging buffers."""
    _tier(monkeypatch, tier)
    monkeypatch.setenv("VSOM_TC_HOST_SLAB_LOG2", "10")
    W, H, D, mean, xall = _row_count_map(vsom, "trained")
    x = xall[:5000]
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean)
    exact = check_against_exact(ctx, x, 0, "slabs")
    t, td, _, _ = run_forms(vsom, ctx, x, 0, exact, f"slabs, tier {tier}")
    assert t == int(tier) and td == int(tier)
    ctx.close()


# ------------------------------------------------------------------------------------------------ Som::topographicError (C++ driver)
def topographic_error(W, bmu, bmu2):
    has = bmu2 != NONE
    dx = np.abs((bmu % W).astype(np.int64) - (bmu2 % W).astype(np.int64))
    dy = np.abs((bmu // W).astype(np.int64) - (bmu2 // W).astype(np.int64))
    return float(np.count_nonzero(has & (np.maximum(dx, dy) != 1))) / len(bmu)


@pytest.mark.parametrize("case", ["k3", "k2"])
def test_som_topographic_error(vsom, po, tmp_path, monkeypatch, case):
    """tests/cpp/topo_driver: Som::topographicError and Som::mapDataSetTopTwo against the rule on the oracle's distances (every row)."""
    monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    if case == "k3":
        W, H, D = 20, 16, 24
        rng = np.random.default_rng(3)
        mean = init_map(W * H, D, 8)
        x = rng.standard_normal((700, D)).astype(F32) * F32(0.5)
    else:
        W, H, D, mean, xall = _row_count_map(vsom, "trained")
        x = xall[:4096]
    n = len(x)
    case_file, out_file = tmp_path / "case.bin", tmp_path / "out.bin"
    with open(case_file, "wb") as f:
        np.array([W, H, D, n], np.int32).tofile(f)
        np.ascontiguousarray(mean, F32).tofile(f)
        np.ascontiguousarray(x, F32).tofile(f)
    r = subprocess.run([TOPO_DRIVER, str(case_file), str(out_file)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = out_file.read_bytes()
    te = np.frombuffer(raw, np.float64, 1)[0]
    o = 8
    b = np.frombuffer(raw, np.uint64, n, o).astype(np.uint32)
    d = np.frombuffer(raw, F32, n, o + 8 * n)
    b2 = np.frombuffer(raw, np.uint64, n, o + 12 * n)
    d2 = np.frombuffer(raw, F32, n, o + 20 * n)
    b2 = np.where(b2 == np.uint64(2**64 - 1), np.uint64(0xFFFFFFFF), b2).astype(np.uint32)
    want = oracle_top2(po, W, H, D, po.ORDER_SEQUENTIAL, mean, x, np.arange(n))
    assert_same((b, d, b2, d2), want, f"{case}: mapDataSetTopTwo vs oracle rule")
    assert te == topographic_error(W, want[0], want[2]), f"{case}: topographicError {te}"
    print(f"{case}: topographic error {te} over {n} rows")
