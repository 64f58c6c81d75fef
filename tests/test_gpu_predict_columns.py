"""Prediction of unobserved columns (vsom_predict_columns / _device, Som::predictColumns).

Every case checks, bit for bit:
- (a) bmu / dist against find_bmu_exact on a second context of the same grid and summation order, Standard, whose mean plane is
  the columns S of the map, with the same hits, on the rows x[:, S];
- (b) mean / sigma against download_state() at the BMU and the predicted columns Q;
- (c) on a subset of rows (first and last rows, rows around the 8192-row probe boundaries, the smallest relative gaps between the
  best and second-best distances), against the findBmu rule on the oracle's distances over the compacted map.
The host and device forms agree; a LANES context gives the REFERENCE bits; the call leaves the state untouched."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import REPO, assert_bit_equal
from test_gpu_benchmark_shapes import PROBE, _row_count_map, synth_chunk
from test_gpu_top2 import oracle_rows, oracle_top2

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

F32 = np.float32
PREDICT_DRIVER = os.path.join(REPO, "tests", "cpp", "predict_driver")


def mask_of(Dm, S):
    m = np.zeros(Dm, np.uint8)
    m[np.asarray(S, np.int64)] = 1
    return m


def scoring_order(order, vsom):
    """Every scoring path sums a LANES context in the REFERENCE order."""
    return vsom.ORDER_REFERENCE if order == vsom.ORDER_LANES else order


def compact_exact(vsom, W, H, order, st, S, xS, min_hits):
    """(a): find_bmu_exact and find_bmu2_exact on the Standard context whose plane is mean[:, S], and its last find_bmu's tier."""
    c = vsom.VsomContext(W, H, len(S), vsom.STANDARD, order)
    c.upload_state(mean=np.ascontiguousarray(st["mean"][:, S]), hits=st["hits"])
    eb, ed = c.find_bmu_exact(xS, min_hits=min_hits)
    e2 = c.find_bmu2_exact(xS, min_hits=min_hits)
    c.close()
    return eb, ed, e2[2], e2[3]


def device_form(vsom, ctx, x, match, min_hits):
    import torch

    n, q = len(x), int(ctx.Dm - int(np.count_nonzero(match)))
    xd = torch.from_numpy(np.ascontiguousarray(x, F32)).cuda()
    b = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    d = torch.empty(max(n, 1), dtype=torch.float32, device="cuda")
    m = torch.empty(max(n * q, 1), dtype=torch.float32, device="cuda")
    s = torch.empty(max(n * q, 1), dtype=torch.float32, device="cuda")
    ctx.predict_columns_device(xd, n, match, b, d, m, s, min_hits=min_hits)
    torch.cuda.synchronize()
    return (b.cpu().numpy()[:n].view(np.uint32), d.cpu().numpy()[:n], m.cpu().numpy()[:n * q].reshape(n, q), s.cpu().numpy()[:n * q].reshape(n, q))


def check_predict(vsom, ctx, x, match, min_hits=0, what="", po=None, probe_rows=True):
    """Host and device forms against (a) and (b), and (c) when po is given.  Returns (host tier, device tier, exact results)."""
    W, H = ctx.W, ctx.H
    S, Q = np.flatnonzero(match), np.flatnonzero(match == 0)
    st = ctx.download_state()
    xS = np.ascontiguousarray(x[:, S])
    eb, ed, e2b, e2d = compact_exact(vsom, W, H, ctx.order, st, S, xS, min_hits)
    if ctx.order == vsom.ORDER_LANES:
        rb, rd, _, _ = compact_exact(vsom, W, H, vsom.ORDER_REFERENCE, st, S, xS, min_hits)
        assert_bit_equal(eb, rb, f"{what}: LANES compact vs REFERENCE bmu")
        assert_bit_equal(ed, rd, f"{what}: LANES compact vs REFERENCE dist")
    hb, hd, hm, hs = ctx.predict_columns(x, match, min_hits=min_hits)
    tier = ctx.last_score_tc
    db, dd, dm, ds = device_form(vsom, ctx, x, match, min_hits)
    tierd = ctx.last_score_tc
    for form, (b, d, m, s) in (("host", (hb, hd, hm, hs)), ("device", (db, dd, dm, ds))):
        assert_bit_equal(b, eb, f"{what}: {form} bmu")
        assert_bit_equal(d, ed, f"{what}: {form} dist")
        assert_bit_equal(m, st["mean"][eb][:, Q] if len(x) else np.empty((0, len(Q)), F32), f"{what}: {form} mean")
        assert_bit_equal(s, st["sigma"][eb][:, Q] if len(x) else np.empty((0, len(Q)), F32), f"{what}: {form} sigma")
    after = ctx.download_state()
    for k in st:
        assert_bit_equal(after[k], st[k], f"{what}: state {k} changed")
    if po is not None and len(x):
        rows = oracle_rows(len(x), ed, e2d) if probe_rows else np.unique(np.r_[np.arange(min(len(x), 64)), np.arange(max(0, len(x) - 64), len(x))])
        want = oracle_top2(po, W, H, len(S), scoring_order(ctx.order, vsom), np.ascontiguousarray(st["mean"][:, S]), xS, rows, hits=st["hits"],
                           min_hits=min_hits)
        g = (eb[rows], ed[rows])
        assert_bit_equal(g[0], want[0], f"{what}: exact bmu vs oracle rule")
        nan = np.isnan(want[1])
        assert np.array_equal(np.isnan(g[1]), nan) and np.array_equal(g[1][~nan].view(np.uint32), want[1][~nan].view(np.uint32)), f"{what}: oracle dist"
    return tier, tierd, (eb, ed)


def trained_ctx(vsom, W, H, D, transform, order, rows=3000, seed=5):
    rng = np.random.default_rng(seed)
    centres = (rng.standard_normal((8, D)) * 3).astype(F32)
    x = (rng.standard_normal((rows, D)) + centres[rng.integers(0, 8, rows)]).astype(F32)
    ctx = vsom.VsomContext(W, H, D, transform, order)
    ctx.upload_state(mean=rng.standard_normal((W * H, D)).astype(F32))
    ctx.train_chunk(x[: rows // 2], 0.3, max(W, H) / 2.0, vsom.EXPONENTIAL)
    ctx.train_chunk(x[rows // 2:], 0.1, 2.0, vsom.EXPONENTIAL)
    return ctx, x


# ------------------------------------------------------------------------------------------------ orders and transformations
@pytest.mark.parametrize("transform", [0, 1])
@pytest.mark.parametrize("order", [0, 1, 2])
def test_orders_and_transforms(vsom, po, order, transform):
    """Standard and Median maps after training, in the REFERENCE, LANES and Eigen orders; K2 (3000 rows) and K3 (700 rows); 25 of
    40 columns scattered, min_hits 0 and 2."""
    ctx, x = trained_ctx(vsom, 24, 20, 40, transform, order)
    match = mask_of(40, np.random.default_rng(order * 2 + transform).choice(40, 25, replace=False))
    for n in (3000, 700):
        for mh in (0, 2):
            t, td, _ = check_predict(vsom, ctx, x[:n], match, mh, f"order {order} transform {transform} n {n} min_hits {mh}", po, probe_rows=False)
            assert t == td and (t == 0) == (n < 1024)
    ctx.close()


# ------------------------------------------------------------------------------------------------ MNIST-shaped rows
def mnist_rows(n, seed):
    rng = np.random.default_rng(seed)
    centres = rng.random((10, 784)).astype(F32)
    cls = rng.integers(0, 10, n)
    x = np.zeros((n, 794), F32)
    x[:, :784] = np.clip(centres[cls] + 0.15 * rng.standard_normal((n, 784)), 0, 1)
    x[np.arange(n), 784 + cls] = 1.0
    return x, cls


def test_mnist_shaped_label_prediction(vsom, po):
    """20 x 20 x 794: 784 'pixels' around ten class centres and a one-hot label, trained through the online step; the ten label
    columns are predicted from the 784 pixels (their values in the rows are never read)."""
    x, cls = mnist_rows(6000, 11)
    ctx = vsom.VsomContext(20, 20, 794, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=np.random.default_rng(3).random((400, 794)).astype(F32))
    for i, (sg, eta) in enumerate(((10.0, 0.5), (5.0, 0.3), (2.0, 0.1))):
        ctx.train_chunk(x[1000 * i:1000 * (i + 1)], eta, sg, vsom.EXPONENTIAL)
    test, tcls = x[3000:].copy(), cls[3000:]
    test[:, 784:] = np.nan
    match = mask_of(794, np.arange(784))
    t, td, _ = check_predict(vsom, ctx, test, match, 0, "mnist-shaped", po)
    assert t in (1, 2) and td == t
    _, _, mean, sigma = ctx.predict_columns(test, match)
    acc = float(np.mean(np.argmax(mean, axis=1) == tcls))
    print(f"mnist-shaped label accuracy {acc:.4f} (tier {t})")
    assert acc > 0.9
    ctx.close()


# ------------------------------------------------------------------------------------------------ bench's trained map, K2's tiers
BIG_N = 1 << 20
_big = {}


def big_case(vsom):
    if "x" not in _big:
        W, H, D, mean, _ = _row_count_map(vsom, "trained")
        S = np.sort(np.random.default_rng(192).choice(D, 192, replace=False))
        _big.update(W=W, H=H, D=D, mean=mean, S=S, x=synth_chunk(BIG_N, D, 1234 + 6))
    return _big


@pytest.mark.parametrize("knob", ["auto", "tier1", "tier2", "single_cta"])
def test_trained_map_tiers(vsom, po, monkeypatch, knob):
    """2^20 rows on bench's trained 128 x 128 x 256 scoring map, |S| = 192 scattered columns, through the probed tier, the forced
    tiers and the single-CTA kernel; the tier is the one find_bmu picks on the compacted context for the same rows."""
    c = big_case(vsom)
    monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    monkeypatch.delenv("VSOM_TC_PAIR", raising=False)
    if knob == "tier1":
        monkeypatch.setenv("VSOM_TC_TIER", "1")
    elif knob == "tier2":
        monkeypatch.setenv("VSOM_TC_TIER", "2")
    elif knob == "single_cta":
        monkeypatch.setenv("VSOM_TC_PAIR", "0")
    ctx = vsom.VsomContext(c["W"], c["H"], c["D"], vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=c["mean"])
    match = mask_of(c["D"], c["S"])
    t, td, _ = check_predict(vsom, ctx, c["x"], match, 0, f"trained map, {knob}", po)
    cc = vsom.VsomContext(c["W"], c["H"], len(c["S"]), vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    cc.upload_state(mean=np.ascontiguousarray(c["mean"][:, c["S"]]))
    cc.find_bmu(np.ascontiguousarray(c["x"][:, c["S"]]))
    want = cc.last_score_tc
    cc.close()
    print(f"{knob}: tier {t} / {td}, compacted find_bmu tier {want}, pair {ctx.last_score_pair}")
    assert t == td == want
    assert t == {"tier1": 1, "tier2": 2}.get(knob, t) and t in (1, 2)
    if knob == "single_cta":
        assert ctx.last_score_pair == 0
    ctx.close()


def test_coincident_map_tier3(vsom, po, monkeypatch):
    """Nodes within 1e-4 of one point: the probes send the rest of the call to the exact scan (tier 3), host and device."""
    monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    W, H, D, mean, x = _row_count_map(vsom, "coincident")
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean)
    match = mask_of(D, np.arange(0, D, 2))
    t, td, _ = check_predict(vsom, ctx, x[: 2 * PROBE + 2], match, 0, "coincident map", po)
    assert t == td == 3
    ctx.close()


# ------------------------------------------------------------------------------------------------ shapes
@pytest.mark.parametrize("m,tier0", [(2048, False), (2049, True)])
def test_wide_map_k2_limit(vsom, m, tier0):
    """Dm = 2560: |S| = 2048 still runs K2, |S| = 2049 runs K3."""
    rng = np.random.default_rng(m)
    ctx = vsom.VsomContext(8, 6, 2560, vsom.STANDARD, vsom.ORDER_REFERENCE)
    ctx.upload_state(mean=rng.standard_normal((48, 2560)).astype(F32))
    x = rng.standard_normal((1100, 2560)).astype(F32)
    match = mask_of(2560, np.sort(rng.choice(2560, m, replace=False)))
    t, td, _ = check_predict(vsom, ctx, x, match, 0, f"Dm 2560, |S| {m}")
    assert t == td and (t == 0) == tier0
    ctx.close()


@pytest.mark.parametrize("n", [0, 1, 1023, 1024, PROBE + 1])
@pytest.mark.parametrize("order", [0, 2])
def test_subset_sizes_and_row_counts(vsom, po, order, n):
    """|S| in {1, 7, 8, 9, Dm - 1} (the Eigen order's block and tail lengths), subsets without the first or the last column."""
    D = 33
    ctx, _ = trained_ctx(vsom, 16, 12, D, vsom.STANDARD, order, rows=2000, seed=order)
    x = synth_chunk(max(n, 1), D, 99 + n)[:n]
    rng = np.random.default_rng(n)
    subsets = [np.sort(rng.choice(D, k, replace=False)) for k in (1, 7, 8, 9, D - 1)]
    subsets += [np.arange(1, D), np.arange(0, D - 1), np.arange(1, D - 1)]
    for S in subsets:
        t, td, _ = check_predict(vsom, ctx, x, mask_of(D, S), 0, f"order {order}, n {n}, |S| {len(S)} first {S[0]} last {S[-1]}", po, probe_rows=False)
        assert t == td
    ctx.close()


def test_full_mask_is_find_bmu(vsom):
    """|S| = Dm: q = 0 and the bits of find_bmu on the original context, host and device."""
    ctx, x = trained_ctx(vsom, 24, 20, 40, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    match = np.ones(40, np.uint8)
    b, d, m, s = ctx.predict_columns(x, match)
    assert m.shape == (len(x), 0) and s.shape == (len(x), 0)
    fb, fd = ctx.find_bmu(x)
    assert_bit_equal(b, fb, "bmu")
    assert_bit_equal(d, fd, "dist")
    db, dd, _, _ = device_form(vsom, ctx, x, match, 0)
    assert_bit_equal(db, fb, "device bmu")
    assert_bit_equal(dd, fd, "device dist")
    ctx.close()


def test_host_slab_boundaries(vsom, monkeypatch):
    """Small host slabs on both host paths: K2's three-buffer pipeline (2^10-row slabs) and the exact scan's (2^9)."""
    monkeypatch.setenv("VSOM_TC_HOST_SLAB_LOG2", "10")
    monkeypatch.setenv("VSOM_EXACT_HOST_SLAB_LOG2", "9")
    ctx, x = trained_ctx(vsom, 24, 20, 40, vsom.STANDARD, vsom.ORDER_REFERENCE, rows=5000)
    match = mask_of(40, np.arange(3, 40, 3))
    t, td, _ = check_predict(vsom, ctx, x, match, 0, "K2 host slabs")
    assert t != 0 and td == t
    t, _, _ = check_predict(vsom, ctx, x[:1000], match, 0, "exact host slabs")
    assert t == 0
    ctx.close()


# ------------------------------------------------------------------------------------------------ special values, min_hits
def test_predicted_columns_are_never_read(vsom, po):
    """NaN, +-inf and garbage in the predicted columns give the outputs of zeros there; a NaN in a matched column follows the
    node-0 rule (BMU 0, NaN distance)."""
    ctx, x = trained_ctx(vsom, 24, 20, 40, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    match = mask_of(40, np.arange(0, 40, 2))
    Q = np.flatnonzero(match == 0)
    zero = x.copy()
    zero[:, Q] = 0
    want = ctx.predict_columns(zero, match)
    for fill in (np.nan, np.inf, -np.inf, 3.0e38):
        y = x.copy()
        y[:, Q] = fill
        got = ctx.predict_columns(y, match)
        for g, w, name in zip(got, want, ("bmu", "dist", "mean", "sigma")):
            assert_bit_equal(g, w, f"{fill} in Q: {name}")
        db, dd, dm, ds = device_form(vsom, ctx, y, match, 0)
        for g, w, name in zip((db, dd, dm, ds), want, ("bmu", "dist", "mean", "sigma")):
            assert_bit_equal(g, w, f"{fill} in Q, device: {name}")
    y = x.copy()
    y[::7, 4] = np.nan
    _, _, (eb, ed) = check_predict(vsom, ctx, y, match, 0, "NaN in a matched column", po, probe_rows=False)
    assert np.all(eb[::7] == 0) and np.all(np.isnan(ed[::7]))
    ctx.close()


def test_min_hits(vsom, po):
    """min_hits after training, and a min_hits no node reaches: only node 0 is eligible."""
    ctx, x = trained_ctx(vsom, 24, 20, 40, vsom.STANDARD, vsom.ORDER_REFERENCE)
    hits = ctx.download_state()["hits"]
    match = mask_of(40, np.arange(10, 40))
    mh = int(np.median(hits[hits > 0]))
    check_predict(vsom, ctx, x, match, mh, f"min_hits {mh}", po, probe_rows=False)
    _, _, (eb, _) = check_predict(vsom, ctx, x, match, int(hits.max()) + 1, "only node 0", po, probe_rows=False)
    assert np.all(eb == 0)
    ctx.close()


# ------------------------------------------------------------------------------------------------ refusals
def _raw_call(vsom, ctx, x, match_ptr, n):
    from importlib import import_module

    binding = import_module(vsom.__name__ + ".binding")
    q = ctx.Dm
    outs = [np.full(n, 0xABABABAB, np.uint32), np.full(n, 7.0, F32), np.full(n * q, 7.0, F32), np.full(n * q, 7.0, F32)]
    keep = [o.copy() for o in outs]
    f32p, u32p = C.POINTER(C.c_float), C.POINTER(C.c_uint32)
    rc = binding.lib().vsom_predict_columns(ctx._h, x.ctypes.data_as(f32p), n, match_ptr, 0, outs[0].ctypes.data_as(u32p), outs[1].ctypes.data_as(f32p),
                                            outs[2].ctypes.data_as(f32p), outs[3].ctypes.data_as(f32p))
    for o, k in zip(outs, keep):
        assert_bit_equal(o, k, "a refused call wrote an output")
    return rc


def _raw_call_device(vsom, ctx, x, match_ptr, n):
    import torch
    from importlib import import_module

    binding = import_module(vsom.__name__ + ".binding")
    xd = torch.from_numpy(x).cuda()
    outs = [torch.full((n,), 5, dtype=torch.int32, device="cuda"), *(torch.full((n * ctx.Dm,), 7.0, device="cuda") for _ in range(3))]
    rc = binding.lib().vsom_predict_columns_device(ctx._h, xd.data_ptr(), n, match_ptr, 0, *(o.data_ptr() for o in outs))
    torch.cuda.synchronize()
    assert bool((outs[0] == 5).all()) and all(bool((o == 7.0).all()) for o in outs[1:]), "a refused device call wrote an output"
    return rc


def test_refusals(vsom):
    """NULL mask, a value of 2, no matched column -> VSOM_ERR_INVALID; a CLR context and a sharded one -> VSOM_ERR_UNSUPPORTED.
    Nothing is written."""
    u8p = C.POINTER(C.c_uint8)
    ctx = vsom.VsomContext(8, 6, 12, vsom.STANDARD, vsom.ORDER_REFERENCE)
    x = np.random.default_rng(0).standard_normal((40, 12)).astype(F32)
    bad2 = mask_of(12, [0, 3])
    bad2[5] = 2
    for what, m in (("NULL", None), ("value 2", bad2), ("all zero", np.zeros(12, np.uint8))):
        ptr = C.cast(None, u8p) if m is None else m.ctypes.data_as(u8p)
        assert _raw_call(vsom, ctx, x, ptr, len(x)) == -1, what
        assert _raw_call_device(vsom, ctx, x, ptr, len(x)) == -1, what
    # the binding refuses a mask that does not hold exactly Dm entries (the library reads Dm bytes and sizes its outputs from them)
    import torch

    xd = torch.from_numpy(x).cuda()
    for what, m in (("too long, a 1 past Dm", np.r_[mask_of(12, [0, 3]), np.uint8(1)]), ("too short", mask_of(12, [0, 3])[:11]),
                    ("column indices", np.array([0, 3], np.uint8)), ("2-d", mask_of(12, [0, 3]).reshape(3, 4))):
        with pytest.raises(ValueError):
            ctx.predict_columns(x, m)
        with pytest.raises(ValueError):
            ctx.predict_columns_device(xd, len(x), m, torch.empty(len(x), dtype=torch.int32, device="cuda"))
    ctx.close()
    clr = vsom.VsomContext(6, 5, 4, vsom.CLR, vsom.ORDER_REFERENCE)
    m = mask_of(clr.Dm, [0, 1])
    assert _raw_call(vsom, clr, np.zeros((10, clr.Dm), F32), m.ctypes.data_as(u8p), 10) == -3
    clr.close()
    ctxs = [vsom.VsomContext(13, 37, 10, vsom.STANDARD, 0, device=0, rank=r, world=2) for r in range(2)]
    for a in ctxs:
        for r, b in enumerate(ctxs):
            a.peer_attach(r, b)
    m = mask_of(10, [1, 2])
    assert _raw_call(vsom, ctxs[0], np.zeros((10, 10), F32), m.ctypes.data_as(u8p), 10) == -3
    assert _raw_call_device(vsom, ctxs[1], np.zeros((10, 10), F32), m.ctypes.data_as(u8p), 10) == -3
    for c in ctxs:
        c.close()


# ------------------------------------------------------------------------------------------------ Som::predictColumns
def test_som_predict_columns_matches_binding(vsom, tmp_path):
    """One epoch of Som::train on a MemoryDataLoader of MNIST-shaped rows, then Som::predictColumns on the same rows
    (tests/cpp/predict_driver), equals predict_columns on a binding context holding the trained state."""
    x, _ = mnist_rows(2500, 21)
    W, H, Din, n = 20, 20, 794, len(x)
    match = mask_of(Din, np.arange(784))
    q = Din - 784
    case, state, out = tmp_path / "case.bin", tmp_path / "state.bin", tmp_path / "out.bin"
    with open(case, "wb") as f:
        f.write(np.array([W, H, Din, 0, 2, n, 1000, 0], np.int32).tobytes())
        f.write(np.array([0.3, 0.1, 6.0, 0.2], np.float64).tobytes())
        f.write(match.tobytes())
        f.write(x.tobytes())
    r = subprocess.run([PREDICT_DRIVER, str(case), str(state), str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    N = W * H
    raw = open(state, "rb").read()
    mean = np.frombuffer(raw, F32, N * Din, 0).reshape(N, Din)
    sigma = np.frombuffer(raw, F32, N * Din, 4 * N * Din).reshape(N, Din)
    weight = np.frombuffer(raw, F32, N, 8 * N * Din)
    hits = np.frombuffer(raw, np.uint64, N, 8 * N * Din + 4 * N)
    o = open(out, "rb").read()
    bmu = np.frombuffer(o, np.uint64, n, 0).astype(np.uint32)
    dist = np.frombuffer(o, F32, n, 8 * n)
    pm = np.frombuffer(o, F32, n * q, 12 * n).reshape(n, q)
    ps = np.frombuffer(o, F32, n * q, 12 * n + 4 * n * q).reshape(n, q)
    ctx = vsom.VsomContext(W, H, Din, vsom.STANDARD, 2)
    ctx.upload_state(mean=mean, sigma=sigma, weight=weight, hits=hits)
    b, d, m, s = ctx.predict_columns(x, match)
    assert_bit_equal(bmu, b, "Som bmu")
    assert_bit_equal(dist, d, "Som dist")
    assert_bit_equal(pm, m, "Som mean")
    assert_bit_equal(ps, s, "Som sigma")
    ctx.close()


# ------------------------------------------------------------------------------------------------ NULL outputs
def test_null_outputs(vsom):
    """Every output may be NULL: the device form without out_bmu (the BMUs then go to staging) and with only sigma, the host form
    with only sigma and with only mean, on K2 (3000 rows) and K3 (700 rows); each equals the call with all four outputs."""
    import torch
    from importlib import import_module

    binding = import_module(vsom.__name__ + ".binding")
    f32p, u32p, u8p = C.POINTER(C.c_float), C.POINTER(C.c_uint32), C.POINTER(C.c_uint8)
    ctx, xall = trained_ctx(vsom, 24, 20, 40, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    match = mask_of(40, np.arange(1, 40, 3))
    q = 40 - int(match.sum())
    for n in (3000, 700):
        x = np.ascontiguousarray(xall[:n])
        b, d, m, s = ctx.predict_columns(x, match)
        xd = torch.from_numpy(x).cuda()
        for want_mean, want_sigma in ((True, False), (False, True), (True, True)):
            om = torch.full((n * q,), 7.0, device="cuda") if want_mean else None
            osg = torch.full((n * q,), 7.0, device="cuda") if want_sigma else None
            ctx.predict_columns_device(xd, n, match, None, None, om, osg)
            torch.cuda.synchronize()
            if om is not None:
                assert_bit_equal(om.cpu().numpy().reshape(n, q), m, f"n {n}, device, no bmu: mean")
            if osg is not None:
                assert_bit_equal(osg.cpu().numpy().reshape(n, q), s, f"n {n}, device, no bmu: sigma")
        for want_mean in (True, False):
            hm = np.full((n, q), 7.0, np.float32)
            hs = np.full((n, q), 7.0, np.float32)
            hb = np.full(n, 0xABABABAB, np.uint32)
            rc = binding.lib().vsom_predict_columns(ctx._h, x.ctypes.data_as(f32p), n, match.ctypes.data_as(u8p), 0, hb.ctypes.data_as(u32p), None,
                                                    hm.ctypes.data_as(f32p) if want_mean else None, None if want_mean else hs.ctypes.data_as(f32p))
            assert rc == 0
            assert_bit_equal(hb, b, f"n {n}, host: bmu")
            if want_mean:
                assert_bit_equal(hm, m, f"n {n}, host, mean only: mean")
                assert np.all(hs == 7.0)
            else:
                assert_bit_equal(hs, s, f"n {n}, host, sigma only: sigma")
                assert np.all(hm == 7.0)
    ctx.close()
