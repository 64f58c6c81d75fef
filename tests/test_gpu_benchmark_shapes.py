"""The online step and scoring against the CPU oracle at the shapes, chunk lengths, row counts and entry points bench.py
measures, and on both sides of the limits where the library changes path.

Online step (K1F and the generic kernel): BASELINE configs 1, 2, 3 and 5 through vsom_train_chunk_device with bench's
initial maps and data; chunks long enough that the exchange tag (t >> 1) & 0xff of both kernels comes back several times;
chunk lengths 1, 2, 3 and either side of 512 and 1024, and chunking invariance; the K1F eligibility edges (a grid side of
4096 and 512 owned nodes per CTA).

Scoring (K2, tensor-core candidate search + exact rescore): rows of 105 / 106 and 317 / 318 dimensions (where the A tile stops
being resident in tiers 2 and 1) up to the largest supported 2048 and the first unsupported 2049; a device call that splits
into three slabs at the shape's own slab cap; the 512 x 512 x 784 map of config 5; batch sizes either side of the dispatch
threshold (1024 rows) and of both probes (8192 rows each), down to the one-row exact-scan remainder; restricted searches
with hit counts and thresholds at and above 2^32; one-node, one-row and one-column maps.

Every result is compared bit for bit, with the oracle running the same reduction order; on large batches K2 is compared
with the exact scan (K3) on every row and with the oracle on the rows where the oracle is cheap."""
import functools
import zlib

import numpy as np
import pytest

from conftest import assert_bit_equal

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

F32 = np.float32
TAG_PERIOD = 512     # both online kernels tag their exchange keys with (t >> 1) & 0xff: a (row, tag) pair recurs every 512 steps
PROBE = 8192         # rows of each K2 probe (score_tc.cu kTcProbeRows)
TC_MIN_ROWS = 1024   # smallest batch the scoring calls send to K2 (score_tc.cu kTcMinRows)


# ------------------------------------------------------------------------------------------------ bench.py's generators
def synth_chunk(n, d, seed):
    """bench.py synth_chunk: x ~ N(mu_c, 1) around 64 cluster centres."""
    rng = np.random.default_rng(seed)
    centres = (rng.standard_normal((64, d)) * 3).astype(F32)
    lab = rng.integers(0, 64, n)
    x = rng.standard_normal((n, d), dtype=F32)
    x += centres[lab]
    return x


def init_map(n_nodes, dm, seed):
    """bench.py init_map: Som::randomInitialize's distribution, multiples of 1/1000 in [-1, 1)."""
    rng = np.random.default_rng(seed)
    return (rng.integers(-1000, 1000, (n_nodes, dm), dtype=np.int16).astype(F32) / F32(1000.0)).astype(F32)


def clr_chunk(n, j, seed):
    """bench.py's config-3 rows: one latent factor, J columns."""
    rng = np.random.default_rng(seed)
    z = rng.standard_normal((n, 1)).astype(F32)
    a = rng.uniform(0.5, 1.5, (1, j)).astype(F32)
    bb = rng.uniform(-1, 1, (1, j)).astype(F32)
    return (a * z + bb + 0.1 * rng.standard_normal((n, j))).astype(F32)


def config1_rows(n, d, seed):
    """bench.py's config-1 rows: integer pixel-like values in [0, 256)."""
    return np.floor(256 * np.random.default_rng(seed).random((n, d), dtype=F32) ** 2).astype(F32)


def small_rows(rng, n, Din, tr):
    if tr == 2:
        z = rng.standard_normal((n, 1)).astype(F32)
        a = rng.uniform(0.5, 1.5, (1, Din)).astype(F32)
        return (a * z + 0.1 * rng.standard_normal((n, Din))).astype(F32)
    return rng.standard_normal((n, Din)).astype(F32)


# ------------------------------------------------------------------------------------------------ helpers
@pytest.fixture(params=["fast", "generic"])
def online_kernel(request, monkeypatch):
    """K1F where it is eligible, and the generic kernel forced through VSOM_ONLINE_KERNEL=generic (read by vsom_create)."""
    if request.param == "generic":
        monkeypatch.setenv("VSOM_ONLINE_KERNEL", "generic")
    else:
        monkeypatch.delenv("VSOM_ONLINE_KERNEL", raising=False)
    return request.param


def _tc_tier(monkeypatch, tier):
    if tier == "auto":
        monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    else:
        monkeypatch.setenv("VSOM_TC_TIER", tier)


def assert_state_equal(ctx, o, what):
    got, want = ctx.download_state(), o.get_state()
    for k in ("mean", "S", "sigma", "weight", "hits"):
        assert_bit_equal(got[k], want[k], f"{what}: {k}")


def train_device(ctx, x, eta, sigma, decay):
    """vsom_train_chunk_device with the outputs in int32 / f32 device buffers that start as all-ones bit patterns, so that an
    output the kernel never writes cannot pass for a right one."""
    import torch

    n = len(x)
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    gb = torch.full((max(n, 1),), -1, dtype=torch.int32, device="cuda")
    gd = torch.full((max(n, 1),), -1, dtype=torch.int32, device="cuda").view(torch.float32)
    ctx.train_chunk_device(xd, n, eta, sigma, decay, gb, gd)
    ctx.synchronize()
    return gb.cpu().numpy()[:n].view(np.uint32), gd.cpu().numpy()[:n]


def train_and_compare(ctx, o, x, eta, sigma, decay, form, what, last=None, state=True):
    """One chunk through the device or the host entry point and through the oracle: per-sample outputs, then the map."""
    ob, od, orr, ol = o.train_rows(x, eta, sigma, decay, last_bmu=None if last is None else last.copy())
    if form == "device":
        assert last is None  # the device form starts every local walk at node 0
        gb, gd = train_device(ctx, x, eta, sigma, decay)
    else:
        gb, gd, gr, gl = ctx.train_chunk(x, eta, sigma, decay, last_bmu=None if last is None else last.copy())
        assert_bit_equal(gr, orr, f"{what}: resid2")
        assert_bit_equal(gl, ol, f"{what}: lastBMU")
    assert_bit_equal(gb, ob, f"{what}: bmu")
    assert_bit_equal(gd, od, f"{what}: dist")
    if state:
        assert_state_equal(ctx, o, what)
    return gb, gd


def bench_config_ctx(vsom, po, W, H, Din, tr, order, init):
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    ctx.upload_state(mean=init)
    o = po.Oracle(W, H, Din, tr, order)  # S, sigma, weight and hits start at zero on both sides
    o.set_state(mean=init)
    return ctx, o


# ------------------------------------------------------------------------------------------------ A.1-A.3: configs 2, 1, 3
@pytest.mark.parametrize("order", [2, 0], ids=["eigen_sse", "seq"])
def test_config2_device_chunks_cross_the_tag_wrap(vsom, po, order, online_kernel):
    """bench's headline call: 64 x 64 x 128 Median, eta 0.05, sigma 32, Exponential, bench's init and data, through
    vsom_train_chunk_device.  2048 samples cross the 512-step tag period three times; a second chunk continues on the carried
    state.  The host-buffer call from the same start state gives the same bits."""
    W, H, D = 64, 64, 128
    init = init_map(W * H, D, 42)
    x = synth_chunk(2048 + 1000, D, 1234 + 2)
    ctx, o = bench_config_ctx(vsom, po, W, H, D, vsom.MEDIAN, order, init)
    assert ctx.planes_resident
    gb, gd = train_and_compare(ctx, o, x[:2048], 0.05, 32.0, vsom.EXPONENTIAL, "device", "chunk 0")
    assert ctx.last_train_fast == (online_kernel == "fast")
    after0 = ctx.download_state()
    train_and_compare(ctx, o, x[2048:], 0.05, 16.0, vsom.EXPONENTIAL, "device", "chunk 1 (carried state)")
    ctx.close()

    hctx = vsom.VsomContext(W, H, D, vsom.MEDIAN, order)
    hctx.upload_state(mean=init)
    hb, hd, _, _ = hctx.train_chunk(x[:2048], 0.05, 32.0, vsom.EXPONENTIAL)
    assert_bit_equal(hb, gb, "host form bmu vs device form")
    assert_bit_equal(hd, gd, "host form dist vs device form")
    got = hctx.download_state()
    for k in ("mean", "S", "sigma", "weight", "hits"):
        assert_bit_equal(got[k], after0[k], f"host form vs device form: {k}")
    hctx.close()


@pytest.mark.parametrize("order", [2, 0], ids=["eigen_sse", "seq"])
def test_config1_device_chunks_cross_the_tag_wrap(vsom, po, order, online_kernel):
    """Config 1 (20 x 20 x 784 Standard, bench's eta 0.1 and sigma 10): in the Eigen order K1F scans each node with eight
    lanes."""
    W, H, D = 20, 20, 784
    init = init_map(W * H, D, 99)
    x = config1_rows(2048 + 600, D, 5)
    ctx, o = bench_config_ctx(vsom, po, W, H, D, vsom.STANDARD, order, init)
    train_and_compare(ctx, o, x[:2048], 0.1, 10.0, vsom.EXPONENTIAL, "device", "chunk 0")
    assert ctx.last_train_fast == (online_kernel == "fast")
    train_and_compare(ctx, o, x[2048:], 0.1, 4.0, vsom.EXPONENTIAL, "device", "chunk 1 (carried state)")
    ctx.close()


def test_config3_clr_device_chunk_crosses_the_tag_wrap(vsom, po, online_kernel):
    """Config 3 (50 x 50 CLR, J = 32: 992 parameters per node, bench's eta 0.001 and sigma 25): 600 samples cross one tag
    period."""
    W, H, J = 50, 50, 32
    Dm = vsom.model_length(J, vsom.CLR)
    init = init_map(W * H, Dm, 99)
    x = clr_chunk(600 + 40, J, 31)
    ctx, o = bench_config_ctx(vsom, po, W, H, J, vsom.CLR, vsom.ORDER_EIGEN_SSE, init)
    train_and_compare(ctx, o, x[:600], 0.001, 25.0, vsom.EXPONENTIAL, "device", "chunk 0")
    assert ctx.last_train_fast == (online_kernel == "fast")
    train_and_compare(ctx, o, x[600:], 0.001, 12.0, vsom.EXPONENTIAL, "device", "chunk 1 (carried state)")
    ctx.close()


# ------------------------------------------------------------------------------------------------ A.4: config 5
@pytest.mark.parametrize("order", [2, 0], ids=["eigen_sse", "seq"])
def test_config5_large_map_online_step_local_walk_and_umatrix(vsom, po, order):
    """The 512 x 512 x 784 map of config 5 (bench's seeds, sigma 16, eta 0.05) on the generic kernel with the planes in HBM and
    about 1772 owned rows per CTA; then a sigma = 1 chunk through the device form (every local walk starts at node 0); then
    the U-matrix."""
    W, H, D = 512, 512, 784
    init = init_map(W * H, D, 4242)
    x = synth_chunk(24 + 32, D, 777)
    ctx, o = bench_config_ctx(vsom, po, W, H, D, vsom.STANDARD, order, init)
    del init
    assert not ctx.planes_resident
    train_and_compare(ctx, o, x[:24], 0.05, 16.0, vsom.EXPONENTIAL, "device", "sigma 16")
    assert not ctx.last_train_fast
    gb, _ = train_and_compare(ctx, o, x[24:], 0.05, 1.0, vsom.EXPONENTIAL, "device", "sigma 1, walks from node 0")
    print(f"config 5 local walks ended at {sorted(set(gb.tolist()))[:8]} ...")
    assert_bit_equal(ctx.update_umatrix(), o.update_umatrix(), "umatrix")
    ctx.close()


# ------------------------------------------------------------------------------------------------ A.5: long chunks
LONG_MAPS = [(16, 12, 8, 0), (16, 12, 8, 1), (16, 12, 6, 2)]


@pytest.mark.parametrize("order", [2, 0], ids=["eigen_sse", "seq"])
@pytest.mark.parametrize("shape", LONG_MAPS, ids=lambda s: "x".join(map(str, s[:3])) + f"-tr{s[3]}")
def test_long_chunks_match_oracle(vsom, po, shape, order, online_kernel):
    """20 000 samples in one chunk at sigma > 1 (the exchange tag wraps 39 times), then 5 000 in the local-walk regime from
    explicit start nodes, through the host-buffer call."""
    W, H, Din, tr = shape
    rng = np.random.default_rng(zlib.crc32(repr((shape, order)).encode()))
    o = po.Oracle(W, H, Din, tr, order)
    o.random_initialize(42, 1.0)
    ctx = vsom.VsomContext(W, H, Din, tr, order)
    st = o.get_state()
    ctx.upload_state(st["mean"], st["S"], st["sigma"], st["weight"], st["hits"])
    x = small_rows(rng, 25000, Din, tr)
    eta = 0.001 if tr == 2 else 0.05
    train_and_compare(ctx, o, x[:20000], eta, 3.0, vsom.EXPONENTIAL, "host", "20000 samples, sigma 3")
    assert ctx.last_train_fast == (online_kernel == "fast")
    starts = rng.integers(0, W * H, 5000).astype(np.uint64)
    train_and_compare(ctx, o, x[20000:], eta, 0.9, vsom.INVERSE_PROPORTIONAL, "host", "5000 samples, sigma 0.9", last=starts)
    ctx.close()


# ------------------------------------------------------------------------------------------------ A.6: chunk-length edges
EDGE_LENGTHS = [1, 2, 3, 511, 512, 513, 1025]
EDGE_MAP = (24, 20, 12)  # 480 nodes: several per CTA on K1F


def _pieces(n):
    """A split of n samples into chunks of uneven lengths (1, 2, 3, 511, ... and the rest)."""
    out, i, k = [], 0, 0
    sizes = [1, 2, 3, 511, 512, 5]
    while i < n:
        s = min(sizes[k % len(sizes)], n - i)
        out.append((i, i + s))
        i, k = i + s, k + 1
    return out


@pytest.mark.parametrize("sigma", [4.0, 1.0], ids=["global", "local_walk"])
@pytest.mark.parametrize("n", EDGE_LENGTHS)
def test_chunk_length_edges_and_chunking_invariance(vsom, po, n, sigma, online_kernel):
    """Chunks of 1, 2, 3, 511, 512, 513 and 1025 samples through the device form against the oracle: the last sample's output
    is emitted after the loop, the sample ring has four slots and the tag period is 512.  The same samples as several chunks,
    and as one chunk per sample, give the same bits."""
    W, H, D = EDGE_MAP
    rng = np.random.default_rng(n)
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.random_initialize(7, 1.0)
    init = o.get_state()
    x = rng.standard_normal((n, D)).astype(F32)

    def fresh():
        c = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
        c.upload_state(init["mean"], init["S"], init["sigma"], init["weight"], init["hits"])
        return c

    ctx = fresh()
    gb, gd = train_and_compare(ctx, o, x, 0.1, sigma, vsom.EXPONENTIAL, "device", f"one chunk of {n}")
    assert ctx.last_train_fast == (online_kernel == "fast")
    whole = ctx.download_state()
    ctx.close()

    for name, pieces in (("uneven chunks", _pieces(n)), ("one sample per chunk", [(i, i + 1) for i in range(n)])):
        c = fresh()
        bs, ds = zip(*(train_device(c, x[a:b], 0.1, sigma, vsom.EXPONENTIAL) for a, b in pieces))
        assert_bit_equal(np.concatenate(bs), gb, f"{name}: bmu")
        assert_bit_equal(np.concatenate(ds), gd, f"{name}: dist")
        got = c.download_state()
        for k in ("mean", "S", "sigma", "weight", "hits"):
            assert_bit_equal(got[k], whole[k], f"{name}: {k}")
        c.close()


# ------------------------------------------------------------------------------------------------ A.7: K1F eligibility edges
def _owned_grid(extra):
    """A map with 512 owned nodes per CTA (extra = 0) or 513 (extra = 1) on this device's K1F grid."""
    import torch

    G = min(torch.cuda.get_device_properties(0).multi_processor_count, 160)  # K1F runs one CTA per SM, at most 160
    return 512 + extra, G


@pytest.mark.parametrize("edge", ["side_4096", "side_4097", "owned_512", "owned_513"])
def test_fast_kernel_eligibility_edges(vsom, po, edge, online_kernel):
    """K1F keys carry 12-bit grid coordinates and one scan lane per owned node: a 4096-wide map and one with 512 owned nodes per
    CTA still run it, one more column or one more node per CTA runs the generic kernel.  Both sides match the oracle."""
    if edge.startswith("side"):
        W, H = int(edge[5:]), 2
        eligible = W <= 4096
    else:
        W, H = _owned_grid(int(edge[6:]) - 512)
        eligible = W == 512
    D = 4
    rng = np.random.default_rng(W * H)
    o = po.Oracle(W, H, D, po.MEDIAN, po.ORDER_EIGEN_SSE)
    o.random_initialize(11, 1.0)
    st = o.get_state()
    ctx = vsom.VsomContext(W, H, D, vsom.MEDIAN, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(st["mean"], st["S"], st["sigma"], st["weight"], st["hits"])
    x = rng.standard_normal((TAG_PERIOD + 77, D)).astype(F32)
    train_and_compare(ctx, o, x[:TAG_PERIOD + 40], 0.1, 3.0, vsom.EXPONENTIAL, "device", f"{W}x{H}")
    assert ctx.last_train_fast == (eligible and online_kernel == "fast"), f"{W}x{H}: K1F ran = {ctx.last_train_fast}"
    train_and_compare(ctx, o, x[TAG_PERIOD + 40:], 0.1, 0.8, vsom.EXPONENTIAL, "host", f"{W}x{H} local walks",
                      last=rng.integers(0, W * H, 37).astype(np.uint64))
    ctx.close()


# ------------------------------------------------------------------------------------------------ B.1: row lengths
ROW_LENGTHS = [105, 106, 317, 318, 1000, 2047, 2048]
ROW_MAP = (20, 20)
ROW_N = 1500


def tc_slab_cap(Dm, split):
    """Rows per K2 slab (score_tc.cu tc_slab_cap): the fp16 operand staging of a slab stays below 2.5 GiB."""
    kpad = ((3 * Dm if split else Dm) + 3 + 15) // 16 * 16
    return max(128, ((5 << 29) // (kpad * 2)) & ~127)


@functools.lru_cache(maxsize=None)
def _row_length_case(vsom, po, D):
    """A 20 x 20 map the online step has clustered (the recipe of test_tensor_core_tiers_and_long_rows), rows from the same
    clusters, and the oracle's answers for every row."""
    W, H = ROW_MAP
    rng = np.random.default_rng(W * D)
    centres = (rng.standard_normal((12, D)) * 2).astype(F32)
    data = lambda k: (centres[rng.integers(0, 12, k)] + 0.4 * rng.standard_normal((k, D))).astype(F32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=(rng.integers(-1000, 1000, (W * H, D)) / 1000).astype(F32))
    for sg, eta in ((W / 3.0, 0.4), (W / 8.0, 0.2), (2.0, 0.1)):
        ctx.train_chunk(data(1500), eta, sg, vsom.EXPONENTIAL)
    st = ctx.download_state()
    ctx.close()
    hits = rng.integers(0, 4, W * H).astype(np.uint64)
    q = data(ROW_N)
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.set_state(mean=st["mean"], hits=hits)
    ob, od = o.find_bmu(q)
    orb = o.find_restricted_bmu(q, 2)
    return st["mean"], hits, centres, q, ob, od, orb


def _score_all_forms(vsom, ctx, q, min_hits, eb, ed, what):
    """find_bmu_batch, find_bmu and find_bmu_batch_device on the same rows, each against the exact scan; returns the batch
    call's (bmu, dist, fallback rows, tier) and the device call's fallback rows and tier."""
    import torch

    n = len(q)
    tb, td, fb = ctx.find_bmu_batch(q, min_hits=min_hits)
    tier = ctx.last_score_tc
    assert_bit_equal(tb, eb, f"{what}: find_bmu_batch bmu vs exact scan")
    assert_bit_equal(td, ed, f"{what}: find_bmu_batch dist vs exact scan")
    hb, hd = ctx.find_bmu(q, min_hits=min_hits)
    assert ctx.last_score_tc == tier, f"{what}: find_bmu ran tier {ctx.last_score_tc}, find_bmu_batch {tier}"
    assert_bit_equal(hb, eb, f"{what}: find_bmu bmu vs exact scan")
    assert_bit_equal(hd, ed, f"{what}: find_bmu dist vs exact scan")
    xd = torch.from_numpy(np.ascontiguousarray(q)).cuda()
    gb = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    gd = torch.full((n,), -1, dtype=torch.int32, device="cuda").view(torch.float32)
    fbd = ctx.find_bmu_batch_device(xd, n, gb, gd, min_hits=min_hits)
    ctx.synchronize()
    tierd = ctx.last_score_tc
    assert_bit_equal(gb.cpu().numpy().view(np.uint32), eb, f"{what}: device bmu vs exact scan")
    assert_bit_equal(gd.cpu().numpy(), ed, f"{what}: device dist vs exact scan")
    assert fb <= n and fbd <= n
    return tb, td, fb, tier, fbd, tierd


@pytest.mark.parametrize("tier", ["1", "2", "auto"])
@pytest.mark.parametrize("D", ROW_LENGTHS)
def test_tensor_core_row_lengths(vsom, po, monkeypatch, D, tier):
    """K2 at row lengths either side of the resident-A limit (Kpad <= 320: D = 317 / 318 in tier 1, 105 / 106 in tier 2), at
    1000 and at the largest supported 2047 / 2048 (tier 2 runs K = 6147 there), host and device forms, global and restricted
    search, against the exact scan and the oracle on every row."""
    _tc_tier(monkeypatch, tier)
    mean, hits, _, q, ob, od, orb = _row_length_case(vsom, po, D)
    W, H = ROW_MAP
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean, hits=hits)
    eb, ed = ctx.find_bmu_exact(q)
    assert ctx.last_score_tc == 0
    assert_bit_equal(eb, ob, "exact scan bmu vs oracle")
    assert_bit_equal(ed, od, "exact scan dist vs oracle")
    tb, td, fb, ran, fbd, rand = _score_all_forms(vsom, ctx, q, 0, eb, ed, f"D={D} tier {tier}")
    print(f"D={D} tier {tier}: ran tier {ran} (device {rand}), {fb} / {fbd} of {len(q)} rows took the exact scan")
    assert ran == rand and ran == (int(tier) if tier != "auto" else ran) and ran in (1, 2)
    assert fb < len(q)
    assert_bit_equal(tb, ob, "K2 bmu vs oracle")
    assert_bit_equal(td, od, "K2 dist vs oracle")
    rb, rd = ctx.find_bmu_exact(q, min_hits=2)
    assert_bit_equal(rb, orb, "restricted exact scan vs oracle")
    _score_all_forms(vsom, ctx, q, 2, rb, rd, f"D={D} tier {tier}, min_hits 2")
    ctx.close()


def test_tensor_core_rejects_rows_longer_than_2048(vsom, po):
    """D = 2049 is past K2's limit: every scoring call runs the exact scan, and says so."""
    import torch

    W, H, D, n = 12, 10, 2049, 1100
    rng = np.random.default_rng(D)
    m = rng.standard_normal((W * H, D)).astype(F32)
    q = (m[rng.integers(0, W * H, n)] + 0.5 * rng.standard_normal((n, D))).astype(F32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=m)
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.set_state(mean=m)
    ob, od = o.find_bmu(q)
    tb, td, fb = ctx.find_bmu_batch(q)
    assert ctx.last_score_tc == 0 and fb == n
    assert_bit_equal(tb, ob, "bmu")
    assert_bit_equal(td, od, "dist")
    xd = torch.from_numpy(q).cuda()
    gb = torch.empty(n, dtype=torch.int32, device="cuda")
    gd = torch.empty(n, dtype=torch.float32, device="cuda")
    fbd = ctx.find_bmu_batch_device(xd, n, gb, gd)
    ctx.synchronize()
    assert ctx.last_score_tc == 0 and fbd == n
    assert_bit_equal(gb.cpu().numpy().view(np.uint32), ob, "device bmu")
    assert_bit_equal(gd.cpu().numpy(), od, "device dist")
    ctx.close()


def test_tensor_core_device_call_splits_at_the_shape_slab_cap(vsom, po, monkeypatch):
    """D = 2048 in tier 2: a slab holds at most 217 856 rows, so 2 x 217 856 + 129 rows run as three slabs with no knob set.
    Every row equals the exact scan, and the rows on each side of both slab boundaries equal the oracle."""
    import torch

    monkeypatch.setenv("VSOM_TC_TIER", "2")
    monkeypatch.delenv("VSOM_TC_SLAB_LOG2", raising=False)
    D = 2048
    cap = tc_slab_cap(D, True)
    assert cap == 217856
    n = 2 * cap + 129
    mean, hits, centres, _, _, _, _ = _row_length_case(vsom, po, D)
    W, H = ROW_MAP
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean, hits=hits)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2048)
    xd = torch.randn((n, D), generator=gen, device="cuda").mul_(0.4)
    xd += torch.from_numpy(centres).cuda()[torch.randint(0, len(centres), (n,), generator=gen, device="cuda")]
    tb = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    td = torch.full((n,), -1, dtype=torch.int32, device="cuda").view(torch.float32)
    fb = ctx.find_bmu_batch_device(xd, n, tb, td)
    ctx.synchronize()
    assert ctx.last_score_tc == 2 and fb < n
    eb = torch.empty(n, dtype=torch.int32, device="cuda")
    ed = torch.empty(n, dtype=torch.float32, device="cuda")
    ctx.find_bmu_exact_device(xd, n, eb, ed)
    ctx.synchronize()
    print(f"{n} rows in three slabs of <= {cap}: {fb} took the exact scan")
    tb, td, eb, ed = (t.cpu().numpy() for t in (tb, td, eb, ed))
    assert_bit_equal(tb, eb, "bmu vs exact scan")
    assert_bit_equal(td, ed, "dist vs exact scan")
    edges = np.r_[0:3, cap - 3:cap + 3, 2 * cap - 3:2 * cap + 3, n - 3:n]
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.set_state(mean=mean, hits=hits)
    ob, od = o.find_bmu(xd[torch.from_numpy(edges).cuda()].cpu().numpy())
    assert_bit_equal(tb[edges].view(np.uint32), ob, "bmu at the slab boundaries vs oracle")
    assert_bit_equal(td[edges], od, "dist at the slab boundaries vs oracle")
    ctx.close()


# ------------------------------------------------------------------------------------------------ B.2: config-5 map scoring
def test_config5_map_scoring(vsom, po):
    """Scoring on a clustered 512 x 512 x 784 map (262 144 nodes): 20 000 rows through the device and the host form, every row
    against the exact scan and the first 64 against the oracle; evaluate; the restricted search with min_hits = 2."""
    import torch

    W, H, D, n, k = 512, 512, 784, 20000, 64
    rng = np.random.default_rng(4242)
    centres = (rng.standard_normal((32, D)) * 2).astype(F32)
    mean = centres[rng.integers(0, 32, W * H)]
    mean += (0.3 * rng.standard_normal((W * H, D), dtype=F32)).astype(F32)
    hits = rng.integers(0, 4, W * H).astype(np.uint64)
    q = (centres[rng.integers(0, 32, n)] + 0.4 * rng.standard_normal((n, D), dtype=F32)).astype(F32)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean, hits=hits)
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.set_state(mean=mean, hits=hits)
    del mean
    ob, od = o.find_bmu(q[:k])
    eb, ed = ctx.find_bmu_exact(q)
    assert_bit_equal(eb[:k], ob, "exact scan bmu vs oracle")
    assert_bit_equal(ed[:k], od, "exact scan dist vs oracle")

    xd = torch.from_numpy(q).cuda()
    gb = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    gd = torch.full((n,), -1, dtype=torch.int32, device="cuda").view(torch.float32)
    fb = ctx.find_bmu_batch_device(xd, n, gb, gd)
    ctx.synchronize()
    print(f"config 5 map: tier {ctx.last_score_tc}, {fb} of {n} rows took the exact scan")
    assert ctx.last_score_tc in (1, 2, 3)
    gb, gd = gb.cpu().numpy().view(np.uint32), gd.cpu().numpy()
    assert_bit_equal(gb, eb, "device bmu vs exact scan")
    assert_bit_equal(gd, ed, "device dist vs exact scan")
    hb, hd = ctx.find_bmu(q)
    assert ctx.last_score_tc
    assert_bit_equal(hb, eb, "host bmu vs exact scan")
    assert_bit_equal(hd, ed, "host dist vs exact scan")

    assert ctx.evaluate(q[:k]) == o.evaluate(q[:k])
    err = 0.0
    for i, d in enumerate(ed):  # Som::evaluate's running mean, in row order
        err += 1.0 / (i + 1.0) * (float(d) - err)
    assert ctx.evaluate(q) == err and ctx.last_score_tc

    orb = o.find_restricted_bmu(q[:k], 2)
    rb, rd = ctx.find_bmu_exact(q, min_hits=2)
    assert_bit_equal(rb[:k], orb, "restricted exact scan vs oracle")
    tb, td, _ = ctx.find_bmu_batch(q, min_hits=2)
    assert ctx.last_score_tc
    assert_bit_equal(tb, rb, "restricted K2 bmu vs exact scan")
    assert_bit_equal(td, rd, "restricted K2 dist vs exact scan")
    ctx.close()


# ------------------------------------------------------------------------------------------------ B.3: row counts
ROW_COUNTS = [1023, 1024, PROBE - 1, PROBE, PROBE + 1, 2 * PROBE, 2 * PROBE + 1, 2 * PROBE + 2]


@functools.lru_cache(maxsize=None)
def _row_count_map(vsom, kind):
    """'trained': bench's scoring map (128 x 128 x 256, random init, 20 000 online steps, sigma 32 -> 2) and bench's scoring rows;
    the tier-1 probe sends it to tier 2.  'coincident': nodes within 1e-4 of one point, hopeless for either tier."""
    if kind == "trained":
        W, H, D = 128, 128, 256
        ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
        ctx.upload_state(mean=init_map(W * H, D, 43))
        centres = (np.random.default_rng(1234 + 4).standard_normal((64, D)) * 3).astype(F32)
        rng = np.random.default_rng(1234 + 40)
        warm = (rng.standard_normal((20000, D), dtype=F32) + centres[rng.integers(0, 64, 20000)]).astype(F32)
        for i, (sg, eta) in enumerate(((32.0, 0.5), (16.0, 0.3), (8.0, 0.2), (4.0, 0.1), (2.0, 0.05))):
            ctx.train_chunk(warm[4000 * i:4000 * (i + 1)], eta, sg, vsom.EXPONENTIAL)
        mean = ctx.download_state()["mean"]
        ctx.close()
        x = synth_chunk(ROW_COUNTS[-1], D, 1234 + 4)
    else:
        W, H, D = 20, 20, 96
        rng = np.random.default_rng(77)
        base = rng.standard_normal(D).astype(F32)
        mean = (base[None, :] + 1e-4 * rng.standard_normal((W * H, D))).astype(F32)
        x = (base[None, :] + rng.standard_normal((ROW_COUNTS[-1], D))).astype(F32)
    return W, H, D, mean, x


@pytest.mark.parametrize("n", ROW_COUNTS)
@pytest.mark.parametrize("kind", ["trained", "coincident"])
def test_scoring_dispatch_and_probe_row_counts(vsom, po, kind, n):
    """Batch sizes either side of 1024 (K3 / K2), of the first probe's 8192 rows and of the second probe, which starts only when
    more than 8192 rows follow the first: on the coincident map it sends the rest to the exact scan (tier 3), one row at
    16 385.  Host and device forms; every row equals the exact scan, the first and last rows equal the oracle."""
    W, H, D, mean, xall = _row_count_map(vsom, kind)
    x = xall[:n]
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean)
    eb, ed = ctx.find_bmu_exact(x)
    tb, td, fb, tier, fbd, tierd = _score_all_forms(vsom, ctx, x, 0, eb, ed, f"{kind}, {n} rows")
    print(f"{kind}, {n} rows: tier {tier} (device {tierd}), {fb} / {fbd} rows took the exact scan")
    if n < TC_MIN_ROWS:
        want = 0
    elif kind == "trained":
        want = 2
    else:
        want = 3 if n > 2 * PROBE else 2
    assert tier == want and tierd == want
    if want == 0:
        assert fb == n and fbd == n
    if want == 3:
        assert fb >= n - 2 * PROBE and fbd >= n - 2 * PROBE
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.set_state(mean=mean)
    rows = np.r_[0:16, PROBE - 2:min(n, PROBE + 2), n - 16:n]
    rows = np.unique(rows[rows < n])
    ob, od = o.find_bmu(x[rows])
    assert_bit_equal(tb[rows], ob, "bmu vs oracle")
    assert_bit_equal(td[rows], od, "dist vs oracle")
    ctx.close()


# ------------------------------------------------------------------------------------------------ B.4: min_hits extremes, tiny grids
BIG = 1 << 32
HITS_CASES = [("node0_only", 2), ("far_corner", 2), ("above_2^32", 2), ("above_2^32", BIG), ("above_2^32", BIG + 1)]


def _hits(case, rng, N):
    if case == "node0_only":
        h = rng.integers(0, 2, N).astype(np.uint64)
        h[0] = 3
    elif case == "far_corner":  # besides node 0 (always the seed), only the last node is eligible
        h = rng.integers(0, 2, N).astype(np.uint64)
        h[0], h[N - 1] = 0, 7
    else:  # hit counts whose low 32 bits alone would rank them differently
        h = rng.choice(np.array([0, 1, 2, BIG - 1, BIG, BIG + 1, 3 * BIG + 2], np.uint64), N)
    return h


@pytest.mark.parametrize("tier", ["1", "2", "auto"])
@pytest.mark.parametrize("case,min_hits", HITS_CASES, ids=[f"{c}-{m}" for c, m in HITS_CASES])
def test_restricted_search_hit_extremes(vsom, po, monkeypatch, case, min_hits, tier):
    """Restricted K2 with one eligible node, with one eligible far corner, and with 64-bit hit counts and thresholds at and
    above 2^32 (a 32-bit hit count or threshold anywhere in the map operand, the rescore, K3 or the fallback scan would change
    which nodes are eligible).  Host and device forms against the oracle on every row."""
    _tc_tier(monkeypatch, tier)
    W, H, D, n = 24, 20, 48, 2048
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    centres = (rng.standard_normal((12, D)) * 2).astype(F32)
    mean = (centres[rng.integers(0, 12, W * H)] + 0.3 * rng.standard_normal((W * H, D))).astype(F32)
    q = (centres[rng.integers(0, 12, n)] + 0.4 * rng.standard_normal((n, D))).astype(F32)
    q[::97] = mean[W * H - 1] + F32(0.01)  # rows next to the far corner
    hits = _hits(case, rng, W * H)
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.set_state(mean=mean, hits=hits)
    orb = o.find_restricted_bmu(q, min_hits)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean, hits=hits)
    rb, rd = ctx.find_bmu_exact(q, min_hits=min_hits)
    assert_bit_equal(rb, orb, "exact scan vs oracle")
    tb, _, fb, ran, _, _ = _score_all_forms(vsom, ctx, q, min_hits, rb, rd, f"{case}, min_hits {min_hits}")
    print(f"{case}, min_hits {min_hits}, tier {tier}: ran tier {ran}, {fb} of {n} rows took the exact scan; "
          f"{len(np.unique(orb))} distinct BMUs")
    assert ran in (1, 2, 3)
    if case == "node0_only":
        assert (orb == 0).all()
    if case == "far_corner":
        assert set(np.unique(orb).tolist()) == {0, W * H - 1}
    ctx.close()


@pytest.mark.parametrize("W,H", [(1, 1), (1, 37), (37, 1)])
def test_tensor_core_tiny_grids(vsom, po, W, H):
    """One node, one column and one row of nodes, 1100 rows (K2 territory): host and device forms, global and restricted, against
    the oracle on every row."""
    D, n = 16, 1100
    rng = np.random.default_rng(W * 100 + H)
    mean = rng.standard_normal((W * H, D)).astype(F32)
    q = (mean[rng.integers(0, W * H, n)] + 0.5 * rng.standard_normal((n, D))).astype(F32)
    hits = rng.integers(0, 3, W * H).astype(np.uint64)
    o = po.Oracle(W, H, D, po.STANDARD, po.ORDER_EIGEN_SSE)
    o.set_state(mean=mean, hits=hits)
    ob, od = o.find_bmu(q)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean, hits=hits)
    _, _, fb, ran, _, _ = _score_all_forms(vsom, ctx, q, 0, ob, od, f"{W}x{H}")
    print(f"{W}x{H}: tier {ran}, {fb} of {n} rows took the exact scan")
    assert ran in (1, 2, 3)
    orb = o.find_restricted_bmu(q, 1)
    rb, rd = ctx.find_bmu_exact(q, min_hits=1)
    assert_bit_equal(rb, orb, "restricted exact scan vs oracle")
    _score_all_forms(vsom, ctx, q, 1, rb, rd, f"{W}x{H}, min_hits 1")
    ctx.close()
