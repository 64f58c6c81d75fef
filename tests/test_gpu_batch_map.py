"""K6, the batch-map trainer (vsom_batch_epoch), against the CPU oracle at the shape bench.py measures and across the launch
configurations launch_batch_epoch chooses on the host.

Phase B's launch shape depends on the map and the row length: chains per thread (cpt 4..8 for Standard / Median, 2..4 for
CLR), neurons per CTA (G <= 8, with a partly filled last CTA), rows per shared-memory batch (R = 32 down to 4) and whether the
neighbourhood table fits in shared memory (<= 4096 entries) or is read from global memory.  Phase A is K2 (tensor-core search,
tiers 1 to 3) or the exact scan on a first epoch, and the local walk from last_bmu[row] afterwards.  The helper k6_launch
restates the host-side choice, and every case asserts that it lands on the configuration it claims to cover; phase A's path is
read back through last_score_tc.

Contract (DESIGN.md section 2): mean, S, sigma, weight and hits bit-identical, NaN positions identical (NaN payload and sign
are not compared), the MSE bit-identical and the returned last_bmu equal.  A shape the trainer refuses returns
VSOM_ERR_UNSUPPORTED and changes nothing.

The oracle dominates the cost.  Each case's oracle trajectory runs once, on a thread pool (ctypes releases the GIL), and
the trajectories of the selected tests are queued when the module starts, so the heavy ones run while the light ones are
checked."""
import collections
import concurrent.futures
import ctypes as C
import functools
import os
import threading

import numpy as np
import pytest

from conftest import assert_bit_equal

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

F32 = np.float32
STD, MED, CLR = 0, 1, 2
ORDERS = pytest.mark.parametrize("order", [2, 0], ids=["eigen_sse", "seq"])
VSOM_ERR_INVALID, VSOM_ERR_UNSUPPORTED = -1, -3
TC_MIN_ROWS = 1024  # smallest first epoch whose BMU search goes through K2 (score_tc.cu kTcMinRows)


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


def batch_leg_rows(n, d, seed):
    """bench.py's batch-map rows: integer pixel-like values in [0, 256)."""
    return np.floor(256 * np.random.default_rng(seed).random((n, d), dtype=F32) ** 2).astype(F32)


def small_rows(rng, n, Din, tr):
    if tr == CLR:
        z = rng.standard_normal((n, 1)).astype(F32)
        a = rng.uniform(0.5, 1.5, (1, Din)).astype(F32)
        return (a * z + 0.1 * rng.standard_normal((n, Din))).astype(F32)
    return rng.standard_normal((n, Din)).astype(F32)


def model_length(Din, tr):
    return Din * (Din - 1) if tr == CLR else Din


# ------------------------------------------------------------------------------------------------ K6's launch shape
def k6_launch(W, H, Din, tr, sms):
    """launch_batch_epoch's host-side choice (batch_map.cu), restated: None when the call is refused, else cpt (chains per
    thread), T (threads per neuron), G (neurons per CTA), last (neurons in the last CTA), R (rows per batch), lut (entries
    of the neighbourhood table over the reference's coordinates, whose y divides by the map height) and lut_smem."""
    Dm = model_length(Din, tr)
    Dq = Dm // 2 if tr == CLR else Dm
    lo, hi = (2, 4) if tr == CLR else (4, 8)
    best = None
    for c in range(lo, hi + 1):  # fewest wasted lanes once T is rounded up to whole warps; ties go to more chains per thread
        t = (-(-Dq // c) + 31) // 32 * 32
        if t <= 736 and (best is None or t * c <= best[0]):
            best = (t * c, c, t)
    if best is None:
        return None
    _, cpt, T = best
    N = W * H
    G, best_rounds = 1, None
    for g in range(1, max(1, min(8, 736 // T)) + 1):  # fewest rounds over the SMs; ties go to more neurons per CTA
        rounds = -(-(-(-N // g)) // sms) * g
        if best_rounds is None or rounds <= best_rounds:
            best_rounds, G = rounds, g
    R = max(4, min(32, (25600 // Din) & ~3))
    if 8 * R * Din > 208 * 1024:
        return None
    my = ((N - 1) - (N - 1) % W) // H
    lut = W * (my + 1)
    return dict(cpt=cpt, T=T, G=G, last=N - (-(-N // G) - 1) * G, R=R, lut=lut, lut_smem=lut <= 4096)


@functools.lru_cache(maxsize=None)
def sm_count():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


G_SIDES_148 = [6, 13, 19, 23, 26, 29, 31, 33]  # square Dm = 8 maps that give G = 1..8 on 148 SMs, partial last CTA for G >= 2


@functools.lru_cache(maxsize=None)
def g_sweep_sides(sms):
    """For G = 1..8, a square Dm = 8 map on which K6 runs G neurons per CTA, with fewer than G in the last CTA when G >= 2."""
    if sms == 148:
        return tuple(G_SIDES_148)
    sides = {}
    for s in range(1, 400):
        c = k6_launch(s, s, 8, STD, sms)
        if c["G"] not in sides and (c["G"] == 1 or c["last"] < c["G"]):
            sides[c["G"]] = s
    return tuple(sides.get(g) for g in range(1, 9))


# ------------------------------------------------------------------------------------------------ comparison
def assert_same(got, want, what):
    """NaN pattern identical, every other value bit for bit."""
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


def assert_state_same(got, want, what):
    for k in ("mean", "S", "sigma", "weight", "hits"):
        assert_same(got[k], want[k], f"{what}: {k}")


# ------------------------------------------------------------------------------------------------ cases and oracle trajectories
# steps: ("epoch", x, sigma, is_first, last_bmu) with last_bmu None (zeros), an array, or "prev" (the previous epoch's
# returned last_bmu); ("score", x) is a find_bmu_batch call on the map as it stands.
Case = collections.namedtuple("Case", "W H Din tr order init steps")


def full_state(N, Dm, mean, hits=None):
    return dict(mean=mean, S=np.zeros((N, Dm), F32), sigma=np.zeros((N, Dm), F32), weight=np.zeros(N, F32),
                hits=np.zeros(N, np.uint64) if hits is None else hits)


def oracle_trajectory(po, case):
    o = po.Oracle(case.W, case.H, case.Din, case.tr, case.order)
    o.set_state(**case.init)
    out, prev = [], None
    for step in case.steps:
        with np.errstate(all="ignore"):
            if step[0] == "score":
                out.append(o.find_bmu(step[1]))
                continue
            _, x, sigma, first, last = step
            mse, prev = o.batch_epoch(x, sigma, first, prev if isinstance(last, str) else last)
        out.append((mse, prev, o.get_state()))
    return out


def case_small(po, W, H, Din, tr, order, n, seed):
    """A random map and n rows; a first epoch at sigma 2.5, then a local-walk epoch at sigma 1.5 from the first epoch's BMUs."""
    rng = np.random.default_rng(seed)
    Dm = model_length(Din, tr)
    x = small_rows(rng, n, Din, tr)
    init = full_state(W * H, Dm, init_map(W * H, Dm, seed), rng.integers(0, 3, W * H).astype(np.uint64))
    return Case(W, H, Din, tr, order, init, [("epoch", x, 2.5, True, None), ("epoch", x, 1.5, False, "prev")])


def case_rows_per_batch(po, Din, R, order):
    """5 x 3 Standard, one context: n = 1100 (>= 1024: K2 up to Dm = 2048, else the exact scan), R - 1, R, R + 1 and 3R + 1 rows,
    alternating first epochs and local walks from random start nodes."""
    W, H = 5, 3
    rng = np.random.default_rng(Din)
    steps = []
    for i, n in enumerate((1100, R - 1, R, R + 1, 3 * R + 1)):
        x = small_rows(rng, n, Din, STD)
        steps.append(("epoch", x, 2.0, i % 2 == 0, None if i % 2 == 0 else rng.integers(0, W * H, n).astype(np.uint64)))
    return Case(W, H, Din, STD, order, full_state(W * H, Din, init_map(W * H, Din, Din)), steps)


def case_lut(po, W, H, Din, n, epochs, order):
    """A random map; a first epoch, then local walks from node 0, then walks from the previous BMUs; sigma 4, 3, 2."""
    rng = np.random.default_rng(W * 1000 + H)
    x = small_rows(rng, n, Din, STD)
    steps = [("epoch", x, 4.0, True, None), ("epoch", x, 3.0, False, None), ("epoch", x, 2.0, False, "prev")][:epochs]
    return Case(W, H, Din, STD, order, full_state(W * H, Din, init_map(W * H, Din, W + H)), steps)


def case_dispatch(po, order):
    """64 x 64 x 128: a first epoch over 1024 rows (K2), then one over 1023 rows (the exact scan)."""
    W, H, D = 64, 64, 128
    x = synth_chunk(2047, D, 64)
    steps = [("epoch", x[:1024], 3.0, True, None), ("epoch", x[1024:], 3.0, True, None)]
    return Case(W, H, D, STD, order, full_state(W * H, D, init_map(W * H, D, 42)), steps)


_TRAINED_LOCK = threading.Lock()


@functools.lru_cache(maxsize=None)
def _bench_scoring_map():
    """bench.py's scoring map (score_map_state): 128 x 128 x 256, init_map(.., 43), 20 000 online steps with sigma 32 -> 2 on the
    scoring distribution, trained on the device (the online step is bit-exact against the oracle, and the oracle would take
    minutes for it); plus the cluster centres of its rows."""
    import importlib

    vsom = importlib.import_module("variational-self-organizing-maps_b200")
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
    return mean


def case_hard(po, kind, order):
    """'coincident': nodes within 1e-4 of one point, 16 385 rows: K2's tier-1 probe, its tier-2 probe and a one-row exact-scan
    remainder (tier 3).  'trained': bench's scoring map and 9000 of bench's scoring rows: the tier-1 probe (8192 rows) sends the
    other 808 to tier 2.  A 32 x 32 x 64 map trained the same way stays in tier 1 (its nodes are far enough apart for one fp16
    value per element), so the smaller map does not cover tier 2."""
    if kind == "coincident":
        W, H, D, n = 20, 20, 96, 16385
        rng = np.random.default_rng(77)
        base = rng.standard_normal(D).astype(F32)
        mean = (base[None, :] + 1e-4 * rng.standard_normal((W * H, D))).astype(F32)
        x = (base[None, :] + rng.standard_normal((n, D))).astype(F32)
    else:
        W, H, D = 128, 128, 256
        with _TRAINED_LOCK:
            mean = _bench_scoring_map()
        x = synth_chunk(9000, D, 1234 + 4)
    return Case(W, H, D, STD, order, full_state(W * H, D, mean), [("epoch", x, 3.0, True, None)])


def smooth_map(W, H, rng, noise=0.02):
    """Dm = 6 models that vary smoothly over the grid (index = y W + x), so that the local walks travel."""
    px, py = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    feats = lambda u, v: np.stack([u, v, 0.1 * u * v, np.sin(0.7 * u), np.cos(0.5 * v), 0.05 * (u - v) ** 2], axis=-1)
    mean = feats(px.ravel(), py.ravel()) + noise * rng.standard_normal((W * H, 6))
    return mean.astype(F32), feats


def case_walk(po, W, H, order):
    """A smooth W x H map; four rows per start node, every node a start; a walk epoch from those starts, then one from the
    BMUs the first returned."""
    rng = np.random.default_rng(W * 100 + H)
    mean, feats = smooth_map(W, H, rng)
    N, reps = W * H, 4
    u, v = rng.uniform(0, W - 1, N * reps), rng.uniform(0, H - 1, N * reps)
    x = (feats(u, v) + 0.05 * rng.standard_normal((N * reps, 6))).astype(F32)
    starts = np.tile(np.arange(N, dtype=np.uint64), reps)
    rng.shuffle(starts)
    return Case(W, H, 6, STD, order, full_state(N, 6, mean), [("epoch", x, 1.5, False, starts), ("epoch", x, 1.2, False, "prev")])


def case_column0(po, order):
    """9 x 7 smooth map, rows next to the right-edge nodes, every walk starting in column 0 of the same grid row: the
    reference's unsigned x - 1 clamps to column W - 1, so the first step can land on the right edge."""
    W, H = 9, 7
    rng = np.random.default_rng(907)
    mean, _ = smooth_map(W, H, rng)
    rows = np.repeat(np.arange(H), 5)
    x = (mean[rows * W + W - 1] + 0.01 * rng.standard_normal((len(rows), 6))).astype(F32)
    starts = (rows * W).astype(np.uint64)
    return Case(W, H, 6, STD, order, full_state(W * H, 6, mean), [("epoch", x, 1.5, False, starts)])


def case_share(po, order):
    """24 x 20 x 48 on one context: find_bmu_batch on 20 000 rows (K2 grows stage slots 6 and 7), a first epoch over 5000 rows
    (K2, then K6 puts its table and coordinates in the same slots), find_bmu_batch again, a first epoch over 3000 rows."""
    W, H, D = 24, 20, 48
    x = synth_chunk(20000, D, 2420)
    steps = [("score", x), ("epoch", x[:5000], 3.0, True, None), ("score", x), ("epoch", x[5000:8000], 2.0, True, None)]
    return Case(W, H, D, STD, order, full_state(W * H, D, init_map(W * H, D, 2420)), steps)


def case_bench(po, order):
    """bench.py's batch-map leg: 20 x 20 x 784 Standard, init_map(400, 784, 99), its pixel-like rows (seed 5), sigma 5: the first
    epoch (global search through K2), the steady-state epoch (walks from node 0, as bench calls it), then walks from the
    second epoch's BMUs.  60 000 rows in bench's default order, 20 000 in the sequential one."""
    W, H, D = 20, 20, 784
    x = batch_leg_rows(60000 if order == 2 else 20000, D, 5)
    steps = [("epoch", x, 5.0, True, None), ("epoch", x, 5.0, False, None), ("epoch", x, 5.0, False, "prev")]
    return Case(W, H, D, STD, order, full_state(W * H, D, init_map(W * H, D, 99)), steps)


def case_bench_median(po, order):
    """The benchmark shape with the Median transformation, 4096 rows: the first epoch runs K2 on a Median map."""
    W, H, D = 20, 20, 784
    x = synth_chunk(4096, D, 7)
    steps = [("epoch", x, 5.0, True, None), ("epoch", x, 5.0, False, "prev")]
    return Case(W, H, D, MED, order, full_state(W * H, D, init_map(W * H, D, 99)), steps)


CASES = dict(small=case_small, rsweep=case_rows_per_batch, lut=case_lut, dispatch=case_dispatch, hard=case_hard, walk=case_walk,
             column0=case_column0, share=case_share, bench=case_bench, bench_median=case_bench_median)
_POOL = concurrent.futures.ThreadPoolExecutor(max_workers=max(2, os.cpu_count() or 2))
_FUTURES = {}


def _build_and_run(po, key):
    case = CASES[key[0]](po, *key[1:])
    return case, oracle_trajectory(po, case)


def oracle_future(po, key):
    if key not in _FUTURES:
        _FUTURES[key] = _POOL.submit(_build_and_run, po, key)
    return _FUTURES[key]


def prefetch(keyfn):
    """Marks a test whose oracle trajectory is queued when the module starts: keyfn(params) -> case key."""
    def deco(f):
        f.oracle_key = keyfn
        return f
    return deco


@pytest.fixture(scope="module", autouse=True)
def _queue_oracle_trajectories(request, po):
    """Queues the trajectories of this module's selected tests, heaviest first, so they overlap the GPU work."""
    keys = []
    for item in request.session.items:
        fn = getattr(getattr(item, "function", None), "oracle_key", None)
        if fn is not None and item.module.__name__ == __name__:
            keys.append(fn(item.callspec.params if hasattr(item, "callspec") else {}))
    heavy = ("hard", "bench", "lut", "share", "bench_median", "dispatch")
    for key in sorted(keys, key=lambda k: heavy.index(k[0]) if k[0] in heavy else len(heavy)):
        oracle_future(po, key)
    yield
    _POOL.shutdown(wait=True, cancel_futures=True)


def run_case(vsom, po, key, what, check=None):
    """The case's steps on a fresh context, each compared with the oracle trajectory; check(i, ctx, gpu_last_bmu) runs after
    step i.  Returns the context (open) and the case."""
    case, want = oracle_future(po, key).result()
    _FUTURES.pop(key, None)
    ctx = vsom.VsomContext(case.W, case.H, case.Din, case.tr, case.order)
    ctx.upload_state(**case.init)
    prev = None
    for i, (step, w) in enumerate(zip(case.steps, want)):
        tag = f"{what}, step {i}"
        if step[0] == "score":
            gb, gd, fb = ctx.find_bmu_batch(step[1])
            print(f"{tag}: find_bmu_batch tier {ctx.last_score_tc}, {fb} of {len(step[1])} rows took the exact scan")
            assert_same(gb, w[0], f"{tag}: find_bmu_batch bmu")
            assert_same(gd, w[1], f"{tag}: find_bmu_batch dist")
            if check:
                check(i, ctx, None)
            continue
        _, x, sigma, first, last = step
        gm, gl = ctx.batch_epoch(x, sigma, first, prev if isinstance(last, str) else last)
        om, ol, ost = w
        tag += f" ({len(x)} rows, sigma {sigma}, {'first epoch' if first else 'local walks'})"
        assert_same(F32(gm), F32(om), f"{tag}: mse")
        assert_same(gl, ol, f"{tag}: last_bmu")
        assert_state_same(ctx.download_state(), ost, tag)
        if check:
            check(i, ctx, gl)
        prev = gl
    return ctx, case


def _expect_tier(i_k2, k2_tiers=(1, 2, 3)):
    """check(): after step i_k2 the first epoch ran K2 (tier in k2_tiers); after every other step last_score_tc is 0."""
    def check(i, ctx, _):
        tier = ctx.last_score_tc
        if i in i_k2:
            assert tier in k2_tiers, f"step {i}: phase A ran tier {tier}, expected K2 in {k2_tiers}"
        else:
            assert tier == 0, f"step {i}: phase A ran tier {tier}, expected the exact scan or the local walks"
    return check


# ------------------------------------------------------------------------------------------------ chains per thread
CPT_CASES = [(STD, 100, 4), (MED, 130, 5), (STD, 170, 6), (MED, 200, 7), (STD, 240, 8), (CLR, 9, 2), (CLR, 20, 3), (CLR, 32, 4), (CLR, 77, 4)]


@ORDERS
@pytest.mark.parametrize("tr,Din,cpt", CPT_CASES, ids=[f"{['std', 'median', 'clr'][t]}{d}-cpt{c}" for t, d, c in CPT_CASES])
@prefetch(lambda p: ("small", 5, 3, p["Din"], p["tr"], p["order"], 97, p["Din"] * 10 + p["tr"]))
def test_chains_per_thread(vsom, po, tr, Din, cpt, order):
    """Every batch_update_kernel instantiation: Standard / Median with 4..8 chains per thread, CLR with 2..4, and CLR at d_in = 77
    (P = 2926 chains on T = 736 threads, the longest model it accepts).  5 x 3 map, 97 rows (three full batches and one row)."""
    cfg = k6_launch(5, 3, Din, tr, sm_count())
    assert cfg["cpt"] == cpt and cfg["R"] == 32, cfg
    if Din == 77:
        assert cfg["T"] == 736
    ctx, _ = run_case(vsom, po, ("small", 5, 3, Din, tr, order, 97, Din * 10 + tr), f"cpt {cpt}, d_in {Din}", _expect_tier(()))
    ctx.close()


# ------------------------------------------------------------------------------------------------ rows per batch
R_CASES = [(801, 28), (1000, 24), (1600, 16), (2048, 12), (2049, 12), (3200, 8), (5888, 4)]


@ORDERS
@pytest.mark.parametrize("Din,R", R_CASES, ids=[f"d{d}-R{r}" for d, r in R_CASES])
@prefetch(lambda p: ("rsweep", p["Din"], p["R"], p["order"]))
def test_rows_per_batch(vsom, po, Din, R, order):
    """Rows longer than 800 values shrink the shared-memory row batches from 32 rows to R; batches of R - 1, R, R + 1 and 3R + 1
    rows and a first epoch over 1100 rows, up to the longest accepted Standard row (5888).  The 1100-row first epoch runs K2 up
    to Dm = 2048 and the exact scan from 2049."""
    cfg = k6_launch(5, 3, Din, STD, sm_count())
    assert cfg["R"] == R, cfg
    k2 = (0,) if Din <= 2048 else ()
    ctx, _ = run_case(vsom, po, ("rsweep", Din, R, order), f"d_in {Din}, R {R}", _expect_tier(k2))
    ctx.close()


# ------------------------------------------------------------------------------------------------ neurons per CTA
@ORDERS
@pytest.mark.parametrize("G", range(1, 9))
@prefetch(lambda p: ("small", g_sweep_sides(sm_count())[p["G"] - 1], g_sweep_sides(sm_count())[p["G"] - 1], 8, STD, p["order"], 150, p["G"]))
def test_neurons_per_cta(vsom, po, G, order):
    """Dm = 8 square maps on which phase B runs G = 1..8 neurons per CTA; for G >= 2 the last CTA holds fewer than G."""
    s = g_sweep_sides(sm_count())[G - 1]
    assert s is not None, f"no square map gives G = {G} on {sm_count()} SMs"
    cfg = k6_launch(s, s, 8, STD, sm_count())
    assert cfg["G"] == G and (G == 1 or cfg["last"] < G), cfg
    ctx, _ = run_case(vsom, po, ("small", s, s, 8, STD, order, 150, G), f"{s}x{s}, G {G} (last CTA {cfg['last']})", _expect_tier(()))
    ctx.close()


def test_neurons_per_cta_sweep_covers_every_g():
    sms = sm_count()
    sides = g_sweep_sides(sms)
    assert {k6_launch(s, s, 8, STD, sms)["G"] for s in sides if s} == set(range(1, 9)), (sms, sides)
    if sms == 148:
        assert list(sides) == G_SIDES_148


# ------------------------------------------------------------------------------------------------ neighbourhood table
LUT_CASES = [(65, 64, 8, 600, 2, 4160), (128, 32, 8, 600, 2, 16000), (128, 128, 16, 3000, 3, 16384), (64, 64, 8, 600, 2, 4096)]


@ORDERS
@pytest.mark.parametrize("W,H,Din,n,epochs,lut", LUT_CASES, ids=[f"{w}x{h}x{d}-lut{lut}" for w, h, d, _, _, lut in LUT_CASES])
@prefetch(lambda p: ("lut", p["W"], p["H"], p["Din"], p["n"], p["epochs"], p["order"]))
def test_neighbourhood_table_placement(vsom, po, W, H, Din, n, epochs, lut, order):
    """The neighbourhood table leaves shared memory above 4096 entries: 65 x 64 (4160), 128 x 32 (the reference's y divides by
    the height, so the table grows to 128 x 125 = 16 000) and 128 x 128 over three epochs read it from global memory;
    64 x 64 (exactly 4096) keeps it in shared memory."""
    cfg = k6_launch(W, H, Din, STD, sm_count())
    assert cfg["lut"] == lut and cfg["lut_smem"] == (lut <= 4096), cfg
    k2 = (0,) if n >= TC_MIN_ROWS else ()
    ctx, _ = run_case(vsom, po, ("lut", W, H, Din, n, epochs, order), f"{W}x{H}x{Din}, table {lut}", _expect_tier(k2))
    ctx.close()


# ------------------------------------------------------------------------------------------------ row counts
PIPE_ROWS = [1, 2, 31, 32, 33, 64, 65, 96, 97]


@ORDERS
@pytest.mark.parametrize("n", PIPE_ROWS)
@prefetch(lambda p: ("small", 12, 12, 8, STD, p["order"], p["n"], 1200 + p["n"]))
def test_row_counts_around_the_pipeline(vsom, po, n, order):
    """12 x 12 x 8 (R = 32): one to four batches, full and partial, through the double-buffered rows and coefficients and the
    three-slot ring of BMU coordinates."""
    assert k6_launch(12, 12, 8, STD, sm_count())["R"] == 32
    ctx, _ = run_case(vsom, po, ("small", 12, 12, 8, STD, order, n, 1200 + n), f"{n} rows", _expect_tier(()))
    ctx.close()


@ORDERS
@prefetch(lambda p: ("dispatch", p["order"]))
def test_first_epoch_dispatch_at_1024_rows(vsom, po, order):
    """64 x 64 x 128: a first epoch over 1024 rows runs K2, the next one over 1023 rows the exact scan, and last_score_tc says
    so each time."""
    ctx, _ = run_case(vsom, po, ("dispatch", order), "dispatch", _expect_tier((0,)))
    ctx.close()


# ------------------------------------------------------------------------------------------------ K2's probes inside an epoch
@ORDERS
@pytest.mark.parametrize("kind,tier", [("coincident", 3), ("trained", 2)])
@prefetch(lambda p: ("hard", p["kind"], p["order"]))
def test_first_epoch_through_k2_probes(vsom, po, kind, tier, order):
    """First epochs on maps where K2's probes change tier: nearly coincident nodes (tier 3: two probes, then a one-row exact
    scan) and bench's trained scoring map (tier 2)."""
    ctx, _ = run_case(vsom, po, ("hard", kind, order), kind, _expect_tier((0,), (tier,)))
    ctx.close()


# ------------------------------------------------------------------------------------------------ local walks
@ORDERS
@pytest.mark.parametrize("W,H", [(9, 7), (7, 9), (1, 37), (37, 1)])
@prefetch(lambda p: ("walk", p["W"], p["H"], p["order"]))
def test_local_walks_from_every_start_node(vsom, po, W, H, order):
    """Every node of 9 x 7, 7 x 9, 1 x 37 and 37 x 1 maps (where W - 1 or H - 1 is 0) as the start of four walks: the node each
    walk ends at, and the map after phase B."""
    def check(i, ctx, gl):
        if i == 0:
            moved = float(np.mean(gl != starts))
            print(f"{W}x{H}: {moved:.0%} of the walks left their start node")
            assert moved > 0.5

    starts = oracle_future(po, ("walk", W, H, order)).result()[0].steps[0][4]
    ctx, _ = run_case(vsom, po, ("walk", W, H, order), f"{W}x{H} walks", check)
    ctx.close()


@ORDERS
@prefetch(lambda p: ("column0", p["order"]))
def test_local_walks_from_column_0_wrap_to_the_right_edge(vsom, po, order):
    """Walks that start in column 0 look at column W - 1 (the reference's unsigned x - 1 clamps there): rows next to the right
    edge end there."""
    def check(i, ctx, gl):
        right = float(np.mean(gl % 9 == 8))
        print(f"{right:.0%} of the walks from column 0 ended in column 8")
        assert right > 0.5

    ctx, _ = run_case(vsom, po, ("column0", order), "walks from column 0", check)
    ctx.close()


def _raw_batch_epoch(vsom, ctx, x, sigma, first, last):
    """vsom_batch_epoch on the caller's own last_bmu array (the binding passes a copy)."""
    b = vsom.binding
    x = np.ascontiguousarray(x, dtype=F32)
    mse = C.c_float(0)
    return vsom.lib().vsom_batch_epoch(ctx._h, b._p(x, b._f32p), len(x), sigma, int(first), b._p(last, b._u64p), C.byref(mse))


@pytest.mark.parametrize("first", [True, False], ids=["first", "later"])
def test_last_bmu_out_of_range_is_refused(vsom, first):
    """A start node equal to N is refused with VSOM_ERR_INVALID, and nothing changes."""
    W, H, D, n = 9, 7, 6, 40
    rng = np.random.default_rng(63)
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(**full_state(W * H, D, init_map(W * H, D, 63), rng.integers(0, 5, W * H).astype(np.uint64)))
    before = ctx.download_state()
    last = rng.integers(0, W * H, n).astype(np.uint64)
    last[n // 2] = W * H
    keep = last.copy()
    assert _raw_batch_epoch(vsom, ctx, rng.standard_normal((n, D)), 2.0, first, last) == VSOM_ERR_INVALID
    assert_bit_equal(last, keep, "last_bmu")
    assert_state_same(ctx.download_state(), before, "after the refused call")
    ctx.close()


# ------------------------------------------------------------------------------------------------ stage slots shared with K2
@ORDERS
@prefetch(lambda p: ("share", p["order"]))
def test_stage_slots_shared_with_scoring(vsom, po, order):
    """K6 keeps its neighbourhood table and BMU coordinates in the stage slots that hold K2's fp16 map operand and row slab:
    scoring, an epoch, scoring again and a smaller epoch on one context each match the oracle."""
    ctx, _ = run_case(vsom, po, ("share", order), "shared stage slots", _expect_tier((0, 1, 2, 3)))
    ctx.close()


# ------------------------------------------------------------------------------------------------ refusals
@pytest.mark.parametrize("first", [True, False], ids=["first", "later"])
@pytest.mark.parametrize("tr,Din", [(STD, 5889), (CLR, 78)], ids=["std5889", "clr78"])
def test_refused_shape_leaves_state_alone(vsom, tr, Din, first):
    """Standard rows of 5889 values and CLR with d_in = 78 (P = 3003) exceed phase B's 736 threads per neuron.  vsom_create
    accepts both; vsom_batch_epoch returns VSOM_ERR_UNSUPPORTED before phase A, so the map, its hit counts and last_bmu stay
    as they were."""
    assert k6_launch(5, 3, Din, tr, sm_count()) is None
    W, H, n = 5, 3, 40
    rng = np.random.default_rng(Din)
    Dm = model_length(Din, tr)
    ctx = vsom.VsomContext(W, H, Din, tr, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(**full_state(W * H, Dm, init_map(W * H, Dm, Din), rng.integers(0, 5, W * H).astype(np.uint64)))
    before = ctx.download_state()
    last = rng.integers(0, W * H, n).astype(np.uint64)
    keep = last.copy()
    x = small_rows(rng, n, Din, tr)
    assert _raw_batch_epoch(vsom, ctx, x, 2.0, first, last) == VSOM_ERR_UNSUPPORTED
    assert_bit_equal(last, keep, "last_bmu")
    assert_state_same(ctx.download_state(), before, "after the refused call")
    with pytest.raises(vsom.VsomError) as e:
        ctx.batch_epoch(x, 2.0, first, last)
    assert e.value.code == VSOM_ERR_UNSUPPORTED and "batch-map trainer" in str(e.value)
    assert_state_same(ctx.download_state(), before, "after the second refused call")
    ctx.close()


# ------------------------------------------------------------------------------------------------ the benchmark leg
@ORDERS
@prefetch(lambda p: ("bench_median", p["order"]))
def test_benchmark_shape_median(vsom, po, order):
    """20 x 20 x 784 Median, 4096 rows: a first epoch through K2 on a Median map, then walks from its BMUs."""
    ctx, _ = run_case(vsom, po, ("bench_median", order), "20x20x784 Median", _expect_tier((0,)))
    ctx.close()


@ORDERS
@prefetch(lambda p: ("bench", p["order"]))
def test_benchmark_leg(vsom, po, order):
    """bench.py's batch-map leg, three epochs: the first (K2), the steady-state epoch bench times (walks from node 0) and one
    more from the second epoch's BMUs."""
    cfg = k6_launch(20, 20, 784, STD, sm_count())
    print(f"20x20x784 on {sm_count()} SMs: {cfg}")
    assert cfg["R"] == 32 and cfg["lut_smem"]
    ctx, _ = run_case(vsom, po, ("bench", order), "bench leg", _expect_tier((0,)))
    ctx.close()
