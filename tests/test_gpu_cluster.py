"""k-means over the map's nodes (vsom_cluster_nodes, VsomContext.cluster_nodes, Som::clusterNodes).

The oracle is a numpy restatement of the header's contract: splitmix64; the block sums and the group sums as Python loops over
blocks and groups, each summed sequentially from 0 (np.cumsum is a running sum), vectorised over components; the f32 distances as
a sequential acc = acc + (m[:, k] - c[k])**2 loop or, in the Eigen order, the restatement of tests/test_oracle_pin.py vectorised
over (centroid, node).  Every case must match it bit for bit: labels, centroids, weights, inertia, iterations and converged."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

from conftest import REPO, assert_bit_equal

F32, F64 = np.float32, np.float64
BLOCK = 1024  # VSOM_CLUSTER_BLOCK
UNIFORM, HITS = 0, 1
M64 = (1 << 64) - 1
CLUSTER_DRIVER = os.path.join(REPO, "tests", "cpp", "cluster_driver")
gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ numpy side of the contract
class Refused(Exception):
    pass


def splitmix_draws(seed, k):
    state, out = seed & M64, []
    for _ in range(k):
        state = (state + 0x9E3779B97F4A7C15) & M64
        z = state
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
        z ^= z >> 31
        out.append(float(z >> 11) * 2.0 ** -53)
    return out


def seq_sum(a):
    """Sequential f64 sum from 0 along axis 0 (vectorised over the other axes)."""
    a = np.asarray(a, F64)
    return np.cumsum(np.concatenate([np.zeros((1,) + a.shape[1:]), a]), axis=0)[-1]


def ordered_sum(term, n, eigen):
    """f32 sum of term(0) .. term(n-1) (arrays of one shape): sequentially from 0, or in Eigen's Packet4f redux order (the statement
    of test_oracle_pin.eigen_sse_sum_numpy, element-wise over the arrays)."""
    if not eigen or n < 4:
        s = term(0).copy() if eigen else np.zeros_like(term(0)) + term(0)
        for i in range(1, n):
            s = s + term(i)
        return s
    a2, a = n // 8 * 8, n // 4 * 4
    p0 = [term(i) for i in range(4)]
    if a > 4:
        p1 = [term(i) for i in range(4, 8)]
        for i in range(8, a2, 8):
            p0 = [p0[j] + term(i + j) for j in range(4)]
            p1 = [p1[j] + term(i + 4 + j) for j in range(4)]
        p0 = [p0[j] + p1[j] for j in range(4)]
        if a > a2:
            p0 = [p0[j] + term(a2 + j) for j in range(4)]
    s = (p0[0] + p0[2]) + (p0[1] + p0[3])
    for i in range(a, n):
        s = s + term(i)
    return s


def dists(mT, c32, eigen):
    """d(p, c_j) for the rows of m (mT = m.T, Dm x N, f32) and the f32 centroids c32 (k x Dm): (k, N) f32."""
    def term(i):
        r = mT[i][None, :] - c32[:, i][:, None]
        return r * r
    return ordered_sum(term, mT.shape[0], eigen)


def restate(m, hits, k, seed, weighting, max_iter, eigen, record=None):
    """The whole call: (labels int32, centroids, weight, inertia, iterations, converged); raises Refused where the call must fail.
    record (a list) gets, per update, the clusters with W_j = 0."""
    m = np.ascontiguousarray(m, F32)
    N, Dm = m.shape
    if not np.isfinite(m).all():
        raise Refused("non-finite")
    mT = np.ascontiguousarray(m.T)
    w = np.ones(N) if weighting == UNIFORM else hits.astype(F64)
    nb = -(-N // BLOCK)

    def block_sums(q):
        return [float(seq_sum(q[b * BLOCK:(b + 1) * BLOCK])) for b in range(nb)]

    # ---- seeding
    u = splitmix_draws(seed, k)
    cent = np.empty((k, Dm), F64)
    D = None
    for j in range(k):
        if j == 0:
            q = w.copy()
        else:
            d = dists(mT, cent[j - 1:j].astype(F32), eigen)[0]
            D = d if D is None else np.where(d < D, d, D)
            q = w * D.astype(F64)
        T = block_sums(q)
        total = float(seq_sum(T))
        if not (total > 0.0 and np.isfinite(total)):
            raise Refused("seeding total")
        target = u[j] * total
        run, blk, last = 0.0, None, None
        for b in range(nb):
            nxt = run + T[b]
            if nxt > target:
                blk = b
                break
            if T[b] > 0.0:
                last = (b, run)
            run = nxt
        if blk is None:
            blk, run = last
        node, lastq = None, None
        for p in range(blk * BLOCK, min(N, (blk + 1) * BLOCK)):
            run = run + float(q[p])
            if run > target:
                node = p
                break
            if q[p] > 0.0:
                lastq = p
        cent[j] = m[node if node is not None else lastq].astype(F64)

    # ---- Lloyd
    def assign(c):
        Dk = dists(mT, c.astype(F32), eigen)
        lab = np.argmin(Dk, axis=0)  # the first minimum: equal distances go to the lower j
        return lab, Dk[lab, np.arange(N)]

    def update(lab, c):
        c = c.copy()
        W = np.zeros(k)
        for j in range(k):
            mem = np.nonzero(lab == j)[0]
            num, wsum = [], []
            for g0 in range(0, len(mem), BLOCK):
                gm = mem[g0:g0 + BLOCK]
                num.append(seq_sum(w[gm][:, None] * m[gm].astype(F64)))
                wsum.append(float(seq_sum(w[gm])))
            W[j] = float(seq_sum(wsum))
            if W[j] != 0.0:
                c[j] = seq_sum(np.array(num).reshape(-1, Dm)) / W[j]
        return c, W

    it, prev = 0, None
    while True:
        it += 1
        lab, d = assign(cent)
        if it > 1 and np.array_equal(lab, prev):
            conv = True
            break
        if it == max_iter:
            conv = False
            break
        cent, W = update(lab, cent)
        if record is not None:
            record.append(np.nonzero(W == 0.0)[0].tolist())
        prev = lab
    _, W = update(lab, cent)
    inertia = float(seq_sum(block_sums(w * d.astype(F64))))
    return lab.astype(np.int32), cent, W, inertia, it, conv


# ------------------------------------------------------------------------------------------------ helpers
def blobs(N, Dm, centres, spread, scale, seed):
    """f32 rows around `centres` random centres: a map whose nodes fall into groups"""
    rng = np.random.default_rng(seed)
    c = rng.standard_normal((centres, Dm)) * scale
    return (c[rng.integers(0, centres, N)] + spread * rng.standard_normal((N, Dm))).astype(F32)


def make_ctx(vsom, W, H, d_in, transform, order, mean, hits=None):
    ctx = vsom.VsomContext(W, H, d_in, transform, order)
    ctx.upload_state(mean=mean, hits=hits)
    return ctx


def check_call(ctx, st, k, seed, weighting, max_iter, what):
    got = ctx.cluster_nodes(k, seed, weighting, max_iter)
    want = restate(st["mean"], st["hits"], k, seed, weighting, max_iter, ctx.order == 2)
    for g, e, name in zip(got[:3], want[:3], ("labels", "centroids", "weight")):
        assert_bit_equal(g, e, f"{what}: {name}")
    assert_bit_equal(np.float64(got[3]), np.float64(want[3]), f"{what}: inertia")
    assert (got[4], got[5]) == (want[4], want[5]), f"{what}: iterations / converged {got[4:]} vs {want[4:]}"
    return got


def assert_state_equal(a, b, what):
    for key in a:
        assert_bit_equal(b[key], a[key], f"{what}: {key}")


ORDERS = {"reference": 0, "lanes": 1, "eigen_sse": 2}


def _cases(vsom):
    """name -> (W, H, d_in, transform, state builder(ctx), [(k, weighting, max_iter, seed)])"""
    return {
        "20x20x784": (20, 20, 784, vsom.STANDARD, lambda: (blobs(400, 784, 12, 20.0, 60.0, 1), None), [(10, UNIFORM, 300, 3)]),
        "64x64x128_median_trained": (64, 64, 128, vsom.MEDIAN, "train", [(16, UNIFORM, 300, 5), (16, HITS, 300, 6)]),
        "50x50_clr_J32": (50, 50, 32, vsom.CLR, lambda: ((np.random.default_rng(4).standard_normal((2500, 992)) * 0.3).astype(F32), None), [(8, UNIFORM, 300, 7)]),
        "128x128x256": (128, 128, 256, vsom.STANDARD, lambda: (blobs(16384, 256, 80, 1.0, 3.0, 2), None), [(64, UNIFORM, 12, 9)]),
        "64x64_k2_groups": (64, 64, 8, vsom.STANDARD, lambda: (blobs(4096, 8, 3, 1.0, 2.0, 3), None), [(2, UNIFORM, 300, 1)]),
        "1x1_k1": (1, 1, 5, vsom.STANDARD, lambda: (np.arange(5, dtype=F32)[None, :], None), [(1, UNIFORM, 300, 0)]),
        "6x5_kN": (6, 5, 3, vsom.STANDARD, lambda: (np.random.default_rng(5).standard_normal((30, 3)).astype(F32), None), [(30, UNIFORM, 300, 2)]),
    }


def build_state(vsom, case, order):
    W, H, d_in, tr, builder, _ = case
    if builder == "train":
        rng = np.random.default_rng(11)
        ctx = vsom.VsomContext(W, H, d_in, tr, order)
        ctx.upload_state(mean=(rng.standard_normal((W * H, d_in)) * 0.1).astype(F32))
        x = blobs(6000, d_in, 20, 0.5, 2.0, 12)
        ctx.train_chunk(x, 0.1, 8.0)
        return ctx
    mean, hits = builder()
    return make_ctx(vsom, W, H, d_in, tr, order, mean, hits)


# ------------------------------------------------------------------------------------------------ restatement self-checks (CPU)
def test_restatement_eigen_order_matches_the_pin():
    """ordered_sum's Eigen order equals test_oracle_pin's statement for every length 1..41; splitmix64's first output for seed 0"""
    from test_oracle_pin import eigen_sse_sum_numpy

    rng = np.random.default_rng(1)
    for n in range(1, 42):
        t = (rng.standard_normal((5, n)) ** 2).astype(F32)
        got = ordered_sum(lambda i: t[:, i], n, True)
        for r in range(5):
            assert got[r] == eigen_sse_sum_numpy(t[r]), (n, r)
    # splitmix64 of state 0: first output 0xE220A8397B1DCDAF
    assert splitmix_draws(0, 1)[0] == float(0xE220A8397B1DCDAF >> 11) * 2.0 ** -53


# ------------------------------------------------------------------------------------------------ device against the restatement
@gpu
@pytest.mark.parametrize("order", list(ORDERS))
@pytest.mark.parametrize("name", ["20x20x784", "64x64x128_median_trained", "50x50_clr_J32", "128x128x256", "64x64_k2_groups", "1x1_k1", "6x5_kN"])
def test_bit_exact_against_restatement(vsom, name, order):
    case = _cases(vsom)[name]
    ctx = build_state(vsom, case, ORDERS[order])
    st = ctx.download_state()
    for k, weighting, max_iter, seed in case[5]:
        got = check_call(ctx, st, k, seed, weighting, max_iter, f"{name} k={k} weighting={weighting}")
        if name == "64x64_k2_groups":
            assert max(np.bincount(got[0])) > BLOCK, "a cluster must span several groups"
    assert_state_equal(st, ctx.download_state(), "state after a successful call")
    ctx.close()


@gpu
@pytest.mark.parametrize("order", ["reference", "eigen_sse"])
@pytest.mark.parametrize("name", ["20x20x784", "50x50_clr_J32", "64x64x128_median_trained"])
def test_assignment_identity(vsom, name, order):
    """The final labels and the distances summed into the inertia are find_bmu_exact's on a k-node Standard context holding
    f32(centroids)."""
    case = _cases(vsom)[name]
    ctx = build_state(vsom, case, ORDERS[order])
    st = ctx.download_state()
    k, weighting, max_iter, seed = case[5][-1]
    labels, cent, _, inertia, _, _ = ctx.cluster_nodes(k, seed, weighting, max_iter)
    ref = vsom.VsomContext(k, 1, ctx.Dm, vsom.STANDARD, ORDERS[order])
    ref.upload_state(mean=cent.astype(F32))
    bmu, dist = ref.find_bmu_exact(st["mean"])
    assert_bit_equal(labels.astype(np.uint32), bmu, "labels vs find_bmu_exact")
    w = np.ones(ctx.N) if weighting == UNIFORM else st["hits"].astype(F64)
    q = w * dist.astype(F64)
    want = seq_sum([float(seq_sum(q[b:b + BLOCK])) for b in range(0, ctx.N, BLOCK)])
    assert_bit_equal(np.float64(inertia), np.float64(want), "inertia from find_bmu_exact's distances")
    ref.close()
    ctx.close()


@gpu
@pytest.mark.parametrize("order", ["reference", "eigen_sse"])
def test_one_iteration_is_the_seeding(vsom, order):
    """max_iter = 1: the centroids are distinct node rows, the labels the assignment to them; repeated calls are identical."""
    W, H, D = 32, 32, 40
    mean = blobs(W * H, D, 25, 0.5, 4.0, 21)
    ctx = make_ctx(vsom, W, H, D, vsom.STANDARD, ORDERS[order], mean)
    st = ctx.download_state()
    a = check_call(ctx, st, 20, 77, UNIFORM, 1, "max_iter 1")
    assert a[4] == 1 and a[5] is False
    rows = {tuple(r) for r in mean.astype(F64)}
    assert all(tuple(c) in rows for c in a[1]), "a centroid is not a node row"
    assert len({tuple(c) for c in a[1]}) == 20, "seeds are distinct"
    ph = ctx.cluster_phases()
    assert ph["assignments"] == 1 and ph["update_ms"] == 0.0 and min(ph["seeding_ms"], ph["assign_ms"], ph["outputs_ms"]) > 0.0, ph
    b = ctx.cluster_nodes(20, 77, UNIFORM, 1)
    for x, y, what in zip(a[:3], b[:3], ("labels", "centroids", "weight")):
        assert_bit_equal(y, x, f"repeat: {what}")
    assert a[3:] == b[3:]
    ctx.close()


def zero_weight_map():
    """An 8 x 8 x 2 map with hits on six nodes"""
    rng = np.random.default_rng(9)
    mean = rng.standard_normal((64, 2)).astype(F32)
    hits = np.zeros(64, np.uint64)
    nodes = rng.choice(64, 6, replace=False)
    hits[nodes] = rng.integers(1, 20, 6)
    return mean, hits


# found by a search over map generators, k and seeds with restate(): in both orders an update meets a cluster without weight
ZERO_WEIGHT_SEED, ZERO_WEIGHT_K = 4, 3


@gpu
@pytest.mark.parametrize("order", ["reference", "eigen_sse"])
def test_hits_weighting(vsom, order):
    """Zero-hit nodes are never seeds and still get labels; the pinned seed has an update with a zero-weight cluster, which keeps its
    centroid, and the device matches the restatement through it."""
    mean, hits = zero_weight_map()
    ctx = make_ctx(vsom, 8, 8, 2, vsom.STANDARD, ORDERS[order], mean, hits)
    st = ctx.download_state()
    for seed in range(6):
        _, cent, _, _, _, _ = ctx.cluster_nodes(ZERO_WEIGHT_K, seed, HITS, 1)
        for c in cent:
            nodes = np.nonzero((mean.astype(F64) == c).all(1))[0]
            assert (hits[nodes] > 0).any(), f"seed {seed}: a zero-hit node was picked"
    record = []
    restate(mean, hits, ZERO_WEIGHT_K, ZERO_WEIGHT_SEED, HITS, 300, ORDERS[order] == 2, record)
    assert any(record), "the pinned case has no zero-weight cluster"
    got = check_call(ctx, st, ZERO_WEIGHT_K, ZERO_WEIGHT_SEED, HITS, 300, "pinned zero-weight case")
    ph = ctx.cluster_phases()
    assert ph["assignments"] == got[4] and ph["update_ms"] > 0.0, ph
    assert ((got[0] >= 0) & (got[0] < ZERO_WEIGHT_K)).all()
    ctx.close()


# ------------------------------------------------------------------------------------------------ refusals
def raw_call(vsom, ctx, k, seed, weighting, max_iter):
    """vsom_cluster_nodes with pre-filled outputs: (rc, outputs)"""
    L = vsom.lib()
    kk = max(k, 1)
    out = dict(labels=np.full(ctx.N, 7, np.int32), centroids=np.full((kk, ctx.Dm), 1.5), weight=np.full(kk, 2.5))
    scalars = (C.c_double(3.5), C.c_int(-9), C.c_int(-8))
    rc = L.vsom_cluster_nodes(ctx._h, k, seed, weighting, max_iter, out["labels"].ctypes.data_as(C.POINTER(C.c_int32)),
                              out["centroids"].ctypes.data_as(C.POINTER(C.c_double)), out["weight"].ctypes.data_as(C.POINTER(C.c_double)),
                              C.byref(scalars[0]), C.byref(scalars[1]), C.byref(scalars[2]))
    return rc, out, tuple(s.value for s in scalars), kk


def assert_refused(vsom, ctx, k, seed, weighting, max_iter, code, what):
    download = ctx.download_state_zero_filled if ctx.world > 1 else ctx.download_state
    before = download()
    rc, out, scalars, _ = raw_call(vsom, ctx, k, seed, weighting, max_iter)
    assert rc == code, f"{what}: rc {rc}"
    assert (out["labels"] == 7).all() and (out["centroids"] == 1.5).all() and (out["weight"] == 2.5).all(), f"{what}: outputs written"
    assert scalars == (3.5, -9, -8), f"{what}: scalar outputs written"
    assert_state_equal(before, download(), what)


@gpu
def test_refusals(vsom):
    rng = np.random.default_rng(5)
    W, H, D = 5, 4, 3
    three = rng.standard_normal((3, D)).astype(F32)
    mean = three[np.arange(W * H) % 3]
    ctx = make_ctx(vsom, W, H, D, vsom.STANDARD, 0, mean)
    labels, cent, weight, inertia, _, _ = ctx.cluster_nodes(3, 1)
    assert inertia == 0.0 and sorted(map(tuple, cent)) == sorted(map(tuple, three.astype(F64)))
    assert_refused(vsom, ctx, 4, 1, UNIFORM, 300, -1, "4 clusters of 3 distinct rows")
    assert_refused(vsom, ctx, 3, 1, HITS, 300, -1, "HITS on a map without data")
    assert_refused(vsom, ctx, 0, 1, UNIFORM, 300, -1, "k = 0")
    assert_refused(vsom, ctx, W * H + 1, 1, UNIFORM, 300, -1, "k = N + 1")
    assert_refused(vsom, ctx, 2, 1, UNIFORM, 0, -1, "max_iter = 0")
    assert_refused(vsom, ctx, 2, 1, 2, 300, -1, "unknown weighting")
    for bad, what in ((np.nan, "NaN"), (np.inf, "+inf"), (-np.inf, "-inf")):
        m = rng.standard_normal((W * H, D)).astype(F32)
        m[W * H - 1, 2] = bad
        ctx.upload_state(mean=m)
        assert_refused(vsom, ctx, 2, 1, UNIFORM, 300, -1, what)
    big = (np.sign(rng.standard_normal((W * H, D))) * 1e20).astype(F32)
    ctx.upload_state(mean=big)
    got = ctx.cluster_nodes(1, 0)  # one pick needs no distance
    assert got[4] >= 1
    assert_refused(vsom, ctx, 2, 1, UNIFORM, 300, -1, "distances overflow at the second pick")
    ctx.close()
    ranks = [vsom.VsomContext(4, 4, 3, vsom.STANDARD, 0, device=0, rank=r, world=2) for r in range(2)]
    for c in ranks:
        assert_refused(vsom, c, 2, 1, UNIFORM, 300, -3, "sharded")
    for c in ranks:
        c.close()


# ------------------------------------------------------------------------------------------------ host API
@gpu
@pytest.mark.parametrize("order,by_hits", [(0, 0), (2, 1)])
def test_host_api(vsom, tmp_path, order, by_hits):
    """Som::clusterNodes (tests/cpp/cluster_driver) after one epoch of Som::train equals the binding's cluster_nodes on the same map."""
    W, H, D, n, chunk, k, max_iter, seed = 12, 10, 6, 600, 200, 5, 300, 1234
    x = blobs(n, D, 6, 0.3, 2.0, 40)
    case, state = tmp_path / "case.bin", tmp_path / "state.bin"
    with open(case, "wb") as f:
        f.write(struct.pack("<10i", W, H, D, 0, order, n, chunk, k, by_hits, max_iter))
        f.write(struct.pack("<Q", seed))
        f.write(struct.pack("<4d", 0.1, 0.05, 3.0, 0.1))
        f.write(np.ascontiguousarray(x, F32).tobytes())
    r = subprocess.run([CLUSTER_DRIVER, str(case), str(state)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.split("\n")
    inertia = float.fromhex(lines[0].split()[1])
    labels = np.array(lines[1].split()[1:], np.int32)
    cent = np.array([[float.fromhex(v) for v in line.split()[2:]] for line in lines[2:2 + k]])
    raw = state.read_bytes()
    N = W * H
    mean = np.frombuffer(raw, F32, N * D, 0).reshape(N, D)
    hits = np.frombuffer(raw, np.uint64, N, 4 * (2 * N * D + N))
    assert hits.sum() == n
    ctx = make_ctx(vsom, W, H, D, vsom.STANDARD, order, mean, hits)
    got = ctx.cluster_nodes(k, seed, by_hits, max_iter)
    assert_bit_equal(labels, got[0], "labels")
    assert_bit_equal(cent, got[1], "centroids")
    assert_bit_equal(np.float64(inertia), np.float64(got[3]), "inertia")
    ctx.close()
