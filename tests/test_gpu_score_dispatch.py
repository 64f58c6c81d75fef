"""The scoring dispatcher (score_rows, csrc/score_tc.cu): the seams between K2's probes, the exact scan of the rows they leave
(tier 3), the host-row slab pipelines and the similarity pass, and the path every call reports.

- vsom_measure_similarity on a map whose nodes nearly coincide: both probes run in 4096-row slabs and the remaining 3077 rows
  take the exact scan in 1024-row slabs, so the per-row similarity pass of every slab must land at its absolute row.
- A table of (last_score_tc, last_score_pair, fallback rows) per call: either side of 1024 rows, forced tiers 1 and 2, the
  single-CTA kernel, tier 3, no rows at all, CLR and Dm = 2049 (always the exact scan), and the batch-map trainer's epochs."""
import numpy as np
import pytest

from conftest import assert_bit_equal
from test_gpu_benchmark_shapes import PROBE, TC_MIN_ROWS

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

F32 = np.float32
TIER3_ROWS = 2 * PROBE + 3 * 1024 + 5


def coincident_map(n):
    """test_gpu_benchmark_shapes._row_count_map's 'coincident' map (nodes within 1e-4 of one point), with n rows."""
    W, H, D = 20, 20, 96
    rng = np.random.default_rng(77)
    base = rng.standard_normal(D).astype(F32)
    mean = (base[None, :] + 1e-4 * rng.standard_normal((W * H, D))).astype(F32)
    x = (base[None, :] + rng.standard_normal((n, D))).astype(F32)
    return W, H, D, mean, x


def test_measure_similarity_tier3_across_slabs(vsom, monkeypatch):
    """Both probes in several host slabs, then the exact scan of the rest in several slabs: BMUs equal the exact scan and every
    row maximum equals test_gpu_parity's numpy formula on them."""
    monkeypatch.delenv("VSOM_TC_TIER", raising=False)
    monkeypatch.setenv("VSOM_TC_HOST_SLAB_LOG2", "12")
    monkeypatch.setenv("VSOM_EXACT_HOST_SLAB_LOG2", "10")
    W, H, D, mean, x = coincident_map(TIER3_ROWS)
    sigma = np.random.default_rng(78).uniform(1e-6, 4e-5, mean.shape).astype(F32)  # about a quarter below the cap of 1e-5
    ctx = vsom.VsomContext(W, H, D, vsom.STANDARD, vsom.ORDER_EIGEN_SSE)
    ctx.upload_state(mean=mean, sigma=sigma)
    eb, _ = ctx.find_bmu_exact(x)
    bmu, row_max = ctx.measure_similarity(x, 3, 0)
    assert ctx.last_score_tc == 3
    assert_bit_equal(bmu, eb, "bmu")
    m, s = mean[eb], sigma[eb]
    sM = np.where(s > F32(0.00001), F32(0.00001), s).astype(F32)
    with np.errstate(all="ignore"):
        delta = (((x - m).astype(F32) / sM).astype(F32) / F32(3)).astype(F32)
    want = np.where(np.isnan(delta), -np.inf, delta).max(axis=1).astype(F32)
    assert_bit_equal(row_max, want, "row maxima")
    ctx.close()


# ------------------------------------------------------------------------------------------------ the path each call reports
def _map(kind):
    """((W, H), Din, transform, mean, rows) of the table's maps; a call takes the first n rows."""
    rng = np.random.default_rng({"random": 1, "clr": 2, "wide": 3}.get(kind, 0))
    if kind == "coincident":
        W, H, D, mean, x = coincident_map(TIER3_ROWS)
        return (W, H), D, 0, mean, x
    if kind == "random":
        W, H, D = 13, 11, 40
        return (W, H), D, 0, rng.standard_normal((W * H, D)).astype(F32), rng.standard_normal((4096, D)).astype(F32)
    if kind == "clr":
        W, H, Din = 13, 11, 6
        z = rng.standard_normal((2048, 1)).astype(F32)
        x = (rng.uniform(0.5, 1.5, (1, Din)) * z + 0.3 * rng.standard_normal((2048, Din))).astype(F32)
        return (W, H), Din, 2, rng.standard_normal((W * H, Din * (Din - 1))).astype(F32), x
    W, H, D = 4, 4, 2049  # one component longer than K2 takes
    return (W, H), D, 0, rng.standard_normal((W * H, D)).astype(F32), rng.standard_normal((1024, D)).astype(F32)


def _call(ctx, entry, x):
    """One scoring call; returns its fallback rows."""
    import torch

    n = len(x)
    if entry == "bmu_host":
        return ctx.find_bmu_batch(x)[2]
    if entry == "bmu2_host":
        return ctx.find_bmu2(x)[4]
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    outs = [torch.empty(n, dtype=torch.int32, device="cuda") for _ in range(4)]
    if entry == "bmu_dev":
        fb = ctx.find_bmu_batch_device(xd, n, outs[0], outs[1].view(torch.float32))
    else:
        fb = ctx.find_bmu2_device(xd, n, outs[0], outs[1].view(torch.float32), outs[2], outs[3].view(torch.float32))
    ctx.synchronize()
    return fb


# (map, rows, environment): "tier" forces VSOM_TC_TIER, "pair0" sets VSOM_TC_PAIR=0.  Settings ending in "after_k2" first run
# 1024 rows through K2 on the same context, so that a call which leaves the report alone is told apart from one that resets it.
SETTINGS = {
    "1023": ("random", 1023, {}),
    "1024": ("random", 1024, {}),
    "tier1": ("random", 4096, {"VSOM_TC_TIER": "1"}),
    "tier2": ("random", 4096, {"VSOM_TC_TIER": "2"}),
    "pair0": ("random", 4096, {"VSOM_TC_PAIR": "0"}),
    "tier3": ("coincident", TIER3_ROWS, {}),
    "n0_after_k2": ("random", 0, {}),
    "clr": ("clr", 2048, {}),
    "dm2049": ("wide", 1024, {}),
}
# the batch-map trainer's phase A: (rows, first epoch)
BATCH = {"first_1023": (1023, True), "first_1024": (1024, True), "later_after_k2": (1024, False)}


def observe(vsom, monkeypatch, entry, setting):
    """(last_score_tc, last_score_pair, fallback rows) after one call; fallback rows is None for the batch-map trainer."""
    for k in ("VSOM_TC_TIER", "VSOM_TC_PAIR", "VSOM_TC_SLAB_LOG2", "VSOM_TC_HOST_SLAB_LOG2", "VSOM_EXACT_HOST_SLAB_LOG2"):
        monkeypatch.delenv(k, raising=False)
    kind, n, env = SETTINGS[setting] if entry != "batch" else ("random", BATCH[setting][0], {})
    (W, H), Din, tr, mean, x = _map(kind)
    ctx = vsom.VsomContext(W, H, Din, tr, vsom.ORDER_REFERENCE)
    ctx.upload_state(mean=mean)
    try:
        if setting.endswith("after_k2"):
            ctx.find_bmu(x[:TC_MIN_ROWS])
            assert ctx.last_score_tc > 0
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        if entry == "batch":
            ctx.batch_epoch(x[:n], 4.0, BATCH[setting][1])
            return ctx.last_score_tc, ctx.last_score_pair, None
        fb = _call(ctx, entry, x[:n])
        return ctx.last_score_tc, ctx.last_score_pair, fb
    finally:
        ctx.close()


# (last_score_tc, last_score_pair, fallback rows) per "entry:setting"; last_score_pair is 1 on a whole B200, which co-schedules
# clusters of two K2 CTAs
EXPECTED = {
    "bmu_host:1023": (0, 0, 1023),
    "bmu_host:1024": (1, 1, 0),
    "bmu_host:tier1": (1, 1, 0),
    "bmu_host:tier2": (2, 1, 0),
    "bmu_host:pair0": (1, 0, 0),
    "bmu_host:tier3": (3, 1, 19461),
    "bmu_host:n0_after_k2": (1, 1, 0),
    "bmu_host:clr": (0, 0, 2048),
    "bmu_host:dm2049": (0, 0, 1024),
    "bmu_dev:1023": (0, 0, 1023),
    "bmu_dev:1024": (1, 1, 0),
    "bmu_dev:tier1": (1, 1, 0),
    "bmu_dev:tier2": (2, 1, 0),
    "bmu_dev:pair0": (1, 0, 0),
    "bmu_dev:tier3": (3, 1, 19461),
    "bmu_dev:n0_after_k2": (0, 0, 0),
    "bmu_dev:clr": (0, 0, 2048),
    "bmu_dev:dm2049": (0, 0, 1024),
    "bmu2_host:1023": (0, 0, 1023),
    "bmu2_host:1024": (1, 1, 0),
    "bmu2_host:tier1": (1, 1, 0),
    "bmu2_host:tier2": (2, 1, 0),
    "bmu2_host:pair0": (1, 0, 0),
    "bmu2_host:tier3": (3, 1, 19461),
    "bmu2_host:n0_after_k2": (1, 1, 0),
    "bmu2_host:clr": (0, 0, 2048),
    "bmu2_host:dm2049": (0, 0, 1024),
    "bmu2_dev:1023": (0, 0, 1023),
    "bmu2_dev:1024": (1, 1, 0),
    "bmu2_dev:tier1": (1, 1, 0),
    "bmu2_dev:tier2": (2, 1, 0),
    "bmu2_dev:pair0": (1, 0, 0),
    "bmu2_dev:tier3": (3, 1, 19461),
    "bmu2_dev:n0_after_k2": (0, 0, 0),
    "bmu2_dev:clr": (0, 0, 2048),
    "bmu2_dev:dm2049": (0, 0, 1024),
    "batch:first_1023": (0, 0, None),
    "batch:first_1024": (1, 1, None),
    "batch:later_after_k2": (0, 0, None),
}


@pytest.mark.parametrize("case", EXPECTED)
def test_reported_path(vsom, monkeypatch, case):
    entry, setting = case.split(":")
    assert observe(vsom, monkeypatch, entry, setting) == EXPECTED[case]
