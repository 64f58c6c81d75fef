"""TEST INFRASTRUCTURE — generates tests/golden/ref_*.npz by driving the reference's OWN code
(oracle/_ref/libvsom_ref.so = the reference's src/*.cpp compiled unmodified, see oracle/Makefile).

Needs the reference's sources to build that library; the fixtures it writes are committed.
Usage: python oracle/gen_golden.py [--restatement]

random_cases / batch_map_cases / eigen_sse_cases are the fresh-input comparisons of tests/test_oracle_pin.py; their
outputs, stored as SHA-256 digests (ref_random.json, ref_batch_map.json, ref_eigen_sse.json), come from the compiled reference, or with --restatement
from oracle/liboracle.so.  The committed three were made with --restatement; oracle/vsom_oracle.c is unchanged since
commit 6ccba42, whose tests compared it with the compiled reference on exactly these inputs, bit for bit.
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import pyoracle as po  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

# name, W, H, Din, transform, decay, eta, rows, sigmas (one train_rows segment each)
CASES = [
    ("std_exp", 12, 9, 17, po.STANDARD, po.EXPONENTIAL, 0.2, 240, (3.0, 1.4, 1.0)),
    ("std_inv", 9, 12, 10, po.STANDARD, po.INVERSE, 0.2, 240, (2.2, 1.3, 1.0)),
    ("med_exp", 8, 8, 33, po.MEDIAN, po.EXPONENTIAL, 0.05, 240, (2.5, 1.2, 1.0)),
    ("med_inv", 5, 7, 4, po.MEDIAN, po.INVERSE, 0.05, 120, (1.9, 1.0)),
    ("clr_exp", 6, 5, 6, po.CLR, po.EXPONENTIAL, 0.01, 200, (2.0, 1.5, 1.0)),
    ("clr_inv", 4, 6, 5, po.CLR, po.INVERSE, 0.01, 160, (1.8, 1.0)),
]


def random_cases(make):
    """Fresh random cases: every transformation and decay, global and local BMU regimes, scoring.  make(W, H, D, tr) -> checker.
    Returns the outputs by name."""
    out = {}
    rng = np.random.default_rng(3)
    for tr in (po.STANDARD, po.MEDIAN, po.CLR):
        for dec in (po.EXPONENTIAL, po.INVERSE):
            W, H, D = int(rng.integers(2, 9)), int(rng.integers(2, 9)), (5 if tr == po.CLR else int(rng.integers(1, 40)))
            c = make(W, H, D, tr)
            c.random_initialize(11, 0.7)
            x = rng.standard_normal((90, D)).astype(np.float32)
            p = f"tr{tr}_dec{dec}_"
            for si, sg in enumerate((2.7, 1.01, 1.0, 0.5)):
                eta = 0.01 if tr == po.CLR else 0.3
                for k, v in zip(("bmu", "dist", "resid2", "last"), c.train_rows(x, eta, sg, dec)):
                    out[f"{p}sigma{si}_{k}"] = v
                for k, v in c.get_state().items():
                    out[f"{p}sigma{si}_{k}"] = v
            for start in (0, W * H - 1, W - 1):
                out[f"{p}local_bmu_from{start}"] = np.int64(c.find_local_bmu(x[0], start))
            out[p + "umatrix"] = c.update_umatrix()
            out[p + "bmd"] = c.find_restricted_bmd(x[1], 1)
            if tr != po.CLR:
                out[p + "evaluate"] = np.float64(c.evaluate(x))
                out[p + "similarity"] = np.int64(c.measure_similarity(x[:30], 3, 0))
    return out


def batch_map_cases(make):
    """The batch-map trainer: non-square maps (the SomIndex(map, index) quirk), several chunks per epoch, U-matrix after each
    epoch and the early return at sigma < 1."""
    out = {}
    rng = np.random.default_rng(21)
    for tr in (po.STANDARD, po.MEDIAN, po.CLR):
        for W, H in ((6, 6), (7, 4), (4, 9)):
            D = 5 if tr == po.CLR else 11
            c = make(W, H, D, tr)
            c.random_initialize(3, 1.0)
            x = rng.standard_normal((90, D)).astype(np.float32)
            p = f"tr{tr}_{W}x{H}_"
            out[p + "mse"] = c.train_batch(x, 40, 5, 3.0, 0.35, True)
            for k, v in c.get_state().items():
                out[p + k] = v
            out[p + "umatrix"] = c.update_umatrix()
    return out


def eigen_sse_cases(make):
    """The whole path in the Eigen SSE2 dot order: training (all transformations, both decays, global and local BMU regimes),
    scoring, evaluate, measureSimilarity, U-matrix, batch-map trainer.  make(W, H, D, tr) -> checker in that order."""
    out = {}
    rng = np.random.default_rng(4)
    for tr in (po.STANDARD, po.MEDIAN, po.CLR):
        for dec in (po.EXPONENTIAL, po.INVERSE):
            W, H, D = int(rng.integers(2, 9)), int(rng.integers(2, 9)), (6 if tr == po.CLR else int(rng.integers(5, 60)))
            c = make(W, H, D, tr)
            c.random_initialize(11, 0.7)
            x = rng.standard_normal((90, D)).astype(np.float32)
            p = f"tr{tr}_dec{dec}_"
            for si, sg in enumerate((2.7, 1.01, 1.0, 0.5)):
                eta = 0.01 if tr == po.CLR else 0.3
                for k, v in zip(("bmu", "dist", "resid2", "last"), c.train_rows(x, eta, sg, dec)):
                    out[f"{p}sigma{si}_{k}"] = v
                for k, v in c.get_state().items():
                    out[f"{p}sigma{si}_{k}"] = v
            out[p + "umatrix"] = c.update_umatrix()
            out[p + "score_bmu"], out[p + "score_dist"] = c.find_bmu(x)
            out[p + "bmd"] = c.find_restricted_bmd(x[1], 1)
            if tr != po.CLR:
                out[p + "evaluate"] = np.float64(c.evaluate(x))
                out[p + "similarity"] = np.int64(c.measure_similarity(x[:30], 3, 0))
    for tr in (po.STANDARD, po.CLR):
        D = 5 if tr == po.CLR else 13
        c = make(7, 4, D, tr)
        c.random_initialize(3, 1.0)
        x = rng.standard_normal((90, D)).astype(np.float32)
        p = f"batch_tr{tr}_"
        out[p + "mse"] = c.train_batch(x, 40, 4, 3.0, 0.35, True)
        for k, v in c.get_state().items():
            out[p + k] = v
    return out


def digests(outputs):
    """Outputs by name -> {name: [dtype, shape, SHA-256 of the bytes]}, in the order they were computed."""
    out = {}
    for k, v in outputs.items():
        a = np.ascontiguousarray(v)
        out[k] = [a.dtype.str, list(np.shape(v)), hashlib.sha256(a.tobytes()).hexdigest()]
    return out


def write_comparison_cases(restatement):
    if restatement:
        seq = lambda W, H, D, tr: po.Oracle(W, H, D, tr)  # noqa: E731
        sse = lambda W, H, D, tr: po.Oracle(W, H, D, tr, po.ORDER_EIGEN_SSE)  # noqa: E731
    else:
        seq, sse = po.Reference, po.ReferenceSse
    for name, fn, make in (("random", random_cases, seq), ("batch_map", batch_map_cases, seq), ("eigen_sse", eigen_sse_cases, sse)):
        with open(os.path.join(OUT, f"ref_{name}.json"), "w") as f:
            json.dump(digests(fn(make)), f, indent=0)
        print(name, "ok")


def main():
    if "--restatement" in sys.argv:
        write_comparison_cases(True)
        return
    if not po.Reference.available():
        po.build(quiet=False)
    assert po.Reference.available(), "oracle/_ref/libvsom_ref.so missing (needs the reference's sources, see oracle/Makefile)"
    os.makedirs(OUT, exist_ok=True)
    write_comparison_cases(False)
    for ci, (name, W, H, Din, tr, dec, eta, rows, sigmas) in enumerate(CASES):
        rng = np.random.default_rng(1000 + ci)
        r = po.Reference(W, H, Din, tr)
        r.random_initialize(42, 1.0)
        init = r.get_state()
        if tr == po.CLR:
            z = rng.standard_normal((rows * len(sigmas), 1)).astype(np.float32)
            a = rng.uniform(0.5, 1.5, (1, Din)).astype(np.float32)
            x = (a * z + 0.1 * rng.standard_normal((rows * len(sigmas), Din))).astype(np.float32)
        else:
            x = rng.standard_normal((rows * len(sigmas), Din)).astype(np.float32)
        out = dict(W=W, H=H, Din=Din, transform=tr, decay=dec, eta=eta, sigmas=np.array(sigmas), rows=rows, x=x, init_mean=init["mean"])
        for si, sg in enumerate(sigmas):
            seg = x[si * rows:(si + 1) * rows]
            bmu, dist, resid2, last = r.train_rows(seg, eta, sg, dec)
            st = r.get_state()
            out[f"bmu{si}"], out[f"dist{si}"], out[f"resid2{si}"], out[f"last{si}"] = bmu, dist, resid2, last
            for k, v in st.items():
                out[f"{k}{si}"] = v
        out["umatrix"] = r.update_umatrix()
        q = x[:64]
        out["score_bmu"], out["score_dist"] = r.find_bmu(q)
        out["restricted_bmu"] = r.find_restricted_bmu(q, 2)
        out["all_dists_row0"] = r.all_dists(q[0])
        if tr != po.CLR:  # Som::evaluate mixes Dm- and Din-sized vectors for CLR (src/Som.cpp:509): undefined in the reference
            out["evaluate"] = np.float64(r.evaluate(q))
        out["eigen_kind"] = np.array(po.Reference.eigen_kind())
        np.savez_compressed(os.path.join(OUT, f"ref_{name}.npz"), **out)
        print(name, "ok", x.shape)
    # a whole Som::train run (epoch schedule + chunked DataSet protocol) on a small map
    rng = np.random.default_rng(77)
    x = rng.standard_normal((150, 9)).astype(np.float32)
    r = po.Reference(7, 6, 9, po.STANDARD)
    r.random_initialize(5, 0.5)
    init = r.get_state()
    mse = r.train(x, 64, 5, 0.3, 0.2, 3.0, 0.15, po.EXPONENTIAL, True)
    st = r.get_state()
    np.savez_compressed(os.path.join(OUT, "ref_train_std_exp.npz"), x=x, init_mean=init["mean"], mse=mse, chunk=64, epochs=5, eta0=0.3, eta_decay=0.2,
                        sigma0=3.0, sigma_decay=0.15, **{f"final_{k}": v for k, v in st.items()})
    print("train ok", mse)


if __name__ == "__main__":
    main()
