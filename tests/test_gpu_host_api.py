"""Drop-in check of the host C++ classes (include/SOM.hpp & co. over libvsom_b200.so): tests/cpp/api_driver.cpp is
one program written against the REFERENCE's public API; it is compiled once against the reference's own headers and
sources (oracle/_ref/api_driver_ref, CPU) and once against this repository's include/ + libvsom_host.so
(tests/cpp/api_driver_b200, B200).  Same input file -> the two output files must be identical byte for byte:
Som::train (epoch schedule, chunked DataSet protocol, metrics), getNeuron / getSigmaNeuron / getWeigthMap /
getBmuHits, updateUMatrix + getUMatrix, evaluate, measureSimilarity, findBmu, findRestrictedBmu,
euclidianWeightedDist, calculateNeighbourhoodWeight, and the Octave-text checkpoint: save() (the file's bytes),
Som(const char*) / getSizeFromFile / load() (the reloaded map and its evaluate()).  The reference build's outputs are
pinned by SHA-256 under tests/golden, so the B200 side runs without the reference's sources."""
import os
import struct
import subprocess

import numpy as np
import pytest

from conftest import REPO

REF_DRIVER = os.path.join(REPO, "oracle", "_ref", "api_driver_ref")
REF_DRIVER_SSE = os.path.join(REPO, "oracle", "_ref", "api_driver_ref_sse")  # reference TUs + stand-in Eigen in Eigen's SSE2 redux order
B200_DRIVER = os.path.join(REPO, "tests", "cpp", "api_driver_b200")
BIG_GOLDEN = os.path.join(REPO, "tests", "golden", "api_driver_big.json")
CASES_GOLDEN = os.path.join(REPO, "tests", "golden", "api_driver_cases.json")

# The LIGHT layout on BASELINE configs[3]'s map: 128x128, D=256, 4096 rows scored (evaluate, measureSimilarity, restricted BMU
# of every row, index) after a short training on the first 192 rows.  The CPU reference needs minutes for this, so its output
# is pinned by SHA-256 (tests/golden/make_api_driver_big.py ran both reference drivers; the hashes are committed).
BIG_CASE = (128, 128, 256, 0, 0, 1, 64, 42, 4096, 0.2, 0.0, 3.0, 0.0)
BIG_TRAIN_ROWS = 192


def make_big_x():
    rng = np.random.default_rng(2026)
    centres = (rng.standard_normal((24, 256)) * 0.6).astype(np.float32)
    return (centres[rng.integers(0, 24, 4096)] + 0.25 * rng.standard_normal((4096, 256))).astype(np.float32)

# W, H, Din, transform, decay, epochs, chunk, seed, n, eta0, etaDecay, sigma0, sigmaDecay
# (the last three schedules decay into the sigma == 1 findLocalBmu regime)
CASES = [
    (9, 7, 12, 0, 0, 4, 50, 42, 130, 0.3, 0.2, 3.0, 0.15),
    (8, 8, 20, 0, 1, 3, 0, 7, 90, 0.3, 0.1, 2.5, 0.2),
    (10, 6, 33, 1, 0, 4, 64, 3, 150, 0.05, 0.1, 3.5, 0.2),
    (7, 9, 6, 2, 0, 3, 40, 11, 100, 0.01, 0.1, 2.2, 0.1),
    (20, 20, 784, 0, 0, 2, 30, 42, 60, 0.1, 0.01, 5.0, 0.3),
    (9, 7, 12, 0, 0, 7, 50, 42, 130, 0.3, 0.2, 2.5, 0.4),
    (11, 8, 16, 1, 1, 6, 33, 5, 100, 0.05, 0.1, 1.8, 0.5),
    (6, 7, 5, 2, 0, 5, 0, 2, 90, 0.01, 0.1, 1.5, 0.6),
    # decay 2 = WeigthDecayFunction::BatchMap: Som::train dispatches to the batch-map trainer
    (8, 8, 12, 0, 2, 5, 50, 42, 130, 0.0, 0.0, 3.0, 0.35),
    (7, 5, 9, 1, 2, 4, 0, 9, 80, 0.0, 0.0, 2.0, 0.2),
]


def write_case(path, case, x, train_rows=0):
    W, H, Din, tr, dec, epochs, chunk, seed, n, eta0, eta_d, s0, s_d = case
    with open(path, "wb") as f:
        f.write(struct.pack("<10i", W, H, Din, tr, dec, epochs, chunk, seed, n, train_rows))
        f.write(struct.pack("<4d", eta0, eta_d, s0, s_d))
        f.write(np.ascontiguousarray(x, np.float32).tobytes())


def make_x(case):
    W, H, Din, tr, *_ = case
    n = case[8]
    rng = np.random.default_rng(sum(case[:9]))
    if tr == 2:
        z = rng.standard_normal((n, 1)).astype(np.float32)
        return (rng.uniform(0.5, 1.5, (1, Din)).astype(np.float32) * z + 0.1 * rng.standard_normal((n, Din))).astype(np.float32)
    return rng.standard_normal((n, Din)).astype(np.float32)


def expected_size(case):
    """Fixed part of the output; the checkpoint text (variable length) and the reloaded map follow."""
    W, H, Din, tr, dec, epochs, chunk, seed, n = case[:9]
    Dm = Din * (Din - 1) if tr == 2 else Din
    N = W * H
    size = 4 * epochs + N * 2 * Dm * 4 + N * 4 + N * 8 + N * 8 + 16
    if tr != 2:
        size += 8 + 4
    size += min(n, 16) * 24
    return size


@pytest.mark.parametrize("case", CASES[:2])
def test_reference_driver_runs_on_cpu(tmp_path, case):
    """CPU only: the reference build of the driver produces an output of the documented layout."""
    if not os.path.exists(REF_DRIVER):
        pytest.skip("oracle/_ref/api_driver_ref not built (oracle/Makefile builds it from the reference's sources)")
    write_case(tmp_path / "case.bin", case, make_x(case))
    subprocess.run([REF_DRIVER, str(tmp_path / "case.bin"), str(tmp_path / "ref.bin")], check=True, timeout=300)
    assert os.path.getsize(tmp_path / "ref.bin") > expected_size(case)


def run_b200(case_path, out_path, order):
    """order: "reference" (sequential dot, = api_driver_ref) or "eigen_sse" (= api_driver_ref_sse); the host classes pick it
    up from VSOM_REDUCTION_ORDER (include/SOM.hpp)."""
    env = dict(os.environ, VSOM_REDUCTION_ORDER=order)
    subprocess.run([B200_DRIVER, str(case_path), str(out_path)], check=True, timeout=600, env=env)


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("order", ["reference", "eigen_sse"])
@pytest.mark.parametrize("case", CASES)
def test_host_api_is_a_drop_in(tmp_path, vsom, case, order):
    """The reference driver's output is pinned by its SHA-256 and length (tests/golden/make_api_driver_cases.py)."""
    import hashlib
    import json

    golden = next(g for g in json.load(open(CASES_GOLDEN)) if tuple(g["case"]) == case)
    vsom.lib()  # builds libvsom_b200.so, libvsom_host.so and the B200 driver when sources are newer
    assert os.path.exists(B200_DRIVER)
    write_case(tmp_path / "case.bin", case, make_x(case))
    assert hashlib.sha256(open(tmp_path / "case.bin", "rb").read()).hexdigest() == golden["case_sha256"], "the case file is not the one the golden was made from"
    run_b200(tmp_path / "case.bin", tmp_path / "b200.bin", order)
    got = open(tmp_path / "b200.bin", "rb").read()
    assert len(got) > expected_size(case) and len(got) == golden[order]["bytes"]
    assert hashlib.sha256(got).hexdigest() == golden[order]["sha256"], f"B200 output differs from the {order} reference driver's"


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("order", ["reference", "eigen_sse"])
def test_host_api_large_map_scoring_takes_the_tensor_core_path(tmp_path, vsom, order):
    """Som::evaluate / measureSimilarity / mapDataSet over 4096 rows at 128x128x256 reach vsom_find_bmu with a batch the
    library scores on the tensor cores (K2); the driver's output must still be the reference's, byte for byte (pinned by the
    committed SHA-256 of the reference drivers' outputs)."""
    import hashlib
    import json

    golden = json.load(open(BIG_GOLDEN))
    vsom.lib()
    write_case(tmp_path / "case.bin", BIG_CASE, make_big_x(), BIG_TRAIN_ROWS)
    assert hashlib.sha256(open(tmp_path / "case.bin", "rb").read()).hexdigest() == golden["case_sha256"], "the case file is not the one the golden was made from"
    run_b200(tmp_path / "case.bin", tmp_path / "b200.bin", order)
    got = open(tmp_path / "b200.bin", "rb").read()
    assert len(got) == golden["bytes"]
    assert hashlib.sha256(got).hexdigest() == golden[order], f"B200 output differs from the {order} reference driver's"
