"""Generates tests/golden/api_driver_cases.json: for every case of tests/test_gpu_host_api.py::CASES, the SHA-256 of the case
file and the SHA-256 and length of the reference drivers' outputs in both dot orders (oracle/_ref/api_driver_ref and
api_driver_ref_sse, the reference's own translation units; oracle/Makefile builds them where the reference's sources are).

  python tests/golden/make_api_driver_cases.py          # the reference drivers, CPU
  python tests/golden/make_api_driver_cases.py --b200   # this repository's tests/cpp/api_driver_b200 on a B200

--b200 gives the reference's bytes only at a commit whose test_host_api_is_a_drop_in compared the B200 driver with the
reference drivers byte for byte and passed.  The committed file was made that way, on a B200, from commit 2078c42, whose
suite had passed that comparison for all ten cases in both orders."""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import test_gpu_host_api as t  # noqa: E402


def sha(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def main():
    b200 = "--b200" in sys.argv
    out = []
    with tempfile.TemporaryDirectory() as d:
        for i, case in enumerate(t.CASES):
            path = os.path.join(d, f"case{i}.bin")
            t.write_case(path, case, t.make_x(case))
            entry = {"case": list(case), "case_sha256": sha(path)}
            for order, drv in (("reference", t.REF_DRIVER), ("eigen_sse", t.REF_DRIVER_SSE)):
                res = os.path.join(d, f"case{i}_{order}.bin")
                if b200:
                    t.run_b200(path, res, order)
                else:
                    subprocess.run([drv, path, res], check=True)
                entry[order] = {"sha256": sha(res), "bytes": os.path.getsize(res)}
            out.append(entry)
            print(entry, flush=True)
    with open(os.path.join(HERE, "api_driver_cases.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
