"""Records tests/golden/ref_digests.json: the sha256 digest of every answer the tests compare with the
reference's own code (oracle_lib.check_ref).  Where oracle/_ref is built for every shape (oracle/build_ref.sh,
from the reference's sources) the answers come from the reference itself; otherwise from the oracle and the
library's host code, which those same comparisons hold bit-identical to the reference where it is built.
The file records which of the two it was.  Run from the repo root after build():
    python tests/golden/make_ref_digests.py
"""
import importlib
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "ref_digests.json")
os.environ["NAVSLAM_RECORD_REF_DIGESTS"] = OUT
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pytest  # noqa: E402

import oracle_lib  # noqa: E402

SHAPES = ("8x8", "5x33", "16x1800", "64x2048")
# cases the tests only ever ran against the oracle: the reference's quadratic quick-select made
# test_tree_build_and_nn_bit_exact skip them while they were compared with the reference
NEVER_COMPARED = ["tree/sorted/20000/"]

if __name__ == "__main__":
    from_ref = all(oracle_lib.ref_available(s) for s in SHAPES)
    tests = [os.path.join(ROOT, "tests", t) for t in ("test_oracle_vs_ref.py", "test_io_formats.py", "test_abi.py")]
    rc = pytest.main(["-q", "-p", "no:cacheprovider", *tests])
    if rc != 0:
        sys.exit(f"make_ref_digests: the tests failed (rc={rc}); nothing written")
    shim_tests = importlib.import_module("test_shim_gpu")
    synth = importlib.import_module("nav-slam_b200.synth")
    oracle = oracle_lib.Oracle()
    for shape, frames in shim_tests.SLAM_STEP_CASES:
        shim_tests.reference_slam_steps(oracle, synth, shape, frames)
    header = {
        "recorded_from": ("the reference's own code (oracle/_ref)" if from_ref else
                          "the oracle and the library's host code, with oracle/_ref absent: every key outside "
                          "never_compared_with_the_reference is an answer those comparisons held bit-identical "
                          "to the reference's where it was built"),
        "never_compared_with_the_reference": [] if from_ref else NEVER_COMPARED,
    }
    oracle_lib.write_recorded(header)
    print(OUT, len(oracle_lib._recorded), "answers,", os.path.getsize(OUT), "bytes")
