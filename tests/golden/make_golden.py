"""Generates the golden data of tests/golden/ from the UNMODIFIED compiled reference (oracle/_ref).

Run where the reference sources exist:   make -C oracle ref && python tests/golden/make_golden.py [npz|digests]

npz:     tests/golden/q8_golden.npz.  For every case of tests/cases.py the reference's own create -> setup -> run
         produces the expected uint8 output (with 0xA5 canaries in the pixel-stride gaps).  Small outputs are stored
         verbatim, MobileNetV2 batch-1 layer outputs as SHA-256 digests.  Inputs are regenerated from the case seed;
         their digest is stored too, so a drifting RNG fails loudly instead of silently.
digests: tests/golden/reference_digests.json (tests/reference.py).  The tests that compare with the reference run with
         the reference in place of the product and record the digest of every answer it gives.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ref as R  # noqa: E402
from tests import cases as CS, util as U  # noqa: E402

# every test that calls tests.reference.expect
DIGEST_TESTS = ["tests/test_gpu_ops.py", "tests/test_ops_oracle.py", "tests/test_chain_check.py",
                "tests/test_oracle.py::test_oracle_matches_compiled_reference_on_device_path_cases",
                "tests/test_oracle.py::test_compiled_reference_q31_matches_oracle"]


def make_npz():
    rf = R.QnnpackHost()
    out = {}
    for case in CS.OPERATOR_CASES + CS.DW_UKERNEL_CASES:
        x, k, b, kw = U.conv_setup(case)
        y = U.run_conv(rf, case, x, k, b, kw)
        out[f"conv/{case['name']}/y"] = y
        out[f"conv/{case['name']}/in_digest"] = np.array(U.digest(x) + U.digest(k) + U.digest(b))
    for case in CS.GEMM_UKERNEL_CASES:
        x, k, b, kw = U.fc_setup(case)
        y = U.run_fc(rf, case, x, k, b, kw)
        out[f"fc/{case['name']}/y"] = y
        out[f"fc/{case['name']}/in_digest"] = np.array(U.digest(x) + U.digest(k) + U.digest(b))
    for entry in CS.MOBILENET_V2:
        case = CS.mobilenet_case(entry, 1)
        x, k, b, kw = U.conv_setup(case)
        y = U.run_conv(rf, case, x, k, b, kw)
        out[f"mnv2/{case['name']}/y_digest"] = np.array(U.digest(y))
        out[f"mnv2/{case['name']}/in_digest"] = np.array(U.digest(x) + U.digest(k) + U.digest(b))
    np.savez_compressed(U.GOLDEN, **out)
    print("wrote", U.GOLDEN, os.path.getsize(U.GOLDEN), "bytes,", len(out), "arrays")


def make_digests():
    import pytest

    import qnnpack_b200.api as A
    from tests import reference as REF

    rf = R.QnnpackHost()
    A._product = rf  # the GPU tests' product fixture now returns the reference: it answers both sides
    REF.RECORD_WITH, REF._table = rf, {}
    rc = pytest.main(["-q", "-p", "no:cacheprovider", "--rootdir", ROOT] + [os.path.join(ROOT, t) for t in DIGEST_TESTS])
    if rc != 0:
        raise SystemExit(f"recording run failed ({rc}); {REF.PATH} left unchanged")
    REF.save()
    print("wrote", REF.PATH, os.path.getsize(REF.PATH), "bytes,", len(REF._table), "digests")


if __name__ == "__main__":
    what = sys.argv[1:] or ["npz", "digests"]
    if "npz" in what:
        make_npz()
    if "digests" in what:
        make_digests()
