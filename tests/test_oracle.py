"""CPU tests: the oracle (C restatement + NumPy restatement) against
  (a) the reference's deterministic Q31 known-answer tests (test/requantization-tester.h),
  (b) golden vectors generated from the unmodified compiled reference (tests/golden/),
  (c) what the compiled reference computed for the same calls (tests/reference.py), and the compiled reference itself
      where oracle/_ref has been built.
"""
import numpy as np
import pytest

from oracle import q8_oracle as O
from tests import cases as CS, reference as REF, util as U


# ---- (a) Q31 known-answer tests, restated from test/requantization-tester.h ---------------------
def _q31(oracle_c, x, scale, zp, qmin=0, qmax=255):
    x = np.asarray(x, dtype=np.int32)
    a = oracle_c.requantize_q31(x, scale, zp, qmin, qmax)
    b = O.q31_requantize_np(x, O.compute_requant_params(scale, zp, qmin, qmax))
    assert np.array_equal(a, b)
    return a


def kat_exact_divide(s, zp):
    """requantization-tester.h:84-109: inputs (clamped_i - zp) << s  ->  outputs clamped_i."""
    max_i = ((2**31 - 1) >> s) + zp
    min_i = -((2**31) >> s) + zp
    ci = np.clip(np.arange(256, dtype=np.int64), min_i, max_i)
    return ((ci - zp) << s).astype(np.int32), ci.astype(np.uint8)


def kat_rounding_up(s, zp):
    """requantization-tester.h:118-144: (i - zp)*2^s - 2^(s-1) + (i <= zp)  ->  i (where it fits int32)."""
    i = np.arange(256, dtype=np.int64)
    x = ((i - zp) << s) - (1 << (s - 1)) + (i <= zp)
    keep = (x >= -(2**31)) & (x < 2**31)
    return x[keep].astype(np.int32), i[keep].astype(np.uint8)


def kat_rounding_away(s, zp):
    """requantization-tester.h:181-215: midpoints towards zero from i round away from zero, back to i.
    The reference's verification loop runs with an unsigned i (:199), so `i - zeroPoint` wraps for
    i < zp and those rows are never asserted; for Q31 they would fail at s=1 (x=-1: the first rounding
    takes -0.5 up to 0), which is the intended double rounding.  Restated as the reference executes it:
    only i >= zp is checked."""
    i = np.arange(256, dtype=np.int64)
    x = (i - zp) << s
    x = np.where(x > 0, x - (1 << (s - 1)), np.where(x < 0, x + (1 << (s - 1)), x))
    keep = (x >= -(2**31)) & (x < 2**31) & (i >= zp)
    return x[keep].astype(np.int32), i[keep].astype(np.uint8)


KAT_ZERO_POINTS = (0, 1, 2, 64, 127, 128, 129, 254, 255)


@pytest.mark.parametrize("s", range(1, 32))
def test_q31_known_answers(oracle_c, s):
    """The Q31 rows of test/requantization.cc:250-310: exact_divide_by_po2, divide_by_po2_with_rounding_up,
    divide_by_po2_with_rounding_away — for every zero point the reference sweeps."""
    scale = np.float32(2.0 ** -s)
    for zp in range(256):
        for kat in (kat_exact_divide, kat_rounding_up, kat_rounding_away):
            x, want = kat(s, zp)
            assert np.array_equal(_q31(oracle_c, x, scale, zp), want), (kat.__name__, s, zp)


def test_q31_special_cases(oracle_c):
    """requantization-tester.h:217-246."""
    for zp in range(256):
        lo = _q31(oracle_c, [np.iinfo(np.int32).min] * 16, np.float32(2.0 ** -32), zp)
        assert lo.min() == max(0, zp - 1)
    hi = _q31(oracle_c, [np.iinfo(np.int32).max] * 16, np.float32(float.fromhex("0x1.FFFFFEp-1")), 255)
    assert (hi == 255).all()


def test_q31_random_is_close_to_exact_scaling(oracle_c):
    """requantization-tester.h:288-328 (approximation <= 0.55) — a property, not a vector."""
    rng = np.random.default_rng(7)
    for zp in (0, 77, 255):
        scale = np.float32(rng.uniform(2.0 ** -20, 2.0 ** -10))
        x = rng.integers(-(2**24), 2**24, 20000).astype(np.int32)
        out = _q31(oracle_c, x, scale, zp).astype(np.float64)
        ideal = np.clip(x.astype(np.float64) * float(scale) + zp, 0, 255)
        assert np.abs(out - ideal).max() <= 0.55


# ---- (b) golden vectors from the compiled reference ----------------------------------------------
@pytest.mark.parametrize("case", CS.OPERATOR_CASES + CS.DW_UKERNEL_CASES, ids=lambda c: c["name"])
def test_c_oracle_matches_golden_conv(oracle_c, golden, case):
    x, k, b, kw = U.conv_setup(case)
    assert str(golden[f"conv/{case['name']}/in_digest"]) == U.digest(x) + U.digest(k) + U.digest(b), "input RNG drifted"
    U.assert_same_bytes(U.run_conv(oracle_c, case, x, k, b, kw), golden[f"conv/{case['name']}/y"], case["name"])


@pytest.mark.parametrize("case", CS.OPERATOR_CASES[::3], ids=lambda c: c["name"])
def test_numpy_oracle_matches_golden_conv(golden, case):
    x, k, b, kw = U.conv_setup(case)
    cin = case["groups"] * case["gic"]
    y = O.convolution2d_nhwc_q8_np(x[..., :cin], k, b, **kw)
    want = golden[f"conv/{case['name']}/y"][..., :case["groups"] * case["goc"]]
    U.assert_same_bytes(y, want, case["name"])


@pytest.mark.parametrize("case", CS.GEMM_UKERNEL_CASES, ids=lambda c: c["name"])
def test_c_oracle_matches_golden_fc(oracle_c, golden, case):
    x, k, b, kw = U.fc_setup(case)
    assert str(golden[f"fc/{case['name']}/in_digest"]) == U.digest(x) + U.digest(k) + U.digest(b), "input RNG drifted"
    U.assert_same_bytes(U.run_fc(oracle_c, case, x, k, b, kw), golden[f"fc/{case['name']}/y"], case["name"])


@pytest.mark.parametrize("entry", CS.MOBILENET_V2[5:], ids=lambda e: e[0])
def test_numpy_oracle_matches_golden_mobilenet(golden, entry):
    """MobileNetV2 layer shapes (bench/convolution.cc:453-537) at batch 1 (the 112x112 ones only on the GPU side)."""
    case = CS.mobilenet_case(entry, 1)
    x, k, b, kw = U.conv_setup(case)
    y = O.convolution2d_nhwc_q8_np(x, k, b, **kw)
    assert U.digest(y) == str(golden[f"mnv2/{case['name']}/y_digest"])


# ---- (c) the compiled reference: recorded, and itself where it exists ------------------------------
@pytest.mark.parametrize("case", CS.OPERATOR_CASES[::4] + CS.DW_UKERNEL_CASES[::4], ids=lambda c: c["name"])
def test_compiled_reference_matches_golden(ref_lib, golden, case):
    x, k, b, kw = U.conv_setup(case)
    U.assert_same_bytes(U.run_conv(ref_lib, case, x, k, b, kw), golden[f"conv/{case['name']}/y"], case["name"])


@pytest.mark.parametrize("case", CS.DW_TC_CASES + CS.STEM_CASES + CS.PERSISTENT_CASES, ids=lambda c: c["name"])
def test_oracle_matches_compiled_reference_on_device_path_cases(oracle_c, case):
    """The GPU tests compare these shapes (tcgen05 depthwise classes, stem loaders, long item sequences) with the C oracle;
    here the oracle is pinned to the unmodified reference on exactly the same inputs."""
    x, k, b, kw = U.conv_setup(case)
    REF.expect(U.run_conv(oracle_c, case, x, k, b, kw), lambda l: U.run_conv(l, case, x, k, b, kw), case["name"])


def test_compiled_reference_q31_matches_oracle(oracle_c):
    rng = np.random.default_rng(3)
    x = rng.integers(-(2**31), 2**31, 1 << 16, dtype=np.int64).astype(np.int32)
    for scale, zp, qmin, qmax in ((0.75, 127, 1, 254), (2.0 ** -11 * 1.3, 3, 0, 255), (2.0 ** -31, 255, 0, 200)):
        got = oracle_c.requantize_q31(x, scale, zp, qmin, qmax)
        for variant in ("scalar", "sse2"):
            REF.expect(got, lambda l: l.requantize_q31(x, scale, zp, qmin, qmax, variant=variant), variant)
