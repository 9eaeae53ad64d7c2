"""CPU: the NumPy restatement of the operators beside the convolution path (oracle/q8_ops_oracle.py) against what the
UNMODIFIED reference computed for the same calls (tests/reference.py) — the same formulas the CUDA kernels implement
(q8_eltwise_sm100.cu)."""
import numpy as np
import pytest

from oracle import q8_ops_oracle as OO
from oracle import q8_oracle as O
from tests import reference as REF, test_gpu_ops as T


@pytest.mark.parametrize("q", [dict(), dict(a_zp=0, b_zp=255, y_zp=3), dict(a_scale=0.25, b_scale=4.0, y_scale=1.3),
                               dict(qmin=128), dict(qmax=128), dict(a_scale=0.004, b_scale=2.3, y_scale=0.9)])
def test_add_restatement(q):
    rng = np.random.default_rng(1)
    batch, channels = 16, 256
    a, b = T._rows(rng, batch, channels, channels), T._rows(rng, batch, channels, channels)
    args = (channels, q.get("a_zp", 121), np.float32(q.get("a_scale", 0.75)), q.get("b_zp", 127), np.float32(q.get("b_scale", 1.25)),
            q.get("y_zp", 133), np.float32(q.get("y_scale", 1.96875)), q.get("qmin", 0), q.get("qmax", 255))
    p = OO.add_params(args[1], args[2], args[3], args[4], args[5], args[6], args[7], args[8])
    REF.expect(OO.add(a, b, p), lambda l: T._run_nc(l, "add_nc_q8", args, batch, channels, a, channels, channels, b, channels))


@pytest.mark.parametrize("width", [1, 7, 8, 49, 100])
def test_global_average_pooling_restatement(width):
    rng = np.random.default_rng(width)
    batch, channels = 3, 40
    x = np.zeros(16 + batch * width * channels + 16, np.uint8)
    xv = x[16:16 + batch * width * channels]
    xv[...] = rng.integers(0, 256, xv.size, dtype=np.uint8)
    for q in (dict(izp=121, ozp=133, qmin=0, qmax=255, **{"is": 1.0}, os=1.0), dict(izp=0, ozp=255, qmin=5, qmax=250, **{"is": 0.01}, os=1.7)):
        got = OO.global_average_pooling(xv.reshape(batch, width, channels), q["izp"], q["is"], q["ozp"], q["os"], q["qmin"], q["qmax"])
        REF.expect(got, lambda l: T._run_gavg(l, batch, width, channels, xv, channels, channels, q), str(q))


@pytest.mark.parametrize("case", T.POOL_CASES, ids=lambda c: "x".join(str(v) for v in c[:4]) + f"_p{c[7][0]}x{c[7][1]}")
@pytest.mark.parametrize("kind", ["avg", "max"])
def test_pooling_restatement(case, kind):
    n, h, w, c, xe, ye, pad, pool, stride, dil = case
    rng = np.random.default_rng(h + w + c)
    buf = np.zeros(16 + n * h * w * c + 16, np.uint8)
    x = buf[16:16 + n * h * w * c]
    x[...] = rng.integers(0, 256, x.size, dtype=np.uint8)
    dils = [(1, 1)] + ([(2, 2)] if kind == "max" and 2 * (pool[0] - 1) + 1 <= h and 2 * (pool[1] - 1) + 1 <= w else [])
    for d in dils:
        q = dict(izp=3, ozp=200, qmin=10, qmax=250, **{"is": 0.3}, os=0.11)
        got = OO.pool2d(x.reshape(n, h, w, c), kind, pad, pool, stride, d, q["izp"], q["is"], q["ozp"], q["os"], q["qmin"], q["qmax"])
        REF.expect(got, lambda l: T._run_pool(l, kind, n, h, w, c, c, c, x, pad, pool, stride, d, q), str(d))


@pytest.mark.parametrize("case", T.DECONV_CASES, ids=lambda c: f"{c[1]}x{c[2]}_g{c[3]}_k{c[8][0]}x{c[8][1]}_s{c[9][0]}x{c[9][1]}_d{c[10][0]}")
def test_deconvolution_restatement(case):
    n, h, w, groups, gic, goc, pad, adj, ks, stride, dil, ye = case
    rng = np.random.default_rng(h * 10 + w + gic)
    buf = np.zeros(16 + n * h * w * groups * gic + 16, np.uint8)
    x = buf[16:16 + n * h * w * groups * gic]
    x[...] = rng.integers(0, 256, x.size, dtype=np.uint8)
    k = rng.integers(0, 256, (groups, gic, ks[0], ks[1], goc), dtype=np.uint8)
    b = rng.integers(-10000, 10000, (groups * goc,), dtype=np.int32)
    q = dict(izp=127, kzp=127, ozp=127, qmin=0, qmax=255, os=float(ks[0] * ks[1] * gic * 40.0))
    acc = OO.deconv_accumulators(x.reshape(n, h, w, groups * gic), k, b, pad, adj, ks, stride, dil, groups, gic, goc, q["izp"], q["kzp"])
    scale = np.float32(1.0) * np.float32(1.0) / np.float32(q["os"])
    got = O.q31_requantize_np(acc.astype(np.int32), O.compute_requant_params(scale, q["ozp"], q["qmin"], q["qmax"]))
    REF.expect(got, lambda l: T._run_deconv(l, x, k, b, n, h, w, groups, gic, goc, pad, adj, ks, stride, dil, q, 0))
