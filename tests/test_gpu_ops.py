"""GPU parity of the operators beside the convolution path (SURVEY.md §8f rows 1, 3, 4) against what the UNMODIFIED
reference computed for the same calls (tests/reference.py): add, global average pooling, average / max pooling, clamp, sigmoid, leaky ReLU, softargmax,
channel shuffle, deconvolution.  Case grids restate test/add.cc, test/global-average-pooling.cc, test/average-pooling.cc,
test/max-pooling.cc, test/clamp.cc, test/sigmoid.cc, test/leaky-relu.cc, test/softargmax.cc, test/channel-shuffle.cc and
test/deconvolution.cc with fixed seeds (the reference draws from std::random_device).  Byte-exact, gaps between rows
(0xA5 canary) untouched."""
import numpy as np
import pytest

from tests import reference as REF

pytestmark = pytest.mark.gpu


def _rows(rng, batch, channels, stride):
    x = rng.integers(0, 256, (batch, stride), dtype=np.uint8)
    return x


def _run_nc(lib, name, create_args, batch, channels, x, x_stride, y_stride, x2=None, x2_stride=None):
    st, op = lib.create(name, *create_args)
    assert st == 0, (name, st)
    y = np.full((batch, y_stride), 0xA5, np.uint8)
    lead = np.zeros(16 + x.size + 16, np.uint8)
    xin = lead[16:16 + x.size].reshape(x.shape)
    xin[...] = x
    if x2 is not None:
        lead2 = np.zeros(16 + x2.size + 16, np.uint8)
        x2in = lead2[16:16 + x2.size].reshape(x2.shape)
        x2in[...] = x2
        st = lib.setup(name, op, batch, xin, x_stride, x2in, x2_stride, y, y_stride)
    else:
        st = lib.setup(name, op, batch, xin, x_stride, y, y_stride)
    assert st == 0, (name, "setup", st)
    assert lib.run(op) == 0
    lib.delete(op)
    return y


NC_SHAPES = [(1, 1, 0, 0), (1, 100, 0, 0), (3, 5, 0, 0), (3, 100, 0, 0), (3, 100, 29, 0), (3, 100, 0, 17), (5, 64, 0, 0),
             (7, 37, 3, 5), (64, 1280, 0, 0), (33, 160, 0, 0)]


@pytest.mark.parametrize("batch,channels,xe,ye", NC_SHAPES)
@pytest.mark.parametrize("q", [dict(), dict(a_zp=0, b_zp=255, y_zp=3), dict(a_scale=0.25, b_scale=4.0, y_scale=1.3),
                               dict(qmin=128), dict(qmax=128), dict(a_scale=0.004, b_scale=2.3, y_scale=0.9)])
def test_add(gpu_lib, batch, channels, xe, ye, q):
    rng = np.random.default_rng(batch * 1000 + channels)
    a = _rows(rng, batch, channels, channels + xe)
    b = _rows(rng, batch, channels, channels + xe + 1)
    args = (channels, q.get("a_zp", 121), np.float32(q.get("a_scale", 0.75)), q.get("b_zp", 127), np.float32(q.get("b_scale", 1.25)),
            q.get("y_zp", 133), np.float32(q.get("y_scale", 1.96875)), q.get("qmin", 0), q.get("qmax", 255))
    def run(l):
        return _run_nc(l, "add_nc_q8", args, batch, channels, a, channels + xe, channels + ye, b, channels + xe + 1)
    got = run(gpu_lib)
    REF.expect(got, run)
    assert (got[:, channels:] == 0xA5).all()


@pytest.mark.parametrize("batch,channels,xe,ye", NC_SHAPES)
def test_clamp_lut_ops(gpu_lib, batch, channels, xe, ye):
    rng = np.random.default_rng(batch * 77 + channels)
    x = _rows(rng, batch, channels, channels + xe)
    cases = [("clamp_nc_u8", (channels, 0, 255)), ("clamp_nc_u8", (channels, 128, 255)), ("clamp_nc_u8", (channels, 17, 200)),
             ("sigmoid_nc_q8", (channels, 121, np.float32(0.75), 0, np.float32(1.0 / 256.0), 0, 255)),
             ("sigmoid_nc_q8", (channels, 0, np.float32(0.03), 0, np.float32(1.0 / 256.0), 128, 250)),
             ("leaky_relu_nc_q8", (channels, np.float32(0.1), 121, np.float32(0.75), 133, np.float32(0.75), 0, 255)),
             ("leaky_relu_nc_q8", (channels, np.float32(0.5), 3, np.float32(1.25), 200, np.float32(0.3), 9, 250)),
             ("softargmax_nc_q8", (channels, np.float32(0.176080), 0, np.float32(1.0 / 256.0))),
             ("softargmax_nc_q8", (channels, np.float32(0.01), 0, np.float32(1.0 / 256.0)))]
    for name, args in cases:
        got = _run_nc(gpu_lib, name, args, batch, channels, x, channels + xe, channels + ye)
        REF.expect(got, lambda l: _run_nc(l, name, args, batch, channels, x, channels + xe, channels + ye), f"{name}{args}")
        assert (got[:, channels:] == 0xA5).all()


@pytest.mark.parametrize("groups,gc", [(2, 1), (2, 37), (3, 5), (4, 16), (5, 7), (7, 24), (2, 160)])
@pytest.mark.parametrize("batch,xe,ye", [(1, 0, 0), (3, 0, 0), (3, 5, 0), (3, 0, 9)])
def test_channel_shuffle(gpu_lib, groups, gc, batch, xe, ye):
    channels = groups * gc
    rng = np.random.default_rng(groups * 100 + gc)
    x = _rows(rng, batch, channels, channels + xe)
    def run(l):
        return _run_nc(l, "channel_shuffle_nc_x8", (groups, gc), batch, channels, x, channels + xe, channels + ye)
    got = run(gpu_lib)
    REF.expect(got, run)
    want = x[:, :channels].reshape(batch, groups, gc).transpose(0, 2, 1).reshape(batch, channels)
    assert np.array_equal(got[:, :channels], want)


def _run_gavg(lib, batch, width, channels, x, x_stride, y_stride, q):
    st, op = lib.create("global_average_pooling_nwc_q8", channels, q["izp"], np.float32(q["is"]), q["ozp"], np.float32(q["os"]),
                        q["qmin"], q["qmax"])
    assert st == 0
    y = np.full((batch, y_stride), 0xA5, np.uint8)
    assert lib.setup("global_average_pooling_nwc_q8", op, batch, width, x, x_stride, y, y_stride) == 0
    assert lib.run(op) == 0
    lib.delete(op)
    return y


@pytest.mark.parametrize("batch,width,channels,xe,ye", [(1, 1, 1, 0, 0), (1, 7, 8, 0, 0), (1, 49, 1280, 0, 0), (3, 49, 160, 0, 0),
                                                        (3, 5, 13, 4, 0), (3, 8, 24, 0, 5), (2, 14, 9, 0, 0), (5, 100, 36, 0, 0),
                                                        (2, 7, 1, 0, 0), (4, 23, 128, 8, 8)])
@pytest.mark.parametrize("q", [dict(), dict(izp=0, ozp=255), dict(**{"is": 0.01}, os=1.7), dict(qmin=128), dict(qmax=128)])
def test_global_average_pooling(gpu_lib, batch, width, channels, xe, ye, q):
    qq = dict(izp=121, ozp=133, qmin=0, qmax=255, **{"is": 1.0}, os=1.0)
    qq.update(q)
    rng = np.random.default_rng(width * 31 + channels)
    xs = channels + xe
    x = np.zeros(16 + batch * width * xs + 16, np.uint8)
    xv = x[16:16 + batch * width * xs]
    xv[...] = rng.integers(0, 256, xv.size, dtype=np.uint8)
    def run(l):
        return _run_gavg(l, batch, width, channels, xv, xs, channels + ye, qq)
    REF.expect(run(gpu_lib), run)


def _run_pool(lib, kind, n, h, w, c, xs, ys, x, pad, pool, stride, dil, q):
    if kind == "avg":
        st, op = lib.create("average_pooling2d_nhwc_q8", *pad, *pool, *stride, c, q["izp"], np.float32(q["is"]), q["ozp"],
                            np.float32(q["os"]), q["qmin"], q["qmax"])
        name = "average_pooling2d_nhwc_q8"
    else:
        st, op = lib.create("max_pooling2d_nhwc_u8", *pad, *pool, *stride, *dil, c, q["qmin"], q["qmax"])
        name = "max_pooling2d_nhwc_u8"
    assert st == 0
    d = (1, 1) if kind == "avg" else dil
    oh = (pad[0] + h + pad[2] - ((pool[0] - 1) * d[0] + 1)) // stride[0] + 1
    ow = (pad[3] + w + pad[1] - ((pool[1] - 1) * d[1] + 1)) // stride[1] + 1
    y = np.full((n, oh, ow, ys), 0xA5, np.uint8)
    assert lib.setup(name, op, n, h, w, x, xs, y, ys, threadpool=True) == 0
    assert lib.run(op) == 0
    lib.delete(op)
    return y


POOL_CASES = [
    # n, h, w, c, xe, ye, pad(t, r, b, l), pool, stride, dilation
    (1, 7, 7, 8, 0, 0, (0, 0, 0, 0), (7, 7), (1, 1), (1, 1)),
    (1, 12, 13, 8, 0, 0, (0, 0, 0, 0), (2, 2), (2, 2), (1, 1)),
    (2, 12, 13, 24, 0, 0, (1, 1, 1, 1), (3, 3), (2, 2), (1, 1)),
    (1, 9, 11, 17, 3, 5, (1, 0, 0, 1), (3, 2), (1, 2), (1, 1)),
    (1, 14, 14, 64, 0, 0, (0, 1, 1, 0), (3, 3), (1, 1), (1, 1)),
    (3, 10, 9, 5, 0, 0, (2, 2, 2, 2), (5, 5), (3, 3), (1, 1)),
    (1, 8, 8, 1, 0, 0, (0, 0, 0, 0), (1, 3), (1, 1), (1, 1)),
    (1, 16, 16, 100, 0, 0, (1, 1, 1, 1), (3, 3), (2, 2), (1, 1)),
]


@pytest.mark.parametrize("case", POOL_CASES, ids=lambda c: "x".join(str(v) for v in c[:4]) + f"_p{c[7][0]}x{c[7][1]}")
@pytest.mark.parametrize("kind", ["avg", "max"])
def test_pooling(gpu_lib, case, kind):
    n, h, w, c, xe, ye, pad, pool, stride, dil = case
    rng = np.random.default_rng(h * 100 + w + c)
    xs, ys = c + xe, c + ye
    buf = np.zeros(16 + n * h * w * xs + 16, np.uint8)
    x = buf[16:16 + n * h * w * xs]
    x[...] = rng.integers(0, 256, x.size, dtype=np.uint8)
    for q in (dict(), dict(izp=3, ozp=200, **{"is": 0.3}, os=0.11), dict(qmin=100, qmax=180)):
        qq = dict(izp=121, ozp=133, qmin=0, qmax=255, **{"is": 1.0}, os=1.0)
        qq.update(q)
        got = _run_pool(gpu_lib, kind, n, h, w, c, xs, ys, x, pad, pool, stride, dil, qq)
        REF.expect(got, lambda l: _run_pool(l, kind, n, h, w, c, xs, ys, x, pad, pool, stride, dil, qq), f"{kind} {q}")
    if kind == "max":  # dilated windows: padded taps read the clamped edge pixel (src/indirection.c:218-224)
        for d in ((2, 2), (1, 3)):
            if (pool[0] - 1) * d[0] + 1 <= h + pad[0] + pad[2] and (pool[1] - 1) * d[1] + 1 <= w + pad[1] + pad[3]:
                qq = dict(qmin=0, qmax=255)
                got = _run_pool(gpu_lib, kind, n, h, w, c, xs, ys, x, pad, pool, stride, d, qq)
                REF.expect(got, lambda l: _run_pool(l, kind, n, h, w, c, xs, ys, x, pad, pool, stride, d, qq), f"max dilated {d}")


def _run_deconv(lib, x, k, b, n, h, w, groups, gic, goc, pad, adj, ks, stride, dil, q, ye):
    st, op = lib.create("deconvolution2d_nhwc_q8", *pad, *adj, *ks, *stride, *dil, groups, gic, goc, q["izp"], np.float32(1.0),
                        q["kzp"], np.float32(1.0), k, b, q["ozp"], np.float32(q["os"]), q["qmin"], q["qmax"])
    assert st == 0, st
    oh = stride[0] * (h - 1) + adj[0] + (ks[0] - 1) * dil[0] + 1 - (pad[0] + pad[2])
    ow = stride[1] * (w - 1) + adj[1] + (ks[1] - 1) * dil[1] + 1 - (pad[1] + pad[3])
    ys = groups * goc + ye
    y = np.full((n, oh, ow, ys), 0xA5, np.uint8)
    assert lib.setup("deconvolution2d_nhwc_q8", op, n, h, w, x, groups * gic, y, ys, threadpool=True) == 0
    assert lib.run(op) == 0
    lib.delete(op)
    return y


DECONV_CASES = [
    # n, h, w, groups, gic, goc, pad, adj, ks, stride, dil, ye
    (1, 8, 9, 1, 15, 17, (0, 0, 0, 0), (0, 0), (1, 1), (1, 1), (1, 1), 0),
    (1, 8, 9, 1, 15, 17, (1, 1, 1, 1), (0, 0), (3, 3), (1, 1), (1, 1), 0),
    (2, 7, 6, 1, 11, 13, (1, 1, 1, 1), (0, 0), (3, 3), (2, 2), (1, 1), 0),
    (1, 7, 6, 1, 11, 13, (1, 1, 1, 1), (1, 1), (3, 3), (2, 2), (1, 1), 5),
    (1, 7, 6, 2, 5, 7, (0, 1, 1, 0), (0, 1), (3, 2), (2, 3), (1, 1), 0),
    (1, 6, 7, 1, 9, 8, (2, 2, 2, 2), (0, 0), (3, 3), (1, 1), (2, 2), 0),
    (1, 5, 5, 1, 32, 16, (0, 0, 0, 0), (0, 0), (2, 2), (2, 2), (1, 1), 0),
]


@pytest.mark.parametrize("case", DECONV_CASES, ids=lambda c: f"{c[1]}x{c[2]}_g{c[3]}_k{c[8][0]}x{c[8][1]}_s{c[9][0]}x{c[9][1]}_d{c[10][0]}")
def test_deconvolution(gpu_lib, case):
    n, h, w, groups, gic, goc, pad, adj, ks, stride, dil, ye = case
    rng = np.random.default_rng(h * 10 + w + gic)
    buf = np.zeros(16 + n * h * w * groups * gic + 16, np.uint8)
    x = buf[16:16 + n * h * w * groups * gic]
    x[...] = rng.integers(0, 256, x.size, dtype=np.uint8)
    k = rng.integers(0, 256, (groups, gic, ks[0], ks[1], goc), dtype=np.uint8)
    b = rng.integers(-10000, 10000, (groups * goc,), dtype=np.int32)
    for q in (dict(), dict(izp=0, kzp=255), dict(qmin=128), dict(qmax=128)):
        qq = dict(izp=127, kzp=127, ozp=127, qmin=0, qmax=255, os=float(ks[0] * ks[1] * gic * 40.0))
        qq.update(q)
        got = _run_deconv(gpu_lib, x, k, b, n, h, w, groups, gic, goc, pad, adj, ks, stride, dil, qq, ye)
        REF.expect(got, lambda l: _run_deconv(l, x, k, b, n, h, w, groups, gic, goc, pad, adj, ks, stride, dil, qq, ye), str(q))
