"""Border-class biases of the depthwise tensor-core kernel in shared memory (DwTcParams::bias_smem, q8_dwconv_umma_sm100.cu).

The planner lists the row classes of the layer's output rows and the column classes of its output columns, and the kernel
copies just those rows of bias_cls into a compact [slots][channels] table.  This replays, on the host, the kernel's two sides
of that table: the copy (slot -> class, from bias_rcls / bias_ccls) and the epilogue's lookup (class -> slot, from
bias_rslot / bias_cslot with the row stride bias_rstride), and checks that every output pixel reads the bias_cls row of its
own class, that every lookup stays inside the table, and that the table fits beside the plan."""
import ctypes as C

import numpy as np
import pytest

SMEM_OPTIN = 232448
CTL_RESERVE = 2048


@pytest.fixture(scope="module")
def lib():
    from qnnpack_b200 import build
    l = C.CDLL(build.build())
    l.qnnp_cuda_debug_plan_dwconv_bias.argtypes = [C.c_int] * 11 + [C.POINTER(C.c_int)]
    return l


def border_bits(o, s, pad, n):
    i0 = o * s - pad
    lo, hi = max(0, -i0), max(0, i0 + 3 - n)
    return 0 if hi >= 3 else ((7 << lo) & 7) & (7 >> hi)


def nib(packed, k):
    return (packed >> (4 * k)) & 15


def plan_bias(lib, c, n, h, w, s, pad, pair, wmode=3):
    oh, ow = (h + 2 * pad[0] - 3) // s + 1, (w + 2 * pad[1] - 3) // s + 1
    out = (C.c_int * 12)()
    if not lib.qnnp_cuda_debug_plan_dwconv_bias(c, n, h, w, oh, ow, s, pad[0], pad[1], wmode, pair, out):
        return None, oh, ow
    keys = "smem off rstride nrc ncc rslot cslot rcls ccls smem_total num_stages stage_bytes".split()
    return {k: int(v) & 0xFFFFFFFF if k in ("rslot", "cslot", "rcls", "ccls") else int(v) for k, v in zip(keys, out)}, oh, ow


def check_lookup(d, c, h, w, s, pad, oh, ow):
    """-> the [slots][c] table the kernel builds from a random bias_cls, after checking every produced pixel's lookup."""
    rng = np.random.default_rng(c + h * 31 + w)
    bias_cls = rng.integers(-(1 << 30), 1 << 30, (64, c), dtype=np.int64)
    slots = d["nrc"] * d["ncc"]
    table = np.stack([bias_cls[nib(d["rcls"], k // d["ncc"]) * 8 + nib(d["ccls"], k % d["ncc"])] for k in range(slots)])
    for oy in range(oh):
        rm = border_bits(oy, s, pad[0], h)
        for ox in range(ow):
            cm = border_bits(ox, s, pad[1], w)
            k = nib(d["rslot"], rm) * d["rstride"] + nib(d["cslot"], cm)
            assert k < slots
            assert np.array_equal(table[k], bias_cls[rm * 8 + cm]), (oy, ox, rm, cm)
    # rows and columns whose outputs are not stored (beyond the image, stacked-image halo) may compute any class bits: their
    # lookup must still land inside the table
    for b in range(8):
        assert nib(d["rslot"], b) * d["rstride"] + nib(d["cslot"], b) < slots
    return table


GEOMETRIES = [
    # (C, N, H, W, stride, pad)
    (32, 2, 112, 112, 1, (1, 1)), (96, 2, 112, 112, 2, (1, 1)), (144, 2, 56, 56, 1, (1, 1)), (192, 2, 28, 28, 1, (1, 1)),
    (192, 2, 28, 28, 2, (1, 1)), (576, 2, 14, 14, 1, (1, 1)), (960, 2, 7, 7, 1, (1, 1)),
    (64, 3, 1, 1, 1, (1, 1)), (64, 3, 2, 2, 1, (1, 1)), (32, 2, 1, 9, 1, (1, 1)), (32, 2, 9, 2, 1, (1, 1)),
    (48, 3, 2, 2, 2, (1, 1)), (32, 2, 9, 12, 1, (0, 0)), (16, 1, 18, 16, 2, (0, 0)), (48, 2, 11, 13, 1, (2, 1)),
    (32, 1, 5, 6, 2, (2, 2)), (176, 2, 18, 18, 1, (1, 1)),
]


@pytest.mark.parametrize("pair", [0, 1])
@pytest.mark.parametrize("c,n,h,w,s,pad", GEOMETRIES)
def test_compact_table_covers_every_class_the_geometry_produces(lib, c, n, h, w, s, pad, pair):
    d, oh, ow = plan_bias(lib, c, n, h, w, s, pad, pair)
    if d is None:
        assert pair and c < 32   # the pair form needs 32 channels
        return
    rset = {border_bits(oy, s, pad[0], h) for oy in range(oh)}
    cset = {border_bits(ox, s, pad[1], w) for ox in range(ow)}
    assert d["smem_total"] <= SMEM_OPTIN - CTL_RESERVE
    if d["smem"]:
        assert (d["nrc"], d["ncc"], d["rstride"]) == (len(rset), len(cset), len(cset))
        assert {nib(d["rcls"], k) for k in range(d["nrc"])} == rset and {nib(d["ccls"], k) for k in range(d["ncc"])} == cset
        assert d["off"] % 16 == 0 and d["off"] + d["nrc"] * d["ncc"] * c * 4 + 1024 == d["smem_total"]
        assert d["off"] >= d["num_stages"] * d["stage_bytes"]      # behind the ring (and the resident weights)
    else:  # the global table: slot = class bits
        assert (d["rstride"], d["nrc"], d["ncc"]) == (8, 8, 8)
    check_lookup(d, c, h, w, s, pad, oh, ow)


def test_nine_classes_for_padding_one(lib):
    """Padding <= 1 on images >= 3 pixels: top / interior / bottom rows times left / interior / right columns at stride 1."""
    d, oh, ow = plan_bias(lib, 144, 4096, 56, 56, 1, (1, 1), 1)
    assert d["smem"] == 1 and d["nrc"] * d["ncc"] == 9


def test_mobilenet_layers_that_carry_the_table(lib):
    """Which MobileNetV2 depthwise plans have room for the table (pair form where the router takes it, i.e. stride 2 or
    all weight blocks resident with >= 4 channel groups; else the 16-channel form) — the layers the go/no-go build sped up."""
    from qnnpack_b200 import mobilenet_v2 as M
    got = {}
    for l in M.layers():
        if l.kind != "dw":
            continue
        d = plan_bias(lib, l.cin, 4096, l.h, l.h, l.stride, (1, 1), 1)[0]
        got[l.name] = d["smem"]
    assert all(got[f"b{i}_dw"] for i in (1, 2, 3, 5, 6, 7))
