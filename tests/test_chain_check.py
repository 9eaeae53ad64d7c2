"""CPU test of the chain gate itself (oracle/chain_check.py): the reference chain run as one batch (byte for byte what
the unmodified reference computed for it) must agree with the chain run image by image through check_graph, and a
corrupted byte must be reported."""
import numpy as np

from oracle import chain_check as CC
from qnnpack_b200 import mobilenet_v2 as M
from tests import reference as REF


def _run_reference_stack(lib, layers, params, batch, x):
    stack = M.Stack(lib, params=params, only=layers)
    cap = stack.max_activation_bytes(batch) + 64
    a, b = np.zeros(cap + 16, np.uint8), np.zeros(cap + 16, np.uint8)
    xin = np.zeros(x.size + 80, np.uint8)
    xin[16:16 + x.size] = x
    bufs = (a[16:], b[16:])
    stack.setup(batch, bufs[0], bufs[1], first_input=xin[16:])
    outs, rows = {}, {}
    def hook(i, after):
        l = layers[i]
        if l.kind == "fc":
            rows[(i, "in" if not after else "out")] = (bufs[(i - 1) % 2] if not after else bufs[i % 2]).copy()
        elif after:
            outs[i] = bufs[i % 2][: batch * l.out_elems_per_image].copy()
    stack.run(hook=hook)
    stack.delete()
    return outs, rows


def test_chain_gate_agrees_with_batched_reference_and_detects_corruption():
    layers = M.layers()[:7] + M.layers()[-2:]   # stem .. b2_dw is a chain; last_1x1 + classifier exercise the row-wise FC
    layers = M.layers()[:4]                     # keep the chain consistent: stem, b1_dw, b1_project, b2_expand
    params = M.make_params(seed=3, only=layers)
    batch = 3
    x = np.random.default_rng(0).integers(0, 256, batch * 224 * 224 * 3, dtype=np.uint8)
    lib, _ = CC._host_lib()
    outs, rows = _run_reference_stack(lib, layers, params, batch, x)
    lib.close()
    REF.expect([outs[i] for i in sorted(outs)], lambda l: [v for _, v in sorted(_run_reference_stack(l, layers, params, batch, x)[0].items())],
               "batched chain")
    e0 = layers[0].in_elems_per_image

    def fetch_out(i, im):
        e = layers[i].out_elems_per_image
        return outs[i][im * e:(im + 1) * e]

    res = CC.check_graph(layers, params, [0, 2], lambda im: x[im * e0:(im + 1) * e0], fetch_out, n_rows=batch)
    assert res["mismatches"] == 0 and res["layers"] == 4 and res["bytes_compared"] > 0
    outs[2][5] ^= 1
    res = CC.check_graph(layers, params, [0, 2], lambda im: x[im * e0:(im + 1) * e0], fetch_out, n_rows=batch)
    assert res["mismatches"] == 1 and res["failed_layers"][0]["layer"] == layers[2].name
