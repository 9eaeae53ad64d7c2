"""TEST INFRASTRUCTURE — byte-exact gate on a whole operator chain at ANY batch size.

The product runs the MobileNetV2 operator graph at the benchmark's batch (4096 images per GPU); its
intermediate tensors are gigabytes, far beyond what the CPU oracle can recompute.  Every operator of the
graph is independent per image, though, so a handful of SAMPLED images pin the run: their input slices go
through the UNMODIFIED reference (oracle/_ref, reference's own SSE2 kernels; or the C restatement when
_ref is absent) layer by layer, and every layer's output slice of those images, copied back from the GPU
buffers, must equal the reference's bytes.  What "expected" means: reference
test/convolution-operator-tester.h:367-464 (accumulate, requantise, clamp) — here produced by the
reference's operators themselves.

Used by bench.py (outside the timed region, "parity_check" in the JSON line) and tests/test_gpu_chain.py.
Never imported by the product package.
"""
from __future__ import annotations

import numpy as np

from qnnpack_b200 import mobilenet_v2 as M


class _OracleOp:
    def __init__(self, kind, args):
        self.kind, self.args, self.io = kind, args, None


class OracleHost:
    """The operators of the MobileNetV2 graph (convolution, fully connected, add, global average pooling) on the C oracle
    and the NumPy restatement of the eltwise operators, behind the part of the qnnpack.h driver that the gate uses.
    Both restatements are pinned to the unmodified reference by the CPU tests (tests/test_oracle.py,
    tests/test_ops_oracle.py), so this is the reference chain wherever oracle/_ref has not been built."""

    def __init__(self):
        from oracle import q8_oracle as O
        self.c = O.COracle()

    def create_convolution(self, kernel, bias, **kw):
        return 0, _OracleOp("conv", (np.array(kernel, np.uint8), np.array(bias, np.int32), kw))

    def create_fully_connected(self, kernel, bias, **kw):
        return 0, _OracleOp("fc", (np.array(kernel, np.uint8), np.array(bias, np.int32), kw))

    def create(self, name, *args):
        return 0, _OracleOp(name, args)

    def setup_convolution(self, op, batch, in_h, in_w, x, in_stride, out, out_stride):
        op.io = (batch, in_h, in_w, x, in_stride, out, out_stride)
        return 0

    def setup_fully_connected(self, op, batch, x, in_stride, out, out_stride):
        op.io = (batch, x, in_stride, out, out_stride)
        return 0

    def setup(self, name, op, *args):
        op.io = args
        return 0

    def run(self, op):
        from oracle import q8_ops_oracle as OPS
        if op.kind == "conv":
            (n, h, w, x, xs, out, ys), (k, b, kw) = op.io, op.args
            y = self.c.convolution(x[:n * h * w * xs].reshape(n, h, w, xs), k, b, out_stride=ys, **kw)
        elif op.kind == "fc":
            (n, x, xs, out, ys), (k, b, kw) = op.io, op.args
            y = self.c.fully_connected(x[:n * xs].reshape(n, xs), k, b, out_stride=ys, **kw)
        elif op.kind == "add_nc_q8":
            (n, a, a_s, b, b_s, out, ys), (c, *q) = op.io, op.args
            assert a_s == b_s == ys == c
            y = OPS.add(a[:n * c], b[:n * c], OPS.add_params(*q))
        elif op.kind == "global_average_pooling_nwc_q8":
            (n, width, x, xs, out, ys), (c, izp, iscale, ozp, oscale, qmin, qmax) = op.io, op.args
            assert xs == ys == c
            y = OPS.global_average_pooling(x[:n * width * c].reshape(n, width, c), izp, iscale, ozp, oscale, qmin, qmax)
        else:
            raise NotImplementedError(op.kind)
        out[:y.size] = y.reshape(-1)
        return 0

    def delete(self, op):
        return 0

    def close(self):
        pass


def _host_lib():
    from oracle import ref as R
    if R.available():
        return R.QnnpackHost(), "oracle/_ref (unmodified reference, SSE2 ukernels)"
    return OracleHost(), "oracle/q8_oracle.c + q8_ops_oracle.py (restatements pinned to the reference)"


def _srcs(nodes, i):
    """Producers of node i's inputs (-1 = the network input).  The conv stack is a plain chain."""
    return M.node_srcs(nodes, i)


class ReferenceChain:
    """The graph's operators created once in the reference library; run() pushes a few images through them."""

    def __init__(self, nodes, params):
        self.lib, self.kind = _host_lib()
        self.nodes = nodes
        self.ops = []
        for node, (kernel, bias) in zip(nodes, params):
            self.ops.append(M.create_node(self.lib, node, kernel, bias))

    def close(self):
        for op in self.ops:
            if op is not None:
                self.lib.delete(op)
        self.lib.close()

    def run_node(self, i, inputs, n):
        """inputs: list of uint8 arrays [n, ...] (NHWC slices of the n sampled images) -> output array."""
        node = self.nodes[i]
        lead = 16  # the reference's SSE2 tails may read a few bytes before a row (src/q8gemm/4x4c2-sse2.c:111-121)
        bufs = []
        for x in inputs:
            b = np.zeros(lead + x.size + 64, np.uint8)
            b[lead:lead + x.size] = x.reshape(-1)
            bufs.append(b[lead:lead + x.size])
        out = np.zeros(n * node.out_elems_per_image + 64, np.uint8)
        M.setup_node(self.lib, node, self.ops[i], n, bufs, out)
        st = self.lib.run(self.ops[i])
        if st != 0:
            raise RuntimeError(f"reference run {node.name} -> status {st}")
        return out[: n * node.out_elems_per_image].copy()


def check_graph(nodes, params, images, fetch_input, fetch_output, fetch_rows=None, n_rows=0, log=None):
    """nodes: M.Layer list in execution order; params: [(kernel, bias)] per node.
    images: sampled image indices.  fetch_input(image) -> the network input slice of that image (uint8).
    fetch_output(i, image) -> output slice of node i for that image as the device produced it.
    fetch_rows(i, "in"|"out", row) -> the conv stack's classifier takes ROWS of the flat previous output, not images:
    one row of its input / output buffer as the device holds it (checked in isolation, input from the device).
    Returns the "parity_check" dict; mismatches > 0 means the device differs from the reference somewhere."""
    chain = ReferenceChain(nodes, params)
    n = len(images)
    ref_out = {}
    per_layer = []
    mism_total = 0
    bytes_total = 0
    try:
        x0 = np.stack([np.asarray(fetch_input(im), np.uint8).reshape(-1) for im in images])
        for i, node in enumerate(nodes):
            if node.kind == "fc" and node.rowwise:
                # rows of the flat previous output, not images: checked in isolation on rows fetched from the device
                rows = sorted({r for r in [0, 1, 48] + list(images) if r < n_rows})
                xin = np.stack([fetch_rows(i, "in", r) for r in rows])
                want = chain.run_node(i, [xin], len(rows)).reshape(len(rows), -1)
                got = np.stack([fetch_rows(i, "out", r) for r in rows])
            else:
                ins = [x0 if s < 0 else ref_out[s] for s in _srcs(nodes, i)]
                want = chain.run_node(i, ins, n).reshape(n, -1)
                ref_out[i] = want
                got = np.stack([np.asarray(fetch_output(i, im), np.uint8).reshape(-1) for im in images])
            bad = int(np.count_nonzero(got != want))
            mism_total += bad
            bytes_total += int(want.size)
            per_layer.append({"layer": node.name, "bytes": int(want.size), "mismatches": bad})
            if log is not None and bad:
                log(f"parity_check: {node.name}: {bad} of {want.size} bytes differ")
            # keep only what later nodes still need
            live = {s for j in range(i + 1, len(nodes)) for s in _srcs(nodes, j)}
            for k in list(ref_out):
                if k not in live:
                    del ref_out[k]
    finally:
        chain.close()
    return {"images": [int(v) for v in images], "layers": len(nodes), "bytes_compared": bytes_total,
            "mismatches": mism_total, "oracle": chain.kind,
            "failed_layers": [p for p in per_layer if p["mismatches"]]}


def check_device_stack(stack, params, batch, x_in, buf_a, buf_b, images, log=None):
    """Runs `stack` (qnnpack_b200.mobilenet_v2.Stack on the product library, already set up with first_input = x_in
    and the ping-pong buffers buf_a / buf_b: torch uint8 CUDA tensors) ONCE more, asynchronously, exactly as the
    benchmark does, copies the sampled images' slice of every layer's output back right after that layer, and compares
    them with the reference chain.  -> "parity_check" dict."""
    import torch

    layers = stack.layers
    bufs = (buf_a, buf_b)
    got = {}
    rows = {}
    fc_rows = sorted({r for r in [0, 1, 48] + list(images) if r < batch})

    def hook(i, after):
        l = layers[i]
        out = bufs[i % 2]  # first_input given: layer 0 writes buf_a, layer 1 buf_b, ...
        if not after:
            if l.kind == "fc":
                src = bufs[(i - 1) % 2]
                rows[(i, "in")] = {r: src[r * l.cin:(r + 1) * l.cin].cpu().numpy() for r in fc_rows}
            return
        if l.kind == "fc":
            rows[(i, "out")] = {r: out[r * l.cout:(r + 1) * l.cout].cpu().numpy() for r in fc_rows}
        else:
            e = l.out_elems_per_image
            got[i] = {im: out[im * e:(im + 1) * e].cpu().numpy() for im in images}

    stack.run(asynchronous=True, hook=hook)
    torch.cuda.synchronize()
    e0 = layers[0].in_elems_per_image
    res = check_graph(layers, params, images,
                      fetch_input=lambda im: x_in[im * e0:(im + 1) * e0].cpu().numpy(),
                      fetch_output=lambda i, im: got[i][im],
                      fetch_rows=lambda i, which, r: rows[(i, which)][r], n_rows=batch, log=log)
    res["batch"] = int(batch)
    return res


def check_device_network(net, params, batch, x_in, buffers, images, log=None):
    """The same gate for the real MobileNetV2 graph (qnnpack_b200.mobilenet_v2.Network: residual adds, global average
    pool, per-image classifier): `buffers` are the torch uint8 CUDA tensors the network was set up with."""
    import torch

    layers = net.layers
    got = {}

    def hook(i, after):
        if after:
            e = layers[i].out_elems_per_image
            out = buffers[net.assign[i]]
            got[i] = {im: out[im * e:(im + 1) * e].cpu().numpy() for im in images}

    net.run(asynchronous=True, hook=hook)
    torch.cuda.synchronize()
    e0 = layers[0].in_elems_per_image
    res = check_graph(layers, params, images, fetch_input=lambda im: x_in[im * e0:(im + 1) * e0].cpu().numpy(),
                      fetch_output=lambda i, im: got[i][im], n_rows=batch, log=log)
    res["batch"] = int(batch)
    return res
