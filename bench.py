#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native q8 hot path (contract: task statement §④ + base contract).

Workload ("step"): one pass of the MobileNetV2-int8 convolution stack — 52 convolutions + classifier,
the layer list of the reference's bench/convolution.cc:453-537 in network order, 300.8 MMAC/image —
over a batch of 4096 synthetic 224x224x3 images PER GPU (BASELINE.json configs[4] is this stack with
the batch sharded over GPUs; configs[1..3], the q8gemm sweep / all conv layers / the depthwise
layers, are subsets of it and are reported from the same timed region in "q8gemm_sweep" and
"per_kernel").  Every operator runs through the qnnpack.h C ABI of libqnnpack.so.

  value    images/s, whole job, inputs resident in HBM, device-timed with CUDA events, max over ranks
  e2e      the same through the same C-ABI calls but with the batch coming from pinned HOST memory and
           the logits read back to the host inside the timed region
  roofline the dominant launch of the step: its algorithmic bytes / its CUDA-event time vs the measured HBM copy
           bandwidth (MEASURED_PEAKS.json); traffic = DRAM bytes of that launch from the committed ncu capture
  cpu_baseline / --impl reference: the UNMODIFIED reference (oracle/_ref, its own SSE2 kernels and
           operator API, pthreadpool over all host cores) on a bounded sample of the same workload

Multi-GPU: one process per GPU (torchrun); the batch dimension shards, the model parameters live on rank 0 and
are replicated with one NCCL broadcast, then every rank packs its own operators; no collective in the timed steps.
"""
from __future__ import annotations

import argparse
import json
import os
import socket
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# dram__bytes_read.sum + dram__bytes_write.sum per launch at batch 4096, from the committed ncu --set full captures
NCU_DRAM_BYTES_PER_LAUNCH = {"stem": 2.209e9, "b1_project": 2.435e9, "b2_expand": 5.705e9, "b1_dw": 3.239e9, "b2_dw": 6.170e9,
                             "b3_dw": 3.791e9}
NCU_DRAM_SOURCE = {"stem": "profiles/r2w_igemm_first3.summary.txt", "b1_project": "profiles/r2w_igemm_first3.summary.txt",
                   "b2_expand": "profiles/r2w_igemm_first3.summary.txt", "b1_dw": "profiles/r2w_dw_umma_first3.summary.txt",
                   "b2_dw": "profiles/r2w_dw_umma_first3.summary.txt", "b3_dw": "profiles/r2w_dw_umma_first3.summary.txt"}
INT8_PEAK_TOPS_NOMINAL = 4500.0  # B200 dense int8 (task statement; not in MEASURED_PEAKS.json)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="images per GPU")
    ap.add_argument("--cpu-batch", type=int, default=0, help="reference arm: images per step (0 = 2 per thread)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip int8 peak / tensor-bound GEMM / latency / host-pointer runs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the logits of the last timed step (rank 0) to DIR/logits.npy "
                    "as float32 [images, 1000]; beyond 64 MB a fixed sample of images, whose indices go to DIR/logits_rows.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.batch < 1:
        ap.error("--steps and --batch must be at least 1, --warmup at least 0")
    return args


DUMP_BYTES_MAX = 64 << 20


def dump_logits(logits, out_dir):
    """logits: uint8 [images, classes] on the host -> DIR/logits.npy (float32), a seeded sample of rows beyond 64 MB."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n, classes = logits.shape
    keep = DUMP_BYTES_MAX // (classes * 4)
    if n > keep:
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        logits = logits[rows]
        np.save(os.path.join(out_dir, "logits_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "logits.npy"), logits.astype(np.float32))


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified compiled reference on the host cores
# ------------------------------------------------------------------------------------------------
def run_reference_stack(steps, warmup, batch, threads):
    import numpy as np
    from oracle import ref as R
    from qnnpack_b200 import mobilenet_v2 as M

    if not R.available():
        raise RuntimeError("oracle/_ref/libqnnpack_ref.so is missing (build it with `make -C oracle ref`)")
    lib = R.QnnpackHost(threads=threads)
    stack = M.Stack(lib, seed=0)
    cap = stack.max_activation_bytes(batch) + 64
    x = np.random.default_rng(1).integers(0, 256, batch * 224 * 224 * 3 + 64, dtype=np.uint8)
    a = np.zeros(cap, np.uint8)
    b = np.zeros(cap, np.uint8)
    stack.setup(batch, a[16:], b[16:], first_input=x[16:])
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        stack.run()
        times.append(time.perf_counter() - t0)
    stack.delete()
    lib.close()
    t = times[warmup:]
    return batch * len(t) / sum(t), sum(t) / len(t)


def reference_main(args, rank, world):
    if rank != 0:
        return
    threads = usable_threads()
    batch = args.cpu_batch or max(16, 2 * threads)
    steps, warmup = max(1, min(args.steps, 5)), max(1, min(args.warmup, 2))
    ips, sec = run_reference_stack(steps, warmup, batch, threads)
    line = {
        "impl": "reference", "metric": "mobilenet_v2_int8_conv_stack_images_per_sec", "value": ips, "unit": "images/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "MobileNetV2-int8 conv stack, 53 operators (BASELINE.json configs[4]; bounded CPU sample)",
                   "batch_per_step": batch, "threads": threads, "host": host_info()},
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": threads, "kind": "reference",
                         "sample": f"{steps} passes of the full 53-operator stack over {batch} images, "
                                   f"unmodified reference (SSE2 ukernels) via oracle/_ref with a {threads}-thread pthreadpool"},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}



def host_info():
    """CPU model, cgroup CPU quota and usable cores of the box (explains the reference arm's box-to-box spread)."""
    info = {"os_cpu_count": os.cpu_count()}
    try:
        info["sched_affinity"] = len(os.sched_getaffinity(0))
    except AttributeError:
        pass
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                info["model"] = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cgroup_" + os.path.basename(path)] = open(path).read().strip()
        except OSError:
            pass
    return info


def usable_threads():
    """Threads the reference arm should use: the cgroup's CPU share when one is set, else the affinity mask."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def measure_tensor_bound_gemm(lib, torch, dev, peak_tops, m=65536, n=4096, k=4096, reps=5, sustained_s=1.5, peak_sustained=None):
    """BASELINE.json metric 1 where the tensor pipe can bind: q8gemm through qnnp_fully_connected_nc_q8 at
    M = 65536, N = K = 4096 (arithmetic intensity 2MNK / (MK + NK + MN) = 3.9 k ops/byte, far above the ridge), device
    pointers, CUDA events; a few output rows are checked bit for bit against the C oracle."""
    import numpy as np
    from oracle import q8_oracle as O
    rng = np.random.default_rng(5)
    w = rng.integers(0, 256, (n, k), dtype=np.uint8)
    b = rng.integers(-10000, 10000, (n,), dtype=np.int32)
    kw = dict(izp=127, input_scale=1.0, kzp=127, kernel_scale=float(np.float32(1.0 / (128.0 * k ** 0.5))), ozp=127, output_scale=1.0)
    st, op = lib.create_fully_connected(w, b, **kw)
    if st != 0:
        return {"error": f"create status {st}"}
    x = torch.randint(0, 256, (m * k,), dtype=torch.uint8, device=dev)
    y = torch.empty(m * n, dtype=torch.uint8, device=dev)
    assert lib.setup_fully_connected(op, m, x.data_ptr(), k, y.data_ptr(), n) == 0
    torch.cuda.synchronize()
    for _ in range(2):
        assert lib.run_async(op) == 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.current_stream()
    e0.record(stream)
    for _ in range(reps):
        assert lib.run_async(op) == 0
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    # the same launch back to back for ~sustained_s seconds: the 1 kW power cap pulls the SM clock down under a saturated
    # tensor pipe (MEASURED_PEAKS.json: bf16 1717 burst / 1472 sustained), so both regimes are reported
    n_sus = max(reps, int(sustained_s * 1e3 / ms))
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    e0.record(stream)
    for _ in range(n_sus):
        assert lib.run_async(op) == 0
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms_sus = e0.elapsed_time(e1) / n_sus
    rows = [0, 1, m // 2 - 1, m - 1]
    xr = np.stack([x[r * k:(r + 1) * k].cpu().numpy() for r in rows])
    want = O.COracle().fully_connected(xr, w, b, **kw)
    got = np.stack([y[r * n:(r + 1) * n].cpu().numpy() for r in rows])
    lib.delete(op)
    tops = 2.0 * m * n * k / ms / 1e9
    tops_sus = 2.0 * m * n * k / ms_sus / 1e9
    return {"m": m, "n": n, "k": k, "ms": ms, "tops": tops, "frac": tops / peak_tops if peak_tops else None,
            "sustained": {"launches": n_sus, "ms": ms_sus, "tops": tops_sus, "frac_of_sustained_peak": tops_sus / peak_sustained if peak_sustained else None,
                          "clocks": clocks},
            "kernel": "q8_gemm2sm_kernel (CTA pairs, cta_group::2 UMMA 256x256x32, SW128 TMA operands)",
            "rows_checked": rows, "mismatches": int(np.count_nonzero(got != want))}


def measure_hbm_by_mix(torch, dev, nbytes=4 << 30, reps=5):
    """HBM bandwidth by access mix, measured live with the device's own fill / copy engines' kernels (torch memset and
    copy): a WRITE-ONLY stream tops out far below the read+write copy figure that MEASURED_PEAKS.json holds, which is what
    bounds the write-heavy 1x1 expansions (6 bytes written per byte read)."""
    x = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    y = torch.empty(nbytes, dtype=torch.uint8, device=dev)

    def timed(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    w_ms = timed(lambda: x.zero_())
    c_ms = timed(lambda: y.copy_(x))
    del x, y
    torch.cuda.empty_cache()
    return {"write_only_gbs": nbytes / 1e6 / w_ms, "copy_gbs": 2 * nbytes / 1e6 / c_ms, "bytes": nbytes,
            "how": "torch memset / device-to-device copy of 4 GiB, CUDA events"}


def measure_small_batch_latency(lib, torch, dev, M, params, batches=(1, 32), iters=50):
    """QNNPACK's own regime: one or a few images.  The 53 asynchronous C-ABI runs of a step are captured once in a CUDA
    graph (launch-bound: ~53 kernels of a few microseconds each) and replayed; the un-captured loop is timed beside it."""
    out = {}
    for b in batches:
        stack = M.Stack(lib, seed=0, params=params)
        cap = stack.max_activation_bytes(b)
        x = torch.randint(0, 256, (b * 224 * 224 * 3,), dtype=torch.uint8, device=dev)
        a_, b_ = torch.empty(cap, dtype=torch.uint8, device=dev), torch.empty(cap, dtype=torch.uint8, device=dev)
        stack.setup(b, a_.data_ptr(), b_.data_ptr(), first_input=x.data_ptr())
        stream = torch.cuda.current_stream()
        for _ in range(3):
            stack.run(asynchronous=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(iters):
            stack.run(asynchronous=True)
        e1.record(stream)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / iters
        eager_ms = e0.elapsed_time(e1) / iters
        entry = {"eager_ms": eager_ms, "eager_host_us_per_launch": wall * 1e6 / len(stack.ops)}
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                stack.run(asynchronous=True)
            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            e0.record(stream)
            for _ in range(iters):
                g.replay()
            e1.record(stream)
            torch.cuda.synchronize()
            entry["graph_ms"] = e0.elapsed_time(e1) / iters
            entry["images_per_s_graph"] = b / (entry["graph_ms"] * 1e-3)
        except Exception as exc:  # graph capture is an optimisation of the caller, not of the library
            entry["graph_error"] = str(exc)[:200]
        out[f"batch_{b}"] = entry
        stack.delete()
    return out


def measure_full_network(lib, torch, dev, M, batch, steps, warmup, peak_gbs):
    """The real MobileNetV2-int8 graph — the 52 convolutions of the headline stack plus the 10 residual adds, the global
    average pool and the per-image classifier (64 qnnpack.h operators) — device-timed like the headline, then gated byte
    for byte against the reference chain on sampled images."""
    from oracle import chain_check as CC
    layers = M.network()
    params = [M.layer_params(l, i)[:2] for i, l in enumerate(layers)]
    net = M.Network(lib, seed=0, params=params)
    cap = net.max_activation_bytes(batch)
    x = torch.randint(0, 256, (batch * 224 * 224 * 3,), dtype=torch.uint8, device=dev)
    bufs = [torch.empty(cap, dtype=torch.uint8, device=dev) for _ in range(net.nbuf)]
    net.setup(batch, [b.data_ptr() for b in bufs], x.data_ptr())
    stream = torch.cuda.current_stream()
    for _ in range(warmup):
        net.run(asynchronous=True)
    torch.cuda.synchronize()
    nl = len(layers)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(nl + 1)] for _ in range(steps)]
    for s_ in range(steps):
        ev[s_][0].record(stream)
        net.run(asynchronous=True, hook=lambda i, after, s_=s_: ev[s_][i + 1].record(stream) if after else None)
    torch.cuda.synchronize()
    ms = ev[0][0].elapsed_time(ev[-1][nl]) / steps
    layer_ms = [statistics.fmean(ev[s_][i].elapsed_time(ev[s_][i + 1]) for s_ in range(steps)) for i in range(nl)]
    images = sorted({0, 1 % batch, max(0, batch // 2 - 1), batch - 1})
    parity = CC.check_device_network(net, params, batch, x, bufs, images)
    by_kind = {}
    for l, t in zip(layers, layer_ms):
        k = by_kind.setdefault(l.kind, {"launches": 0, "ms": 0.0, "gb": 0.0})
        k["launches"] += 1
        k["ms"] += t
        k["gb"] += l.algorithmic_bytes(batch) / 1e9
    for k in by_kind.values():
        k["frac_of_hbm_peak"] = k["gb"] * 1e3 / k["ms"] / peak_gbs
    net.delete()
    return {"operators": nl, "batch": batch, "ms_per_step": ms, "images_per_s": batch / (ms * 1e-3), "buffers": net.nbuf,
            "algorithmic_gb": net.total_bytes(batch) / 1e9, "by_kind": by_kind,
            "parity_check": {k: parity[k] for k in ("images", "layers", "bytes_compared", "mismatches", "oracle")}}


def measure_e2e_plugin(lib, M, params, batch=64, steps=3):
    """The stock caller's path (reference bench/convolution.cc:83-97 loop): qnnp_setup_* with HOST pointers and a
    synchronous qnnp_run_operator per layer — every layer's input and output cross PCIe inside the call."""
    import numpy as np
    stack = M.Stack(lib, seed=0, params=params)
    cap = stack.max_activation_bytes(batch) + 64
    x = np.random.default_rng(1).integers(0, 256, batch * 224 * 224 * 3 + 64, dtype=np.uint8)
    a, b = np.zeros(cap, np.uint8), np.zeros(cap, np.uint8)
    stack.setup(batch, a[16:], b[16:], first_input=x[16:])
    stack.run()
    t0 = time.perf_counter()
    for _ in range(steps):
        stack.run()
    dt = (time.perf_counter() - t0) / steps
    stack.delete()
    moved = sum(l.in_elems_per_image + l.out_elems_per_image for l in stack.layers) * batch
    return {"value": batch / dt, "unit": "images/s", "batch": batch, "ms_per_step": dt * 1e3, "pcie_bytes_per_step": int(moved),
            "note": "host pointers, synchronous qnnp_run_operator per layer (pageable memory): every activation crosses "
                    "PCIe twice; device pointers + qnnp_cuda_run_operator_async is the intended integration (e2e above)"}


def b200_main(args, rank, local_rank, world):
    import faulthandler

    import numpy as np
    import torch
    import torch.distributed as dist

    faulthandler.dump_traceback_later(240, exit=False)  # a hung collective or kernel leaves a stack trace on stderr
    # stdout must carry exactly one line, the JSON.  Native libraries write to file descriptor 1 behind Python's back
    # (NCCL prints its version banner there), so fd 1 is pointed at stderr for the duration of the run and the result
    # goes to a private duplicate of the original stdout.
    sys.stdout.flush()
    result_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    os.environ["QNNP_CUDA_DEVICE"] = str(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    import qnnpack_b200
    from qnnpack_b200 import mobilenet_v2 as M

    lib = qnnpack_b200.load()  # raises if the extension or the GPU is missing: no fallback
    # A dedicated (non-default) stream carries every launch, copy and event of the benchmark; the
    # library is told to enqueue on it (NULL would select the library's own stream instead).
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    lib.set_stream(stream.cuda_stream)

    B = args.batch
    # one-time replication of the model parameters: rank 0 -> all, one NCCL broadcast (NVLink/NVSwitch); every rank
    # then plans and packs its own operators from identical numbers
    params = M.make_params(seed=0, zero=(rank != 0))
    bcast_bytes = 0
    if world > 1:
        from qnnpack_b200 import shard as S
        bcast_bytes = S.replicate_params_from_rank0([a for kb in params for a in kb], device=dev)
        torch.cuda.synchronize()
    stack = M.Stack(lib, seed=0, params=params)

    cap = stack.max_activation_bytes(B)
    # seeded, so that two builds given the same arguments see the same images (--dump-outputs)
    x_in = torch.randint(0, 256, (B * 224 * 224 * 3,), dtype=torch.uint8, device=dev,
                         generator=torch.Generator(device=dev).manual_seed(0))
    buf_a = torch.empty(cap, dtype=torch.uint8, device=dev)
    buf_b = torch.empty(cap, dtype=torch.uint8, device=dev)
    final = stack.setup(B, buf_a.data_ptr(), buf_b.data_ptr(), first_input=x_in.data_ptr())
    logits_dev = (buf_a, buf_b)[final][: B * 1000]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    nl = len(stack.layers)
    for _ in range(args.warmup):
        stack.run(asynchronous=True)
    barrier()

    # ---- timed region: K steps, inputs resident in HBM ------------------------------------------------
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(nl + 1)] for _ in range(args.steps)]
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.launch_count()
    barrier()
    for s in range(args.steps):
        ev[s][0].record(stream)
        stack.run(asynchronous=True, hook=lambda i, after, s=s: ev[s][i + 1].record(stream) if after else None)
    barrier()
    launches = lib.launch_count() - launches0
    clocks = sampler.stop()
    total_ms = ev[0][0].elapsed_time(ev[-1][nl])
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * B * args.steps / (total_ms * 1e-3)

    # per-layer times (mean over steps) from the same timed region
    layer_ms = [statistics.fmean(ev[s][i].elapsed_time(ev[s][i + 1]) for s in range(args.steps)) for i in range(nl)]

    # the last timed step's logits, before anything below reuses the activation buffers
    if args.dump_outputs and rank == 0:
        dump_logits(logits_dev.view(B, 1000).cpu().numpy(), args.dump_outputs)

    # ---- e2e: batch from pinned host memory, logits back to the host, inside the timed region ---------
    # The public API is driven the way a serving loop would drive it: step i+1's images are copied host->device
    # on a copy stream (into the other of two device input buffers) while step i computes; the first layer is
    # re-setup each step with the buffer that holds its images (setup only records pointers); logits return
    # over the compute stream.  Every step's H2D, 53 C-ABI runs and D2H are inside the timed region.
    e2e = None
    if not args.no_e2e:
        x_host = torch.randint(0, 256, (B * 224 * 224 * 3,), dtype=torch.uint8).pin_memory()
        y_host = torch.empty(B * 1000, dtype=torch.uint8).pin_memory()
        x_dev = [x_in, torch.empty_like(x_in)]
        copy_stream = torch.cuda.Stream(device=dev)
        h2d_done = [torch.cuda.Event() for _ in range(2)]
        free_ev = [torch.cuda.Event() for _ in range(2)]
        stem, stem_op = stack.layers[0], stack.ops[0]

        def e2e_steps(n):
            for s in range(n):
                b = s % 2
                with torch.cuda.stream(copy_stream):
                    if s >= 2:
                        copy_stream.wait_event(free_ev[b])      # the stem of step s-2 has consumed this buffer
                    x_dev[b].copy_(x_host, non_blocking=True)
                    h2d_done[b].record(copy_stream)
                stream.wait_event(h2d_done[b])
                st = lib.setup_convolution(stem_op, B, stem.h, stem.h, x_dev[b].data_ptr(), stem.cin, buf_a.data_ptr(), stem.cout)
                assert st == 0
                stack.run(asynchronous=True, hook=lambda i, after, b=b: free_ev[b].record(stream) if (after and i == 0) else None)
                y_host.copy_(logits_dev, non_blocking=True)
            stream.synchronize()  # the caller owns every result when the loop returns

        e2e_steps(2)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        e2e_steps(args.steps)
        e1.record(stream)
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": world * B * args.steps / (float(t.item()) * 1e-3), "unit": "images/s",
               "h2d_bytes_per_step": int(x_host.numel()), "d2h_bytes_per_step": int(y_host.numel()),
               "note": "H2D of step i+1 overlaps the compute of step i (two device input buffers, copy stream)"}
        # restore the stem's input for anything that runs afterwards
        lib.setup_convolution(stem_op, B, stem.h, stem.h, x_in.data_ptr(), stem.cin, buf_a.data_ptr(), stem.cout)

    # ---- parity gate on the benchmarked configuration (outside every timed region) -------------------------------
    # The step is run once more, exactly as timed (device pointers, asynchronous launches, same batch); the first, second,
    # middle and last image's slice of EVERY layer's output is copied back right after that layer and compared byte for
    # byte with the unmodified reference (oracle/_ref; where it has not been built, the oracle restatements pinned to it)
    # pushed through the same operators image by image.
    parity = None
    if not args.no_parity_check:
        from oracle import chain_check as CC
        images = sorted({0, 1 % B, B // 2 - 1 if B >= 2 else 0, B - 1})
        parity = CC.check_device_stack(stack, params, B, x_in, buf_a, buf_b, images,
                                       log=lambda m: print(m, file=sys.stderr, flush=True))
        parity["rank"] = rank
        if parity["mismatches"] != 0:
            print(f"bench.py: PARITY FAILURE on rank {rank}: {json.dumps(parity)}", file=sys.stderr, flush=True)
            os._exit(3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- side measurements (rank 0, outside every timed region) ---------------------------------------------------------
    extras = {}
    if not args.no_extras:
        try:
            tops, ms = lib.measure_int8_peak(20000, 3)
            extras["int8_peak"] = {"tops": tops, "ms_per_launch": ms, "how": "qnnp_cuda_measure_int8_peak: smem-resident tcgen05.mma "
                                   "kind::i8 loop, 148 CTAs x 160000 UMMAs of 128x256x32 (q8_peak_sm100.cu)"}
            sampler = ClockSampler(local_rank)
            sampler.start()
            tops_s, ms_s = lib.measure_int8_peak(20000, 140)  # ~1.5 s back to back
            extras["int8_peak_sustained"] = {"tops": tops_s, "ms_per_launch": ms_s, "launches": 140, "clocks": sampler.stop()}
            extras["tensor_bound_gemm"] = measure_tensor_bound_gemm(lib, torch, dev, tops, peak_sustained=tops_s)
            if world == 1:
                extras["hbm_by_mix"] = measure_hbm_by_mix(torch, dev)
                extras["full_network"] = measure_full_network(lib, torch, dev, M, B, min(args.steps, 5), 2, measured_peaks()[0])
                extras["small_batch_latency"] = measure_small_batch_latency(lib, torch, dev, M, params)
                extras["e2e_plugin_host_pointers"] = measure_e2e_plugin(lib, M, params)
        except Exception as exc:
            extras["error"] = str(exc)[:300]

    # ---- reporting (rank 0) -----------------------------------------------------------------------------
    peak_gbs, peak_src = measured_peaks()
    kinds = {"igemm": ("conv", "pw", "fc"), "dwconv3x3": ("dw",)}
    per_kernel = {}
    for kname, ks in kinds.items():
        idx = [i for i, l in enumerate(stack.layers) if l.kind in ks]
        ms = sum(layer_ms[i] for i in idx)
        by = sum(stack.layers[i].algorithmic_bytes(B) for i in idx)
        ops = sum(stack.layers[i].ops(B) for i in idx)
        per_kernel[kname] = {"launches_per_step": len(idx), "ms_per_step": ms, "share_of_step": ms / sum(layer_ms),
                             "algorithmic_gb": by / 1e9, "achieved_gbs": by / 1e6 / ms, "frac_of_hbm_peak": by / 1e6 / ms / peak_gbs,
                             "tops": ops / 1e9 / ms}
    ig = per_kernel["igemm"]
    # roofline: the dominant LAUNCH of the step (largest CUDA-event time), with its algorithmic bytes; `traffic` is
    # that launch's dram__bytes_read + dram__bytes_write from the committed `ncu --set full` capture (profiles/),
    # valid for the default batch only
    dom = max(range(nl), key=lambda i: layer_ms[i])
    dl = stack.layers[dom]
    kname = {"dw": "q8_dwconv3x3 (tcgen05 block-diagonal UMMA or dp4a streaming kernel, see layers[])",
             "conv": "q8_igemm_kernel<conv> (tcgen05 kind::i8 implicit GEMM, fused Q31 epilogue)"}.get(
                 dl.kind, "q8_igemm_kernel<gemm> (tcgen05 kind::i8, TMA loads, fused Q31 epilogue)")
    dom_gbs = dl.algorithmic_bytes(B) / 1e6 / layer_ms[dom]
    roofline = {"kernel": kname, "layer": dl.name, "bound": "hbm", "achieved": dom_gbs, "peak": peak_gbs, "unit": "GB/s",
                "frac": dom_gbs / peak_gbs,
                "traffic": NCU_DRAM_BYTES_PER_LAUNCH.get(dl.name) if B == 4096 else None,
                "traffic_source": NCU_DRAM_SOURCE.get(dl.name) if B == 4096 else None,
                "algorithmic_bytes": dl.algorithmic_bytes(B), "ms": layer_ms[dom], "peak_source": peak_src,
                "all_igemm_launches": {"achieved": ig["achieved_gbs"], "frac": ig["achieved_gbs"] / peak_gbs,
                                       "launches_per_step": ig["launches_per_step"]},
                "note": "achieved = algorithmic bytes of the step's slowest launch / its mean CUDA-event duration in the "
                        "timed region; per_kernel / layers[] carry every other launch"}
    # BASELINE.json configs[1]: q8gemm sweep = the distinct 1x1 / FC shapes, each once
    seen, sw_ops, sw_ms, sweep_rows = set(), 0.0, 0.0, []
    for i, l in enumerate(stack.layers):
        if l.kind in ("pw", "fc") and (l.h, l.cin, l.cout) not in seen:
            seen.add((l.h, l.cin, l.cout))
            sw_ops += l.ops(B); sw_ms += layer_ms[i]
            bound_ms = max(l.ops(B) / (INT8_PEAK_TOPS_NOMINAL * 1e9), l.algorithmic_bytes(B) / (peak_gbs * 1e6))
            sweep_rows.append({"layer": l.name, "m": B * l.out_h * l.out_h if l.kind != "fc" else B, "n": l.cout, "k": l.cin,
                               "ms": layer_ms[i], "tops": l.ops(B) / 1e9 / layer_ms[i],
                               "gbs": l.algorithmic_bytes(B) / 1e6 / layer_ms[i], "frac_of_roofline": bound_ms / layer_ms[i]})
    int8_peak = (extras.get("int8_peak") or {}).get("tops")
    q8gemm = {"tops": sw_ops / 1e9 / sw_ms, "pct_of_int8_peak_nominal": 100.0 * sw_ops / 1e9 / sw_ms / INT8_PEAK_TOPS_NOMINAL,
              "int8_peak_tops_nominal": INT8_PEAK_TOPS_NOMINAL, "int8_peak_tops_measured": int8_peak,
              "pct_of_int8_peak_measured": (100.0 * sw_ops / 1e9 / sw_ms / int8_peak) if int8_peak else None,
              "tensor_bound": extras.get("tensor_bound_gemm"), "shapes": sweep_rows,
              "note": "every MobileNetV2 shape is HBM-bound (frac_of_roofline per shape); tensor_bound is the GEMM where the "
                      "int8 tensor pipe can bind"}
    layers_out = [{"layer": l.name, "kind": l.kind, "ms": layer_ms[i], "gbs": l.algorithmic_bytes(B) / 1e6 / layer_ms[i],
                   "tops": l.ops(B) / 1e9 / layer_ms[i]} for i, l in enumerate(stack.layers)]
    # Second reading of the roofline: a launch cannot finish before its OUTPUT has been written at the write-only rate
    # either.  bound = max(all bytes / copy peak, output bytes / write-only peak); informative, `roofline` keeps the contract.
    mixed = None
    wo = (extras.get("hbm_by_mix") or {}).get("write_only_gbs")
    if wo:
        tot_bound = 0.0
        for i, l in enumerate(stack.layers):
            out_b = B * l.cout * (1 if l.kind == "fc" else l.out_h * l.out_h)
            bound = max(l.algorithmic_bytes(B) / (peak_gbs * 1e6), out_b / (wo * 1e6))
            layers_out[i]["mixed_bound_ms"] = bound
            layers_out[i]["frac_of_mixed_bound"] = bound / layer_ms[i]
            tot_bound += bound
        mixed = {"write_only_gbs": wo, "stack_bound_ms": tot_bound, "stack_frac": tot_bound / ms_per_step,
                 "note": "per launch max(bytes / copy peak, output bytes / write-only peak); see layers[].frac_of_mixed_bound"}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            threads = usable_threads()
            cb = args.cpu_batch or max(16, 2 * threads)
            ips, sec = run_reference_stack(3, 1, cb, threads)
            scaling = {}
            for t in sorted({1, max(1, threads // 4), threads}):
                if t != threads:
                    scaling[str(t)] = run_reference_stack(1, 1, max(4, min(cb, 2 * t)), t)[0]
            scaling[str(threads)] = ips
            cpu = {"value": ips, "unit": "images/s", "cores": threads, "kind": "reference",
                   "sample": f"3 passes of the full 53-operator stack over {cb} images, unmodified reference "
                             f"(oracle/_ref, SSE2 ukernels) with a {threads}-thread pthreadpool",
                   "thread_scaling_images_per_s": scaling, "host": host_info()}
        except Exception as exc:  # the baseline is informative; never let it take the GPU numbers down
            cpu = {"value": None, "unit": "images/s", "cores": 0, "kind": "reference", "sample": f"failed: {exc}"}

    line = {
        "metric": "mobilenet_v2_int8_conv_stack_images_per_sec", "value": value, "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "MobileNetV2-int8 conv stack (53 operators, 300.8 MMAC/image; BASELINE.json configs[4], "
                               "containing the q8gemm sweep configs[1], all conv layers configs[2] and the depthwise layers configs[3])",
                   "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                   "l2": "every layer streams activations far larger than the 126 MB L2 (no flush needed)",
                   "quantization": "zero points 127, requant scale 1/(128*sqrt(K)), clamp 0..255",
                   "weights_broadcast_bytes": bcast_bytes},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "parity_check": parity, "extras": extras,
        "roofline": roofline, "cpu_baseline": cpu, "q8gemm_sweep": q8gemm, "per_kernel": per_kernel, "layers": layers_out,
        "stack_ops_g": stack.total_ops(B) / 1e9, "stack_algorithmic_gb": stack.total_bytes(B) / 1e9,
        "stack_frac_of_hbm_roofline": (stack.total_bytes(B) / 1e6 / peak_gbs) / ms_per_step,
        "stack_mixed_bound": mixed,
    }
    print(json.dumps(line), file=result_out, flush=True)
    faulthandler.cancel_dump_traceback_later()
    if world > 1:
        dist.destroy_process_group()


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def main():
    args = parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1 and "RANK" not in os.environ:
        # convenience: `python bench.py --gpus N` re-launches itself under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(free_port()), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_main(args, rank, world)
    else:
        b200_main(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
