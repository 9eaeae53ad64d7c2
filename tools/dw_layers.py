"""Per-layer timing of the 17 depthwise layers of mobilenet_v2.Stack, alone, for A/B comparisons on one GPU.

Each arm is a library build and/or a set of environment knobs.  Arms run in alternation, ROUNDS times, each run in a
fresh process (the knobs are read when an operator is planned), so that drift of the card or of other work on the host
hits every arm alike.  Per layer and run: WARMUP launches, then REPS back-to-back launches between two CUDA events.
Every run also checksums each layer's output, so arms that must compute the same thing can be checked to do so.

    python tools/dw_layers.py --arm old=lib/old.so --arm new= --rounds 3 --json out.json
    python tools/dw_layers.py --arm pair= --arm nopair=:QNNP_CUDA_DW_NO_PAIR=1

An arm is NAME=[LIBRARY][:KEY=VALUE[,KEY=VALUE...]]; an empty LIBRARY is the in-tree libqnnpack.so.  The table gives the
median ms over the rounds, the spread (max - min) of the rounds, and the fraction of the mixed bound: max(all bytes / copy
bandwidth, output bytes / write-only bandwidth), both bandwidths measured at the start of the call.  The card's name,
power limit and clocks are read in the same call.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dw_layers():
    sys.path.insert(0, ROOT)
    from qnnpack_b200 import mobilenet_v2 as M
    return [(i, l) for i, l in enumerate(M.layers()) if l.kind == "dw"]


def checksum(torch, t):
    """Position-weighted sums of the output's 32-bit words, reduced on the GPU (the outputs are up to 1.6 GB)."""
    h = hashlib.sha256()
    v = t.view(torch.int32)
    for i in range(0, v.numel(), 1 << 26):
        c = v[i:i + (1 << 26)].to(torch.int64)
        w = torch.arange(i + 1, i + 1 + c.numel(), device=c.device, dtype=torch.int64)
        h.update(f"{int(c.sum())},{int((c * w).sum())};".encode())
    return h.hexdigest()[:16]


def child_layers(args):
    import torch

    sys.path.insert(0, ROOT)
    from qnnpack_b200 import api, mobilenet_v2 as M

    lib = api.QnnpackLibrary(args.lib or api.PRODUCT_LIB)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    lib.set_stream(stream.cuda_stream)
    B = args.batch
    layers = dw_layers()
    cap = max(B * l.h * l.h * l.cin for _, l in layers)
    x = torch.randint(0, 256, (cap,), dtype=torch.uint8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    y = torch.empty(cap, dtype=torch.uint8, device="cuda")
    rows = []
    for i, l in layers:
        kernel, bias, _ = M.layer_params(l, i)  # the parameters bench.py gives this layer (seed 0)
        op = M.create_node(lib, l, kernel, bias)
        M.setup_node(lib, l, op, B, [x.data_ptr()], y.data_ptr())
        for _ in range(args.warmup):
            assert lib.run_async(op) == 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.reps):
            lib.run_async(op)
        e1.record(stream)
        torch.cuda.synchronize()
        rows.append({"layer": l.name, "ms": e0.elapsed_time(e1) / args.reps, "kernel": lib.kernel_name(op),
                     "checksum": checksum(torch, y[:B * l.out_h * l.out_h * l.cout])})
        lib.delete(op)
    print(json.dumps(rows))


def child_peaks(args):
    import torch

    n = 4 << 30
    a, b = torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
    a.fill_(1)

    def timed(fn, reps=5):
        fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    copy_gbs = 2 * n / 1e6 / timed(lambda: b.copy_(a))
    wo_gbs = n / 1e6 / timed(lambda: b.fill_(3))
    print(json.dumps({"copy_gbs": copy_gbs, "write_only_gbs": wo_gbs}))


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return dict(zip(q.split(","), [f.strip() for f in out.split(",")])) if out else {}


def run_child(mode, lib, env, args):
    cmd = [sys.executable, os.path.abspath(__file__), "--child", mode, "--batch", str(args.batch), "--reps", str(args.reps),
           "--warmup", str(args.warmup)] + (["--lib", lib] if lib else [])
    proc = subprocess.run(cmd, capture_output=True, text=True, env={**os.environ, **env}, timeout=args.timeout)
    if proc.returncode != 0:
        sys.stderr.write(proc.stderr[-4000:])
        raise RuntimeError(f"{mode} run failed ({proc.returncode}): lib={lib or 'in-tree'} env={env}")
    return json.loads(proc.stdout.strip().splitlines()[-1])


def parse_arm(spec):
    name, _, rest = spec.partition("=")
    lib, _, envs = rest.partition(":")
    env = dict(kv.split("=", 1) for kv in envs.split(",") if kv)
    return name, (os.path.abspath(lib) if lib else ""), env


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--arm", action="append", default=[], help="NAME=[LIBRARY][:KEY=VALUE,...] (repeatable)")
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--timeout", type=int, default=900)
    ap.add_argument("--json", help="write every run and the summary here")
    ap.add_argument("--child", choices=["layers", "peaks"], help=argparse.SUPPRESS)
    ap.add_argument("--lib", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if min(args.batch, args.reps, args.rounds) < 1 or args.warmup < 0:
        ap.error("--batch, --reps and --rounds must be >= 1, --warmup >= 0")
    if args.child == "layers":
        return child_layers(args)
    if args.child == "peaks":
        return child_peaks(args)

    arms = [parse_arm(a) for a in (args.arm or ["current="])]
    info = {"before": gpu_info()}
    peaks = run_child("peaks", "", {}, args)
    runs = {name: [] for name, _, _ in arms}
    for r in range(args.rounds):
        for name, lib, env in arms if r % 2 == 0 else arms[::-1]:  # ABBA...: neither arm always runs first
            runs[name].append(run_child("layers", lib, env, args))
            print(f"round {r} {name}: {sum(x['ms'] for x in runs[name][-1]):.3f} ms", file=sys.stderr, flush=True)
    info["after"] = gpu_info()

    B = args.batch
    summary = {}
    for name, _, _ in arms:
        rows = []
        for k, (_, l) in enumerate(dw_layers()):
            ms = [run[k]["ms"] for run in runs[name]]
            out_b = B * l.out_h * l.out_h * l.cout
            bound = max(l.algorithmic_bytes(B) / (peaks["copy_gbs"] * 1e6), out_b / (peaks["write_only_gbs"] * 1e6))
            digests = sorted({run[k]["checksum"] for run in runs[name]})
            rows.append({"layer": l.name, "shape": f"{l.h}x{l.h}x{l.cin} s{l.stride}", "ms": statistics.median(ms),
                         "spread": max(ms) - min(ms), "mixed_bound_ms": bound, "frac_of_mixed_bound": bound / statistics.median(ms),
                         "kernel": runs[name][0][k]["kernel"], "checksums": digests})
        totals = [sum(x["ms"] for x in run) for run in runs[name]]
        summary[name] = {"layers": rows, "total_ms": statistics.median(totals), "total_spread": max(totals) - min(totals)}

    print(f"# {info['before'].get('name', '?')}, power limit {info['before'].get('power.limit', '?')}, "
          f"max SM clock {info['before'].get('clocks.max.sm', '?')}, SM clock before/after {info['before'].get('clocks.sm', '?')} / "
          f"{info['after'].get('clocks.sm', '?')}; batch {B}, {args.reps} launches per layer and run, {args.rounds} rounds; "
          f"copy {peaks['copy_gbs']:.0f} GB/s, write-only {peaks['write_only_gbs']:.0f} GB/s")
    names = [a[0] for a in arms]
    print("layer    shape            " + "".join(f"{n + ' ms':>12}{'±':>7}{'bound':>7}" for n in names) + "  outputs")
    for k, (_, l) in enumerate(dw_layers()):
        cells = "".join(f"{summary[n]['layers'][k]['ms']:12.4f}{summary[n]['layers'][k]['spread']:7.4f}"
                        f"{summary[n]['layers'][k]['frac_of_mixed_bound']:7.2f}" for n in names)
        same = len({d for n in names for d in summary[n]["layers"][k]["checksums"]}) == 1
        print(f"{l.name:8} {summary[names[0]]['layers'][k]['shape']:16} {cells}  {'same' if same else 'DIFFER'}")
    print("total                     " + "".join(f"{summary[n]['total_ms']:12.4f}{summary[n]['total_spread']:7.4f}{'':7}" for n in names))
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"gpu": info, "peaks": peaks, "batch": B, "reps": args.reps, "rounds": args.rounds,
                       "arms": {n: {"lib": lib, "env": env} for n, lib, env in arms}, "summary": summary, "runs": runs}, f, indent=1)


if __name__ == "__main__":
    main()
