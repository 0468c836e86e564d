"""Timing of sample-granular calls of the one-block-latency convolver (LowLatencyConvolver.process_samples) on one GPU, DEVICE buffers.

    python tools/lowlat_samples_time.py [--out profiles] [--quick] [--parent TREE] [--parts cost,trade,noregress]

Writes <out>/r04_lowlat_samples_cost.json, r04_lowlat_samples_trade.json and (with --parent) r04_lowlat_samples_noregress.json, each
with the GPU name and power limit:
  - cost per call, for call lengths {1, 32, 64, 128, 256, B/2, B} at C5 (1024 channels, 2^20 taps, B = 1024) and stereo (2 channels,
    2^17 taps, B = 512): stream time per call (CUDA events around a run of calls with no host synchronisation, ended by synchronize),
    host wall per call with a synchronize after every call (p50 / p99), and the mean duration of each kernel the calls launch
    (torch.profiler, in a run of its own);
  - the trade at a target latency of 64 samples: B = 64 with whole-block calls against B = 1024 with 64-sample calls, in
    channel-Msamples/s, at 1024 channels x 2^20 taps and at stereo x 2^17 taps;
  - no regression: tools/lowlat_time.py's C5 measurement at one block per call for the tree at TREE (the parent commit, built) and this
    tree, alternating, each in a process of its own.
Every shape is warmed up with at least 2 T_n blocks of whole-block calls (every level runs), then with calls of the measured length.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from lowlat_time import gpu_info, impulse, pct  # noqa: E402


def load(tree):
    sys.path.insert(0, tree)
    import __graft_entry__ as entry

    pkg = entry.load_package()
    if pkg.device_count() < 1:
        raise SystemExit("lowlat_samples_time.py needs a CUDA device")
    pkg.set_device(0)
    return pkg


def make(pkg, torch, C, B, taps, seed=1):
    conv = pkg.LowLatencyConvolver("float32")
    conv.set_stream(torch.cuda.current_stream())
    conv.impulse(impulse(torch, C, taps, seed), B)
    return conv


class Feed:
    """consecutive calls of `n` samples from a [C][L] device signal (wrapping around), each into its own [C][n] buffer pair"""

    def __init__(self, torch, x, n, nbuf=64):
        C, L = x.shape
        starts = [(i * n) % (L - n) for i in range(nbuf)]
        self.ins = [x[:, s : s + n].contiguous() for s in starts]
        self.outs = [torch.empty_like(v) for v in self.ins]
        self.i = 0

    def __call__(self, conv):
        k = self.i % len(self.ins)
        conv.process_samples(self.ins[k], self.outs[k])
        self.i += 1


def warm(torch, conv, C, B, x):
    T = conv.layout(int(conv.cfg.partitions), B)["frame_blocks"]
    blocks = max(8, 2 * max(T or (1,)))
    xb = torch.empty((C, 8 * B), device="cuda")
    for t in range(0, blocks, 8):
        conv(xb.copy_(x[:, : 8 * B]))
    conv.synchronize()
    return blocks


def stream_time(torch, conv, feed, calls):
    s = torch.cuda.current_stream()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(s)
    for _ in range(calls):
        feed(conv)
    conv.synchronize()
    end.record(s)
    end.synchronize()
    return start.elapsed_time(end) / 1e3


def wall(conv, feed, calls):
    out = []
    for _ in range(calls):
        t0 = time.perf_counter()
        feed(conv)
        conv.synchronize()
        out.append((time.perf_counter() - t0) * 1e6)
    return {"p50_us": pct(out, 50), "p99_us": pct(out, 99), "max_us": float(max(out)), "calls": calls}


def kernel_means(torch, conv, feed, calls):
    """mean duration (us) and count of every kernel launched by `calls` calls, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile

    conv.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            feed(conv)
        conv.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and ev.count > 0 and getattr(ev, "device_time_total", 0) > 0:
            name = ev.key.split("(")[0].split("<")[0].replace("void ", "").strip()
            d = out.setdefault(name, {"count": 0, "total_us": 0.0})
            d["count"] += ev.count
            d["total_us"] += ev.device_time_total
    for d in out.values():
        d["mean_us"] = d["total_us"] / d["count"]
        d["per_call_us"] = d["total_us"] / calls
    return out


def cost(pkg, torch, C, B, taps, lengths, quick):
    x = torch.rand((C, 64 * B), device="cuda") * 2 - 1
    conv = make(pkg, torch, C, B, taps)
    res = {"shape": {"channels": C, "block": B, "taps": taps}, "layout": conv.layout(taps // B, B), "device_bytes": conv.device_bytes(),
           "calls": []}
    warmed = warm(torch, conv, C, B, x)
    for n in lengths:
        # whole blocks' worth of calls, so level releases and completing segments are in the average as often as a stream has them
        calls = max(64 if quick else 256, (4 if quick else 16) * B // n)
        feed = Feed(torch, x, n)
        stream_time(torch, conv, feed, min(calls, 4 * B // n + 16))  # warm-up at this length
        sec = stream_time(torch, conv, feed, calls)
        r = {"samples_per_call": n, "calls_timed": calls, "stream_us_per_call": sec / calls * 1e6,
             "channel_msamples_s": C * n * calls / sec / 1e6, "host_wall_per_call_sync": wall(conv, feed, min(calls, 2000))}
        try:
            r["kernels"] = kernel_means(torch, conv, feed, min(calls, 4 * B // n + 8))
        except Exception as exc:  # the timings above stand without it
            r["kernels"] = f"unavailable: {exc}"
        res["calls"].append(r)
        print(json.dumps({"C": C, "B": B, "n": n, "stream_us_per_call": r["stream_us_per_call"],
                          "wall_p50_us": r["host_wall_per_call_sync"]["p50_us"]}), flush=True)
    res["warmup_blocks"] = warmed
    conv.close()
    return res


def throughput(pkg, torch, C, B, taps, n, blocks, quick):
    """channel-Msamples/s of calls of n samples over `blocks` blocks after the warm-up"""
    x = torch.rand((C, 64 * max(B, 64)), device="cuda") * 2 - 1
    conv = make(pkg, torch, C, B, taps)
    warmed = warm(torch, conv, C, B, x)
    feed = Feed(torch, x, n)
    calls = blocks * B // n
    stream_time(torch, conv, feed, min(calls, 256))
    sec = stream_time(torch, conv, feed, calls)
    out = {"block": B, "samples_per_call": n, "layout": conv.layout(taps // B, B), "warmup_blocks": warmed, "calls_timed": calls,
           "channel_msamples_s": C * n * calls / sec / 1e6, "stream_us_per_call": sec / calls * 1e6,
           "host_wall_per_call_sync": wall(conv, feed, min(calls, 1000))}
    conv.close()
    return out


def c5_one_block(tree, quick):
    """tools/lowlat_time.py's C5 lowlat_default measurement with the package of `tree`"""
    import torch

    from lowlat_time import lowlat, measure

    pkg = load(tree)
    C, B, taps = (64, 256, 1 << 15) if quick else (1024, 1024, 1 << 20)
    x = torch.rand((64 if quick else 256, C, B), device="cuda") * 2 - 1
    y = torch.empty_like(x)
    conv = lowlat(pkg, impulse(torch, C, taps), B)
    r = measure(pkg, torch, conv, C, B, x, y, 256, 256 if quick else 1024, 64 if quick else 200)
    conv.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--quick", action="store_true", help="small sizes: checks the script end to end, numbers mean nothing")
    ap.add_argument("--parent", help="a built tree of the parent commit, for the no-regression comparison")
    ap.add_argument("--parts", default="cost,trade,noregress", help="comma-separated subset of cost, trade, noregress")
    ap.add_argument("--c5-one-block", metavar="TREE", help=argparse.SUPPRESS)  # one side of the comparison, in its own process
    args = ap.parse_args()

    if args.c5_one_block:
        print(json.dumps(c5_one_block(args.c5_one_block, args.quick)))
        return

    import torch

    parts = set(args.parts.split(","))
    pkg = load(ROOT)
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    if "cost" in parts:
        measure_cost(pkg, torch, info, args)
    if "trade" in parts:
        measure_trade(pkg, torch, info, args)
    if "noregress" in parts:
        if not args.parent:
            raise SystemExit("the noregress part needs --parent")
        measure_noregress(info, args)


def measure_cost(pkg, torch, info, args):
    shapes = [(64, 256, 1 << 15), (2, 512, 1 << 15)] if args.quick else [(1024, 1024, 1 << 20), (2, 512, 1 << 17)]
    res = dict(info, method=__doc__.split("Writes")[1].split("  - the trade")[0].strip(), shapes=[])
    for C, B, taps in shapes:
        res["shapes"].append(cost(pkg, torch, C, B, taps, sorted({1, 32, 64, 128, 256, B // 2, B}), args.quick))
        torch.cuda.empty_cache()
    with open(os.path.join(args.out, "r04_lowlat_samples_cost.json"), "w") as f:
        json.dump(res, f, indent=1)


def measure_trade(pkg, torch, info, args):
    trade = dict(info, latency_samples=64, method=(
        "DEVICE buffers, events around a run of calls with no host synchronisation, ended by synchronize; (a) B = 64, one 64-sample "
        "block per call, (b) B = 1024, 64-sample calls (16 per block); default schedule for each"), shapes=[])
    for C, taps in ([(64, 1 << 15), (2, 1 << 15)] if args.quick else [(1024, 1 << 20), (2, 1 << 17)]):
        a = throughput(pkg, torch, C, 64, taps, 64, 256 if args.quick else 4096, args.quick)
        torch.cuda.empty_cache()
        b = throughput(pkg, torch, C, 1024, taps, 64, 16 if args.quick else 256, args.quick)
        torch.cuda.empty_cache()
        winner = "a: B = 64, whole blocks" if a["channel_msamples_s"] > b["channel_msamples_s"] else "b: B = 1024, 64-sample calls"
        trade["shapes"].append({"channels": C, "taps": taps, "a_block_64": a, "b_block_1024_calls_64": b, "faster": winner,
                                "ratio_b_over_a": b["channel_msamples_s"] / a["channel_msamples_s"]})
        print(json.dumps({"C": C, "a": a["channel_msamples_s"], "b": b["channel_msamples_s"], "faster": winner}), flush=True)
    with open(os.path.join(args.out, "r04_lowlat_samples_trade.json"), "w") as f:
        json.dump(trade, f, indent=1)


def measure_noregress(info, args):
    runs = []
    for rnd in range(3):
        for name, tree in (("parent", os.path.abspath(args.parent)), ("this", ROOT)):
            cmd = [sys.executable, os.path.abspath(__file__), "--c5-one-block", tree] + (["--quick"] if args.quick else [])
            p = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
            if p.returncode != 0:
                raise SystemExit(f"{name} run failed:\n{p.stdout[-2000:]}\n{p.stderr[-3000:]}")
            r = json.loads(p.stdout.strip().splitlines()[-1])
            runs.append({"round": rnd, "tree": name, "channel_msamples_s": r["channel_msamples_s"], "us_per_block": r["us_per_block"]})
            print(json.dumps(runs[-1]), flush=True)
    summary = {k: {"median_channel_msamples_s": float(np.median([r["channel_msamples_s"] for r in runs if r["tree"] == k])),
                   "runs": [r["channel_msamples_s"] for r in runs if r["tree"] == k]} for k in ("parent", "this")}
    summary["this_over_parent"] = summary["this"]["median_channel_msamples_s"] / summary["parent"]["median_channel_msamples_s"]
    noreg = dict(info, method="tools/lowlat_time.py lowlat_default at C5 (one block per call), parent and this tree alternating, "
                 "one process per run, 3 rounds", runs=runs, summary=summary)
    with open(os.path.join(args.out, "r04_lowlat_samples_noregress.json"), "w") as f:
        json.dump(noreg, f, indent=1)
    print(json.dumps({"this_over_parent": summary["this_over_parent"]}))


if __name__ == "__main__":
    main()
