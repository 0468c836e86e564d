"""Timing of the one-block-latency convolver (LowLatencyConvolver) on one GPU, one block per call, DEVICE buffers.

    python tools/lowlat_time.py [--out profiles] [--quick]

Writes <out>/r03_lowlat_c5.json, r03_lowlat_c3.json and r03_lowlat_sweep.json, each with the GPU name and power limit:
  - C5 (1024 channels, 2^20 taps, B = 1024): steady throughput (CUDA events over a run of one-block calls, side streams included by a
    final synchronize), host wall time per call with a synchronize after every call (p50 / p99 / max), the direct-form Convolver at one
    block per call in the same run, fused against unfused head, device_bytes;
  - C3 (stereo, B = 512, 2^17 taps): microseconds per block, host and device;
  - the schedule sweep T_1 in {2, 4, 8, 16} x ratio {4, 8} on C5 that decides the library default.
Every timed shape is warmed up first (at least 2 T_n blocks, so every level runs). The input is [blocks][C][B] on the device; at C5 one
block of filter and delay line alone is 8.6 GB for the direct form and 0.3 GB for the head, beyond the 126 MB L2.
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
sys.path.insert(0, ROOT)


def gpu_info():
    import torch

    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else None
    except Exception as exc:  # the number is still worth keeping without it
        info["power_limit_and_max_sm_clock"] = f"unavailable: {exc}"
    return info


def impulse(torch, channels, taps, seed=1):
    g = torch.Generator(device="cuda").manual_seed(seed)
    ir = torch.rand((channels, taps), generator=g, device="cuda", dtype=torch.float32) * 2 - 1
    return ir / ir.pow(2).sum(dim=1).max().sqrt()


def pct(v, q):
    return float(np.percentile(np.asarray(v), q))


def time_blocks(torch, conv, x, y, first, count):
    """device time of `count` one-block calls starting at block `first` (events on the caller's stream; synchronize waits for every
    side stream before the end event is read)"""
    s = torch.cuda.current_stream()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(s)
    for t in range(first, first + count):
        conv(x[t % x.shape[0]], y[t % y.shape[0]])
    conv.synchronize()
    end.record(s)
    end.synchronize()
    return start.elapsed_time(end) / 1e3


def wall_per_call(conv, x, y, first, count):
    out = []
    for t in range(first, first + count):
        t0 = time.perf_counter()
        conv(x[t % x.shape[0]], y[t % y.shape[0]])
        conv.synchronize()
        out.append((time.perf_counter() - t0) * 1e6)
    return {"p50_us": pct(out, 50), "p99_us": pct(out, 99), "max_us": float(max(out)), "calls": count}


def measure(pkg, torch, conv, channels, block, x, y, warm, steady, walls):
    s = torch.cuda.current_stream()
    conv.set_stream(s)
    time_blocks(torch, conv, x, y, 0, warm)
    sec = time_blocks(torch, conv, x, y, warm, steady)
    res = {
        "blocks_timed": steady,
        "device_s": sec,
        "us_per_block": sec / steady * 1e6,
        "channel_msamples_s": channels * block * steady / sec / 1e6,
        "host_wall_per_call_sync": wall_per_call(conv, x, y, warm + steady, walls),
        "device_bytes": int(conv.device_bytes()),
    }
    return res


def lowlat(pkg, ir, block, frame_blocks=None, unfused=False):
    if unfused:
        os.environ["NEO_B200_LOWLAT_UNFUSED"] = "1"
    try:
        conv = pkg.LowLatencyConvolver("float32", frame_blocks=frame_blocks)
        conv.impulse(ir, block)
    finally:
        os.environ.pop("NEO_B200_LOWLAT_UNFUSED", None)
    return conv


def schedule(t1, ratio, parts):
    out, t = [], t1
    while t <= 512 and len(out) < 4 and 2 * t < parts:
        out.append(t)
        t *= ratio
    return tuple(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--quick", action="store_true", help="small sizes: checks the script end to end, numbers mean nothing")
    args = ap.parse_args()

    import torch

    import __graft_entry__ as entry

    pkg = entry.load_package()
    if pkg.device_count() < 1:
        raise SystemExit("lowlat_time.py needs a CUDA device")
    pkg.set_device(0)
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()

    C, B, taps = (64, 256, 1 << 15) if args.quick else (1024, 1024, 1 << 20)
    P = taps // B
    nbuf = 64 if args.quick else 256  # [blocks][C][B] device input: 1 GB at C5
    x = torch.rand((nbuf, C, B), device="cuda") * 2 - 1
    y = torch.empty_like(x)
    ir = impulse(torch, C, taps)
    steady, walls = (256, 64) if args.quick else (1024, 200)

    c5 = dict(info, shape={"channels": C, "block": B, "taps": taps, "partitions": P}, method=(
        "one block per call, DEVICE buffers [C][B]; throughput = CUDA events around `blocks_timed` calls after a warm-up of 2 T_n "
        "blocks, ended by synchronize (side streams included); host wall = perf_counter around call + synchronize"))
    default = pkg.LowLatencyConvolver.layout(P, B)
    warm = max(256, 2 * max(default["frame_blocks"] or (1,)))
    conv = lowlat(pkg, ir, B)
    c5["lowlat_default"] = dict(layout=default, **measure(pkg, torch, conv, C, B, x, y, warm, steady, walls))
    conv.close()
    conv = lowlat(pkg, ir, B, unfused=True)
    c5["lowlat_default_unfused_head"] = measure(pkg, torch, conv, C, B, x, y, warm, steady, walls)
    conv.close()
    torch.cuda.empty_cache()
    direct = pkg.Convolver(pkg.UPOLS, "float32", pkg.DIAGONAL, max_blocks=1)
    direct.impulse(ir, B)
    c5["direct_form_1_block"] = measure(pkg, torch, direct, C, B, x, y, 32, 128 if not args.quick else 64, 50)
    direct.close()
    torch.cuda.empty_cache()
    c5["speedup_vs_direct"] = c5["lowlat_default"]["channel_msamples_s"] / c5["direct_form_1_block"]["channel_msamples_s"]
    c5["realtime_factor_48khz"] = c5["lowlat_default"]["channel_msamples_s"] * 1e6 / C / 48000.0
    with open(os.path.join(args.out, "r03_lowlat_c5.json"), "w") as f:
        json.dump(c5, f, indent=1)
    print(json.dumps({"c5_lowlat": c5["lowlat_default"]["channel_msamples_s"], "c5_direct": c5["direct_form_1_block"]["channel_msamples_s"]}))

    sweep = dict(info, shape=c5["shape"], method="as r03_lowlat_c5.json lowlat_default, per schedule", runs=[])
    for t1 in (2, 4, 8, 16):
        for ratio in (4, 8):
            fb = schedule(t1, ratio, P)
            conv = lowlat(pkg, ir, B, frame_blocks=fb)
            warm_s = max(256, 2 * max(fb))
            r = measure(pkg, torch, conv, C, B, x, y, warm_s, max(steady, 2 * max(fb)), 32)
            conv.close()
            sweep["runs"].append(dict(t1=t1, ratio=ratio, frame_blocks=fb, **r))
            print(json.dumps({"sweep": fb, "channel_msamples_s": r["channel_msamples_s"]}), flush=True)
    best = max(sweep["runs"], key=lambda r: r["channel_msamples_s"])
    sweep["best"] = {"frame_blocks": best["frame_blocks"], "channel_msamples_s": best["channel_msamples_s"]}
    with open(os.path.join(args.out, "r03_lowlat_sweep.json"), "w") as f:
        json.dump(sweep, f, indent=1)
    del x, y, ir
    torch.cuda.empty_cache()

    # C3: stereo, B = 512, 2^17 taps
    C3, B3, taps3 = 2, 512, 1 << 17
    x3 = torch.rand((256, C3, B3), device="cuda") * 2 - 1
    y3 = torch.empty_like(x3)
    ir3 = impulse(torch, C3, taps3)
    c3 = dict(info, shape={"channels": C3, "block": B3, "taps": taps3, "partitions": taps3 // B3},
              reference_direct_form="profiles/r01_c3_latency.json: 20.5 us device / 35.7 us host per block")
    conv = lowlat(pkg, ir3, B3)
    c3["lowlat_default"] = dict(layout=pkg.LowLatencyConvolver.layout(taps3 // B3, B3), **measure(pkg, torch, conv, C3, B3, x3, y3, 256, 2048, 500))
    conv.close()
    direct = pkg.Convolver(pkg.UPOLS, "float32", pkg.DIAGONAL, max_blocks=1)
    direct.impulse(ir3, B3)
    c3["direct_form_1_block"] = measure(pkg, torch, direct, C3, B3, x3, y3, 64, 2048, 500)
    direct.close()
    with open(os.path.join(args.out, "r03_lowlat_c3.json"), "w") as f:
        json.dump(c3, f, indent=1)
    print(json.dumps({"c3_lowlat_us": c3["lowlat_default"]["us_per_block"], "c3_direct_us": c3["direct_form_1_block"]["us_per_block"]}))


if __name__ == "__main__":
    main()
