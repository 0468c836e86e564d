"""Cost of switching the one-block-latency convolver to a new impulse response with a crossfade (LowLatencyConvolver.stage_impulse /
crossfade) on one GPU, DEVICE buffers, one block per call.

    python tools/lowlat_crossfade_time.py [--out profiles] [--quick] [--parent TREE] [--parts phases,noregress]

Writes <out>/r05_lowlat_crossfade_phases.json and (with --parent) r05_lowlat_crossfade_noregress.json, each with the GPU name, power
limit and max SM clock read in the same run:
  - phases, at C5 (1024 channels, 2^20 taps, B = 1024) and stereo (2 channels, 2^17 taps, B = 512), default schedule:
      staging time: host wall of stage_impulse from HOST (pageable) and DEVICE input, each called while 2 T_n blocks of whole-block
      calls are still enqueued (the streams busy), 3 times each;
      stream time per block (CUDA events around a run of one-block calls with no host synchronisation, ended by synchronize) in each
      phase: steady state (nothing staged), the delay window (from the crossfade call to start: level work run for both filters) and
      the fade (FADE_BLOCKS blocks: head run for both filters), over 3 crossfades;
      host wall per one-block call with a synchronize after each (p50 / p99) in steady state and during a fade;
      device bytes before and after the first stage.
  - no regression: tools/lowlat_time.py's C5 measurement at one block per call (via tools/lowlat_samples_time.py --c5-one-block) for the
    tree at TREE (the parent commit, built) and this tree, alternating, one process per run, 3 rounds.
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

from lowlat_samples_time import load  # noqa: E402
from lowlat_time import gpu_info, impulse, pct  # noqa: E402

FADE_BLOCKS = 64


def run_blocks(torch, conv, x, y, count, pos):
    """stream time (s) of `count` one-block calls, and the new block position"""
    s = torch.cuda.current_stream()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(s)
    for t in range(pos, pos + count):
        conv(x[t % x.shape[0]], y[t % y.shape[0]])
    conv.synchronize()
    end.record(s)
    end.synchronize()
    return start.elapsed_time(end) / 1e3, pos + count


def wall_blocks(conv, x, y, count, pos):
    out = []
    for t in range(pos, pos + count):
        t0 = time.perf_counter()
        conv(x[t % x.shape[0]], y[t % y.shape[0]])
        conv.synchronize()
        out.append((time.perf_counter() - t0) * 1e6)
    return {"p50_us": pct(out, 50), "p99_us": pct(out, 99), "max_us": float(max(out)), "calls": count}, pos + count


def phases(pkg, torch, C, B, taps, quick):
    x = torch.rand((64, C, B), device="cuda") * 2 - 1
    y = torch.empty_like(x)
    conv = pkg.LowLatencyConvolver("float32")
    conv.set_stream(torch.cuda.current_stream())
    conv.impulse(impulse(torch, C, taps, seed=1), B)
    levels = conv.layout(taps // B, B)["frame_blocks"]
    busy = 2 * max(levels or (1,))
    irs = [impulse(torch, C, taps, seed=2 + i) for i in range(2)]
    host_ir = irs[0].cpu().numpy()
    res = {"shape": {"channels": C, "block": B, "taps": taps}, "layout": conv.layout(taps // B, B), "fade_blocks": FADE_BLOCKS,
           "device_bytes_before_stage": conv.device_bytes()}
    _, pos = run_blocks(torch, conv, x, y, 2 * busy, 0)  # warm-up: every level runs

    steady, pos = run_blocks(torch, conv, x, y, 4 * busy, pos)
    res["steady_stream_us_per_block"] = steady / (4 * busy) * 1e6
    res["steady_wall_per_call_sync"], pos = wall_blocks(conv, x, y, 200 if quick else 1000, pos)

    stage = {"host": [], "device": []}
    for _ in range(3):
        for kind, ir in (("host", host_ir), ("device", irs[0])):
            for t in range(pos, pos + busy):  # enqueued, not waited for
                conv(x[t % x.shape[0]], y[t % y.shape[0]])
            pos += busy
            t0 = time.perf_counter()
            conv.stage_impulse(ir)
            stage[kind].append((time.perf_counter() - t0) * 1e3)
    conv.synchronize()
    res["stage_wall_ms"] = {k: {"runs": v, "median": float(np.median(v))} for k, v in stage.items()}
    res["stage_busy_blocks_enqueued"] = busy
    res["device_bytes_after_stage"] = conv.device_bytes()

    delay, fade, after, walls = [], [], [], []
    for r in range(3):
        if r > 0:
            conv.stage_impulse(irs[r % 2])
        start = conv.crossfade(FADE_BLOCKS * B)
        n = start // B - pos
        sec, pos = run_blocks(torch, conv, x, y, n, pos)
        delay.append({"blocks": n, "stream_us_per_block": sec / n * 1e6})
        if r == 2:  # host wall per call inside the fade
            w, pos = wall_blocks(conv, x, y, FADE_BLOCKS, pos)
            walls.append(w)
        else:
            sec, pos = run_blocks(torch, conv, x, y, FADE_BLOCKS, pos)
            fade.append({"blocks": FADE_BLOCKS, "stream_us_per_block": sec / FADE_BLOCKS * 1e6})
        sec, pos = run_blocks(torch, conv, x, y, busy, pos)
        after.append({"blocks": busy, "stream_us_per_block": sec / busy * 1e6})
    res["delay_window"] = delay
    res["fade"] = fade
    res["after_fade"] = after
    res["fade_wall_per_call_sync"] = walls[0]
    res["summary_stream_us_per_block"] = {
        "steady": res["steady_stream_us_per_block"],
        "delay_window": float(np.mean([d["stream_us_per_block"] for d in delay])),
        "fade": float(np.mean([d["stream_us_per_block"] for d in fade])),
        "after_fade": float(np.mean([d["stream_us_per_block"] for d in after])),
    }
    conv.close()
    print(json.dumps({"C": C, "B": B, "stream_us_per_block": res["summary_stream_us_per_block"], "stage_ms": {k: v["median"] for k, v in res["stage_wall_ms"].items()},
                      "device_bytes": [res["device_bytes_before_stage"], res["device_bytes_after_stage"]]}), flush=True)
    return res


def measure_noregress(info, args):
    runs = []
    for rnd in range(3):
        for name, tree in (("parent", os.path.abspath(args.parent)), ("this", ROOT)):
            cmd = [sys.executable, os.path.join(ROOT, "tools", "lowlat_samples_time.py"), "--c5-one-block", tree] + (["--quick"] if args.quick else [])
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
    with open(os.path.join(args.out, "r05_lowlat_crossfade_noregress.json"), "w") as f:
        json.dump(noreg, f, indent=1)
    print(json.dumps({"this_over_parent": summary["this_over_parent"]}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--quick", action="store_true", help="small sizes: checks the script end to end, numbers mean nothing")
    ap.add_argument("--parent", help="a built tree of the parent commit, for the no-regression comparison")
    ap.add_argument("--parts", default="phases,noregress", help="comma-separated subset of phases, noregress")
    args = ap.parse_args()

    import torch

    parts = set(args.parts.split(","))
    pkg = load(ROOT)
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    if "phases" in parts:
        shapes = [(64, 256, 1 << 15), (2, 512, 1 << 15)] if args.quick else [(1024, 1024, 1 << 20), (2, 512, 1 << 17)]
        res = dict(info, method=__doc__.split("  - no regression")[0].split("Writes")[1].strip(), shapes=[])
        for C, B, taps in shapes:
            res["shapes"].append(phases(pkg, torch, C, B, taps, args.quick))
            torch.cuda.empty_cache()
        with open(os.path.join(args.out, "r05_lowlat_crossfade_phases.json"), "w") as f:
            json.dump(res, f, indent=1)
    if "noregress" in parts:
        if not args.parent:
            raise SystemExit("the noregress part needs --parent")
        measure_noregress(info, args)


if __name__ == "__main__":
    main()
