"""Cost of switching the convolver bank to a new impulse response with a crossfade (Convolver.stage_impulse / crossfade) on one GPU,
DEVICE buffers, at BASELINE config 5's shape (1024 channels, 2^20 taps, B = 1024).

    python tools/conv_crossfade_time.py [--out profiles] [--quick] [--parent TREE] [--parts phases,noregress]

Writes <out>/r06_conv_crossfade_phases.json and (with --parent) r06_conv_crossfade_noregress.json, each with the GPU name, power limit
and max SM clock read in the same run:
  - phases, for frame mode T = 256 and the direct form at T = 16 and T = 1:
      device time per call (CUDA events around a run of calls on the handle's stream, no host synchronisation in between) steady (nothing
      staged), with a filter staged but no crossfade requested, in fade calls (every sample of the call inside the fade: both filters)
      and after the switch;
      host wall of stage_impulse from HOST pageable memory and from DEVICE memory, 3 times each (the stream idle);
      device bytes before and after the first stage.
  - no regression: device time per call of frame mode T = 256 and the direct form T = 16 with nothing staged, for the tree at TREE (the
    parent commit, built) and this tree, alternating, one process per run, 3 rounds.
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

from lowlat_time import gpu_info, impulse  # noqa: E402

MODES = {"frame256": (256, True), "direct16": (16, False), "direct1": (1, False)}


def load(tree):
    sys.path.insert(0, tree)
    import __graft_entry__ as entry

    pkg = entry.load_package()
    if pkg.device_count() < 1:
        raise SystemExit("conv_crossfade_time.py needs a CUDA device")
    pkg.set_device(0)
    return pkg


def make(pkg, torch, C, B, taps, T, frame):
    conv = pkg.Convolver(pkg.UPOLS, "float32", pkg.DIAGONAL, max_blocks=T, frame_blocks=T if frame else 0)
    conv.set_stream(torch.cuda.current_stream())
    conv.impulse(impulse(torch, C, taps, seed=1), B)
    x = torch.rand((C, T * B), device="cuda") * 2 - 1
    return conv, x, torch.empty_like(x)


def per_call(torch, conv, x, y, count):
    """device time (s) per call over `count` calls"""
    s = torch.cuda.current_stream()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(s)
    for _ in range(count):
        conv(x, y)
    end.record(s)
    end.synchronize()
    return start.elapsed_time(end) / 1e3 / count


def calls_for(T, quick):
    return (4 if quick else 16) if T >= 16 else (16 if quick else 128)


def phases(pkg, torch, C, B, taps, mode, quick):
    T, frame = MODES[mode]
    conv, x, y = make(pkg, torch, C, B, taps, T, frame)
    n = calls_for(T, quick)
    per_call(torch, conv, x, y, 3)  # warm-up
    res = {"mode": mode, "blocks_per_call": T, "frame_mode": frame, "calls_per_measurement": n, "device_bytes_before_stage": conv.device_bytes()}
    res["steady_ms"] = per_call(torch, conv, x, y, n) * 1e3
    ir_host = impulse(torch, C, taps, seed=2).cpu().numpy()
    ir_dev = impulse(torch, C, taps, seed=3)
    torch.cuda.synchronize()
    stage = {"host_pageable": [], "device": []}
    for _ in range(3):
        for kind, ir in (("host_pageable", ir_host), ("device", ir_dev)):
            t0 = time.perf_counter()
            conv.stage_impulse(ir)
            stage[kind].append((time.perf_counter() - t0) * 1e3)
    res["stage_wall_ms"] = {k: {"runs": v, "median": float(np.median(v))} for k, v in stage.items()}
    res["device_bytes_after_stage"] = conv.device_bytes()
    res["staged_ms"] = per_call(torch, conv, x, y, n) * 1e3
    fade, after = [], []
    for r in range(3):
        if r > 0:
            conv.stage_impulse(ir_dev)
        conv.crossfade(n * T * B)  # the next n calls lie wholly inside the fade
        fade.append(per_call(torch, conv, x, y, n) * 1e3)
        after.append(per_call(torch, conv, x, y, n) * 1e3)
    res["fade_ms"] = {"runs": fade, "median": float(np.median(fade))}
    res["after_switch_ms"] = {"runs": after, "median": float(np.median(after))}
    conv.close()
    print(json.dumps({"mode": mode, "steady_ms": res["steady_ms"], "staged_ms": res["staged_ms"], "fade_ms": res["fade_ms"]["median"],
                      "after_ms": res["after_switch_ms"]["median"], "stage_ms": {k: v["median"] for k, v in res["stage_wall_ms"].items()},
                      "device_bytes": [res["device_bytes_before_stage"], res["device_bytes_after_stage"]]}), flush=True)
    return res


def one_steady(tree, mode, quick):
    """the no-regression sample: device time per call with nothing staged, in a process of its own"""
    import torch

    pkg = load(tree)
    C, B, taps = (64, 1024, 1 << 15) if quick else (1024, 1024, 1 << 20)
    T, frame = MODES[mode]
    conv, x, y = make(pkg, torch, C, B, taps, T, frame)
    n = calls_for(T, quick)
    per_call(torch, conv, x, y, 3)
    ms = per_call(torch, conv, x, y, n) * 1e3
    conv.close()
    print(json.dumps({"mode": mode, "ms_per_call": ms, "channel_msamples_s": C * T * B / (ms * 1e3)}))


def measure_noregress(info, args):
    runs = []
    for rnd in range(3):
        for mode in ("frame256", "direct16"):
            for name, tree in (("parent", os.path.abspath(args.parent)), ("this", ROOT)):
                cmd = [sys.executable, os.path.abspath(__file__), "--one", mode, tree] + (["--quick"] if args.quick else [])
                p = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
                if p.returncode != 0:
                    raise SystemExit(f"{name} run failed:\n{p.stdout[-2000:]}\n{p.stderr[-3000:]}")
                r = json.loads(p.stdout.strip().splitlines()[-1])
                runs.append({"round": rnd, "mode": mode, "tree": name, "ms_per_call": r["ms_per_call"], "channel_msamples_s": r["channel_msamples_s"]})
                print(json.dumps(runs[-1]), flush=True)
    summary = {}
    for mode in ("frame256", "direct16"):
        s = {}
        for k in ("parent", "this"):
            v = [r["ms_per_call"] for r in runs if r["tree"] == k and r["mode"] == mode]
            s[k] = {"median_ms_per_call": float(np.median(v)), "runs": v, "spread_ms": float(max(v) - min(v))}
        s["this_over_parent"] = s["this"]["median_ms_per_call"] / s["parent"]["median_ms_per_call"]
        summary[mode] = s
    noreg = dict(info, method="device time per call with nothing staged, C5 shape, DEVICE buffers; parent and this tree alternating, one "
                 "process per run, 3 rounds", runs=runs, summary=summary)
    with open(os.path.join(args.out, "r06_conv_crossfade_noregress.json"), "w") as f:
        json.dump(noreg, f, indent=1)
    print(json.dumps({m: summary[m]["this_over_parent"] for m in summary}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--quick", action="store_true", help="small sizes: checks the script end to end, numbers mean nothing")
    ap.add_argument("--parent", help="a built tree of the parent commit, for the no-regression comparison")
    ap.add_argument("--parts", default="phases,noregress", help="comma-separated subset of phases, noregress")
    ap.add_argument("--one", nargs=2, metavar=("MODE", "TREE"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.one:
        one_steady(args.one[1], args.one[0], args.quick)
        return

    import torch

    parts = set(args.parts.split(","))
    pkg = load(ROOT)
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    if "phases" in parts:
        C, B, taps = (64, 1024, 1 << 15) if args.quick else (1024, 1024, 1 << 20)
        res = dict(info, method=__doc__.split("  - no regression")[0].split("Writes")[1].strip(), shape={"channels": C, "block": B, "taps": taps},
                   modes=[])
        for mode in MODES:
            res["modes"].append(phases(pkg, torch, C, B, taps, mode, args.quick))
            torch.cuda.empty_cache()
        with open(os.path.join(args.out, "r06_conv_crossfade_phases.json"), "w") as f:
            json.dump(res, f, indent=1)
    if "noregress" in parts:
        if not args.parent:
            raise SystemExit("the noregress part needs --parent")
        measure_noregress(info, args)


if __name__ == "__main__":
    main()
