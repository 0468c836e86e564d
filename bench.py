#!/usr/bin/env python
"""bench.py -- the reference's headline workload on B200 (BASELINE.json):
"UPOLS channel-Msamples/s (B=1024, 2^20 taps); batched FFT GB/s vs HBM peak".

    python bench.py --gpus N --steps K --warmup W [--frame T | --frame 0 --blocks T] [--layout GcxGp] [--impl reference]
                    [--dump-outputs DIR]

A step is one call of the convolver bank: T consecutive blocks of 1024 samples for each of the 1024 channels, each channel convolved
with its own 2^20-tap impulse response (P = 1024 partitions) -- BASELINE config 5. T = 1 is the reference's streaming call (one block
per call); T > 1 hands the bank T blocks at once (the CLI / offline case, extra/cli/src/convolver.cpp:42-55). Two forms of T > 1: the
direct form (--frame 0 --blocks T) reuses every filter partition T times in the MAC kernel (FP32-bound from T = 16); frame mode
(--frame T, the default, T = 256) evaluates the sum over partitions by a second overlap-save level along block time
(neo-dsp_b200/csrc/conv_frame.cuh), HBM-bound again. Same results within the float32 tolerance either way; every number states its mode.

  value        whole-job channel-Msamples/s, inputs resident in HBM, CUDA events on the launching streams, max over ranks
  e2e          the same through the C-ABI call with HOST (pinned) buffers: H2D and D2H inside the timed region
  roofline     the dominant kernel (spectral MAC): algorithmic bytes per launch / event-timed duration vs measured HBM peak
  cpu_baseline the reference's own CPU convolver (oracle/_ref) on this box's host cores, bounded sample (N=1, rank 0)
  fft_sweep    batched rfft/irfft float32 N=2^10..2^16 (BASELINE config 2), GB/s against the same HBM peak, CPU pair beside it
  configs      BASELINE configs 1, 3, 4 (c2c N=1024 batch 1; stereo reverb; 64x64 matrix) with the reference CPU figure beside each

N > 1 (torchrun, one rank per GPU): the bank lives in the LIBRARY (neo_b200_bank_*). Layout Gc x Gp: Gc channel groups, inside a
group the partitions of every impulse response are sharded Gp ways and the partial spectra are summed over NVLink (BASELINE config 5:
"partitions sharded across GPUs with NVLink NCCL reduce of partial spectra" -- NEO_B200_BANK_EXCHANGE=collective does it with
ncclReduceScatter; the default moves the rows with the copy engines and sums them inside the c2r kernel, which measured faster); every
rank moves only 1/N of the input and output rows over its own host link and the shards of a group exchange input rows over NVLink.
Default Gp = 2. Total work is fixed: "scaling": "strong". The line also carries the no-collective layout (Gc = N),
BASELINE config 4 sharded by output channel, the FFT batch split over the ranks, and `parity_rel_l2`: rank 0's rows of a multi-step
run compared with a single direct-form handle on the same inputs, outside the timed region (the run fails above 1e-5).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CHANNELS, BLOCK, TAPS = 1024, 1024, 1 << 20
PARTS = TAPS // BLOCK
METRIC = "UPOLS channel-Msamples/s (B=1024, 2^20 taps); batched FFT GB/s vs HBM peak"
UNIT = "channel-Msamples/s"
WORKLOAD = "C5: 1024 channels x 2^20-tap IR each, UPOLS B=1024 (P=1024, K=1025), white-noise input"
PARITY_TOL = 1e-5  # north_star: relative L2 vs neo's own convolver, float32
DUMP_BYTES = 32 << 20  # --dump-outputs writes at most this much output


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---- reference arm (the reference's own CPU code, oracle/_ref) -------------------------------------------------------------------
_CPU_INPUTS: dict = {}


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def timing_ref():
    """(library, how it was compiled) of the reference build that is timed here, or (None, None) when it did not travel."""
    from oracle import pyoracle

    got = pyoracle.ref_timing()
    return got if got is not None else (None, None)


def cpu_conv(channels: int, blocks: int, threads: int, kind: int, block: int = BLOCK, parts: int = PARTS):
    """The reference's own convolver (oracle/_ref when it travelled, else the C restatement) on the host cores:
    `channels` independent convolvers, own filter memory each, `blocks` blocks; returns (channel-Msamples/s, kind, threads)."""
    from oracle import pyoracle

    bins = block + 1
    key = (channels, blocks, block, parts)
    if key not in _CPU_INPUTS:
        rng = np.random.default_rng(11)
        one = (rng.uniform(-1, 1, size=(parts, 2 * bins)).astype(np.float32) * np.float32(1e-3)).view(np.complex64)
        filt = np.empty((channels, parts, bins), dtype=np.complex64)  # own memory per channel, as in the real workload
        filt[:] = one[None]
        sig = rng.uniform(-1, 1, size=(channels, blocks * block)).astype(np.float32)
        _CPU_INPUTS.clear()
        _CPU_INPUTS[key] = (filt, sig)
    filt, sig0 = _CPU_INPUTS[key]
    sig = sig0.copy()
    ref, _ = timing_ref()
    if ref is not None:
        seconds = ref.conv_bench(kind, filt, parts * bins, sig, threads)
        how = "reference"
    else:
        orc = pyoracle.oracle()
        start = time.perf_counter()
        orc.convolve_blocks(0, filt, sig)
        seconds = time.perf_counter() - start
        how, threads = "port", 1
    return channels * blocks * block / seconds / 1e6, how, threads


def run_reference(args, rank: int):
    if rank != 0:
        return
    cores = host_cores()
    sample = max(cores, min(2 * cores, 128))
    blocks = 32
    vals = []
    for _ in range(args.warmup):
        cpu_conv(min(sample, cores), 4, cores, 2)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, how, used = cpu_conv(sample, blocks, cores, 2)
        vals.append(v)
    wall = time.perf_counter() - t0
    value = float(np.mean(vals))
    _, flags = timing_ref()
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / max(1, args.steps),
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "blocks_per_call": 1},
        "cpu_baseline": {
            "value": value,
            "unit": UNIT,
            "cores": used,
            "kind": how,
            "sample": f"{sample} of 1024 channels x {blocks} blocks per step, own random filter per channel, "
                      f"neo::split_upols_convolver (the reference's faster dense form), {flags}, no xsimd; worker threads are created "
                      "before the clock starts",
        },
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---- helpers shared by both GPU paths ---------------------------------------------------------------------------------------------
def mode_name(frame: int, T: int) -> str:
    if frame > 0:
        return f"frame mode: {T} blocks per call, sum over partitions by overlap-save along block time (frame transforms of length {2 * T})"
    return "streaming (reference call shape)" if T == 1 else f"time-batched direct form, {T} blocks per call"


def impulse_rows(torch, first: int, count: int, taps: int = TAPS, seed: int = 1100):
    """rows [first, first+count) of the bank's random impulse responses on the current device. One generator seed per channel, so any
    rank regenerates any row; scaled to unit expected energy (normalize_impulse's common factor to within 0.2 % for white noise)."""
    out = torch.empty((count, taps), device="cuda", dtype=torch.float32)
    gen = torch.Generator(device="cuda")
    for i in range(count):
        gen.manual_seed(seed + first + i)
        out[i].uniform_(-1.0, 1.0, generator=gen)
    out *= float(np.sqrt(3.0 / taps))
    return out


def signal_rows(torch, first: int, count: int, samples: int, seed: int = 1300):
    out = torch.empty((count, samples), device="cuda", dtype=torch.float32)
    gen = torch.Generator(device="cuda")
    for i in range(count):
        gen.manual_seed(seed + first + i)
        out[i].uniform_(-1.0, 1.0, generator=gen)
    return out


def frame_bytes_per_channel(T: int, q_local: int) -> int:
    """algorithmic bytes of the fused frame kernel per channel and launch: the two frames' level-1 spectra (2T rows of B) read, Q
    filter rows and Q-1 older ring slots of 2T x (B+1) bins read, the new ring slot and the T result rows written"""
    bins = BLOCK + 1
    return 8 * (bins * 2 * T * 2 * q_local + 3 * T * BLOCK)


def direct_bytes_per_channel(T: int, parts_local: int) -> int:
    """SURVEY 8d: 16*K*P bytes per channel-block at T=1; with T blocks per launch the filter is read once and P+T-1 delay-line rows
    serve all T blocks; plus the T accumulator rows written"""
    return 8 * (BLOCK + 1) * (parts_local + (parts_local + T - 1) + T)


def fft_sweep(pkg, torch, peak, share: int = 1, reps: int = 10):
    """BASELINE config 2: batched rfft / irfft float32, N = 2^10..2^16, batch = 2^29/N (2 GiB in per pass) / share."""
    out = []
    x = torch.rand((1 << 29) // share, device="cuda", dtype=torch.float32) * 2 - 1
    for order in range(10, 17):
        n = 1 << order
        batch = (1 << 29) // n // share
        plan = pkg.RFFTPlan(order, "float32")
        plan.set_stream(torch.cuda.current_stream())
        xin = x.view(batch, n)
        spec = torch.empty((batch, n // 2 + 1), dtype=torch.complex64, device="cuda")
        back = torch.empty_like(xin)
        bytes_pass = batch * (4 * n + 8 * (n // 2 + 1))
        res = {"n": n, "batch": batch}
        for name, fn in (("r2c", lambda: plan.rfft(xin, out=spec)), ("c2r", lambda: plan.irfft(spec, out=back))):
            for _ in range(3):
                fn()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
            ev[0].record()
            for i in range(reps):
                fn()
                ev[i + 1].record()
            torch.cuda.synchronize()
            ms = float(np.median([ev[i].elapsed_time(ev[i + 1]) for i in range(reps)]))
            res[name + "_ms"] = ms
            res[name + "_gbs"] = bytes_pass / ms / 1e6
            res[name + "_frac"] = res[name + "_gbs"] / peak
        out.append(res)
        plan.close()
        del spec, back
    del x
    torch.cuda.empty_cache()
    return out


def fft_cpu_baseline(sweep):
    """The reference's rfft+irfft pair (what extra/benchmark/src/rfft.cpp:22-31 times) on the host, 1 thread and all cores, 16 MiB of
    rows per size, with the bytes convention of the GPU sweep (4N + 8(N/2+1) per direction)."""
    ref, flags = timing_ref()
    if ref is None:
        return None
    cores = host_cores()
    rng = np.random.default_rng(2)
    for res in sweep:
        n = res["n"]
        order = n.bit_length() - 1
        pair_bytes = 2 * (4 * n + 8 * (n // 2 + 1))
        out = {}
        for threads in (1, cores):
            batch = max(threads * 4, (1 << (22 if threads > 1 else 20)) // n)
            data = rng.uniform(-1, 1, size=(batch, n)).astype(np.float32)
            sec = ref.rfft_bench(order, data, threads)
            out[f"pair_gbs_{threads}_threads" if threads > 1 else "pair_gbs_1_thread"] = batch * pair_bytes / sec / 1e9
        res["cpu_reference"] = out
    return {"cores": cores, "kind": "reference", "build": flags,
            "what": "neo::fft::rfft_plan rfft + irfft round trips (fallback plan, no xsimd), GB/s with the sweep's byte convention"}


# ---- BASELINE configs 1, 3, 4 (one GPU) ---------------------------------------------------------------------------------------------
def gpu_time(torch, fn, reps, warm=3):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps  # ms


def config_c1(pkg, torch):
    """c2c complex<float> N=1024: forward + inverse (+1/N) round trips. batch 1 through host buffers is the reference's call shape
    (extra/benchmark/src/fft.cpp:22-29); the batched device figure is the one the HBM roofline applies to (16 N bytes per transform)."""
    ref, flags = timing_ref()
    x = np.random.default_rng(1).uniform(-1, 1, size=2048).astype(np.float32)
    cpu_us = None
    if ref is not None:
        reps = 20000
        cpu_us = ref.c2c_bench(10, x.copy(), reps) / reps * 1e6
    plan = pkg.FFTPlan(10, np.complex64)
    buf = x.view(np.complex64).copy()
    for _ in range(20):
        plan(buf, pkg.FORWARD)
    t0 = time.perf_counter()
    for _ in range(300):
        plan(buf, pkg.FORWARD)
        plan(buf, pkg.BACKWARD)
    host_us = (time.perf_counter() - t0) / 300 * 1e6
    plan.set_stream(torch.cuda.current_stream())
    one = torch.randn((1, 1024), dtype=torch.complex64, device="cuda")
    dev_us = gpu_time(torch, lambda: (plan(one, pkg.FORWARD), plan(one, pkg.BACKWARD)), reps=200, warm=20) * 1e3
    batch = 1 << 18
    dx = torch.randn((batch, 1024), dtype=torch.complex64, device="cuda")
    ms = gpu_time(torch, lambda: (plan(dx, pkg.FORWARD), plan(dx, pkg.BACKWARD)), reps=20)
    plan.close()
    return {
        "workload": "C1: c2c complex<float> N=1024, forward + inverse per round trip",
        "reference_cpu_us_per_roundtrip_1_core": cpu_us,
        "reference_build": flags,
        "b200_host_call_us_per_roundtrip_batch1": host_us,
        "b200_device_us_per_roundtrip_batch1": dev_us,
        "b200_device_batched_ns_per_roundtrip": ms * 1e6 / batch,
        "b200_device_batched_gbs": 2 * 2 * batch * 1024 * 8 / ms / 1e6,
        "note": "one 8 KiB transform per call is launch + PCIe latency on a GPU (two kernel launches and four 8 KiB copies per round trip); "
                "the batched figure is what the HBM roofline applies to",
    }


def config_c3(pkg, torch):
    """UPOLS stereo, B=512, 2^17-tap IR (P=256): state is L2-resident (2 x 2.1 MB), so the bound is launch latency, not HBM."""
    B, L, C = 512, 1 << 17, 2
    ir = impulse_rows(torch, 0, C, L, seed=3100)
    res = {"workload": "C3: UPOLS stereo, B=512, 2^17-tap IR per channel (P=256)"}
    for frame, T in ((0, 1), (0, 16), (64, 64)):
        conv = pkg.Convolver(pkg.UPOLS, "float32", pkg.DIAGONAL, max_blocks=T, frame_blocks=frame)
        conv.set_stream(torch.cuda.current_stream())
        conv.impulse(ir, B)
        xin = torch.rand((C, T * B), device="cuda") * 2 - 1
        yout = torch.empty_like(xin)
        ms = gpu_time(torch, lambda: conv(xin, out=yout), reps=200 if T == 1 else 50, warm=10)
        entry = {"device_us_per_block": ms * 1e3 / T, "realtime_x_48k": (B * T / 48000.0) / (ms * 1e-3),
                 "channel_msamples_s": C * B * T / ms / 1e3}
        if T == 1:  # the reference's own call: one block of pageable host memory in, the same block out
            hx = np.random.default_rng(3).uniform(-1, 1, size=(C, B)).astype(np.float32)
            for _ in range(20):
                conv(hx)
            t0 = time.perf_counter()
            for _ in range(300):
                conv(hx)
            entry["host_call_us_per_block"] = (time.perf_counter() - t0) / 300 * 1e6
        res[f"frame{T}" if frame else f"T{T}"] = entry
        conv.close()
    cores = host_cores()
    v1, how, _ = cpu_conv(C, 400, 1, 2, block=B, parts=L // B)
    v2, _, used = cpu_conv(C, 400, min(C, cores), 2, block=B, parts=L // B)
    _, flags = timing_ref()
    res["cpu_reference"] = {"kind": how, "build": flags, "us_per_block_1_core": C * B / v1, "us_per_block_2_threads": C * B / v2 if used > 1 else None,
                            "channel_msamples_s_1_core": v1, "what": "2 x neo::split_upols_convolver, 400 blocks"}
    return res


def config_c4(pkg, torch, peak):
    """64-in x 64-out convolution matrix, B=256, 2^16-tap IRs (P=256, K=257): per block-step 8*64*64*256*257 = 2.156 GFLOP; at T=1 the
    2.156 GB filter set streams once per block-step (HBM roofline), time-batched the contraction is FP32-bound, in frame mode the
    second-level filter set streams once per T blocks."""
    B, L, O, I = 256, 1 << 16, 64, 64
    P, K = L // B, B + 1
    ir = impulse_rows(torch, 0, O * I, L, seed=4100).view(O, I, L)
    res = {"workload": "C4: 64-in x 64-out convolution matrix, B=256, 2^16-tap IRs (P=256)", "flop_per_block_step": 8 * O * I * P * K,
           "filter_bytes": 8 * K * P * O * I}
    for frame, T in ((0, 1), (0, 16), (64, 64)):
        conv = pkg.Convolver(pkg.UPOLS, "float32", pkg.MATRIX, max_blocks=T, frame_blocks=frame)
        conv.set_stream(torch.cuda.current_stream())
        conv.impulse(ir, B)
        xin = torch.rand((I, T * B), device="cuda") * 2 - 1
        yout = torch.empty((O, T * B), device="cuda")
        reps = 20
        for _ in range(3):
            conv(xin, out=yout)
        conv.profile(True)
        conv.profile_read()
        ms = gpu_time(torch, lambda: conv(xin, out=yout), reps=reps, warm=0)
        _, mac_ms, _, _, _, _ = conv.profile_read(frame_phases=True)
        mac = mac_ms / reps
        entry = {"ms_per_block_step": ms / T, "realtime_x_48k": (B * T / 48000.0) / (ms * 1e-3), "mac_ms_per_call": mac}
        if frame:
            stream_bytes = 8 * K * 2 * T * ((P + T - 1) // T) * O * I
            entry["mac_filter_stream_gbs"] = stream_bytes / mac / 1e6
            entry["mac_frac_of_hbm"] = entry["mac_filter_stream_gbs"] / peak
        else:
            entry["mac_fp32_tflops"] = 8.0 * K * P * O * I * T / mac / 1e9
            if T == 1:
                entry["mac_filter_stream_gbs"] = 8 * K * P * O * I / mac / 1e6
                entry["mac_frac_of_hbm"] = entry["mac_filter_stream_gbs"] / peak
        res[f"frame{T}" if frame else f"T{T}"] = entry
        conv.close()
    del ir
    torch.cuda.empty_cache()
    # reference: 64 x 64 independent convolvers summed per output (uniform_partitioned_convolver.hpp:48-65); a slice of 4 outputs x 64
    # inputs is timed and scaled by 16 (the convolvers are independent)
    cores = host_cores()
    slice_convs, blocks = 4 * I, 8
    v1, how, _ = cpu_conv(slice_convs, blocks, 1, 2, block=B, parts=P)
    vn, _, used = cpu_conv(slice_convs, blocks, cores, 2, block=B, parts=P)
    _, flags = timing_ref()
    per_step = O * I * B  # convolver-samples per block-step of the whole matrix
    res["cpu_reference"] = {"kind": how, "build": flags, "ms_per_block_step_1_core": per_step / v1 / 1e3,
                            f"ms_per_block_step_{used}_threads": per_step / vn / 1e3,
                            "what": f"{slice_convs} of 4096 neo::split_upols_convolver x {blocks} blocks, scaled to the full matrix"}
    return res


# ---- unchanged-driver shape: one facade convolver per channel, one block per call, pageable memory ---------------------------------
def unchanged_driver(channels: int, blocks: int):
    """tests/cpp/unchanged_driver: the per-channel loop of extra/cli/src/convolver.cpp:37-55 / extra/benchmark/src/convolution.cpp:28-40
    compiled against include/neo_b200.hpp (one neo::b200::upols_convolver per channel, one block per call, std::vector memory)."""
    import subprocess

    exe = os.path.join(ROOT, "tests", "cpp", "unchanged_driver")
    if not os.path.exists(exe):
        return None
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = os.path.join(ROOT, "neo-dsp_b200") + os.pathsep + env.get("LD_LIBRARY_PATH", "")
    try:
        proc = subprocess.run([exe, str(channels), str(blocks), str(BLOCK), str(TAPS)], capture_output=True, text=True, timeout=300, env=env)
        return json.loads(proc.stdout.strip().splitlines()[-1]) if proc.returncode == 0 else {"error": proc.stderr[-300:]}
    except Exception as exc:  # measurement aid: never take the headline line down
        return {"error": str(exc)}


# ---- one GPU ---------------------------------------------------------------------------------------------------------------------
def build_conv(pkg, torch, stream, T, frame, channels=CHANNELS, first=0):
    conv = pkg.Convolver(pkg.UPOLS, "float32", pkg.DIAGONAL, max_blocks=T, frame_blocks=frame)
    conv.set_stream(stream)
    ir = impulse_rows(torch, first, channels)
    conv.impulse(ir, BLOCK)
    del ir
    torch.cuda.empty_cache()
    return conv


def host_link_probe(torch, hx, hy, iters: int = 8):
    """GB/s per direction of pinned H2D + D2H copies running at the same time (the bound of every e2e number here)"""
    dx, dy = torch.empty(hx.shape, dtype=hx.dtype, device="cuda"), torch.empty(hy.shape, dtype=hy.dtype, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    best = 0.0
    for _ in range(iters):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        s1.wait_event(e0)
        s2.wait_event(e0)
        with torch.cuda.stream(s1):
            dx.copy_(hx, non_blocking=True)
        with torch.cuda.stream(s2):
            hy.copy_(dy, non_blocking=True)
        torch.cuda.current_stream().wait_stream(s1)
        torch.cuda.current_stream().wait_stream(s2)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, hx.numel() * hx.element_size() / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del dx, dy
    return best


def e2e_host(conv, hx, hy, steps):
    """the C-ABI call a reference-side caller makes: HOST buffers in, HOST buffers out, returns when hy holds the result"""
    T = hx.shape[1] // BLOCK
    for _ in range(2):
        conv(hx, out=hy)
    t0 = time.perf_counter()
    for _ in range(steps):
        conv(hx, out=hy)
    return CHANNELS * BLOCK * T * steps / (time.perf_counter() - t0) / 1e6


def run_single(args, pkg, torch, emit, peak, peak_src):
    stream = torch.cuda.current_stream()
    frame = args.frame
    T = frame if frame > 0 else args.blocks
    # BASELINE config 2 runs first: its passes are short bursts and are compared with the burst copy bandwidth, so they are taken
    # before the sustained convolver loop pulls the part into its power cap
    sweep = None if args.no_fft_sweep else fft_sweep(pkg, torch, peak)

    conv = build_conv(pkg, torch, stream, T, frame)
    nbuf = 4 if T <= 256 else 2
    gen = torch.Generator(device="cuda").manual_seed(13)
    xs = [torch.rand((CHANNELS, T * BLOCK), device="cuda", dtype=torch.float32, generator=gen) * 2 - 1 for _ in range(nbuf)]
    ys = torch.empty((CHANNELS, T * BLOCK), device="cuda", dtype=torch.float32)
    warm = max(3, args.warmup)
    for i in range(warm):
        conv(xs[i % nbuf], out=ys)
    torch.cuda.synchronize()
    launches0 = pkg.kernel_launches()
    conv.profile(True)
    conv.profile_read()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clocks:
        torch.cuda.synchronize()
        start.record()
        for i in range(args.steps):
            conv(xs[i % nbuf], out=ys)
        stop.record()
        torch.cuda.synchronize()
    ms_total = start.elapsed_time(stop)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, torch, ys)
    ms_r2c, ms_mac, ms_c2r, mac_launches = conv.profile_read()
    conv.profile(False)
    launches = pkg.kernel_launches() - launches0
    value = CHANNELS * BLOCK * T * args.steps / (ms_total * 1e-3) / 1e6

    # ---- e2e: HOST buffers through the C ABI; pinned (copies overlap the kernels) and pageable (what std::vector / numpy hands over) ----
    n_e2e = max(3, min(args.steps, 20))
    hx = torch.rand((CHANNELS, T * BLOCK), dtype=torch.float32).pin_memory()
    hy = torch.empty((CHANNELS, T * BLOCK), dtype=torch.float32).pin_memory()
    e2e_pinned = e2e_host(conv, hx.numpy(), hy.numpy(), n_e2e)
    px, py = np.array(hx.numpy(), copy=True), np.empty((CHANNELS, T * BLOCK), dtype=np.float32)
    e2e_pageable = e2e_host(conv, px, py, max(3, n_e2e // 2))
    io_bytes = CHANNELS * T * BLOCK * 4
    e2e = {"value": e2e_pinned, "unit": UNIT, "h2d_bytes_per_step": io_bytes, "d2h_bytes_per_step": io_bytes, "steps": n_e2e,
           "host_memory": "pinned", "blocks_per_call": T}
    # what bounds it: the host link with both directions busy (plain pinned copies of the same buffers, no kernels)
    link = host_link_probe(torch, hx, hy)
    e2e["host_link"] = {"both_directions_gbs_each": link, "achieved_gbs_each": e2e_pinned * 1e6 * 4 / 1e9,
                        "what": "cudaMemcpyAsync H2D and D2H of the step's 1 GiB buffers on two streams at once, GB/s per direction, best of 8 "
                                "(a momentary figure: the host side is shared with the box's other GPUs); e2e moves the same bytes, so achieved / "
                                "both_directions is its fraction of the link"}
    del hx, hy, px, py

    # ---- roofline of the dominant kernel (spectral MAC), from the event-timed launches inside the timed region ----
    if frame > 0:
        q = (PARTS + T - 1) // T
        alg_bytes_launch = CHANNELS * frame_bytes_per_channel(T, q)
        kernel_name = (f"frame_fused_kernel<float, LOGL={(2 * T).bit_length() - 1}{', 32 points per thread' if T >= 512 or (T == 256 and q <= 2) else ''}>"
                       " (frame transform + ring insert + MAC + inverse frame transform)")
    else:
        alg_bytes_launch = CHANNELS * direct_bytes_per_channel(T, PARTS)
        kernel_name = "fdl_mac_stream_kernel<float>" if T == 1 else f"fdl_mac_tma_kernel (T={T})"
    mac_ms_avg = ms_mac / max(1, mac_launches)
    achieved = alg_bytes_launch / (mac_ms_avg * 1e-3) / 1e9 if mac_ms_avg > 0 else 0.0
    fp32 = CHANNELS * 8.0 * (BLOCK + 1) * PARTS * T / (mac_ms_avg * 1e-3) / 1e12 if frame == 0 and mac_ms_avg > 0 else None
    traffic, traffic_src = ncu_traffic(f"frame_fused_T{T}_G1" if frame > 0 else f"fdl_mac_T{T}_G1")
    roofline = {
        "kernel": kernel_name, "bound": "hbm", "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
        "algorithmic_bytes_per_launch": alg_bytes_launch, "launch_ms": mac_ms_avg,
        "share_of_step": ms_mac / ms_total if ms_total > 0 else None, "fp32_tflops": fp32,
        "phases_ms_per_step": {"r2c_fdl_insert": ms_r2c / args.steps, "mac": ms_mac / args.steps, "c2r_discard": ms_c2r / args.steps},
    }
    # the forward / inverse block transforms as HBM streams: T*B reals in, T*B complex out per channel (and back)
    io_alg = CHANNELS * T * BLOCK * 12
    if ms_r2c > 0 and ms_c2r > 0:
        roofline["r2c_frac_of_hbm"] = io_alg / (ms_r2c / args.steps * 1e-3) / 1e9 / peak
        roofline["c2r_frac_of_hbm"] = io_alg / (ms_c2r / args.steps * 1e-3) / 1e9 / peak

    modes = None
    e2e_modes = {f"frame{T}" if frame > 0 else f"T{T}": {"pinned": e2e_pinned, "pageable": e2e_pageable, "unit": UNIT}}
    if not args.no_modes:
        # the other call shapes, measured the same way (fewer steps), so every number on the line states its T
        conv.close()
        del conv, xs, ys
        torch.cuda.empty_cache()
        tag = f"frame{T}" if frame > 0 else f"T{T}"
        modes = {tag: {"value": value, "unit": UNIT, "mac_algorithmic_gbs": achieved, "mac_fp32_tflops": fp32}}
        for f_other, t_other in [(0, 1), (0, 16), (64, 64), (256, 256), (512, 512)]:
            if (f_other, t_other) == (frame, T):
                continue
            c2 = build_conv(pkg, torch, stream, t_other, f_other)
            x2 = torch.rand((CHANNELS, t_other * BLOCK), device="cuda", dtype=torch.float32) * 2 - 1
            y2 = torch.empty_like(x2)
            for _ in range(max(3, args.warmup)):
                c2(x2, out=y2)
            c2.profile(True)
            c2.profile_read()
            n2 = 30 if t_other == 1 else 10
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(n2):
                c2(x2, out=y2)
            e1.record()
            torch.cuda.synchronize()
            _, mac2, _, nl2 = c2.profile_read()
            ms2 = e0.elapsed_time(e1)
            if f_other > 0:
                alg2 = CHANNELS * frame_bytes_per_channel(t_other, (PARTS + t_other - 1) // t_other)
                flops2 = None
            else:
                alg2 = CHANNELS * direct_bytes_per_channel(t_other, PARTS)
                flops2 = CHANNELS * 8.0 * (BLOCK + 1) * PARTS * t_other / (mac2 / max(1, nl2) * 1e-3) / 1e12
            name2 = f"frame{t_other}" if f_other > 0 else f"T{t_other}"
            modes[name2] = {"value": CHANNELS * BLOCK * t_other * n2 / (ms2 * 1e-3) / 1e6, "unit": UNIT,
                            "mac_algorithmic_gbs": alg2 / (mac2 / max(1, nl2) * 1e-3) / 1e9, "mac_fp32_tflops": flops2, "steps": n2}
            if (f_other, t_other) in ((0, 1), (0, 16)):  # e2e per mode: the reference's streaming call and the direct form
                hx = torch.rand((CHANNELS, t_other * BLOCK), dtype=torch.float32).pin_memory()
                hy = torch.empty((CHANNELS, t_other * BLOCK), dtype=torch.float32).pin_memory()
                n3 = 30 if t_other == 1 else 10
                pinned = e2e_host(c2, hx.numpy(), hy.numpy(), n3)
                px, py = np.array(hx.numpy(), copy=True), np.empty((CHANNELS, t_other * BLOCK), dtype=np.float32)
                e2e_modes[name2] = {"pinned": pinned, "pageable": e2e_host(c2, px, py, n3), "unit": UNIT}
                del hx, hy, px, py
            c2.close()
            del c2, x2, y2
            torch.cuda.empty_cache()
    else:
        conv.close()
        del conv, xs, ys
        torch.cuda.empty_cache()

    configs = None
    if not args.no_configs:
        configs = {"C1": config_c1(pkg, torch), "C3": config_c3(pkg, torch), "C4": config_c4(pkg, torch, peak)}

    cores = host_cores()
    sample = max(cores, min(2 * cores, 128))
    v_split, how, used = cpu_conv(sample, 16, cores, 2)
    v_aos, _, _ = cpu_conv(sample, 16, cores, 0)
    v_one, _, _ = cpu_conv(2, 16, 1, 2)
    _, flags = timing_ref()
    cpu_baseline = {
        "value": max(v_split, v_aos), "unit": UNIT, "cores": used, "kind": how, "value_1_core": v_one,
        "sample": f"{sample} of 1024 channels x 16 blocks, own random filter per channel; split_upols_convolver {v_split:.2f}, "
                  f"upols_convolver {v_aos:.2f} {UNIT} on {used} threads, split_upols_convolver {v_one:.2f} on 1 core ({flags}, no xsimd)",
    }
    driver = None if args.no_configs else unchanged_driver(32, 24)
    if driver is not None and "channel_msamples_s" in driver:
        e2e_modes["unchanged_driver"] = driver
    fft_cpu = fft_cpu_baseline(sweep) if sweep is not None else None

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": WORKLOAD, "blocks_per_call": T, "mode": mode_name(frame, T), "sharding": "none",
            "l2": "working set per step (filter + delay line, 17-41 GB) exceeds the 126 MB L2; 4 rotating input buffers",
            "realtime_x_aggregate_48k": value * 1e6 / 48000.0, "realtime_x_wall_1024ch_48k": value * 1e6 / CHANNELS / 48000.0,
        },
        "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu_baseline,
        "e2e_modes": e2e_modes,
    }
    if modes is not None:
        line["modes"] = modes
    if sweep is not None:
        line["fft_sweep"] = sweep
        if fft_cpu is not None:
            line["fft_sweep_cpu_baseline"] = fft_cpu
    if configs is not None:
        line["configs"] = configs
    emit(line)


def dump_outputs(directory: str, torch, y) -> None:
    """--dump-outputs: what the last timed step handed back, y[channels][T*B] float32, as `directory`/output.npy. Above DUMP_BYTES
    a fixed seeded sample of whole channel rows (ascending order) is written, and where one row alone exceeds it, each row's leading
    samples. The inputs are seeded, so two builds run with the same arguments can be compared output for output."""
    rows = max(1, min(y.shape[0], DUMP_BYTES // (y.shape[1] * y.element_size())))
    cols = min(y.shape[1], DUMP_BYTES // (rows * y.element_size()))
    pick = np.sort(np.random.default_rng(0).choice(y.shape[0], rows, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "output.npy"), y[torch.as_tensor(pick, device=y.device), :cols].cpu().numpy())


def ncu_traffic(key: str, scale: int = 1):
    """(bytes, source): dram__bytes_read.sum + dram__bytes_write.sum per launch from an ncu --set full capture of this kernel
    (profiles/traffic.json names the capture); `scale` multiplies per-channel entries. (None, None) when never captured."""
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            entry = json.load(f).get(key)
        if isinstance(entry, dict):
            return entry["bytes"] * scale, "ncu capture, not measured in this run: " + entry["capture"]
    return None, None


# ---- N GPUs: the library's bank --------------------------------------------------------------------------------------------------
def parse_layout(text: str, world: int):
    if text:
        gc, gp = (int(v) for v in text.lower().split("x"))
    else:
        gp = 2 if world % 2 == 0 else 1
        gc = world // gp
    if gc * gp != world:
        raise SystemExit(f"--layout {text}: {gc} x {gp} != {world} ranks")
    return gc, gp


def make_bank(pkg, torch, dist, rank, world, local, layout, T, frame, topology=None, outputs=CHANNELS, inputs=CHANNELS, block=BLOCK,
              taps=TAPS, seed=1100):
    topology = pkg.DIAGONAL if topology is None else topology
    uid = [pkg.bank_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    bank = pkg.Bank(pkg.UPOLS, "float32", topology, outputs, inputs, block, taps // block, max_blocks=T, frame_blocks=frame, layout=layout,
                    rank=rank, world=world, unique_id=uid[0], device=local)
    info = bank.ranks[0]
    if topology == pkg.DIAGONAL:
        ir = impulse_rows(torch, info["group_first"], info["group_count"], taps, seed)
    else:
        ir = impulse_rows(torch, info["group_first"] * inputs, info["group_count"] * inputs, taps, seed).view(info["group_count"], inputs, taps)
    bank.impulse([ir])
    del ir
    torch.cuda.empty_cache()
    return bank, info


def run_bank_timed(bank, xs, ys, steps, device: bool):
    """`steps` pipelined steps (three in flight: the copy-in of step i+2 and the copy-out of step i-1 overlap the kernels of step i);
    returns device milliseconds (CUDA events on the bank's streams) and wall seconds"""
    t0 = time.perf_counter()
    bank.timer_start()
    for i in range(steps):
        bank.submit([xs[i % len(xs)]], [ys[i % len(ys)]])
        if i >= 2:
            bank.wait()
    ms = bank.timer_stop()
    return ms, time.perf_counter() - t0


def measure_layout(args, pkg, torch, dist, rank, world, local, layout, T, frame, steps, want_e2e=True, want_parity=True):
    """value / e2e / roofline / parity of BASELINE config 5 on a Gc x Gp bank. Every rank calls; every rank gets the dict."""
    bank, info = make_bank(pkg, torch, dist, rank, world, local, layout, T, frame)
    n_in, n_out = info["in_count"], info["out_count"]
    xs = [torch.rand((n_in, T * BLOCK), device="cuda", dtype=torch.float32) * 2 - 1 for _ in range(4)]
    ys = [torch.empty((n_out, T * BLOCK), device="cuda", dtype=torch.float32) for _ in range(3)]
    max_over_ranks = lambda v: float(_allreduce_max(torch, dist, v))
    warm = max(3, args.warmup)
    torch.cuda.synchronize()  # the bank's streams do not wait for torch's: the inputs above must be complete
    run_bank_timed(bank, xs, ys, warm, True)
    dist.barrier()
    torch.cuda.synchronize()
    launches0 = pkg.kernel_launches()
    bank.profile(True)
    bank.profile_read(0)
    with ClockSampler(local) as clocks:
        dist.barrier()
        ms_total, _ = run_bank_timed(bank, xs, ys, steps, True)
        dist.barrier()
    ms_total = max_over_ranks(ms_total)
    ms_r2c, ms_mac, ms_c2r, _, _, mac_launches = bank.profile_read(0)
    bank.profile(False)
    launches = pkg.kernel_launches() - launches0
    value = CHANNELS * BLOCK * T * steps / (ms_total * 1e-3) / 1e6
    res = {"value": value, "unit": UNIT, "steps": steps, "ms_per_step": ms_total / steps, "blocks_per_call": T, "mode": mode_name(frame, T),
           "layout": f"{layout[0]} channel groups x {layout[1]} partition shards", "clocks": clocks.summary(), "gpu_launches": launches,
           "device_bytes_per_rank": bank.device_bytes(0), "realtime_x_wall_1024ch_48k": value * 1e6 / CHANNELS / 48000.0}

    # roofline of the dominant kernel on THIS rank: its share of the channels and partitions
    parts_local = info["partition_end"] - info["partition_begin"]
    if frame > 0:
        alg = info["group_count"] * frame_bytes_per_channel(T, (parts_local + T - 1) // T)
    else:
        alg = info["group_count"] * direct_bytes_per_channel(T, parts_local)
    mac_ms = ms_mac / max(1, mac_launches)
    peak, peak_src = measured_peaks()
    q_local = (parts_local + T - 1) // T if frame > 0 else 0
    traffic, traffic_src = ncu_traffic(f"frame_fused_T{T}_Q{q_local}_per_channel", info["group_count"]) if frame > 0 else (None, None)
    if traffic is None and frame > 0 and layout[1] == 1 and info["group_count"] > 0:  # unsharded partitions: the one-GPU kernel on fewer channels
        whole, traffic_src = ncu_traffic(f"frame_fused_T{T}_G1")
        traffic = whole * info["group_count"] // CHANNELS if whole is not None else None
    res["roofline"] = {
        "kernel": (("frame_fused_kernel<float, 32 points per thread>" if q_local <= 2 or T >= 512 else "frame_fused_kernel<float>") if T >= 256
                   else "frame_fused_kernel<float>") if frame > 0 else "fdl_mac kernel",
        "bound": "hbm", "unit": "GB/s", "peak": peak, "peak_source": peak_src,
        "achieved": alg / (mac_ms * 1e-3) / 1e9 if mac_ms > 0 else 0.0, "frac": (alg / (mac_ms * 1e-3) / 1e9 / peak) if mac_ms > 0 else 0.0,
        "algorithmic_bytes_per_launch": alg, "launch_ms": mac_ms, "rank": rank,
        "traffic": traffic, "traffic_source": traffic_src,
        "phases_ms_per_step": {"r2c_fdl_insert": ms_r2c / steps, "mac": ms_mac / steps, "c2r_discard": ms_c2r / steps},
        "share_of_step": (ms_mac / steps) / (ms_total / steps) if ms_total > 0 else None,
    }

    if want_e2e:
        # end to end: every rank moves ITS 1/N of the rows between pinned host memory and the device, three steps in flight
        hx = [torch.rand((n_in, T * BLOCK), dtype=torch.float32).pin_memory().numpy() for _ in range(3)]
        hy = [torch.empty((n_out, T * BLOCK), dtype=torch.float32).pin_memory().numpy() for _ in range(3)]
        run_bank_timed(bank, hx, hy, 4, False)
        n_e2e = max(4, min(steps, 20))
        dist.barrier()
        _, wall = run_bank_timed(bank, hx, hy, n_e2e, False)
        dist.barrier()
        wall = max_over_ranks(wall)
        res["e2e"] = {"value": CHANNELS * BLOCK * T * n_e2e / wall / 1e6, "unit": UNIT, "h2d_bytes_per_step": CHANNELS * T * BLOCK * 4,
                      "d2h_bytes_per_step": CHANNELS * T * BLOCK * 4, "steps": n_e2e, "host_memory": "pinned",
                      "per_rank": f"each rank copies {n_in} of {CHANNELS} rows in and {n_out} out per step; shards of a group all-gather over NVLink"}
        del hx, hy

    if want_parity:
        res["parity_rel_l2"] = bank_parity(pkg, torch, dist, bank, info, rank, T, frame)
    bank.close()
    del bank, xs, ys
    torch.cuda.empty_cache()
    return res


def bank_parity(pkg, torch, dist, bank, info, rank, T, frame):
    """Fresh state, then enough steps that every partition shard contributes history (the delayed shards start from zeros); rank 0's
    rows are compared with a single-device direct-form handle on the same inputs (the reference's own sum order per partition,
    uniform_partitioned_convolver.hpp:55-61 with fdl_index.hpp:28-31). Outside every timed region."""
    steps = max(2, min(5, PARTS // T + 1))
    bank.reset()
    x_all = signal_rows(torch, info["in_first"], info["in_count"], steps * T * BLOCK)
    ys = []
    for s in range(steps):
        y = torch.empty((info["out_count"], T * BLOCK), device="cuda", dtype=torch.float32)
        x = x_all[:, s * T * BLOCK : (s + 1) * T * BLOCK].contiguous()
        torch.cuda.synchronize()  # the bank runs on its own streams: its device inputs must be complete when it is called
        bank([x], [y])
        ys.append(y)
    got = torch.cat(ys, dim=1)
    err = torch.zeros(1, device="cuda", dtype=torch.float64)
    if rank == 0:
        tb = 16
        ref = pkg.Convolver(pkg.UPOLS, "float32", pkg.DIAGONAL, max_blocks=tb)
        ref.set_stream(torch.cuda.current_stream())
        ir = impulse_rows(torch, info["out_first"], info["out_count"])
        ref.impulse(ir, BLOCK)
        del ir
        want = torch.empty_like(got)
        xr = x_all if info["in_first"] == info["out_first"] else signal_rows(torch, info["out_first"], info["out_count"], steps * T * BLOCK)
        torch.cuda.synchronize()
        blk = torch.empty((info["out_count"], tb * BLOCK), device="cuda", dtype=torch.float32)
        for pos in range(0, steps * T, tb):
            ref(xr[:, pos * BLOCK : (pos + tb) * BLOCK].contiguous(), out=blk)
            want[:, pos * BLOCK : (pos + tb) * BLOCK] = blk
        torch.cuda.synchronize()
        err[0] = (got.double() - want.double()).norm() / want.double().norm()
        ref.close()
    dist.broadcast(err, src=0)
    return float(err.item())


def _allreduce_max(torch, dist, v):
    t = torch.tensor([v], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item()


def sharded_c4(args, pkg, torch, dist, rank, world, local):
    """BASELINE config 4 sharded by output channel (SURVEY 8e row 3): rank r holds H[outputs of group r][all 64 inputs]; the 64 input
    rows are all-gathered (each rank brings 64/N of them), no collective on the output side."""
    B, L, O, I = 256, 1 << 16, 64, 64
    out = {"workload": "C4: 64-in x 64-out convolution matrix, B=256, 2^16-tap IRs, sharded by output channel", "layout": f"{world} output groups x 1"}
    for frame, T in ((0, 1), (64, 64)):
        bank, info = make_bank(pkg, torch, dist, rank, world, local, (world, 1), T, frame, topology=pkg.MATRIX, outputs=O, inputs=I, block=B, taps=L, seed=4100)
        xs = [torch.rand((info["in_count"], T * B), device="cuda", dtype=torch.float32) * 2 - 1 for _ in range(3)]
        ys = [torch.empty((info["out_count"], T * B), device="cuda", dtype=torch.float32) for _ in range(3)]
        steps = 30 if T == 1 else 10
        torch.cuda.synchronize()
        run_bank_timed(bank, xs, ys, 3, True)
        dist.barrier()
        ms, _ = run_bank_timed(bank, xs, ys, steps, True)
        ms = _allreduce_max(torch, dist, ms)
        entry = {"ms_per_block_step": ms / steps / T, "realtime_x_48k": (B * T / 48000.0) / (ms / steps * 1e-3)}
        # parity: rank 0's outputs against one unsharded matrix handle holding just those outputs
        bank.reset()
        nsteps = 3
        x_all = signal_rows(torch, info["in_first"], info["in_count"], nsteps * T * B, seed=4300)
        got = []
        for s in range(nsteps):
            y = torch.empty((info["out_count"], T * B), device="cuda", dtype=torch.float32)
            x = x_all[:, s * T * B : (s + 1) * T * B].contiguous()
            torch.cuda.synchronize()  # the bank's own streams do not wait for torch's
            bank([x], [y])
            got.append(y)
        got = torch.cat(got, dim=1)
        err = torch.zeros(1, device="cuda", dtype=torch.float64)
        if rank == 0:
            ref = pkg.Convolver(pkg.UPOLS, "float32", pkg.MATRIX, max_blocks=T if T <= 16 else 16)
            ref.set_stream(torch.cuda.current_stream())
            ir = impulse_rows(torch, info["out_first"] * I, info["out_count"] * I, L, 4100).view(info["out_count"], I, L)
            ref.impulse(ir, B)
            xin = signal_rows(torch, 0, I, nsteps * T * B, seed=4300)
            want = torch.empty_like(got)
            tb = T if T <= 16 else 16
            torch.cuda.synchronize()
            for pos in range(0, nsteps * T, tb):
                blk = torch.empty((info["out_count"], tb * B), device="cuda", dtype=torch.float32)
                ref(xin[:, pos * B : (pos + tb) * B].contiguous(), out=blk)
                want[:, pos * B : (pos + tb) * B] = blk
            torch.cuda.synchronize()
            err[0] = (got.double() - want.double()).norm() / want.double().norm()
            ref.close()
        dist.broadcast(err, src=0)
        entry["parity_rel_l2"] = float(err.item())
        out[f"frame{T}" if frame else f"T{T}"] = entry
        bank.close()
        del bank, xs, ys
        torch.cuda.empty_cache()
    return out


def bind_to_gpu_numa_node(local: int):
    """pin this rank's threads to the CPUs next to its GPU (NVML's ideal affinity) BEFORE any pinned host memory is allocated, so the
    staging buffers are first-touched on the GPU's own NUMA node and the ranks do not all pull through one socket"""
    try:
        import pynvml

        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        return sorted(os.sched_getaffinity(0))
    except Exception:
        return None


def run_sharded(args, pkg, torch, dist, emit, rank, world, local, peak, peak_src):
    cpus = bind_to_gpu_numa_node(local)
    frame = args.frame
    layout = parse_layout(args.layout, world)
    if frame > 0:
        frame = min(frame, PARTS // layout[1])  # a shard starts on a frame boundary of the partition axis
    T = frame if frame > 0 else args.blocks
    main = measure_layout(args, pkg, torch, dist, rank, world, local, layout, T, frame, args.steps)
    alt = c4 = sweep = f512 = None
    if not args.no_modes:
        # the same layout at 512 blocks per call (the longest frame): fewer second-level partitions per shard, the best absolute throughput
        if 0 < frame < 512 and PARTS // layout[1] >= 512:
            try:
                f512 = measure_layout(args, pkg, torch, dist, rank, world, local, layout, 512, 512, max(5, min(args.steps, 10)),
                                      want_e2e=False, want_parity=True)
            except Exception as exc:  # an extra: never let it take the line down (every rank raises or none does: same code, same sizes)
                f512 = {"error": f"{type(exc).__name__}: {exc}"}
        # the no-collective layout of the same workload (SURVEY 8e row 2), same code path with Gp = 1
        if layout[1] != 1:
            alt = measure_layout(args, pkg, torch, dist, rank, world, local, (world, 1), args.frame or args.blocks, args.frame,
                                 max(5, min(args.steps, 20)), want_e2e=True, want_parity=True)
        c4 = sharded_c4(args, pkg, torch, dist, rank, world, local)
        # BASELINE config 2 with the batch split over the ranks (SURVEY 8e row 1): no collective, aggregate = N x per-rank bytes / slowest rank
        mine = fft_sweep(pkg, torch, peak, share=world, reps=5)
        times = torch.tensor([[r["r2c_ms"], r["c2r_ms"]] for r in mine], device="cuda", dtype=torch.float64)
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        sweep = []
        for r, (t_f, t_b) in zip(mine, times.tolist()):
            bytes_all = world * r["batch"] * (4 * r["n"] + 8 * (r["n"] // 2 + 1))
            sweep.append({"n": r["n"], "batch_per_rank": r["batch"], "r2c_gbs": bytes_all / t_f / 1e6, "c2r_gbs": bytes_all / t_b / 1e6,
                          "r2c_frac_of_aggregate_hbm": bytes_all / t_f / 1e6 / (world * peak), "c2r_frac_of_aggregate_hbm": bytes_all / t_b / 1e6 / (world * peak)})
    if rank == 0:
        worst = main["parity_rel_l2"]
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {
                "workload": WORKLOAD, "blocks_per_call": T, "mode": main["mode"],
                "sharding": f"library bank (neo_b200_bank_*, one rank per process): {main['layout']}; exchange = "
                            + {"dma": "copy engines over NVLink (CUDA IPC mappings): input rows into the other shards' rings, partial spectra into "
                                      "the owner's inbox, summed inside the owner's c2r kernel; one-word ncclAllGather per step as the gate",
                               "kernel": "peer stores from inside the fused frame kernel into the owner's inbox, summed inside its c2r kernel",
                               "collective": "ncclAllGather of the input rows, ncclReduceScatter of the partial spectra"}.get(
                                   os.environ.get("NEO_B200_BANK_EXCHANGE", "dma"), "see NEO_B200_BANK_EXCHANGE")
                            + "; three steps in flight",
                "layout": {"channel_groups": layout[0], "partition_shards": layout[1]},
                "l2": "working set per rank and step (filter + delay line, several GB) exceeds the 126 MB L2; 4 rotating input buffers",
                "realtime_x_aggregate_48k": main["value"] * 1e6 / 48000.0, "realtime_x_wall_1024ch_48k": main["realtime_x_wall_1024ch_48k"],
                "host_cpus_rank0": f"{len(cpus)} CPUs next to GPU 0 (NVML affinity)" if cpus else "default affinity",
            },
            "clocks": main["clocks"], "e2e": main.get("e2e"), "gpu_launches": main["gpu_launches"], "roofline": main["roofline"],
            "parity_rel_l2": main["parity_rel_l2"], "parity_tolerance": PARITY_TOL,
            "device_bytes_per_rank": main["device_bytes_per_rank"],
        }
        if f512 is not None:
            line["modes"] = {"frame512": f512}
            if "parity_rel_l2" in f512:
                worst = max(worst, f512["parity_rel_l2"])
        if alt is not None:
            line["channel_sharded"] = alt
            worst = max(worst, alt["parity_rel_l2"])
        if c4 is not None:
            line["configs"] = {"C4_sharded": c4}
            worst = max([worst] + [v["parity_rel_l2"] for v in c4.values() if isinstance(v, dict)])
        if sweep is not None:
            line["fft_sweep_sharded"] = sweep
        emit(line)
        if not (worst <= PARITY_TOL):
            raise SystemExit(f"parity check failed: rel L2 {worst:.3e} > {PARITY_TOL:g}")


def run_ours(args):
    # stdout carries exactly ONE JSON line: native libraries (NCCL's version banner) write to fd 1 too, so fd 1 is pointed at
    # stderr for the duration of the run and the line goes to the saved descriptor
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    import torch
    import torch.distributed as dist

    import __graft_entry__ as entry

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    pkg = entry.load_package()
    if pkg.device_count() < 1:
        raise SystemExit("no CUDA device: neo_b200 has no CPU fallback")
    pkg.set_device(local)
    peak, peak_src = measured_peaks()
    if args.fft_only:  # development aid: just the BASELINE config 2 sweep
        emit({"fft_sweep": fft_sweep(pkg, torch, peak)})
        return
    if world == 1:
        run_single(args, pkg, torch, emit, peak, peak_src)
        return
    # NCCL prints its version banner on stdout at NCCL_DEBUG=VERSION/INFO; stdout carries exactly one JSON line
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    try:
        run_sharded(args, pkg, torch, dist, emit, rank, world, local, peak, peak_src)
    finally:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--blocks", type=int, default=16, help="direct form (--frame 0): blocks per call T (1 = the reference's streaming call)")
    ap.add_argument("--frame", type=int, default=256,
                    help="frame mode: blocks per call T (power of two, 2..512), second overlap-save level along block time; 0 = direct form")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layout", default="", help="N > 1: GcxGp = channel groups x partition shards (default: Gp = 2)")
    ap.add_argument("--no-fft-sweep", action="store_true")
    ap.add_argument("--fft-only", action="store_true")
    ap.add_argument("--no-modes", action="store_true", help="skip the other call shapes / layouts")
    ap.add_argument("--no-configs", action="store_true", help="skip BASELINE configs 1, 3, 4 and the unchanged-driver run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the convolver output of the last timed step to DIR/output.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.gpus != 1 or args.impl != "ours" or args.fft_only):
        ap.error("--dump-outputs writes the one-GPU convolver's output: use it with --gpus 1 and --impl ours, without --fft-only")
    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")))
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
