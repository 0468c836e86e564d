"""GPU: sample-granular calls of the one-block-latency convolver (LowLatencyConvolver.process_samples,
neo_b200_lowlat_process_samples). Calls of any length against an exact float64 convolution at every head size, the bit-level
guarantees at block boundaries, zero added latency, mixing with whole-block calls, reset and set_filter mid-block, memory kinds and
odd row offsets, one launch per call inside a block, a wide bank, the C++ facade's process() and the argument errors."""
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_lowlat_gpu import run
from test_lowlat_reference_gpu import BOUND, DELAY_ATOL, assert_same_bits, block_errors, ref_convolve

pytestmark = pytest.mark.gpu

F32, F64 = "float32", "float64"
HEAD_G = {F32: {6: 8, 7: 4, 8: 4, 9: 2, 10: 1, 11: 1, 12: 1}, F64: {6: 8, 7: 4, 8: 2, 9: 1, 10: 1, 11: 1}}


def ragged(B, total, seed):
    """call lengths summing to `total`: 1, B - 1, B, B + 1 and odd lengths first, then seeded draws from [1, 3 B]"""
    rng = np.random.default_rng(seed)
    lens = [1, B - 1, B, B + 1, 2 * B + 1, 3] + [int(v) for v in rng.integers(1, 3 * B + 1, size=4 * total // B + 8)]
    out, left = [], total
    for n in lens:
        if left == 0:
            break
        out.append(min(n, left))
        left -= out[-1]
    if left:
        out.append(left)
    return out


def run_samples(conv, sig, lengths):
    """feed sig[C][n] through process_samples with the given call lengths (HOST buffers, in place)"""
    out = sig.copy()
    pos = 0
    for n in lengths:
        chunk = np.ascontiguousarray(out[:, pos : pos + n])
        conv.process_samples(chunk)
        out[:, pos : pos + n] = chunk
        pos += n
    assert pos == sig.shape[1]
    return out


def random_case(channels, taps, n, dtype, seed):
    rng = np.random.default_rng(seed)
    ir = rng.uniform(-1, 1, size=(channels, taps)).astype(dtype)
    ir /= np.sqrt((ir.astype(np.float64) ** 2).sum(axis=1).max())
    return ir, rng.uniform(-1, 1, size=(channels, n)).astype(dtype)


def convolver(gpu, dtype, fb, ir, B, monkeypatch=None, env=None):
    if env:
        monkeypatch.setenv(env, "1")
    conv = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    conv.impulse(ir, B)
    if env:
        monkeypatch.delenv(env)
    return conv


def assert_reference(name, got, want, B, dtype):
    total = float(np.linalg.norm(got.astype(np.float64) - want) / np.linalg.norm(want))
    pad = ((0, 0), (0, -want.shape[1] % B))  # a stream that ends inside a block: its last block is zero-padded on both sides
    err = block_errors(np.pad(np.asarray(got, dtype=np.float64), pad), np.pad(want, pad), B)
    c, b = np.unravel_index(np.argmax(err), err.shape)
    print(f"[lowlat-samples] {name}: overall {total:.2e}, worst (channel {c}, block {b}) {err[c, b]:.2e}")
    assert total <= BOUND[dtype][0], f"{name}: overall relative L2 {total:.2e}"
    assert err[c, b] <= BOUND[dtype][1], f"{name}: worst (channel {c}, block {b}) relative L2 {err[c, b]:.2e}"


def case(dtype, B, C, P, fb, blocks, env=None):
    return (dtype, B, C, P, fb, blocks, env)


# (dtype, block, channels, partitions, frame_blocks, blocks, environment). Fused head sizes run 2 G + 1 channels (a ragged last CTA).
# Measured maxima over every case on one B200 (1000 W), against BOUND: float 3.3e-7 overall / 5.6e-7 worst (channel, block) (the
# latter at B = 2), double 7.7e-16 / 1.7e-15 -- the same order as whole-block calls.
CASES = (
    [case(F32, 1 << g, 2 * G + 1, 12 if g <= 10 else 6, (2, 4) if g <= 10 else (2,), 16 if g <= 10 else 10) for g, G in HEAD_G[F32].items()]
    + [case(F64, 1 << g, 2 * G + 1, 12 if g <= 10 else 6, (2, 4) if g <= 10 else (2,), 16 if g <= 10 else 10) for g, G in HEAD_G[F64].items()]
    + [case(F32, B, 3, 12, (2, 4), 16) for B in (2, 8, 32)]
    + [case(F64, B, 3, 12, (2, 4), 16) for B in (2, 8, 32)]
    + [case(F32, 8192, 2, 6, (2,), 10), case(F64, 4096, 2, 6, (2,), 10)]
    + [case(F32, 256, 3, 12, (2, 4), 16, "NEO_B200_LOWLAT_UNFUSED"), case(F64, 128, 3, 12, (2, 4), 16, "NEO_B200_LOWLAT_UNFUSED")]
    + [case(F32, 64, 3, 40, (2, 4, 16), 56), case(F32, 64, 3, 40, (2, 4, 8, 16), 56), case(F64, 64, 3, 40, (2, 4, 8, 16), 56)]
    + [case(F32, 128, 3, 12, (8,), 20), case(F64, 128, 3, 16, (8,), 20)]  # P <= 2 T_1: head only
)


def case_id(c):
    dtype, B, C, P, fb, blocks, env = c
    return f"{dtype}-B{B}-C{C}-P{P}-T{'x'.join(map(str, fb))}" + ("-unfused" if env else "")


@pytest.mark.parametrize("c", CASES, ids=[case_id(c) for c in CASES])
def test_ragged_calls_against_float64_reference(gpu, monkeypatch, c):
    dtype, B, C, P, fb, blocks, env = c
    taps = P * B - B // 2
    ir, sig = random_case(C, taps, blocks * B, dtype, seed=CASES.index(c))
    lengths = ragged(B, blocks * B, seed=CASES.index(c))
    conv = convolver(gpu, dtype, fb, ir, B, monkeypatch, env)
    got = run_samples(conv, sig, lengths)
    conv.close()
    assert_reference(case_id(c), got, ref_convolve(ir, sig), B, dtype)


def split_starts(lengths, B):
    """for each block, the position inside it where the call segment that completes it starts"""
    starts, pos = {}, 0
    for n in lengths:
        begin, end = pos, pos + n
        for b in range(begin // B, (end - 1) // B + 1):
            if (b + 1) * B <= end:
                starts[b] = max(begin - b * B, 0)
        pos = end
    return starts


@pytest.mark.parametrize("env", [None, "NEO_B200_LOWLAT_UNFUSED"], ids=["fused", "unfused"])
def test_bit_guarantees(gpu, monkeypatch, env):
    dtype, B, C, fb, blocks = F32, 128, 5, (2, 4), 40
    taps = 14 * B - 3
    ir, sig = random_case(C, taps, blocks * B, dtype, seed=11)
    conv = convolver(gpu, dtype, fb, ir, B, monkeypatch, env)
    whole = run(conv, sig, B)

    # 1. whole-block calls through process_samples give the bits of process
    conv.reset()
    assert_same_bits("whole blocks through process_samples", run_samples(conv, sig, [B, 3 * B] * (blocks // 4)), whole, B)

    # 2. the segment that completes a block gives the whole-block bits from its start to the block's end
    lengths = ragged(B, blocks * B, seed=12)
    conv.reset()
    split = run_samples(conv, sig, lengths)
    starts = split_starts(lengths, B)
    assert len(starts) == blocks and any(s > 0 for s in starts.values())
    for b, s in starts.items():
        assert_same_bits(f"block {b} from {s}", split[:, b * B + s : (b + 1) * B], whole[:, b * B + s : (b + 1) * B], B)

    # 3. after a split sequence that returns to a block boundary, everything is the whole-block bits
    k = 23 * B
    head = ragged(B, k, seed=13)
    conv.reset()
    first = run_samples(conv, sig[:, :k], head)
    rest = run(conv, np.ascontiguousarray(sig[:, k:]), B, pattern=(1, 3))
    assert_same_bits("after a boundary", rest, whole[:, k:], B)
    starts = split_starts(head, B)
    for b, s in starts.items():
        assert_same_bits(f"prefix block {b}", first[:, b * B + s : (b + 1) * B], whole[:, b * B + s : (b + 1) * B], B)

    # the same ragged sequence twice with a reset between, and with NEO_B200_LOWLAT_SYNC, gives the same bits
    conv.reset()
    assert_same_bits("ragged again after reset", run_samples(conv, sig, lengths), split, B)
    conv.close()
    monkeypatch.setenv("NEO_B200_LOWLAT_SYNC", "1")
    sync = convolver(gpu, dtype, fb, ir, B, monkeypatch, env)
    monkeypatch.delenv("NEO_B200_LOWLAT_SYNC")
    assert_same_bits("ragged under NEO_B200_LOWLAT_SYNC", run_samples(sync, sig, lengths), split, B)
    sync.close()


@pytest.mark.parametrize("dtype", [F32, F64])
def test_zero_added_latency(gpu, dtype):
    # a unit impulse at a random sample, one sample per call: ir[c][0] comes back in the call that delivers the impulse, the rest of
    # the impulse response in the calls that follow (across every level hand-off: taps > 2 T_n B)
    B, C, fb = 64, 2, (2, 4)
    taps = 12 * B - 5
    rng = np.random.default_rng(21)
    ir = rng.uniform(-1, 1, size=(C, taps)).astype(dtype)
    t0 = int(rng.integers(B + 1, 3 * B))
    n = t0 + taps + 3
    conv = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    conv.impulse(ir, B)
    got = np.empty((C, n), dtype=dtype)
    for t in range(n):
        x = np.zeros((C, 1), dtype=dtype)
        if t == t0:
            x[:] = 1
        conv.process_samples(x)
        got[:, t] = x[:, 0]
        if t == t0:
            assert np.abs(x[:, 0].astype(np.float64) - ir[:, 0]).max() <= DELAY_ATOL[dtype], (x[:, 0], ir[:, 0])
    conv.close()
    want = np.zeros((C, n))
    want[:, t0 : t0 + taps] = ir
    err = float(np.abs(got - want).max())
    print(f"[lowlat-samples] unit impulse at {t0}, one-sample calls, {dtype}: max |error| {err:.2e}")
    assert err <= DELAY_ATOL[dtype]


def test_mixing_with_whole_blocks_reset_and_set_filter(gpu, orc):
    dtype, B, C, fb, blocks = F32, 64, 3, (2, 8), 60
    taps = 30 * B - 7
    ir, sig = random_case(C, taps, blocks * B, dtype, seed=31)
    ir2, _ = random_case(C, taps, B, dtype, seed=32)
    want = ref_convolve(ir, sig)
    conv = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    conv.impulse(ir, B)
    out = sig.copy()
    pos = 0
    for n, whole in [(B + 5, False), (4 * B, True), (7, False), (B, True), (3 * B + 1, False), (16 * B, True)]:
        chunk = np.ascontiguousarray(out[:, pos : pos + n])
        if whole:
            conv(chunk)  # whole blocks, starting in the middle of a block
        else:
            conv.process_samples(chunk)
        out[:, pos : pos + n] = chunk
        pos += n
    rest = np.ascontiguousarray(out[:, pos:])
    conv.process_samples(rest)
    out[:, pos:] = rest
    assert_reference("whole-block calls on a handle mid-block", out, want, B, dtype)

    # reset, set_filter and set_impulse on a handle left mid-block: the output of a fresh handle
    lengths = ragged(B, 20 * B, seed=33)
    part = np.ascontiguousarray(sig[:, : 20 * B])
    fresh = run_samples(convolver(gpu, dtype, fb, ir, B), part, lengths)
    conv.process_samples(np.ascontiguousarray(sig[:, : B // 2 + 3]))
    conv.reset()
    assert_same_bits("reset mid-block", run_samples(conv, part, lengths), fresh, B)
    H2 = orc.uniform_partition(ir2, B)
    other = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    other.filter(H2)
    fresh2 = run_samples(other, part, lengths)
    conv.process_samples(np.ascontiguousarray(sig[:, : 2 * B + 9]))
    gpu._check(gpu.library().neo_b200_lowlat_set_filter(conv._h, H2.ctypes.data, gpu.HOST))
    assert_same_bits("set_filter mid-block", run_samples(conv, part, lengths), fresh2, B)
    conv.process_samples(np.ascontiguousarray(sig[:, :5]))
    gpu._check(gpu.library().neo_b200_lowlat_set_impulse(conv._h, ir.ctypes.data, taps, gpu.HOST))
    assert_same_bits("set_impulse mid-block", run_samples(conv, part, lengths), fresh, B)


def test_memory_kinds_and_odd_offsets(gpu):
    import torch

    dtype, B, C, fb = F32, 256, 4, (2, 8)
    taps = 40 * B - 1
    total = 30 * B + 17
    ir, sig = random_case(C, taps, total, dtype, seed=41)
    lengths = ragged(B, total, seed=42)
    assert any(n % 2 for n in lengths)
    conv = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    conv.impulse(ir, B)
    pageable = run_samples(conv, sig, lengths)
    assert_reference("HOST pageable, in place", pageable, ref_convolve(ir, sig), B, dtype)

    conv.reset()  # pinned, out of place
    pinned = np.empty_like(sig)
    pos = 0
    for n in lengths:
        xi = torch.from_numpy(np.ascontiguousarray(sig[:, pos : pos + n])).pin_memory()
        yo = torch.empty_like(xi).pin_memory()
        conv.process_samples(xi.numpy(), yo.numpy())
        pinned[:, pos : pos + n] = yo.numpy()
        pos += n
    assert_same_bits("HOST pinned, out of place", pinned, pageable, B)
    conv.close()

    # DEVICE on a torch stream: rows of odd length start at odd element offsets; every other call also starts the whole buffer at an
    # odd element offset. In place and out of place alternate.
    stream = torch.cuda.Stream()
    dev = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    dev.set_stream(stream)
    with torch.cuda.stream(stream):
        dev.impulse(torch.from_numpy(ir).cuda(), B)
        x = torch.from_numpy(sig).cuda()
        y = torch.empty_like(x)
        pos = 0
        for i, n in enumerate(lengths):
            buf = torch.empty(C * n + 1, dtype=x.dtype, device=x.device)
            xi = buf[i % 2 : i % 2 + C * n].view(C, n)
            xi.copy_(x[:, pos : pos + n])
            if i % 3 == 0:
                dev.process_samples(xi)
                y[:, pos : pos + n] = xi
            else:
                yo = torch.empty((C, n), dtype=x.dtype, device=x.device)
                dev.process_samples(xi, yo)
                y[:, pos : pos + n] = yo
            pos += n
    dev.synchronize()
    stream.synchronize()
    assert_same_bits("DEVICE, odd offsets", y.cpu().numpy(), pageable, B)
    dev.close()


def test_one_launch_per_call_inside_a_block(gpu):
    import torch

    dtype, B, C, fb = F32, 512, 8, (4, 16)
    ir, sig = random_case(C, 40 * B, 8 * B, dtype, seed=51)
    conv = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    s = torch.cuda.current_stream()
    conv.set_stream(s)
    conv.impulse(ir, B)
    x = torch.from_numpy(sig).cuda()
    conv(x[:, : 5 * B].contiguous())  # blocks 0..4; block 3 completed a frame of the first level
    pos = 5 * B
    for n in (1, 1, 2, 63, B - 100, 30):  # all inside block 5
        seg = x[:, pos : pos + n].contiguous()
        out = torch.empty_like(seg)
        before = gpu.kernel_launches()
        conv.process_samples(seg, out)
        assert gpu.kernel_launches() - before == 1, n
        pos += n
    conv.synchronize()


def test_wide_bank(gpu):
    import torch

    # 1024 channels, B = 1024, P = 80: the default schedule gives levels T = 8 over [16, 64) and T = 32 over [64, 80)
    C, B, P, blocks = 1024, 1024, 80, 100
    taps = P * B
    assert gpu.LowLatencyConvolver.layout(P, B)["levels"] == [(16, 64), (64, 80)]
    g = torch.Generator(device="cuda")
    g.manual_seed(61)
    ir = torch.rand((C, taps), generator=g, device="cuda") * 2 - 1
    ir /= torch.linalg.vector_norm(ir, dim=1, dtype=torch.float64).max().float()
    x = torch.rand((C, blocks * B), generator=g, device="cuda") * 2 - 1
    y = torch.empty_like(x)
    s = torch.cuda.current_stream()
    conv = gpu.LowLatencyConvolver(F32)
    conv.set_stream(s)
    conv.impulse(ir, B)
    pos = 0
    for n in ragged(B, blocks * B, seed=62):
        seg = x[:, pos : pos + n].contiguous()
        conv.process_samples(seg)
        y[:, pos : pos + n] = seg
        pos += n
    conv.synchronize()
    rows = sorted(set([0, 1, C - 1] + [int(v) for v in np.random.default_rng(63).integers(2, C - 1, size=5)]))
    idx = torch.tensor(rows, device="cuda")
    want = ref_convolve(ir[idx].cpu().numpy(), x[idx].cpu().numpy())
    assert_reference(f"wide bank, channels {rows}", y[idx].cpu().numpy(), want, B, F32)
    conv.close()


def test_cpp_facade_process(gpu, tmp_path):
    src = os.path.join(ROOT, "tests", "cpp", "lowlat_samples_check.cpp")
    exe = str(tmp_path / "lowlat_samples_check")
    # the flags tests/cpp/Makefile builds its C++ checks with
    text = open(os.path.join(ROOT, "tests", "cpp", "Makefile")).read()
    cuda = re.search(r"^CUDA\s*\?=\s*(\S+)", text, re.M).group(1)
    flags = re.search(r"^CXXFLAGS\s*:=\s*(.*)$", text, re.M).group(1).replace("$(CUDA)", os.environ.get("CUDA", cuda)).split()
    lib = os.path.join(ROOT, "neo-dsp_b200")
    cxx = os.environ.get("CXX", "g++")
    subprocess.run([cxx, *flags, "-o", exe, src, "-L", lib, "-lneo_b200", f"-Wl,-rpath,{lib}"], check=True)
    proc = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-2000:]
    assert "lowlat samples ok" in proc.stdout


def test_argument_errors(gpu):
    lib = gpu.library()
    B, C = 64, 2
    ir = np.ones((C, 4 * B), dtype=np.float32)
    x = np.zeros((C, 5), dtype=np.float32)
    conv = gpu.LowLatencyConvolver(F32)
    conv._create(C, B, 4)  # a handle with no filter
    assert lib.neo_b200_lowlat_process_samples(conv._h, x.ctypes.data, x.ctypes.data, 5, gpu.HOST) == 1
    assert "no filter" in lib.neo_b200_last_error().decode()
    gpu._check(lib.neo_b200_lowlat_set_impulse(conv._h, ir.ctypes.data, 4 * B, gpu.HOST))
    assert lib.neo_b200_lowlat_process_samples(conv._h, x.ctypes.data, x.ctypes.data, 0, gpu.HOST) == 1
    assert "samples" in lib.neo_b200_last_error().decode()
    assert lib.neo_b200_lowlat_process_samples(conv._h, None, x.ctypes.data, 5, gpu.HOST) == 1
    assert "null buffer" in lib.neo_b200_last_error().decode()
    assert lib.neo_b200_lowlat_process_samples(None, x.ctypes.data, x.ctypes.data, 5, gpu.HOST) == 1
    assert "null" in lib.neo_b200_last_error().decode()
    with pytest.raises(ValueError):
        conv.process_samples(np.zeros((C, 0), dtype=np.float32))
    conv.process_samples(x)  # the handle still works after the refusals
    assert np.array_equal(x, np.zeros_like(x))
    conv.close()
    with pytest.raises(RuntimeError):
        gpu.LowLatencyConvolver(F32).process_samples(x)
