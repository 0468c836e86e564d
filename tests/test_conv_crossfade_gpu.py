"""GPU: switching the convolver bank to a new impulse response mid-stream (Convolver.stage_filter / stage_impulse / crossfade,
neo_b200_conv_stage_* / _crossfade). The crossfade against a float64 blend of two exact convolutions in the direct form (every MAC
kernel) and frame mode, both topologies and dtypes, the wide c2r; fade lengths and start positions; the bit guarantees, with HOST channel
groups and a misaligned DEVICE output; launch counts; chains and cancels; the C++ facade's crossfade_to and every error."""
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, TOL, rel_l2
from test_lowlat_crossfade_gpu import ref_fade
from test_lowlat_reference_gpu import assert_same_bits, random_case, ref_convolve

pytestmark = pytest.mark.gpu

F32, F64 = "float32", "float64"
INVALID, UNSUPPORTED = 1, 2  # NEO_B200_ERR_INVALID, NEO_B200_ERR_UNSUPPORTED


def matrix_case(outputs, inputs, taps, n, dtype, seed):
    rng = np.random.default_rng(seed)
    ir = rng.uniform(-1, 1, size=(outputs, inputs, taps)).astype(dtype)
    ir /= np.sqrt((ir.astype(np.float64) ** 2).sum(axis=(1, 2)).max())
    return ir, rng.uniform(-1, 1, size=(inputs, n)).astype(dtype)


def ref_bank(ir, sig):
    """ref_convolve per channel (diagonal ir [C][L]) or summed over inputs (matrix ir [O][I][L])"""
    if ir.ndim == 2:
        return ref_convolve(ir, sig)
    return np.stack([sum(ref_convolve(ir[o, i][None], sig[i][None])[0] for i in range(ir.shape[1])) for o in range(ir.shape[0])])


def bank(gpu, dtype, topology, ir, B, T, frame):
    conv = gpu.Convolver(gpu.UPOLS, dtype, topology, max_blocks=T, frame_blocks=T if frame else 0)
    conv.impulse(ir, B)
    return conv


def run_calls(conv, sig, call, actions=None, outputs=None):
    """HOST calls of `call` samples; actions[i](conv) runs before call i. Returns the output and what the actions returned."""
    outputs = outputs or sig.shape[0]
    out = np.empty((outputs, sig.shape[1]), dtype=sig.dtype)
    got = {}
    for i, pos in enumerate(range(0, sig.shape[1], call)):
        if actions and i in actions:
            got[i] = actions[i](conv)
        x = np.ascontiguousarray(sig[:, pos : pos + call])
        y = np.empty((outputs, call), dtype=sig.dtype)
        conv(x, y)
        out[:, pos : pos + call] = y
    return out, got


def assert_reference(name, got, want, call, dtype):
    total = rel_l2(got, want)
    worst = max(rel_l2(got[:, s : s + call], want[:, s : s + call]) for s in range(0, want.shape[1], call))
    print(f"[conv-crossfade] {name}: overall {total:.2e}, worst call {worst:.2e}")
    assert total <= TOL[dtype], f"{name}: relative L2 {total:.2e}"
    assert worst <= 2 * TOL[dtype], f"{name}: worst call relative L2 {worst:.2e}"


def case(dtype, topology, B, T, frame, P, calls):
    return (dtype, topology, B, T, frame, P, calls)


D, M = "diag", "matrix"
# (dtype, topology, block, blocks per call, frame mode, partitions, calls). Direct form: T = 1 (stream kernel), 4 (Toeplitz), 16
# (Toeplitz below B = 128, TMA from it), 32 (TMA); frame mode: T = 16, 64, 256, fused for diagonal banks, three kernels for matrix banks;
# B = 1024 float takes the wide c2r
CASES = [
    case(F32, D, 64, 1, False, 10, 40),
    case(F32, D, 64, 4, False, 10, 12),
    case(F32, D, 64, 16, False, 20, 5),
    case(F32, D, 256, 16, False, 20, 5),
    case(F32, D, 128, 32, False, 40, 4),
    case(F32, M, 64, 1, False, 6, 30),
    case(F32, M, 32, 4, False, 9, 10),
    case(F64, D, 32, 1, False, 7, 30),
    case(F64, D, 64, 4, False, 10, 12),
    case(F64, M, 32, 4, False, 9, 10),
    case(F32, D, 1024, 1, False, 6, 12),
    case(F32, D, 1024, 16, False, 20, 4),
    case(F32, D, 64, 16, True, 40, 6),
    case(F32, D, 32, 64, True, 150, 4),
    case(F32, D, 32, 256, True, 520, 3),
    case(F32, M, 64, 16, True, 40, 6),
    case(F64, D, 64, 16, True, 40, 6),
    case(F64, M, 32, 64, True, 150, 4),
    case(F32, D, 1024, 16, True, 40, 4),
]


def case_id(c):
    dtype, top, B, T, frame, P, calls = c
    return f"{dtype}-{top}-B{B}-T{T}-{'frame' if frame else 'direct'}-P{P}"


def make(gpu, c, seed):
    """(conv, ir_a, ir_b, sig, outputs); ir_b is a few partitions shorter than ir_a"""
    dtype, top, B, T, frame, P, calls = c
    taps = P * B - B // 2
    if top == D:
        C = 3
        ir_a, sig = random_case(C, taps, calls * T * B, dtype, seed=seed)
        ir_b, _ = random_case(C, taps - 2 * B - 3, B, dtype, seed=seed + 100)
        return bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, frame), ir_a, ir_b, sig, C
    O, I = 4, 3
    ir_a, sig = matrix_case(O, I, taps, calls * T * B, dtype, seed=seed)
    ir_b, _ = matrix_case(O, I, taps - 2 * B - 3, B, dtype, seed=seed + 100)
    return bank(gpu, dtype, gpu.MATRIX, ir_a, B, T, frame), ir_a, ir_b, sig, O


@pytest.mark.parametrize("c", CASES, ids=[case_id(c) for c in CASES])
def test_crossfade_against_float64_reference(gpu, c):
    # the fade is requested before call 1 and starts half a call and 5 samples later (inside a call, inside a block), lasting a call and
    # 7 samples: it covers calls partly, wholly and not at all
    dtype, top, B, T, frame, P, calls = c
    conv, ir_a, ir_b, sig, outputs = make(gpu, c, seed=CASES.index(c))
    call = T * B
    delay = call // 2 + 5
    fade = call + 7
    out, got = run_calls(conv, sig, call, {1: lambda h: (h.stage_impulse(ir_b), h.crossfade(fade, delay))[1]}, outputs)
    conv.close()
    start = got[1]
    assert start == call + delay and start + fade < sig.shape[1]
    want = ref_fade(ref_bank(ir_a, sig), ref_bank(ir_b, sig), start, fade)
    assert_reference(case_id(c), out, want, call, dtype)


@pytest.mark.parametrize("frame", [False, True], ids=["direct", "frame"])
@pytest.mark.parametrize("fade", [0, 1, 37, 3 * 256 + 5], ids=["hard", "one", "short", "calls"])
@pytest.mark.parametrize("where", ["boundary", "in-call", "in-block", "ahead"])
def test_fade_lengths_and_start_positions(gpu, frame, fade, where):
    # calls of 4 blocks of 64: start on a call boundary, inside a call on a block boundary, inside a block, and several calls ahead
    dtype, B, T, C, P, calls = F32, 64, 4, 3, 16, 16
    call = T * B
    ir_a, sig = random_case(C, P * B - 9, calls * call, dtype, seed=71)
    ir_b, _ = random_case(C, P * B - 9, B, dtype, seed=72)
    delay = {"boundary": 0, "in-call": 2 * B, "in-block": B + 17, "ahead": 3 * call + 2 * B + 9}[where]
    conv = bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, frame)
    out, got = run_calls(conv, sig, call, {2: lambda h: (h.stage_impulse(ir_b), h.crossfade(fade, delay))[1]})
    conv.close()
    assert got[2] == 2 * call + delay
    want = ref_fade(ref_convolve(ir_a, sig), ref_convolve(ir_b, sig), got[2], fade)
    assert_reference(f"fade {fade} at {where}", out, want, call, dtype)


def guarantee_run(gpu, dtype, B, T, frame, ir_a, ir_b, sig, k, delay, fade):
    """(out, start) of HOST calls with the crossfade requested before call k"""
    conv = bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, frame)
    out, got = run_calls(conv, sig, T * B, {k: lambda h: (h.stage_impulse(ir_b), h.crossfade(fade, delay))[1]})
    conv.close()
    return out, got[k]


@pytest.mark.parametrize("frame", [False, True], ids=["direct", "frame"])
def test_bit_guarantees(gpu, frame):
    dtype, B, T, C, calls = F32, 128, 4, 5, 12
    call = T * B
    taps = (32 if frame else 14) * B - 3
    ir_a, sig = random_case(C, taps, calls * call, dtype, seed=91)
    ir_b, _ = random_case(C, taps, B, dtype, seed=92)
    plain, _ = run_calls(bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, frame), sig, call)
    other, _ = run_calls(bank(gpu, dtype, gpu.DIAGONAL, ir_b, B, T, frame), sig, call)
    got, start = guarantee_run(gpu, dtype, B, T, frame, ir_a, ir_b, sig, 3, call + B + 37, 2 * call + 11)
    end = start + 2 * call + 11
    assert 0 < start and end < calls * call
    # 1. before start: the handle without a crossfade; 2. from start + fade: a handle given B, fed the same calls
    assert_same_bits("before start", got[:, :start], plain[:, :start], B)
    assert_same_bits("from the end of the fade", got[:, end:], other[:, end:], B)
    assert not np.array_equal(got[:, start:end], plain[:, start:end])


@pytest.mark.parametrize("frame", [False, True], ids=["direct", "frame"])
def test_host_channel_groups_pinned_pageable_and_device(gpu, frame):
    import torch

    # 512 channels, 4 blocks per call: the HOST call is cut into channel groups; pinned, pageable and DEVICE (aligned, and offset by two
    # floats, which rules out the wide c2r's 16-byte rows) give the same bits
    dtype, B, T, C, calls = F32, 1024, 4, 512, 6
    call = T * B
    taps = 12 * B - 5
    ir_a, sig = random_case(C, taps, calls * call, dtype, seed=101)
    ir_b, _ = random_case(C, taps - B, B, dtype, seed=102)
    k, delay, fade = 2, B + 300, call + B + 3
    pageable, start = guarantee_run(gpu, dtype, B, T, frame, ir_a, ir_b, sig, k, delay, fade)

    conv = bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, frame)
    pin = torch.empty((C, call), dtype=torch.float32).pin_memory().numpy()
    pout = torch.empty((C, call), dtype=torch.float32).pin_memory().numpy()
    pinned = np.empty_like(sig)
    for i in range(calls):
        if i == k:
            conv.stage_impulse(ir_b)
            assert conv.crossfade(fade, delay) == start
        pin[:] = sig[:, i * call : (i + 1) * call]
        conv(pin, pout)
        pinned[:, i * call : (i + 1) * call] = pout
    conv.close()
    assert_same_bits("HOST pinned", pinned, pageable, B)

    s = torch.cuda.current_stream()
    x = torch.from_numpy(sig).cuda()
    for offset in (0, 2):
        conv = bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, frame)
        conv.set_stream(s)
        xin = torch.empty((C, call), dtype=torch.float32, device="cuda")
        raw = torch.empty(C * call + offset, dtype=torch.float32, device="cuda")
        yout = raw[offset:].view(C, call)
        dev = np.empty_like(sig)
        for i in range(calls):
            if i == k:
                conv.stage_impulse(ir_b)
                assert conv.crossfade(fade, delay) == start
            xin.copy_(x[:, i * call : (i + 1) * call])
            conv(xin, yout)
            dev[:, i * call : (i + 1) * call] = yout.cpu().numpy()
        conv.close()
        if offset == 0:
            assert_same_bits("DEVICE", dev, pageable, B)
        else:
            # the cta_fft c2r on both sides: guarantees 1 and 2 against handles running the same kernel
            plain = bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, frame)
            other = bank(gpu, dtype, gpu.DIAGONAL, ir_b, B, T, frame)
            ya, yb = np.empty_like(sig), np.empty_like(sig)
            for h, y in ((plain, ya), (other, yb)):
                h.set_stream(s)
                for i in range(calls):
                    xin.copy_(x[:, i * call : (i + 1) * call])
                    h(xin, yout)
                    y[:, i * call : (i + 1) * call] = yout.cpu().numpy()
                h.close()
            assert_same_bits("offset DEVICE before start", dev[:, :start], ya[:, :start], B)
            assert_same_bits("offset DEVICE after the fade", dev[:, start + fade :], yb[:, start + fade :], B)
            want = ref_fade(ref_convolve(ir_a[:3], sig[:3]), ref_convolve(ir_b[:3], sig[:3]), start, fade)
            assert_reference("offset DEVICE", dev[:3], want, call, dtype)


def test_launch_counts(gpu):
    import torch

    # a staged but not started fade, and calls after the switch, launch what the plain handle launches; a call inside the fade adds
    # one MAC and one c2r
    dtype, B, T, C = F32, 256, 4, 8
    call = T * B
    ir_a, sig = random_case(C, 20 * B, 12 * call, dtype, seed=131)
    ir_b, _ = random_case(C, 20 * B, B, dtype, seed=132)
    s = torch.cuda.current_stream()
    x = torch.from_numpy(sig).cuda()
    y = torch.empty((C, call), dtype=torch.float32, device="cuda")

    def counts(conv, first, n):
        res = []
        for i in range(first, first + n):
            before = gpu.kernel_launches()
            conv(x[:, i * call : (i + 1) * call].contiguous(), y)
            res.append(gpu.kernel_launches() - before)
        return res

    plain = bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, False)
    plain.set_stream(s)
    base = counts(plain, 0, 1)[0]
    plain.close()
    conv = bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, False)
    conv.set_stream(s)
    assert counts(conv, 0, 2) == [base, base]
    conv.stage_impulse(ir_b)
    assert counts(conv, 2, 1) == [base]  # staged only
    assert conv.crossfade(call + 10, 2 * call + B) == 5 * call + B
    assert counts(conv, 3, 2) == [base, base]  # before start
    inside = counts(conv, 5, 2)
    assert inside == [base + 2, base + 2]  # [5 call + B, 6 call + B + 10): one more MAC and c2r each
    assert counts(conv, 7, 3) == [base] * 3  # after the switch
    conv.synchronize()
    conv.close()


def test_chain_shorter_response_and_stage_filter(gpu, orc):
    # A -> B (stage_filter) -> C (stage_impulse, shorter: zero-padded), in frame mode; the spare set is reused, device bytes stay put
    dtype, B, T, C, P, calls = F32, 64, 8, 3, 30, 14
    call = T * B
    taps = P * B - 7
    ir_a, sig = random_case(C, taps, calls * call, dtype, seed=141)
    ir_b, _ = random_case(C, taps, B, dtype, seed=142)
    ir_c, _ = random_case(C, (P - 9) * B + 5, B, dtype, seed=143)
    conv = bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, True)
    sizes = []

    def step(stage, fade, delay):
        def go(h):
            before = h.device_bytes()
            stage(h)
            sizes.append((before, h.device_bytes()))
            return h.crossfade(fade, delay), fade
        return go

    out, marks = run_calls(conv, sig, call, {2: step(lambda h: h.stage_filter(orc.uniform_partition(ir_b, B)), 2 * B, 5),
                                             6: step(lambda h: h.stage_impulse(ir_c), call + 3, call + 1)})
    conv.close()
    assert sizes[0][1] > sizes[0][0] and sizes[1][1] == sizes[1][0] == sizes[0][1]
    y = ref_fade(ref_convolve(ir_a, sig), ref_convolve(ir_b, sig), *marks[2])
    want = ref_fade(y, ref_convolve(ir_c, sig), *marks[6])
    assert_reference("A -> B -> C", out, want, call, dtype)


@pytest.mark.parametrize("when", ["delay", "fade"])
def test_reset_set_filter_and_set_impulse_cancel(gpu, orc, when):
    dtype, B, T, C, calls = F32, 64, 4, 3, 6
    call = T * B
    taps = 10 * B - 1
    ir_a, sig = random_case(C, taps, calls * call, dtype, seed=151)
    ir_b, _ = random_case(C, taps, B, dtype, seed=152)
    fresh_a, _ = run_calls(bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, False), sig, call)
    fresh_b, _ = run_calls(bank(gpu, dtype, gpu.DIAGONAL, ir_b, B, T, False), sig, call)
    H_b = orc.uniform_partition(ir_b, B)
    filtered = gpu.Convolver(gpu.UPOLS, dtype, gpu.DIAGONAL, max_blocks=T)
    filtered.filter(H_b)  # H_b from the host partitioner: its own bits, unlike impulse(ir_b)
    fresh_h, _ = run_calls(filtered, sig, call)
    filtered.close()
    conv = bank(gpu, dtype, gpu.DIAGONAL, ir_a, B, T, False)
    lib = gpu.library()
    for cancel in ("reset", "set_filter", "set_impulse"):
        conv.reset()
        conv(np.ascontiguousarray(sig[:, :call]), np.empty((C, call), dtype=dtype))
        conv.stage_impulse(ir_b)
        assert conv.crossfade(2 * call, call + 5) == 2 * call + 5
        # into the delay (before start) or into the fade (past start, before its end)
        for _ in range(1 if when == "delay" else 2):
            conv(np.ascontiguousarray(sig[:, :call]), np.empty((C, call), dtype=dtype))
        if cancel == "reset":
            conv.reset()  # keeps A: the fade had not ended
            assert_same_bits(f"reset during the {when}", run_calls(conv, sig, call)[0], fresh_a, B)
        elif cancel == "set_filter":
            gpu._check(lib.neo_b200_conv_set_filter(conv._h, H_b.ctypes.data, gpu.HOST))
            assert_same_bits(f"set_filter during the {when}", run_calls(conv, sig, call)[0], fresh_h, B)
            gpu._check(lib.neo_b200_conv_set_impulse(conv._h, ir_a.ctypes.data, taps, gpu.HOST))
        else:
            gpu._check(lib.neo_b200_conv_set_impulse(conv._h, ir_b.ctypes.data, taps, gpu.HOST))
            assert_same_bits(f"set_impulse during the {when}", run_calls(conv, sig, call)[0], fresh_b, B)
            gpu._check(lib.neo_b200_conv_set_impulse(conv._h, ir_a.ctypes.data, taps, gpu.HOST))
        # nothing is staged any more
        assert lib.neo_b200_conv_crossfade(conv._h, 0, 0, None) == INVALID
    # reset after the fade ended keeps B
    conv.stage_impulse(ir_b)
    conv.crossfade(0)
    conv.reset()
    assert_same_bits("reset after the switch", run_calls(conv, sig, call)[0], fresh_b, B)
    conv.close()


def test_cpp_facade_crossfade_to(gpu, tmp_path):
    src = os.path.join(ROOT, "tests", "cpp", "conv_crossfade_check.cpp")
    exe = str(tmp_path / "conv_crossfade_check")
    # the flags tests/cpp/Makefile builds its C++ checks with
    text = open(os.path.join(ROOT, "tests", "cpp", "Makefile")).read()
    cuda = re.search(r"^CUDA\s*\?=\s*(\S+)", text, re.M).group(1)
    flags = re.search(r"^CXXFLAGS\s*:=\s*(.*)$", text, re.M).group(1).replace("$(CUDA)", os.environ.get("CUDA", cuda)).split()
    lib = os.path.join(ROOT, "neo-dsp_b200")
    cxx = os.environ.get("CXX", "g++")
    subprocess.run([cxx, *flags, "-o", exe, src, "-L", lib, "-lneo_b200", f"-Wl,-rpath,{lib}"], check=True)
    proc = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-2000:]
    assert "conv crossfade ok" in proc.stdout


def test_argument_errors(gpu, orc):
    import torch

    lib = gpu.library()
    B, C, P, T = 64, 2, 8, 4
    ir = np.ones((C, P * B), dtype=np.float32)
    H = np.zeros((C, P, B + 1), dtype=np.complex64)
    x = np.zeros((C, T * B), dtype=np.float32)
    start = gpu._sz(0)

    def refused(status, code, text):
        assert status == code, (status, text)
        assert text in lib.neo_b200_last_error().decode()

    conv = gpu.Convolver(gpu.UPOLS, F32, gpu.DIAGONAL, max_blocks=T)
    conv._create(C, C, B, P)  # a handle with no filter
    refused(lib.neo_b200_conv_stage_impulse(conv._h, ir.ctypes.data, P * B, gpu.HOST), INVALID, "no filter")
    refused(lib.neo_b200_conv_stage_filter(conv._h, H.ctypes.data, gpu.HOST), INVALID, "no filter")
    gpu._check(lib.neo_b200_conv_set_impulse(conv._h, ir.ctypes.data, P * B, gpu.HOST))
    refused(lib.neo_b200_conv_crossfade(conv._h, 0, 10, gpu.C.byref(start)), INVALID, "nothing staged")
    refused(lib.neo_b200_conv_stage_impulse(conv._h, ir.ctypes.data, B - 1, gpu.HOST), INVALID, "shorter than one block")
    long_ir = np.ones((C, (P + 1) * B), dtype=np.float32)
    refused(lib.neo_b200_conv_stage_impulse(conv._h, long_ir.ctypes.data, (P + 1) * B, gpu.HOST), INVALID, "partitions")
    refused(lib.neo_b200_conv_stage_impulse(conv._h, None, P * B, gpu.HOST), INVALID, "null")
    refused(lib.neo_b200_conv_stage_filter(None, H.ctypes.data, gpu.HOST), INVALID, "null")
    refused(lib.neo_b200_conv_crossfade(None, 0, 0, None), INVALID, "null")
    with pytest.raises(ValueError):
        conv.stage_impulse(long_ir)
    with pytest.raises(ValueError):
        conv.stage_impulse(ir.astype(np.float64))
    with pytest.raises(ValueError):
        conv.stage_impulse(ir[:1].copy())
    with pytest.raises(ValueError):
        conv.stage_filter(H[:, :-1].copy())
    with pytest.raises(ValueError):
        conv.stage_filter(H.astype(np.complex128))
    with pytest.raises(ValueError):
        conv.crossfade(-1)
    with pytest.raises(ValueError):
        conv.crossfade(10, -1)
    conv.stage_impulse(ir)
    conv.stage_impulse(ir)  # staging again before a crossfade replaces the staged set
    assert conv.crossfade(400, 3 * T * B) == 3 * T * B  # [768, 1168)
    refused(lib.neo_b200_conv_crossfade(conv._h, 0, 10, gpu.C.byref(start)), INVALID, "pending or running")
    refused(lib.neo_b200_conv_stage_impulse(conv._h, ir.ctypes.data, P * B, gpu.HOST), INVALID, "pending or running")  # pending
    # the split and windowed forms have no whole output to blend
    xd = torch.zeros((C, T * B), dtype=torch.float32, device="cuda")
    refused(lib.neo_b200_conv_forward(conv._h, xd.data_ptr(), T, gpu.DEVICE), INVALID, "crossfade")
    refused(lib.neo_b200_conv_forward_range(conv._h, xd.data_ptr(), T, 0, C, 1), INVALID, "crossfade")
    refused(lib.neo_b200_conv_inverse(conv._h, xd.data_ptr(), xd.data_ptr(), 0, C, 1, gpu.DEVICE), INVALID, "crossfade")
    refused(lib.neo_b200_conv_process_window(conv._h, xd.data_ptr(), xd.data_ptr(), 0, gpu.DEVICE), INVALID, "crossfade")
    for _ in range(4):  # to 1024
        conv(x.copy(), np.empty_like(x))
    refused(lib.neo_b200_conv_stage_filter(conv._h, H.ctypes.data, gpu.HOST), INVALID, "pending or running")  # running
    y = np.empty_like(x)
    conv(x, y)  # the handle still works after the refusals, and the fade has ended
    assert np.array_equal(y, np.zeros_like(y))
    gpu._check(lib.neo_b200_conv_forward(conv._h, x.ctypes.data, T, gpu.HOST))
    conv.close()
    with pytest.raises(RuntimeError):
        gpu.Convolver(gpu.UPOLS, F32).stage_impulse(ir)

    # overlap-add, sparse filters and partition-sharded handles: UNSUPPORTED
    ola = gpu.Convolver(gpu.UPOLA, F32, gpu.DIAGONAL)
    ola.impulse(ir, B)
    refused(lib.neo_b200_conv_stage_impulse(ola._h, ir.ctypes.data, P * B, gpu.HOST), UNSUPPORTED, "overlap-add")
    refused(lib.neo_b200_conv_crossfade(ola._h, 0, 0, None), UNSUPPORTED, "overlap-add")
    ola.close()
    Hs = orc.uniform_partition(ir, B)
    sparse = gpu.Convolver(gpu.UPOLS, F32, gpu.DIAGONAL)
    sparse.filter_sparse(Hs, np.abs(Hs) > 0)
    refused(lib.neo_b200_conv_stage_filter(sparse._h, Hs.ctypes.data, gpu.HOST), UNSUPPORTED, "set_filter_csr")
    sparse.close()
    shard = gpu.Convolver(gpu.UPOLS, F32, gpu.DIAGONAL, partition_range=(0, P // 2))
    shard.filter(Hs)
    refused(lib.neo_b200_conv_stage_filter(shard._h, Hs.ctypes.data, gpu.HOST), UNSUPPORTED, "partition-sharded")
    shard.close()
