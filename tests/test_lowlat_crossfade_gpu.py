"""GPU: switching the one-block-latency convolver to a new impulse response mid-stream (LowLatencyConvolver.stage_filter /
stage_impulse / crossfade, neo_b200_lowlat_stage_* / _crossfade). The crossfade against a float64 blend of two exact convolutions at
every head size, fade lengths and call positions, the start rule, the bit guarantees, chains and cancels, memory kinds, launch counts,
a wide bank, the C++ facade's crossfade_to and the argument errors."""
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_lowlat_reference_gpu import assert_same_bits, ref_convolve
from test_lowlat_samples_gpu import HEAD_G, assert_reference, random_case, ragged, run_samples, split_starts

pytestmark = pytest.mark.gpu

F32, F64 = "float32", "float64"
INVALID = 1  # NEO_B200_ERR_INVALID


def expected_start(pos, B, levels):
    """the first sample of a fade requested when `pos` samples have been delivered: the next sample with no levels, else the block
    b0 = max_i (floor(b / T_i) + 2) T_i, b the block holding the next sample"""
    if not levels:
        return pos
    return max((pos // B // t + 2) * t for t in levels) * B


def ref_fade(y, y_next, start, fade):
    """y before start, y + g (y_next - y) with g = (t - start) / fade inside the fade, y_next from start + fade on"""
    t = np.arange(y.shape[1])
    g = np.clip((t - start) / fade, 0.0, 1.0) if fade > 0 else (t >= start).astype(np.float64)
    return y + g * (y_next - y)


def fade_run(conv, sig, lengths, k, stage, fade):
    """process_samples (HOST, in place) with the given call lengths; before call k, stage(conv) then crossfade(fade). Returns the
    output and the start crossfade returned."""
    out, pos, start = sig.copy(), 0, None
    for i, n in enumerate(lengths):
        if i == k:
            stage(conv)
            start = conv.crossfade(fade)
        chunk = np.ascontiguousarray(out[:, pos : pos + n])
        conv.process_samples(chunk)
        out[:, pos : pos + n] = chunk
        pos += n
    return out, start


def convolver(gpu, dtype, fb, ir, B, monkeypatch=None, env=None):
    for e in env or ():
        monkeypatch.setenv(e, "1")
    conv = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    conv.impulse(ir, B)
    for e in env or ():
        monkeypatch.delenv(e)
    return conv


def levels_of(gpu, P, B, fb):
    return gpu.LowLatencyConvolver.layout(P, B, fb)["frame_blocks"]


def case(dtype, B, C, P, fb, blocks, env=None):
    return (dtype, B, C, P, fb, blocks, env)


UNFUSED = ("NEO_B200_LOWLAT_UNFUSED",)
# (dtype, block, channels, partitions, frame_blocks, blocks, environment), as the sample-granular tests: every fused head size with
# 2 G + 1 channels, the unfused sizes, the unfused knob, one to four levels and a head-only schedule
CASES = (
    [case(F32, 1 << g, 2 * G + 1, 12 if g <= 10 else 6, (2, 4) if g <= 10 else (2,), 16 if g <= 10 else 10) for g, G in HEAD_G[F32].items()]
    + [case(F64, 1 << g, 2 * G + 1, 12 if g <= 10 else 6, (2, 4) if g <= 10 else (2,), 16 if g <= 10 else 10) for g, G in HEAD_G[F64].items()]
    + [case(F32, B, 3, 12, (2, 4), 16) for B in (2, 8, 32)]
    + [case(F64, B, 3, 12, (2, 4), 16) for B in (2, 8, 32)]
    + [case(F32, 8192, 2, 6, (2,), 10), case(F64, 4096, 2, 6, (2,), 10)]
    + [case(F32, 256, 3, 12, (2, 4), 16, UNFUSED), case(F64, 128, 3, 12, (2, 4), 16, UNFUSED)]
    + [case(F32, 64, 3, 40, (2,), 56), case(F32, 64, 3, 40, (2, 4, 16), 56), case(F32, 64, 3, 40, (2, 4, 8, 16), 56)]
    + [case(F64, 64, 3, 40, (2, 4, 8, 16), 56)]
    + [case(F32, 128, 3, 12, (8,), 20), case(F64, 128, 3, 16, (8,), 20), case(F32, 8, 3, 12, (8,), 20, UNFUSED)]  # head only
)


def case_id(c):
    dtype, B, C, P, fb, blocks, env = c
    return f"{dtype}-B{B}-C{C}-P{P}-T{'x'.join(map(str, fb))}" + ("-unfused" if env else "")


@pytest.mark.parametrize("c", CASES, ids=[case_id(c) for c in CASES])
def test_crossfade_against_float64_reference(gpu, monkeypatch, c):
    # ragged calls; the crossfade is requested mid-block (after 1, B - 1, B, B + 1 samples: position 3 B + 1) and fades over 3 B + 7
    # samples, across level-frame boundaries
    dtype, B, C, P, fb, blocks, env = c
    seed = CASES.index(c)
    taps = P * B - B // 2
    ir_a, sig = random_case(C, taps, blocks * B, dtype, seed=seed)
    ir_b, _ = random_case(C, taps, B, dtype, seed=seed + 100)
    lengths = ragged(B, blocks * B, seed=seed)
    fade = 3 * B + 7
    conv = convolver(gpu, dtype, fb, ir_a, B, monkeypatch, env)
    got, start = fade_run(conv, sig, lengths, 4, lambda h: h.stage_impulse(ir_b), fade)
    conv.close()
    assert start == expected_start(sum(lengths[:4]), B, levels_of(gpu, P, B, fb))
    assert start + fade <= blocks * B
    want = ref_fade(ref_convolve(ir_a, sig), ref_convolve(ir_b, sig), start, fade)
    assert_reference(f"{case_id(c)} start {start}", got, want, B, dtype)


@pytest.mark.parametrize("fade", [0, 1, 37, 127, 5 * 128 + 3])
@pytest.mark.parametrize("where", ["boundary", "mid-block"])
def test_fade_lengths_and_call_positions(gpu, fade, where):
    dtype, B, C, P, fb, blocks = F32, 128, 3, 24, (2, 4), 40
    ir_a, sig = random_case(C, P * B - 9, blocks * B, dtype, seed=71)
    ir_b, _ = random_case(C, P * B - 9, B, dtype, seed=72)
    lengths = [5 * B] + ragged(B, blocks * B - 5 * B, seed=73) if where == "boundary" else [5 * B + 17] + ragged(B, blocks * B - 5 * B - 17, seed=73)
    conv = convolver(gpu, dtype, fb, ir_a, B)
    got, start = fade_run(conv, sig, lengths, 1, lambda h: h.stage_impulse(ir_b), fade)
    assert start == expected_start(lengths[0], B, fb) == 12 * B
    want = ref_fade(ref_convolve(ir_a, sig), ref_convolve(ir_b, sig), start, fade)
    assert_reference(f"fade {fade} at a {where}", got, want, B, dtype)
    conv.close()


@pytest.mark.parametrize(
    "P,fb", [(24, (2, 4)), (40, (2, 4, 16)), (70, (2, 4, 8, 16)), (40, None), (12, (8,))], ids=["T2x4", "T2x4x16", "T2x4x8x16", "default", "head-only"]
)
def test_start_rule(gpu, P, fb):
    # the returned start for a sweep of call positions (each behind ragged calls, then cancelled by reset)
    B, C = 64, 2
    ir, sig = random_case(C, P * B, 80 * B, F32, seed=81)
    levels = levels_of(gpu, P, B, fb)
    assert (fb == (8,)) == (not levels)
    conv = convolver(gpu, F32, fb, ir, B)
    positions = sorted(set([0, 1, B - 1, B, 2 * B, 7 * B + 5, 8 * B, 31 * B + 63, 32 * B] + [int(v) for v in np.random.default_rng(82).integers(2, 70 * B, 12)]))
    for pos in positions:
        conv.reset()
        if pos:
            run_samples(conv, np.ascontiguousarray(sig[:, :pos]), ragged(B, pos, seed=pos))
        conv.stage_impulse(ir)
        assert conv.crossfade(B) == expected_start(pos, B, levels), pos
    conv.close()
    # the examples DESIGN §4.7 gives for the default schedule
    assert gpu.LowLatencyConvolver.layout(1024, 1024)["frame_blocks"] == (8, 32, 128)
    starts = [expected_start(b * 1024, 1024, (8, 32, 128)) // 1024 - b for b in range(0, 1024)]
    assert (min(starts), max(starts)) == (129, 256)
    assert gpu.LowLatencyConvolver.layout(256, 512)["frame_blocks"] == (8, 32)
    starts = [expected_start(b * 512, 512, (8, 32)) // 512 - b for b in range(0, 256)]
    assert (min(starts), max(starts)) == (33, 64)


@pytest.mark.parametrize("env", [None, UNFUSED], ids=["fused", "unfused"])
def test_bit_guarantees(gpu, monkeypatch, env):
    dtype, B, C, fb, blocks = F32, 128, 5, (2, 4), 40
    taps = 14 * B - 3
    ir_a, sig = random_case(C, taps, blocks * B, dtype, seed=91)
    ir_b, _ = random_case(C, taps, B, dtype, seed=92)
    lengths = ragged(B, blocks * B, seed=93)
    k, fade = 5, 2 * B + 11
    plain = run_samples(convolver(gpu, dtype, fb, ir_a, B, monkeypatch, env), sig, lengths)
    other = run_samples(convolver(gpu, dtype, fb, ir_b, B, monkeypatch, env), sig, lengths)
    conv = convolver(gpu, dtype, fb, ir_a, B, monkeypatch, env)
    got, start = fade_run(conv, sig, lengths, k, lambda h: h.stage_impulse(ir_b), fade)
    end = start + fade
    assert 0 < start and end < blocks * B
    # 1. before start: the handle without a crossfade; 2. from start + fade: a handle given B, fed the same calls
    assert_same_bits("before start", got[:, :start], plain[:, :start], B)
    assert_same_bits("from the end of the fade", got[:, end:], other[:, end:], B)
    assert not np.array_equal(got[:, start:end], plain[:, start:end])
    # the same calls again after a reset (which dropped nothing: the fade ended, B is current): B's bits throughout
    conv.reset()
    assert_same_bits("after reset, B is current", run_samples(conv, sig, lengths), other, B)
    conv.close()
    # 3. NEO_B200_LOWLAT_SYNC: the same bits
    sync = convolver(gpu, dtype, fb, ir_a, B, monkeypatch, ("NEO_B200_LOWLAT_SYNC",) + (env or ()))
    assert_same_bits("NEO_B200_LOWLAT_SYNC", fade_run(sync, sig, lengths, k, lambda h: h.stage_impulse(ir_b), fade)[0], got, B)
    sync.close()
    # whole-block calls against the ragged split: the segment that completes a block is the whole-block computation, fade included
    pos = sum(lengths[:k])
    whole_lengths = [pos - pos % B] + [B] * (blocks - pos // B)
    whole = convolver(gpu, dtype, fb, ir_a, B, monkeypatch, env)
    wgot, wstart = fade_run(whole, sig, whole_lengths, 1, lambda h: h.stage_impulse(ir_b), fade)
    whole.close()
    assert wstart == start
    for b, s in split_starts(lengths, B).items():
        assert_same_bits(f"block {b} from {s}", got[:, b * B + s : (b + 1) * B], wgot[:, b * B + s : (b + 1) * B], B)


def test_chain_shorter_response_and_stage_filter(gpu, orc):
    # A -> B (stage_filter) -> C (stage_impulse, shorter: zero-padded); the spare set is reused, device bytes stay put
    dtype, B, C, P, fb, blocks = F32, 64, 3, 30, (2, 8), 120
    taps = P * B - 7
    ir_a, sig = random_case(C, taps, blocks * B, dtype, seed=101)
    ir_b, _ = random_case(C, taps, B, dtype, seed=102)
    ir_c, _ = random_case(C, (P - 9) * B + 5, B, dtype, seed=103)
    conv = convolver(gpu, dtype, fb, ir_a, B)
    out, pos, marks = sig.copy(), 0, []
    for n, action in [(3 * B + 5, None), (40 * B, ("filter", 2 * B)), (B - 3, ("impulse", 5 * B + 1)), (76 * B - 2, None)]:
        if action:
            kind, fade = action
            before = conv.device_bytes()  # (HOST calls grow the handle's staging buffers with their length: read right around the stage)
            if kind == "filter":
                conv.stage_filter(orc.uniform_partition(ir_b, B))
            else:
                conv.stage_impulse(ir_c)
            marks.append((conv.crossfade(fade), fade))
            if len(marks) == 1:
                assert conv.device_bytes() > before  # the spare set
            else:
                assert conv.device_bytes() == before  # reused
        chunk = np.ascontiguousarray(out[:, pos : pos + n])
        conv.process_samples(chunk)
        out[:, pos : pos + n] = chunk
        pos += n
    assert pos == blocks * B and marks[1][0] + marks[1][1] < pos
    y = ref_fade(ref_convolve(ir_a, sig), ref_convolve(ir_b, sig), *marks[0])
    want = ref_fade(y, ref_convolve(ir_c, sig), *marks[1])
    assert_reference("A -> B -> C", out, want, B, dtype)
    conv.close()


@pytest.mark.parametrize("when", ["delay", "fade"])
def test_reset_and_set_impulse_cancel(gpu, when):
    dtype, B, C, fb, blocks = F32, 64, 3, (2, 8), 40
    taps = 24 * B - 1
    ir_a, sig = random_case(C, taps, blocks * B, dtype, seed=111)
    ir_b, _ = random_case(C, taps, B, dtype, seed=112)
    lengths = ragged(B, 20 * B, seed=113)
    part = np.ascontiguousarray(sig[:, : 20 * B])
    fresh_a = run_samples(convolver(gpu, dtype, fb, ir_a, B), part, lengths)
    fresh_b = run_samples(convolver(gpu, dtype, fb, ir_b, B), part, lengths)
    conv = convolver(gpu, dtype, fb, ir_a, B)
    for cancel in ("reset", "set_impulse"):
        conv.reset()
        conv.process_samples(np.ascontiguousarray(sig[:, : 2 * B + 3]))
        conv.stage_impulse(ir_b)
        start = conv.crossfade(4 * B)
        assert start == 16 * B
        # into the delay (before start) or into the fade (past start, before its end)
        n = start - (2 * B + 3) - 5 if when == "delay" else start - (2 * B + 3) + 2 * B
        conv.process_samples(np.ascontiguousarray(sig[:, :n]))
        if cancel == "reset":
            conv.reset()  # keeps A: the fade had not ended
            assert_same_bits(f"reset during the {when}", run_samples(conv, part, lengths), fresh_a, B)
        else:
            gpu._check(gpu.library().neo_b200_lowlat_set_impulse(conv._h, ir_b.ctypes.data, taps, gpu.HOST))
            assert_same_bits(f"set_impulse during the {when}", run_samples(conv, part, lengths), fresh_b, B)
            gpu._check(gpu.library().neo_b200_lowlat_set_impulse(conv._h, ir_a.ctypes.data, taps, gpu.HOST))
        # nothing is staged any more
        assert gpu.library().neo_b200_lowlat_crossfade(conv._h, 0, None) == INVALID
    conv.close()


def test_memory_kinds(gpu, orc):
    import torch

    dtype, B, C, fb, blocks = F32, 256, 4, (2, 8), 48
    taps = 40 * B - 1
    ir_a, sig = random_case(C, taps, blocks * B, dtype, seed=121)
    ir_b, _ = random_case(C, taps, B, dtype, seed=122)
    H = orc.uniform_partition(ir_b, B)
    lengths = ragged(B, blocks * B, seed=123)
    pinned = torch.from_numpy(ir_b).pin_memory()
    ir_dev, H_dev = torch.from_numpy(ir_b).cuda(), torch.from_numpy(H).cuda()
    torch.cuda.synchronize()  # the handles below run on streams of their own
    results = {}
    for name, stage in [
        ("impulse pageable", lambda h: h.stage_impulse(ir_b)),
        ("impulse pinned", lambda h: h.stage_impulse(pinned.numpy())),
        ("impulse device", lambda h: h.stage_impulse(ir_dev)),
        ("filter pageable", lambda h: h.stage_filter(H)),
        ("filter device", lambda h: h.stage_filter(H_dev)),
    ]:
        conv = convolver(gpu, dtype, fb, ir_a, B)
        results[name], start = fade_run(conv, sig, lengths, 6, stage, 3 * B)
        conv.close()
    want = ref_fade(ref_convolve(ir_a, sig), ref_convolve(ir_b, sig), start, 3 * B)
    assert_reference("staged from HOST pageable", results["impulse pageable"], want, B, dtype)
    for name, got in results.items():
        assert_same_bits(name, got, results["impulse pageable"] if "impulse" in name else results["filter pageable"], B)

    # DEVICE processing on a torch stream, staged from a device tensor mid-stream
    stream = torch.cuda.Stream()
    dev = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    dev.set_stream(stream)
    with torch.cuda.stream(stream):
        dev.impulse(torch.from_numpy(ir_a).cuda(), B)
        x = torch.from_numpy(sig).cuda()
        y = torch.empty_like(x)
        pos = 0
        for i, n in enumerate(lengths):
            if i == 6:
                dev.stage_impulse(ir_dev)
                assert dev.crossfade(3 * B) == start
            seg = x[:, pos : pos + n].contiguous()
            dev.process_samples(seg)
            y[:, pos : pos + n] = seg
            pos += n
    dev.synchronize()
    stream.synchronize()
    assert_same_bits("DEVICE on a torch stream", y.cpu().numpy(), results["impulse pageable"], B)
    dev.close()


def test_launch_counts(gpu):
    import torch

    # fused head: one launch per call inside a block outside the fade window, two inside it; staging adds none to processing
    dtype, B, C, fb = F32, 512, 8, (4, 16)
    ir_a, sig = random_case(C, 40 * B, 64 * B, dtype, seed=131)
    ir_b, _ = random_case(C, 40 * B, B, dtype, seed=132)
    conv = gpu.LowLatencyConvolver(dtype, frame_blocks=fb)
    s = torch.cuda.current_stream()
    conv.set_stream(s)
    conv.impulse(ir_a, B)
    x = torch.from_numpy(sig).cuda()

    def call(pos, n):
        seg = x[:, pos : pos + n].contiguous()
        out = torch.empty_like(seg)
        before = gpu.kernel_launches()
        conv.process_samples(seg, out)
        return gpu.kernel_launches() - before

    conv(x[:, : 5 * B].contiguous())
    conv.stage_impulse(ir_b)
    start = conv.crossfade(2 * B + 100)
    assert start == 32 * B
    assert [call(5 * B + p, n) for p, n in ((0, 1), (1, 63), (64, B - 100))] == [1, 1, 1]  # staged, before start
    conv.process_samples(x[:, 6 * B - 36 : 32 * B].contiguous())
    assert [call(32 * B + p, n) for p, n in ((0, 1), (1, 63), (64, B - 100))] == [2, 2, 2]  # inside the fade
    conv.process_samples(x[:, 33 * B - 36 : 34 * B].contiguous())
    # the fade ends at 34 B + 100: a call that straddles the end still runs both sides, the next ones run B alone
    assert [call(34 * B + p, n) for p, n in ((0, 99), (99, 2), (101, 1), (102, 63))] == [2, 2, 1, 1]
    conv.synchronize()
    conv.close()


def test_wide_bank(gpu):
    import torch

    # 1024 channels, B = 1024, P = 80: the default schedule, levels T = 8 and T = 32
    C, B, P, blocks = 1024, 1024, 80, 100
    taps = P * B
    g = torch.Generator(device="cuda")
    g.manual_seed(141)
    ir_a = torch.rand((C, taps), generator=g, device="cuda") * 2 - 1
    ir_a /= torch.linalg.vector_norm(ir_a, dim=1, dtype=torch.float64).max().float()
    ir_b = torch.rand((C, taps - 3 * B - 1), generator=g, device="cuda") * 2 - 1
    ir_b /= torch.linalg.vector_norm(ir_b, dim=1, dtype=torch.float64).max().float()
    x = torch.rand((C, blocks * B), generator=g, device="cuda") * 2 - 1
    y = torch.empty_like(x)
    s = torch.cuda.current_stream()
    conv = gpu.LowLatencyConvolver(F32)
    conv.set_stream(s)
    conv.impulse(ir_a, B)
    pos, start, fade = 0, None, 5 * B + 300
    for i, n in enumerate(ragged(B, blocks * B, seed=142)):
        if i == 8:
            conv.stage_impulse(ir_b)
            start = conv.crossfade(fade)
            assert start == expected_start(pos, B, (8, 32))
        seg = x[:, pos : pos + n].contiguous()
        conv.process_samples(seg)
        y[:, pos : pos + n] = seg
        pos += n
    conv.synchronize()
    assert start + fade < blocks * B
    rows = sorted(set([0, 1, C - 1] + [int(v) for v in np.random.default_rng(143).integers(2, C - 1, size=5)]))
    idx = torch.tensor(rows, device="cuda")
    xs = x[idx].cpu().numpy()
    want = ref_fade(ref_convolve(ir_a[idx].cpu().numpy(), xs), ref_convolve(ir_b[idx].cpu().numpy(), xs), start, fade)
    assert_reference(f"wide bank, channels {rows}", y[idx].cpu().numpy(), want, B, F32)
    conv.close()


def test_cpp_facade_crossfade_to(gpu, tmp_path):
    src = os.path.join(ROOT, "tests", "cpp", "lowlat_crossfade_check.cpp")
    exe = str(tmp_path / "lowlat_crossfade_check")
    # the flags tests/cpp/Makefile builds its C++ checks with
    text = open(os.path.join(ROOT, "tests", "cpp", "Makefile")).read()
    cuda = re.search(r"^CUDA\s*\?=\s*(\S+)", text, re.M).group(1)
    flags = re.search(r"^CXXFLAGS\s*:=\s*(.*)$", text, re.M).group(1).replace("$(CUDA)", os.environ.get("CUDA", cuda)).split()
    lib = os.path.join(ROOT, "neo-dsp_b200")
    cxx = os.environ.get("CXX", "g++")
    subprocess.run([cxx, *flags, "-o", exe, src, "-L", lib, "-lneo_b200", f"-Wl,-rpath,{lib}"], check=True)
    proc = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-2000:]
    assert "lowlat crossfade ok" in proc.stdout


def test_argument_errors(gpu):
    lib = gpu.library()
    B, C, P = 64, 2, 24
    ir = np.ones((C, P * B), dtype=np.float32)
    H = np.zeros((C, P, B + 1), dtype=np.complex64)
    x = np.zeros((C, 5), dtype=np.float32)
    start = gpu._sz(0)

    def refused(status, text):
        assert status == INVALID
        assert text in lib.neo_b200_last_error().decode()

    conv = gpu.LowLatencyConvolver(F32, frame_blocks=(2, 4))
    conv._create(C, B, P)  # a handle with no filter
    refused(lib.neo_b200_lowlat_stage_impulse(conv._h, ir.ctypes.data, P * B, gpu.HOST), "no filter")
    refused(lib.neo_b200_lowlat_stage_filter(conv._h, H.ctypes.data, gpu.HOST), "no filter")
    gpu._check(lib.neo_b200_lowlat_set_impulse(conv._h, ir.ctypes.data, P * B, gpu.HOST))
    refused(lib.neo_b200_lowlat_crossfade(conv._h, 10, gpu.C.byref(start)), "nothing staged")
    refused(lib.neo_b200_lowlat_stage_impulse(conv._h, ir.ctypes.data, B - 1, gpu.HOST), "shorter than one block")
    long_ir = np.ones((C, (P + 1) * B), dtype=np.float32)
    refused(lib.neo_b200_lowlat_stage_impulse(conv._h, long_ir.ctypes.data, (P + 1) * B, gpu.HOST), "partitions")
    refused(lib.neo_b200_lowlat_stage_impulse(conv._h, None, P * B, gpu.HOST), "null")
    refused(lib.neo_b200_lowlat_stage_filter(None, H.ctypes.data, gpu.HOST), "null")
    refused(lib.neo_b200_lowlat_crossfade(None, 0, None), "null")
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
    conv.stage_impulse(ir)
    conv.stage_impulse(ir)  # staging again before a crossfade replaces the staged set
    assert conv.crossfade(100) == 8 * B
    refused(lib.neo_b200_lowlat_crossfade(conv._h, 10, gpu.C.byref(start)), "already pending or running")
    refused(lib.neo_b200_lowlat_stage_impulse(conv._h, ir.ctypes.data, P * B, gpu.HOST), "pending or running")  # pending
    conv.process_samples(np.zeros((C, 8 * B + 3), dtype=np.float32))
    refused(lib.neo_b200_lowlat_stage_filter(conv._h, H.ctypes.data, gpu.HOST), "pending or running")  # running
    conv.process_samples(x)  # the handle still works after the refusals
    assert np.array_equal(x, np.zeros_like(x))
    conv.close()
    with pytest.raises(RuntimeError):
        gpu.LowLatencyConvolver(F32).stage_impulse(ir)
