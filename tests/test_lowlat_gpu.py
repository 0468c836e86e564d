"""GPU: the one-block-latency convolver (LowLatencyConvolver, neo_b200_lowlat_*) against the oracle's upols convolver, the direct-form
bank, itself (call shapes, stream timing, head forms) and the reference CLI's per-channel loop through the C++ facade."""
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, TOL, rel_l2
from test_conv_gpu import make_case

pytestmark = pytest.mark.gpu


def run(conv, sig, block, pattern=(1,)):
    """feed sig[C][n] through `conv` with the given sequence of blocks per call (HOST buffers, in place)"""
    out = sig.copy()
    pos, i = 0, 0
    while pos < sig.shape[1]:
        n = min(pattern[i % len(pattern)], (sig.shape[1] - pos) // block)
        chunk = np.ascontiguousarray(out[:, pos : pos + n * block])
        conv(chunk)
        out[:, pos : pos + n * block] = chunk
        pos += n * block
        i += 1
    return out


def oracle_case(orc, channels, taps, block, nblocks, real=np.float32, seed=0):
    ir, sig = make_case(orc, channels, taps, block, nblocks, real, seed)
    H = orc.uniform_partition(ir, block)
    return ir, H, sig, orc.convolve_blocks(0, H, sig)


def worst_block(got, want, block):
    errs = []
    for b in range(want.shape[1] // block):
        w = want[:, b * block : (b + 1) * block]
        if np.linalg.norm(w) > 0:
            errs.append(rel_l2(got[:, b * block : (b + 1) * block], w))
    return max(errs)


# (name, channels, block, partitions, frame_blocks, blocks, dtype); every case runs >= 5 T_n blocks
CASES = [
    ("tiny_block", 3, 2, 9, (2,), 24, np.float32),
    ("head_only", 3, 64, 12, (8,), 20, np.float32),
    ("ragged_last_level", 2, 128, 45, (4, 16), 96, np.float32),
    ("three_levels", 2, 64, 70, (2, 4, 16), 96, np.float32),
    ("block_1024_default", 2, 1024, 200, None, 170, np.float32),
    ("largest_block_unfused", 2, 8192, 7, (2,), 12, np.float32),
    ("f64_two_levels", 2, 64, 30, (2, 8), 48, np.float64),
    ("f64_block_2048", 2, 2048, 20, (4,), 24, np.float64),
]


@pytest.mark.parametrize("name,channels,block,parts,fb,nblocks,real", CASES, ids=[c[0] for c in CASES])
def test_oracle_parity(gpu, orc, name, channels, block, parts, fb, nblocks, real):
    ir, H, sig, want = oracle_case(orc, channels, parts * block - block // 2 if block > 2 else parts * block, block, nblocks, real)
    assert H.shape[1] == parts
    conv = gpu.LowLatencyConvolver(real, frame_blocks=fb)
    conv.filter(H)
    got = run(conv, sig, block)
    key = np.dtype(real).name
    assert rel_l2(got, want) <= TOL[key]
    if real == np.float32:
        assert worst_block(got, want, block) <= 2e-5
    conv.close()


def test_against_direct_form_bank(gpu, orc):
    import torch

    C, B, P, nblocks = 64, 256, 64, 48
    ir, sig = make_case(orc, C, P * B, B, nblocks)
    direct = gpu.Convolver(gpu.UPOLS, "float32", gpu.DIAGONAL, max_blocks=1)
    direct.impulse(ir, B)
    low = gpu.LowLatencyConvolver("float32")
    low.impulse(ir, B)
    assert gpu.LowLatencyConvolver.layout(P, B)["levels"] == [(16, 64)]  # default schedule: T = 8 only
    x = torch.from_numpy(sig).cuda()
    a, b = torch.empty_like(x), torch.empty_like(x)
    s = torch.cuda.current_stream()
    direct.set_stream(s)
    low.set_stream(s)
    for t in range(nblocks):
        blk = x[:, t * B : (t + 1) * B].contiguous()
        ya, yb = torch.empty_like(blk), torch.empty_like(blk)
        direct(blk, ya)
        low(blk, yb)
        a[:, t * B : (t + 1) * B] = ya
        b[:, t * B : (t + 1) * B] = yb
    low.synchronize()
    torch.cuda.synchronize()
    assert rel_l2(b.cpu().numpy(), a.cpu().numpy()) <= 1e-5
    direct.close()
    low.close()


def test_bit_identical_call_shapes_and_runs(gpu, orc):
    ir, H, sig, want = oracle_case(orc, 3, 40 * 128, 128, 80)
    conv = gpu.LowLatencyConvolver("float32", frame_blocks=(2, 8))
    conv.filter(H)
    one = run(conv, sig, 128)
    conv.reset()
    mixed = run(conv, sig, 128, pattern=(1, 3, 2, 7, 1, 16, 5))
    conv.filter(H)
    again = run(conv, sig, 128)
    assert np.array_equal(one, mixed)
    assert np.array_equal(one, again)
    assert rel_l2(one, want) <= TOL["float32"]


def test_sync_knob_gives_the_same_bits(gpu, orc, monkeypatch):
    ir, H, sig, _ = oracle_case(orc, 4, 70 * 64, 64, 96)
    conv = gpu.LowLatencyConvolver("float32", frame_blocks=(2, 4, 16))
    conv.filter(H)
    asynchronous = run(conv, sig, 64, pattern=(1, 5, 2))
    monkeypatch.setenv("NEO_B200_LOWLAT_SYNC", "1")
    sync = gpu.LowLatencyConvolver("float32", frame_blocks=(2, 4, 16))
    sync.filter(H)
    monkeypatch.delenv("NEO_B200_LOWLAT_SYNC")
    assert np.array_equal(asynchronous, run(sync, sig, 64, pattern=(1, 5, 2)))


@pytest.mark.parametrize("real,block", [(np.float32, 256), (np.float64, 128)])
def test_unfused_head_knob(gpu, orc, monkeypatch, real, block):
    ir, H, sig, want = oracle_case(orc, 3, 33 * block, block, 40, real)
    fused = gpu.LowLatencyConvolver(real, frame_blocks=(4,))
    fused.filter(H)
    monkeypatch.setenv("NEO_B200_LOWLAT_UNFUSED", "1")
    unfused = gpu.LowLatencyConvolver(real, frame_blocks=(4,))
    unfused.filter(H)
    monkeypatch.delenv("NEO_B200_LOWLAT_UNFUSED")
    a, b = run(fused, sig, block), run(unfused, sig, block, pattern=(2, 1))
    key = np.dtype(real).name
    assert rel_l2(a, want) <= TOL[key] and rel_l2(b, want) <= TOL[key]
    assert rel_l2(a, b) <= TOL[key]


def test_memory_kinds_reset_and_impulse(gpu, orc):
    import torch

    C, B, nblocks = 4, 256, 40
    ir, H, sig, want = oracle_case(orc, C, 50 * B, B, nblocks)
    conv = gpu.LowLatencyConvolver("float32", frame_blocks=(2, 8))
    conv.filter(H)
    pageable = run(conv, sig, B, pattern=(1, 2))
    assert rel_l2(pageable, want) <= TOL["float32"]

    conv.reset()
    pinned_in = torch.from_numpy(sig).pin_memory()
    pinned_out = torch.empty_like(pinned_in).pin_memory()
    for t in range(nblocks):  # one-block calls out of place through pinned host memory
        xi = pinned_in[:, t * B : (t + 1) * B].contiguous().pin_memory()
        yo = torch.empty_like(xi).pin_memory()
        conv(xi.numpy(), yo.numpy())
        pinned_out[:, t * B : (t + 1) * B] = yo
    assert np.array_equal(pinned_out.numpy(), pageable)

    stream = torch.cuda.Stream()
    dev = gpu.LowLatencyConvolver("float32", frame_blocks=(2, 8))
    dev.set_stream(stream)
    dev.impulse(torch.from_numpy(ir).cuda(), B)
    with torch.cuda.stream(stream):
        x = torch.from_numpy(sig).cuda()
        y = torch.empty_like(x)
        for t in range(0, nblocks, 4):
            part = torch.empty((C, 4 * B), dtype=x.dtype, device=x.device)
            dev(x[:, t * B : (t + 4) * B].contiguous(), part)
            y[:, t * B : (t + 4) * B] = part
    dev.synchronize()
    stream.synchronize()
    assert rel_l2(y.cpu().numpy(), pageable) <= TOL["float32"]

    host_ir = gpu.LowLatencyConvolver("float32", frame_blocks=(2, 8))
    host_ir.impulse(ir, B)
    assert rel_l2(run(host_ir, sig, B), pageable) <= TOL["float32"]


def test_one_launch_per_block_call(gpu, orc):
    import torch

    B = 512
    ir, H, sig, _ = oracle_case(orc, 8, 40 * B, B, 8)
    conv = gpu.LowLatencyConvolver("float32", frame_blocks=(4, 16))
    conv.filter(H)
    x = torch.from_numpy(sig).cuda()
    s = torch.cuda.current_stream()
    conv.set_stream(s)
    for t in range(5):  # blocks 0..4: block 3 completes a frame of the first level
        conv(x[:, t * B : (t + 1) * B].contiguous())
    blk = x[:, 5 * B : 6 * B].contiguous()
    out = torch.empty_like(blk)
    before = gpu.kernel_launches()
    conv(blk, out)  # block 5 completes no frame
    assert gpu.kernel_launches() - before == 1
    conv.synchronize()


def test_cpp_facade_low_latency_convolver(gpu, tmp_path):
    src = os.path.join(ROOT, "tests", "cpp", "lowlat_facade_check.cpp")
    exe = str(tmp_path / "lowlat_facade_check")
    # the flags tests/cpp/Makefile builds its C++ checks with
    text = open(os.path.join(ROOT, "tests", "cpp", "Makefile")).read()
    cuda = re.search(r"^CUDA\s*\?=\s*(\S+)", text, re.M).group(1)
    flags = re.search(r"^CXXFLAGS\s*:=\s*(.*)$", text, re.M).group(1).replace("$(CUDA)", os.environ.get("CUDA", cuda)).split()
    lib = os.path.join(ROOT, "neo-dsp_b200")
    cxx = os.environ.get("CXX", "g++")
    subprocess.run([cxx, *flags, "-o", exe, src, "-L", lib, "-lneo_b200", f"-Wl,-rpath,{lib}"], check=True)
    proc = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-2000:]
    assert "lowlat facade ok" in proc.stdout
