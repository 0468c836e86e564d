"""The one-block-latency convolver (LowLatencyConvolver, neo_b200_lowlat_*) against an exact float64 convolution: every fused head
size with a ragged last CTA, every unfused block size, every level frame size, four levels, the partition counts around the
schedule, delayed unit impulses across every hand-off, the C5 geometry and a 1024-channel bank whose level frames run alongside
many head blocks. The reference and the case table are checked without a device."""
import numpy as np
import pytest

from conftest import TOL, rel_l2
from test_lowlat_gpu import run

F32, F64 = "float32", "float64"

# channels per CTA of lowlat_head_kernel<T, LOGM> (fft_cfg<T, LOGM>::G), for LOGM = log2(B)
HEAD_G = {F32: {6: 8, 7: 4, 8: 4, 9: 2, 10: 1, 11: 1, 12: 1}, F64: {6: 8, 7: 4, 8: 2, 9: 1, 10: 1, 11: 1}}
UNFUSED = {F32: (2, 4, 8, 16, 32, 8192), F64: (2, 4, 8, 16, 32, 4096)}

# (relative L2 over the whole output, relative L2 of the worst (channel, block)) against ref_convolve. Measured maxima over every
# case below on one B200 (1000 W): float 3.9e-7 / 1.9e-6 (the latter at B = 2), double 8.1e-16 / 6.3e-15
BOUND = {F32: (2e-6, 1e-5), F64: (1e-14, 5e-14)}
# largest |error| of a delayed unit impulse (input uniform in [-1, 1]); measured maxima float 9.5e-7, double 1.2e-15
DELAY_ATOL = {F32: 5e-6, F64: 1e-14}


def ref_convolve(ir, sig):
    """y[c][n] = sum_k ir[c][k] sig[c][n - k] for n < len(sig): the exact causal linear convolution, truncated to the signal
    length, in float64 from the upcast inputs (rfft / irfft at a power of two >= n + L - 1, one channel at a time)."""
    ir, sig = np.asarray(ir, dtype=np.float64), np.asarray(sig, dtype=np.float64)
    n, taps = sig.shape[1], ir.shape[1]
    m = 1 << (n + taps - 2).bit_length()
    out = np.empty(sig.shape, dtype=np.float64)
    for c in range(sig.shape[0]):
        out[c] = np.fft.irfft(np.fft.rfft(sig[c], m) * np.fft.rfft(ir[c], m), m)[:n]
    return out


def random_case(channels, taps, n, dtype, seed):
    """uniform(-1, 1) impulse responses scaled to at most unit energy, and uniform(-1, 1) input"""
    rng = np.random.default_rng(seed)
    ir = rng.uniform(-1, 1, size=(channels, taps)).astype(dtype)
    ir /= np.sqrt((ir.astype(np.float64) ** 2).sum(axis=1).max())
    return ir, rng.uniform(-1, 1, size=(channels, n)).astype(dtype)


def block_errors(got, want, block):
    """[C][blocks] relative L2 error of each (channel, block). A block whose reference norm is below a quarter of its channel's
    RMS block norm is measured against that quarter instead, so a (near) zero reference block is held to an absolute bound."""
    C = want.shape[0]
    g = np.asarray(got, dtype=np.float64).reshape(C, -1, block)
    w = np.asarray(want, dtype=np.float64).reshape(C, -1, block)
    den = np.linalg.norm(w, axis=2)
    floor = 0.25 * np.sqrt(np.mean(den**2, axis=1, keepdims=True))
    return np.linalg.norm(g - w, axis=2) / np.maximum(den, np.maximum(floor, np.finfo(np.float64).tiny))


def assert_close(name, got, want, block, overall, per_block):
    total = rel_l2(got, want)
    err = block_errors(got, want, block)
    c, b = np.unravel_index(np.argmax(err), err.shape)
    where = f"{name}: worst (channel {c}, block {b}) relative L2 {err[c, b]:.2e}"
    print(f"[lowlat-ref] {name}: overall {total:.2e}, {where.split(': ', 1)[1]}")
    assert total <= overall, f"{where}; over all channels {total:.2e} > {overall:.0e}"
    assert err[c, b] <= per_block, f"{where} > {per_block:.0e}"


def assert_same_bits(name, got, want, block):
    """bit-identical outputs; a failure names the first differing (channel, block)"""
    got, want = np.asarray(got), np.asarray(want)
    if not np.array_equal(got, want):
        c, s = np.argwhere(got != want)[0]
        raise AssertionError(f"{name}: first difference at channel {c}, block {s // block} (sample {s})")


def case(dtype, B, C, P, frame_blocks, blocks, via="impulse", cut=None):
    """(dtype, block, channels, taps, frame_blocks, blocks, via): taps = P B - cut, by default half a block short of P partitions"""
    return (dtype, B, C, P * B - (B // 2 if cut is None else cut), frame_blocks, blocks, via)


# Fused head sizes run 2 G + 1 channels (three CTAs, the last with one live channel); every level frame size 2..512 appears per
# dtype; None is the library's default schedule. `via`: impulse(ir, B) or filter(orc.uniform_partition(ir, B)).
GEOMETRY = [
    case(F32, 64, 17, 70, (2, 4, 16), 64),
    case(F32, 128, 9, 1100, None, 1600),  # default -> (8, 32, 128, 512)
    case(F32, 256, 9, 300, (4, 64), 200, "filter"),
    case(F32, 512, 5, 520, (16, 128), 400),
    case(F32, 1024, 3, 600, (8, 256), 800),
    case(F32, 2048, 3, 40, (2, 8), 32, "filter"),
    case(F32, 4096, 3, 20, (2, 4), 20),
    case(F32, 2, 3, 1100, None, 1600),
    case(F32, 4, 3, 70, (2, 32), 100, "filter"),
    case(F32, 8, 3, 150, (8, 64), 200),
    case(F32, 16, 3, 40, (2, 4, 8, 16), 52),
    case(F32, 32, 3, 9, (4,), 16),  # P = 2 T_1 + 1: a one-partition level
    case(F32, 8192, 3, 9, (2,), 8),
    case(F64, 64, 17, 90, (2, 8, 32), 112),
    case(F64, 128, 9, 40, (4, 16), 64, "filter"),
    case(F64, 256, 5, 1030, (8, 512), 1600),
    case(F64, 512, 3, 40, (2, 4, 8, 16), 64),
    case(F64, 1024, 3, 200, (16, 64), 216),
    case(F64, 2048, 3, 7, (2,), 12),
    case(F64, 2, 3, 1100, None, 1600),  # default -> (8, 32, 128, 512)
    case(F64, 4, 3, 17, (8,), 32, "filter"),  # P = 2 T_1 + 1
    case(F64, 8, 3, 600, (16, 256), 800),
    case(F64, 16, 3, 40, (2, 4, 8, 16), 52),
    case(F64, 32, 3, 10, (4,), 16),
    case(F64, 4096, 3, 5, (2,), 8),
]

# partition counts at the edges of the schedule
EDGES = [
    case(F32, 64, 17, 1, (8,), 12, cut=0),  # P = 1: taps = B
    case(F64, 1024, 3, 12, (8,), 16),  # P < 2 T_1: head only
    case(F32, 1024, 3, 16, (8,), 16, cut=0),  # P = 2 T_1: the level is dropped
    case(F64, 64, 17, 16, None, 24, cut=0),  # P = 2 T_1 of the default schedule
    case(F32, 1024, 3, 17, None, 32),  # P = 2 T_1 + 1 of the default schedule
    case(F32, 64, 17, 32, (2, 4, 16), 16, cut=0),  # P = 2 T_n: the last level is dropped
    case(F64, 1024, 3, 32, (2, 4, 16), 16, "filter"),
]

CASES = GEOMETRY + EDGES


def case_id(c):
    dtype, B, C, taps, fb, blocks, via = c
    sched = "-".join(map(str, fb)) if fb else "default"
    return f"{'f32' if dtype == F32 else 'f64'}_B{B}_C{C}_P{num_parts(taps, B)}_L{taps}_T{sched}{'_H' if via == 'filter' else ''}"


def fused(dtype, B):
    return int(B).bit_length() - 1 in HEAD_G[dtype]


def num_parts(taps, B):
    return -(-taps // B)


def test_ref_convolve_is_the_exact_linear_convolution(orc):
    # thought of as B = 64: L < B, L not a multiple of B, L > n, and the one-tap and one-sample edges
    for seed, (C, taps, n) in enumerate([(2, 5, 256), (3, 100, 192), (1, 333, 97), (2, 1000, 200), (2, 1, 17), (1, 64, 64), (2, 37, 1)]):
        ir, sig = random_case(C, taps, n, np.float64, seed)
        got = ref_convolve(ir, sig)
        assert got.shape == sig.shape
        for c in range(C):
            want = np.convolve(ir[c], sig[c])[:n]
            assert np.linalg.norm(got[c] - want) <= 1e-13 * np.linalg.norm(want), (C, taps, n, c)
            direct = orc.direct_convolve(sig[c], ir[c], n)
            assert np.linalg.norm(got[c] - direct) <= 1e-13 * np.linalg.norm(direct), (C, taps, n, c)
    # float32 inputs are upcast, not convolved in float32
    ir, sig = random_case(2, 300, 500, np.float32, 9)
    want = np.stack([np.convolve(ir[c].astype(np.float64), sig[c].astype(np.float64))[:500] for c in range(2)])
    assert np.linalg.norm(ref_convolve(ir, sig) - want) <= 1e-13 * np.linalg.norm(want)


def test_block_errors_name_the_channel_and_block():
    want = np.ones((3, 4 * 8))
    want[1, 16:24] = 0  # a zero reference block is held to an absolute bound
    got = want.copy()
    got[2, 9] += 1e-3
    err = block_errors(got, want, 8)
    assert np.unravel_index(np.argmax(err), err.shape) == (2, 1)
    assert err[1, 2] == 0 and np.isfinite(err).all()
    with pytest.raises(AssertionError, match=r"case-x: worst \(channel 2, block 1\)"):
        assert_close("case-x", got, want, 8, 1e-3, 1e-5)
    with pytest.raises(AssertionError, match="channel 2, block 1 "):
        assert_same_bits("case-y", got, want, 8)


def test_case_table_covers_the_schedule(pkg):
    # the coverage the GPU cases below are meant to have, checked against the library's own schedule
    levels = {F32: set(), F64: set()}
    seen = {F32: {}, F64: {}}
    edges = set()
    for c in CASES:
        dtype, B, C, taps, fb, blocks, via = c
        P = num_parts(taps, B)
        lay = pkg.LowLatencyConvolver.layout(P, B, fb, dtype)
        live = lay["frame_blocks"]
        levels[dtype].update(live)
        seen[dtype].setdefault(B, []).append(C)
        t1 = fb[0] if fb else 8
        # every level delivers at least two frames into both plane slots
        assert blocks >= (3 * live[-1] + live[0] if live else 4), case_id(c)
        if fused(dtype, B):
            assert C == max(2 * HEAD_G[dtype][B.bit_length() - 1] + 1, 3), case_id(c)
        last = lay["levels"][-1] if live else None
        for label, holds in [
            (("4 levels", dtype), len(live) == 4),
            (("default 4 levels", dtype), fb is None and P > 1024 and live == (8, 32, 128, 512)),
            ("P = 1", P == 1),
            ("head only", P < 2 * t1),
            ("P = 2 T_1", P == 2 * t1),
            ("P = 2 T_1 + 1", P == 2 * t1 + 1 and lay["levels"] == [(2 * t1, 2 * t1 + 1)]),
            ("ragged last level", bool(live) and (last[1] - last[0]) % live[-1] != 0),
            ("P = 2 T_n", bool(fb) and 0 < len(live) < len(fb) and P == 2 * fb[len(live)]),
            ("taps % B", taps % B != 0),
        ]:
            if holds:
                edges.add(label)
    for dtype in (F32, F64):
        assert levels[dtype] >= {2 << i for i in range(9)}, (dtype, sorted(levels[dtype]))
        assert set(seen[dtype]) >= set(1 << g for g in HEAD_G[dtype]) | set(UNFUSED[dtype]), (dtype, sorted(seen[dtype]))
        assert ("4 levels", dtype) in edges and ("default 4 levels", dtype) in edges, dtype
        assert BOUND[dtype][0] <= TOL[dtype]
    assert edges >= {"P = 1", "head only", "P = 2 T_1", "P = 2 T_1 + 1", "ragged last level", "P = 2 T_n", "taps % B"}, edges


def make_convolver(gpu, orc, dtype, frame_blocks, ir, B, via):
    conv = gpu.LowLatencyConvolver(dtype, frame_blocks=frame_blocks)
    if via == "filter":
        conv.filter(orc.uniform_partition(ir, B))
    else:
        conv.impulse(ir, B)
    return conv


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[case_id(c) for c in CASES])
def test_against_float64_reference(gpu, orc, monkeypatch, case):
    dtype, B, C, taps, fb, blocks, via = case
    name = case_id(case)
    ir, sig = random_case(C, taps, blocks * B, dtype, seed=CASES.index(case))
    want = ref_convolve(ir, sig)
    live = gpu.LowLatencyConvolver.layout(num_parts(taps, B), B, fb, dtype)["frame_blocks"]

    # (a) one block per call against the reference, per (channel, block)
    conv = make_convolver(gpu, orc, dtype, fb, ir, B, via)
    one = run(conv, sig, B)
    assert_close(name, one, want, B, *BOUND[dtype])
    # (b) a ragged call pattern, including a call of a whole last-level frame, gives the same bits
    conv.reset()
    assert_same_bits(f"{name} ragged calls", run(conv, sig, B, pattern=(1, 3, 2, live[-1] if live else 4, 1, 7)), one, B)
    conv.close()
    # (c) all level work on the head's stream gives the same bits
    monkeypatch.setenv("NEO_B200_LOWLAT_SYNC", "1")
    sync = make_convolver(gpu, orc, dtype, fb, ir, B, via)
    monkeypatch.delenv("NEO_B200_LOWLAT_SYNC")
    assert_same_bits(f"{name} NEO_B200_LOWLAT_SYNC", run(sync, sig, B), one, B)
    sync.close()
    # (d) the unfused head meets the same bound
    if fused(dtype, B):
        monkeypatch.setenv("NEO_B200_LOWLAT_UNFUSED", "1")
        unfused = make_convolver(gpu, orc, dtype, fb, ir, B, via)
        monkeypatch.delenv("NEO_B200_LOWLAT_UNFUSED")
        assert_close(f"{name} unfused", run(unfused, sig, B, pattern=(2, 1)), want, B, *BOUND[dtype])
        unfused.close()


def handoff_delays(B, frame_blocks, taps):
    """0, 1, B - 1, B, B + 1, then 2 T_i B - 1, 2 T_i B, 2 T_i B + 1 for every level (head -> level, level -> level), and L - 1"""
    return [0, 1, B - 1, B, B + 1] + [2 * t * B + k for t in frame_blocks for k in (-1, 0, 1)] + [taps - 1]


def delayed_impulse_run(gpu, dtype, B, taps, frame_blocks, delays, blocks, seed):
    ird = np.zeros((len(delays), taps), dtype=dtype)
    for c, d in enumerate(delays):
        ird[c, d] = 1
    sig = np.random.default_rng(seed).uniform(-1, 1, size=(len(delays), blocks * B)).astype(dtype)
    conv = gpu.LowLatencyConvolver(dtype, frame_blocks=frame_blocks)
    conv.impulse(ird, B)
    out = run(conv, sig, B)
    conv.close()
    n = blocks * B
    worst = 0.0
    for c, d in enumerate(delays):
        err = float(np.abs(out[c].astype(np.float64) - np.concatenate([np.zeros(d), sig[c, : n - d]])).max())
        worst = max(worst, err)
        assert err <= DELAY_ATOL[dtype], f"{dtype} B={B}: unit impulse at tap {d} (channel {c}): max |error| {err:.2e}"
    print(f"[lowlat-ref] delayed impulses {dtype} B={B} T={frame_blocks}: max |error| {worst:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F32, F64])
def test_delayed_impulses_cross_every_hand_off(gpu, dtype):
    # an off-by-one-block or off-by-one-frame in any level's timing moves one of these delays
    B, fb, taps, blocks = 64, (2, 4, 16, 64), 160 * 64 - 17, 224  # 224 > 3 T_n + T_1 and > P: L - 1 is reached
    assert gpu.LowLatencyConvolver.layout(num_parts(taps, B), B, fb, dtype)["levels"] == [(4, 8), (8, 32), (32, 128), (128, 160)]
    delayed_impulse_run(gpu, dtype, B, taps, fb, handoff_delays(B, fb, taps), blocks, seed=3)


@pytest.mark.gpu
def test_c5_geometry(gpu):
    # BASELINE config 5 per channel: B = 1024, 2^20 taps, default schedule (8, 32, 128); 1152 blocks reach d = L - 1
    B, taps, blocks = 1024, 1 << 20, 1152
    fb = gpu.LowLatencyConvolver.layout(taps // B, B)["frame_blocks"]
    assert fb == (8, 32, 128)
    delays = handoff_delays(B, fb, taps)
    delays.append(int(np.random.default_rng(4).integers(B + 2, taps - 1)))
    assert len(delays) == 16
    delayed_impulse_run(gpu, F32, B, taps, None, delays, blocks, seed=5)

    ir, sig = random_case(2, taps, blocks * B, F32, seed=6)
    conv = gpu.LowLatencyConvolver(F32)
    conv.impulse(ir, B)
    got = run(conv, sig, B)
    conv.close()
    assert_close("C5 geometry, 2 channels", got, ref_convolve(ir, sig), B, *BOUND[F32])


def run_device(conv, X, Y, start, stop, pattern=(1,)):
    """blocks start .. stop - 1 of X [blocks][C][B] into Y on the current torch stream, with the given blocks per call; no host
    synchronisation. One-block calls read and write X[t] / Y[t] in place, longer calls go through [C][n B] copies."""
    import torch

    C, B = X.shape[1], X.shape[2]
    t, i = start, 0
    while t < stop:
        n = min(pattern[i % len(pattern)], stop - t)
        if n == 1:
            conv(X[t], Y[t])
        else:
            x = X[t : t + n].transpose(0, 1).reshape(C, n * B)
            y = torch.empty_like(x)
            conv(x, y)
            Y[t : t + n] = y.view(C, n, B).transpose(0, 1)
        t, i = t + n, i + 1


def assert_same_device_bits(name, got, want):
    import torch

    torch.cuda.synchronize()
    if not torch.equal(got, want):
        b, c, s = (int(v) for v in (got != want).nonzero()[0])
        raise AssertionError(f"{name}: first difference at channel {c}, block {b} (sample {s})")


@pytest.mark.gpu
@pytest.mark.parametrize("frame_blocks,levels", [(None, [(16, 64), (64, 256), (256, 1024)]), ((2,), [(4, 1024)])],
                         ids=["c5_schedule", "slow_level"])
def test_wide_bank_stream_ordering(gpu, monkeypatch, frame_blocks, levels):
    # 1024 channels, B = 256, 2^18 taps: P = 1024. With no host synchronisation between one-block calls each level frame runs on
    # its side stream alongside head blocks; a missing or misplaced event wait shows up as a difference from NEO_B200_LOWLAT_SYNC,
    # where all work is on one stream.
    # - c5_schedule: C5's default schedule (8, 32, 128), whose T = 128 frames overlap many head blocks. Its levels finish well
    #   within their frame period, so the head seldom has to wait.
    # - slow_level: one T = 2 level over partitions [4, 1024). Each of its frames takes far longer than the host takes to issue
    #   the next two blocks, so the head stream is held back only by its event waits.
    import torch

    C, B, taps, blocks = 1024, 256, 1 << 18, 640
    assert gpu.LowLatencyConvolver.layout(taps // B, B, frame_blocks)["levels"] == levels
    mid = 383  # (mid + 1) % 128 == 0 (and % 2 == 0): a frame of the last level has just been released to its side stream
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    g = torch.Generator(device="cuda")
    g.manual_seed(20)
    with torch.cuda.stream(s1):
        irs = []
        for _ in range(2):
            ir = torch.rand((C, taps), generator=g, device="cuda") * 2 - 1
            ir /= torch.linalg.vector_norm(ir, dim=1, dtype=torch.float64).max().float()
            irs.append(ir)
        X = torch.rand((blocks, C, B), generator=g, device="cuda") * 2 - 1
        Y0, Y1 = torch.empty_like(X), torch.empty_like(X)

    def fresh(ir):
        conv = gpu.LowLatencyConvolver(F32, frame_blocks=frame_blocks)
        conv.set_stream(s1)
        conv.impulse(ir, B)
        return conv

    with torch.cuda.stream(s1):
        conv = fresh(irs[0])
        print(f"[lowlat-ref] wide bank {frame_blocks}: device_bytes {conv.device_bytes() / 1e9:.2f} GB")
        run_device(conv, X, Y0, 0, blocks)

        rows = [0, 1, 511, 512, 1021, 1022, 1023, int(np.random.default_rng(8).integers(2, 511))]
        idx = torch.tensor(rows, device="cuda")
        y = Y0[:, idx].permute(1, 0, 2).reshape(len(rows), -1).cpu().numpy()
        x = X[:, idx].permute(1, 0, 2).reshape(len(rows), -1).cpu().numpy()
        assert_close(f"wide bank {frame_blocks}, channels {rows}", y, ref_convolve(irs[0][idx].cpu().numpy(), x), B, *BOUND[F32])

        # set_stream to a second stream right after block `mid`, then continue there
        conv.reset()
        run_device(conv, X, Y1, 0, mid + 1)
        s2.wait_stream(s1)
        conv.set_stream(s2)
        with torch.cuda.stream(s2):
            run_device(conv, X, Y1, mid + 1, blocks)
        s1.wait_stream(s2)
        conv.set_stream(s1)
        assert_same_device_bits("set_stream after block 383", Y1, Y0)

        # reset() right after block `mid`, then replay from block 0
        conv.reset()
        run_device(conv, X, Y1, 0, mid + 1)
        conv.reset()
        Y1.zero_()
        run_device(conv, X, Y1, 0, blocks)
        assert_same_device_bits("reset after block 383 and replay", Y1, Y0)

        # a mixed call pattern from block `mid` + 1 on, starting with a whole T = 128 frame in one call
        conv.reset()
        Y1.zero_()
        run_device(conv, X, Y1, 0, mid + 1)
        run_device(conv, X, Y1, mid + 1, blocks, pattern=(128, 1, 3, 2, 7, 32))
        assert_same_device_bits("mixed calls after block 383", Y1, Y0)

        # neo_b200_lowlat_set_impulse on the live handle right after block `mid`: the blocks that follow are a fresh start with the
        # second impulse response
        conv.reset()
        run_device(conv, X, Y1, 0, mid + 1)
        gpu._check(gpu.library().neo_b200_lowlat_set_impulse(conv._h, irs[1].data_ptr(), taps, gpu.DEVICE))
        run_device(conv, X, Y1, mid + 1, blocks)
        conv.close()
        other = fresh(irs[1])
        Y0b = torch.empty_like(X)
        run_device(other, X, Y0b, mid + 1, blocks)
        other.close()
        assert_same_device_bits("set_impulse on the live handle", Y1[mid + 1 :], Y0b[mid + 1 :])
        del Y0b

        monkeypatch.setenv("NEO_B200_LOWLAT_SYNC", "1")
        sync = fresh(irs[0])
        monkeypatch.delenv("NEO_B200_LOWLAT_SYNC")
        Y1.zero_()
        run_device(sync, X, Y1, 0, blocks)
        sync.close()
        assert_same_device_bits("NEO_B200_LOWLAT_SYNC", Y1, Y0)
