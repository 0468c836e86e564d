"""GPU: parity of the CUDA partitioned-convolver bank with the oracle (= the reference's upols/upola convolvers, one per
channel) through the C ABI, block by block including the zero-history warm-up blocks."""
import numpy as np
import pytest

from conftest import TOL, rel_l2

pytestmark = pytest.mark.gpu


def make_case(orc, channels, taps, block, nblocks, real=np.float32, seed=0):
    ir = np.stack([orc.noise(taps, 11 + seed + c, real) for c in range(channels)])
    if real == np.float32:
        ir = orc.normalize_impulse(ir)
    else:
        ir = ir / np.sqrt((ir**2).sum(axis=1).max())
    sig = np.stack([orc.noise(block * nblocks, 13 + seed + c, real) for c in range(channels)])
    return ir, sig


def run_bank(conv, sig, block, pattern):
    """feed sig[C][n] through the bank with the given sequence of blocks-per-call"""
    out = sig.copy()
    pos = 0
    i = 0
    while pos < sig.shape[1]:
        t = min(pattern[i % len(pattern)], (sig.shape[1] - pos) // block)
        chunk = np.ascontiguousarray(out[:, pos : pos + t * block])
        conv(chunk)
        out[:, pos : pos + t * block] = chunk
        pos += t * block
        i += 1
    return out


@pytest.mark.parametrize("name,kind", [("upols", 0), ("upola", 1)])
@pytest.mark.parametrize("tag,real", [("f32", np.float32), ("f64", np.float64)])
def test_golden_vectors_from_the_reference(gpu, golden, name, kind, tag, real):
    B, L, NB = (int(v) for v in golden["conv/block"])
    H, sig, want = golden[f"conv/{tag}/H"], golden[f"conv/{tag}/signal"], golden[f"conv/{tag}/{name}"]
    for pattern in ([1], [2], [3, 1], [12]):
        conv = gpu.Convolver(kind, real, gpu.DIAGONAL, max_blocks=max(pattern))
        conv.filter(H)
        got = run_bank(conv, sig, B, pattern)
        assert rel_l2(got, want) <= TOL[np.dtype(real).name], pattern
        conv.close()
    # split_* aliases and upola_v2 (block-sized calls) compute the same thing (dense_convolver.hpp:28-41)
    assert rel_l2(golden[f"conv/{tag}/split_{name}"], want) <= 1e-6
    if kind == 1:
        assert rel_l2(golden[f"conv/{tag}/upola_v2"], want) <= 1e-6


@pytest.mark.parametrize("block,taps,channels,nblocks", [
    (2, 7, 3, 9), (8, 8, 2, 6), (16, 100, 3, 40), (128, 1000, 3, 24), (512, 512 * 17, 2, 40), (1024, 1024 * 33 - 5, 2, 45),
    (4096, 4096 * 3, 1, 7),
])
def test_upols_matches_oracle_streaming_and_batched(gpu, orc, block, taps, channels, nblocks):
    ir, sig = make_case(orc, channels, taps, block, nblocks)
    H = orc.uniform_partition(ir, block)
    want = orc.convolve_blocks(0, H, sig)
    for pattern in ([1], [1, 2, 5, 16, 7, 1, 3], [32]):
        conv = gpu.Convolver(gpu.UPOLS, np.float32, gpu.DIAGONAL, max_blocks=32)
        conv.filter(H)
        got = run_bank(conv, sig, block, pattern)
        assert rel_l2(got, want) <= 1e-5, (pattern, rel_l2(got, want))
        conv.close()
    # against direct convolution too (the gap SURVEY section 4 names)
    direct = np.stack([orc.direct_convolve(sig[c], ir[c], sig.shape[1]) for c in range(channels)])
    assert rel_l2(got, direct) <= 1e-5


@pytest.mark.parametrize("block,taps", [(16, 100), (256, 256 * 9 - 3)])
def test_upola_and_f64(gpu, orc, block, taps):
    for real in (np.float32, np.float64):
        ir, sig = make_case(orc, 2, taps, block, 20, real)
        H = orc.uniform_partition(ir, block)
        for kind in (0, 1):
            want = orc.convolve_blocks(kind, H, sig)
            for pattern in ([1], [4, 1, 8]):
                conv = gpu.Convolver(kind, real, gpu.DIAGONAL, max_blocks=8)
                conv.filter(H)
                assert rel_l2(run_bank(conv, sig, block, pattern), want) <= TOL[np.dtype(real).name], (real, kind, pattern)
                conv.close()


def test_identity_filter_passes_signal(gpu, orc):
    # convolution/uniform_partitioned_convolver_test.cpp:35-75
    for block in (128, 256, 512, 1024):
        H = np.zeros((1, 3, block + 1), dtype=np.complex64)
        H[0, 0, :] = 1
        sig = orc.noise(block * 20, 7, np.float32)[None, :]
        for kind in (gpu.UPOLS, gpu.UPOLA):
            conv = gpu.Convolver(kind, np.float32)
            conv.filter(H)
            assert np.allclose(run_bank(conv, sig, block, [1]), sig, atol=1e-5)
            conv.close()


def test_uniform_partition_matches_oracle(gpu, orc, golden):
    B, L, _ = (int(v) for v in golden["conv/block"])
    for tag, real in (("f32", np.float32), ("f64", np.float64)):
        got = gpu.uniform_partition(golden[f"conv/{tag}/ir"], B)
        assert got.shape == golden[f"conv/{tag}/H"].shape
        assert rel_l2(got, golden[f"conv/{tag}/H"]) <= TOL[np.dtype(real).name]
    for L in (4096, 4095):  # convolution/uniform_partition_test.cpp:8-38
        ir = np.stack([orc.noise(L, 3 + c, np.float32) for c in range(2)])
        got = gpu.uniform_partition(ir, 128)
        assert got.shape == (2, 32, 129)
        assert rel_l2(got, orc.uniform_partition(ir, 128)) <= 1e-5
    with pytest.raises(RuntimeError):
        gpu.uniform_partition(np.zeros((1, 100), dtype=np.float32), 128)  # L < B underflows in the reference
    with pytest.raises(RuntimeError):
        gpu.uniform_partition(np.zeros((1, 300), dtype=np.float32), 96)   # B must be a power of two


def test_impulse_entry_equals_filter_entry(gpu, orc):
    ir, sig = make_case(orc, 3, 700, 64, 16)
    a = gpu.Convolver(gpu.UPOLS, np.float32, max_blocks=4)
    a.filter(orc.uniform_partition(ir, 64))
    b = gpu.Convolver(gpu.UPOLS, np.float32, max_blocks=4)
    b.impulse(ir, 64)
    ya, yb = run_bank(a, sig, 64, [4]), run_bank(b, sig, 64, [4])
    assert rel_l2(yb, ya) <= 2e-6


@pytest.mark.parametrize("block,taps,channels,thr", [(128, 1000, 3, 0.05), (16, 16 * 41 - 3, 2, 0.2), (1024, 1024 * 6, 2, 0.02), (4, 40, 2, 0.3)])
def test_sparse_filters_csr_device_layout(gpu, orc, golden, block, taps, channels, thr):
    # sparse_upols / sparse_upola (sparse_convolver.hpp:14-22): the CSR matrices of neo::csr_matrix go to the device, which keeps
    # and multiplies only the stored elements (multiply_add.hpp:306-324). Oracle = the reference's sparse convolvers (kinds 5, 6).
    ir, sig = make_case(orc, channels, taps, block, 13)
    H = orc.uniform_partition(ir, block)
    keep = (np.abs(H.real) > thr) | (np.abs(H.imag) > thr)
    assert 0 < keep.sum() < keep.size
    for kind in (0, 1):
        want = orc.convolve_blocks_sparse(5 + kind, H, sig, thr)
        for pattern in ([1], [3, 1, 4]):
            conv = gpu.Convolver(kind, np.float32, gpu.DIAGONAL, max_blocks=4)
            conv.filter_sparse(H, keep)
            # the containers handed over are the reference's own, bit for bit (channel 0 checked against the oracle's csr_matrix)
            rows, cols, vals = orc.csr_build(H[0], thr)
            n0 = int(rows[-1])
            assert np.array_equal(conv.csr[0][0], rows) and np.array_equal(conv.csr[1][:n0], cols) and np.array_equal(conv.csr[2][:n0], vals)
            got = run_bank(conv, sig, block, pattern)
            assert rel_l2(got, want) <= 1e-5, (kind, pattern, rel_l2(got, want))
            sparse_bytes = conv.device_bytes()
            conv.filter(H)  # a dense filter replaces the sparse one (and the other way round)
            assert rel_l2(run_bank(conv, sig, block, pattern), orc.convolve_blocks(kind, H, sig)) <= 1e-5
            if keep.mean() < 0.8 and block >= 128:
                assert sparse_bytes < conv.device_bytes()
            conv.close()
    # a wide bank through the host pipeline (channel groups, T = 4 per call) and with device buffers
    irw, sigw = make_case(orc, 48, 32 * 5, 32, 8)
    Hw = orc.uniform_partition(irw, 32)
    keepw = (np.abs(Hw.real) > 0.1) | (np.abs(Hw.imag) > 0.1)
    wantw = orc.convolve_blocks_sparse(5, Hw, sigw, 0.1)
    conv = gpu.Convolver(gpu.UPOLS, np.float32, gpu.DIAGONAL, max_blocks=4)
    conv.filter_sparse(Hw, keepw)
    assert rel_l2(run_bank(conv, sigw, 32, [4]), wantw) <= 1e-5
    conv.reset()
    import torch

    conv.set_stream(torch.cuda.current_stream())  # device buffers: the input copies and the read-backs below are on torch's stream
    x = torch.from_numpy(sigw).cuda()
    y = torch.empty_like(x[:, : 4 * 32])
    outs = []
    for s in range(2):
        conv(x[:, s * 128 : (s + 1) * 128].contiguous(), out=y)
        outs.append(y.cpu().numpy())
    conv.close()
    assert rel_l2(np.concatenate(outs, axis=1), wantw) <= 1e-5
    # float64, and a filter whose predicate keeps nothing in some channels / everything in others
    ir64, sig64 = make_case(orc, 2, 300, 32, 9, np.float64)
    H64 = orc.uniform_partition(ir64, 32)
    keep64 = np.ones(H64.shape, dtype=bool)
    keep64[1] = False
    conv = gpu.Convolver(gpu.UPOLS, np.float64, gpu.DIAGONAL, max_blocks=2)
    conv.filter_sparse(H64, keep64)
    got = run_bank(conv, sig64, 32, [2, 1])
    conv.close()
    want = orc.convolve_blocks(0, H64, sig64)
    assert rel_l2(got[0], want[0]) <= 1e-12 and not got[1].any()
    # the golden vectors of the compiled reference
    gthr = float(golden["sparse/threshold"][0])
    Hg, sg = golden["conv/f32/H"], golden["conv/f32/signal"]
    for kind, name in ((0, "upols"), (1, "upola")):
        conv = gpu.Convolver(kind, np.float32, gpu.DIAGONAL)
        conv.filter_sparse(Hg, (np.abs(Hg.real) > gthr) | (np.abs(Hg.imag) > gthr))
        assert rel_l2(run_bank(conv, sg, 32, [1]), golden[f"sparse/{name}"]) <= 1e-5
        conv.close()


@pytest.mark.parametrize("bits", [8, 16])
def test_compressed_fdl_on_the_device(gpu, orc, golden, bits):
    # compressed_fdl (compressed_fdl.hpp:17-52): the device stores the reference's integers (bit-exact) and reads rows back as its
    # compressed_accessor does; golden = the compiled reference's read-back
    fdl = gpu.CompressedFDL(4, 257, "float32", bits)
    x = golden["cfdl/noise_in"]
    fdl.insert(x, 2)
    assert np.array_equal(fdl.raw(2), orc.compress_row(x, bits).astype(fdl.raw(2).dtype))
    assert np.array_equal(fdl.row(2), golden[f"cfdl/{bits}/noise_out"])
    assert not fdl.raw(0).any() and not fdl.row(3).any()  # untouched rows are zero, like the reference's value-initialised storage
    fdl.close()
    kat = gpu.CompressedFDL(4, 8, "float32", bits)
    kat.insert(golden["cfdl/kat_in"], 0)
    assert np.array_equal(kat.row(0), golden[f"cfdl/{bits}/kat_out"])
    kat.close()
    # double-precision rows: val * (float) max is a double product there
    xd = (orc.noise(100, 5, np.complex128) * 0.999).astype(np.complex128)
    fd = gpu.CompressedFDL(2, 100, "float64", bits)
    fd.insert(xd, 1)
    q = orc.compress_row(xd, bits)
    assert np.array_equal(fd.raw(1), q.astype(fd.raw(1).dtype))
    top = 127 if bits == 8 else 32767
    assert np.array_equal(fd.row(1).view(np.float64).reshape(-1, 2), q.astype(np.float64) * (1.0 / top))
    with pytest.raises(RuntimeError):
        fd.insert(xd, 2)  # past the last row
    fd.close()


def test_filter_swap_and_reset(gpu, orc):
    ir, sig = make_case(orc, 2, 500, 32, 10)
    ir2, _ = make_case(orc, 2, 300, 32, 10, seed=50)
    H, H2 = orc.uniform_partition(ir, 32), orc.uniform_partition(ir2, 32)
    conv = gpu.Convolver(gpu.UPOLS, np.float32)
    conv.filter(H)
    first = run_bank(conv, sig, 32, [1])
    conv.reset()
    assert np.array_equal(run_bank(conv, sig, 32, [1]), first)  # reset restores the zero-history state exactly
    conv.filter(H2)  # filter() may be called again to swap IRs; all state is re-created (uniform_partitioned_convolver.hpp:38-45)
    assert rel_l2(run_bank(conv, sig, 32, [1]), orc.convolve_blocks(0, H2, sig)) <= 1e-5


def test_matrix_topology_equals_sum_of_reference_convolvers(gpu, orc):
    # 3 inputs x 2 outputs: every (o, i) pair is one reference convolver, outputs summed per o (SURVEY 8d C4)
    O, I, B, L, NB = 2, 3, 64, 64 * 9, 14
    ir = np.stack([np.stack([orc.noise(L, 100 + 10 * o + i, np.float32) for i in range(I)]) for o in range(O)])
    ir /= np.sqrt((ir**2).sum(axis=2).max())
    sig = np.stack([orc.noise(B * NB, 13 + i, np.float32) for i in range(I)])
    want = np.zeros((O, B * NB), dtype=np.float64)
    for o in range(O):
        H = orc.uniform_partition(ir[o], B)
        want[o] = orc.convolve_blocks(0, H, sig).astype(np.float64).sum(axis=0)
    Hm = np.stack([orc.uniform_partition(ir[o], B) for o in range(O)])
    for pattern in ([1], [2, 4, 1]):
        conv = gpu.Convolver(gpu.UPOLS, np.float32, gpu.MATRIX, max_blocks=4)
        conv.filter(Hm)
        got = np.zeros((O, B * NB), dtype=np.float32)
        pos, i = 0, 0
        while pos < B * NB:
            t = min(pattern[i % len(pattern)], NB - pos // B)
            got[:, pos : pos + t * B] = conv(np.ascontiguousarray(sig[:, pos : pos + t * B]))
            pos += t * B
            i += 1
        assert rel_l2(got, want) <= 1e-5, pattern
        conv.close()


def test_wide_bank_host_pipeline_and_device_path_agree_with_oracle(gpu, orc):
    # >= 128 channels and >= 4 blocks per call: host-buffer calls are cut into channel groups and pipelined over copy streams
    import torch

    C, B, P, NB = 160, 64, 5, 16
    ir, sig = make_case(orc, C, B * P - 3, B, NB)
    H = orc.uniform_partition(ir, B)
    want = orc.convolve_blocks(0, H, sig)
    for pattern in ([4], [8, 4, 1, 3]):
        conv = gpu.Convolver(gpu.UPOLS, np.float32, gpu.DIAGONAL, max_blocks=8)
        conv.filter(H)
        assert rel_l2(run_bank(conv, sig, B, pattern), want) <= 1e-5, pattern
        conv.close()
    conv = gpu.Convolver(gpu.UPOLA, np.float32, gpu.DIAGONAL, max_blocks=8)
    conv.filter(H)
    assert rel_l2(run_bank(conv, sig, B, [8]), orc.convolve_blocks(1, H, sig)) <= 1e-5
    conv.close()
    # same bank with device-resident buffers on a caller-provided stream
    conv = gpu.Convolver(gpu.UPOLS, np.float32, gpu.DIAGONAL, max_blocks=8)
    conv.set_stream(torch.cuda.current_stream())
    conv.filter(torch.from_numpy(H).cuda())
    dx = torch.from_numpy(sig).cuda()
    dy = torch.empty_like(dx)
    for pos in range(0, NB, 8):
        chunk = dx[:, pos * B : (pos + 8) * B].contiguous()
        out = torch.empty_like(chunk)
        conv(chunk, out=out)
        dy[:, pos * B : (pos + 8) * B] = out
    torch.cuda.synchronize()
    assert rel_l2(dy.cpu().numpy(), want) <= 1e-5


def test_matrix_topology_four_outputs_per_thread_path(gpu, orc):
    # outputs % 4 == 0 selects the output-tiled streaming MAC (T = 1) for the matrix topology
    O, I, B, L, NB = 8, 3, 128, 128 * 6, 9
    ir = np.stack([np.stack([orc.noise(L, 300 + 10 * o + i, np.float32) for i in range(I)]) for o in range(O)])
    ir /= np.sqrt((ir**2).sum(axis=2).max())
    sig = np.stack([orc.noise(B * NB, 13 + i, np.float32) for i in range(I)])
    want = np.stack([orc.convolve_blocks(0, orc.uniform_partition(ir[o], B), sig).astype(np.float64).sum(axis=0) for o in range(O)])
    conv = gpu.Convolver(gpu.UPOLS, np.float32, gpu.MATRIX, max_blocks=2)
    conv.impulse(ir, B)
    got = np.zeros((O, B * NB), dtype=np.float32)
    for b in range(NB):
        got[:, b * B : (b + 1) * B] = conv(np.ascontiguousarray(sig[:, b * B : (b + 1) * B]))
    assert rel_l2(got, want) <= 1e-5


def test_partition_sharded_handles_sum_to_the_whole(gpu, orc):
    # one long IR split over "devices": partial spectra add up; inverse runs on the sum (SURVEY 8e, last row)
    import torch

    C, B, P, NB, T = 4, 128, 12, 18, 3
    ir, sig = make_case(orc, C, B * P - 17, B, NB)
    H = orc.uniform_partition(ir, B)
    want = orc.convolve_blocks(0, H, sig)
    shards = [(0, 5), (5, 6), (6, 12)]
    convs = []
    for lo, hi in shards:
        c = gpu.Convolver(gpu.UPOLS, np.float32, gpu.DIAGONAL, max_blocks=T, partition_range=(lo, hi))
        c.filter(H)
        convs.append(c)
    got = np.zeros_like(sig)
    for pos in range(0, NB, T):
        x = torch.from_numpy(np.ascontiguousarray(sig[:, pos * B : (pos + T) * B])).cuda()
        total = None
        for c in convs:
            c.forward(x)
            c.synchronize()
            part = c.spectra_tensor(T).clone()
            total = part if total is None else total + part
        y = torch.empty_like(x)
        # the channel range is split too: outputs [0,1) on "rank" 0, [1,4) on "rank" 2
        convs[0].inverse(total[0:1].contiguous(), y[0:1], 0, 1, T)
        convs[2].inverse(total[1:4].contiguous(), y[1:4], 1, 3, T)
        convs[0].synchronize()
        convs[2].synchronize()
        got[:, pos * B : (pos + T) * B] = y.cpu().numpy()
    assert rel_l2(got, want) <= 1e-5
    with pytest.raises(RuntimeError):
        convs[0](np.zeros((C, B), dtype=np.float32))  # a sharded handle has no complete process()


def test_small_bank_splits_partitions_across_ctas(gpu, orc):
    # 1 channel x 256 partitions: the partition loop is split over CTAs and partial planes are summed in the c2r load
    ir, sig = make_case(orc, 1, 256 * 256, 256, 12)
    H = orc.uniform_partition(ir, 256)
    want = orc.convolve_blocks(0, H, sig)
    for pattern in ([1], [4]):
        conv = gpu.Convolver(gpu.UPOLS, np.float32, max_blocks=4)
        conv.filter(H)
        assert rel_l2(run_bank(conv, sig, 256, pattern), want) <= 1e-5
        conv.close()


def test_full_size_partitions_north_star_shape(gpu, orc):
    # BASELINE config 5 geometry (B=1024, 2^20 taps -> P=1024, K=1025) on a 2-channel slice, full oracle parity,
    # plus a size-independent property on more channels: an IR that is a unit impulse at tap d delays the input by d.
    B, L, NB = 1024, 1 << 20, 12
    ir, sig = make_case(orc, 2, L, B, NB)
    conv = gpu.Convolver(gpu.UPOLS, np.float32, max_blocks=4)
    conv.impulse(ir, B)
    got = run_bank(conv, sig, B, [1, 4, 2])
    want = orc.convolve_blocks(0, orc.uniform_partition(ir, B), sig)
    assert rel_l2(got, want) <= 1e-5
    conv.close()

    C = 16
    delays = [(c * 65521 + 3) % (NB * B // 2) for c in range(C)]
    ird = np.zeros((C, L), dtype=np.float32)
    for c, d in enumerate(delays):
        ird[c, d] = 1
    sigd = np.stack([orc.noise(B * NB, 200 + c, np.float32) for c in range(C)])
    conv = gpu.Convolver(gpu.UPOLS, np.float32, max_blocks=12)
    conv.impulse(ird, B)
    out = run_bank(conv, sigd, B, [12])
    for c, d in enumerate(delays):
        expect = np.concatenate([np.zeros(d, dtype=np.float32), sigd[c, : B * NB - d]])
        assert np.allclose(out[c], expect, atol=2e-5), c


def test_error_contract(gpu, orc):
    conv = gpu.Convolver(gpu.UPOLS, np.float32, max_blocks=2)
    with pytest.raises(RuntimeError):
        conv.filter(np.zeros((1, 3, 97), dtype=np.complex64))  # B = 96 is not a power of two
    H = np.zeros((2, 3, 65), dtype=np.complex64)
    conv.filter(H)
    with pytest.raises(ValueError):
        conv(np.zeros((2, 100), dtype=np.float32))  # not a whole number of blocks
    with pytest.raises(RuntimeError):
        conv(np.zeros((2, 64 * 3), dtype=np.float32))  # more blocks than max_blocks
    assert conv.device_bytes() > 0


def test_python_convolve_front_end(gpu, orc):
    # extra/python/test/test.py:25-40: delta patch returns the signal; unsupported modes raise RuntimeError
    sig = orc.noise(1000, 5, np.float32)
    for method in ("upols", "upola"):
        out = gpu.convolve(sig, np.array([1.0], dtype=np.float32), method=method)
        assert out.shape == (1000,) and np.allclose(out, sig, atol=1e-5)
        ir = orc.noise(300, 6, np.float32)
        full = gpu.convolve(sig, ir, method=method)
        assert full.shape == (1299,)
        assert rel_l2(full, np.convolve(sig.astype(np.float64), ir.astype(np.float64))) < 1e-5
    for mode in ("valid", "same"):
        with pytest.raises(RuntimeError):
            gpu.convolve(sig, sig, mode=mode)
    assert gpu.convolve(np.zeros(0, dtype=np.float32), sig).size == 0  # empty-input edge case (direct_convolve_test.cpp)


def test_baseline_config4_full_size_matrix_routing(gpu, orc):
    # BASELINE config 4 at full size: 64 in x 64 out, B=256, 2^16-tap IRs (2.2 GB of filter spectra). Property: an impulse-response
    # matrix of unit impulses h[o][i] = delta(n - d(o,i)) * g(o,i) makes every output a gain-weighted sum of delayed inputs.
    import torch

    O = I = 64
    B, L, NB = 256, 1 << 16, 8
    rng = np.random.default_rng(5)
    delays = rng.integers(0, B * NB // 2, size=(O, I))
    gains = rng.uniform(-1, 1, size=(O, I)).astype(np.float32)
    ir = torch.zeros((O, I, L), device="cuda")
    oo, ii = np.meshgrid(np.arange(O), np.arange(I), indexing="ij")
    ir[torch.from_numpy(oo.ravel()).cuda(), torch.from_numpy(ii.ravel()).cuda(), torch.from_numpy(delays.ravel()).cuda()] = torch.from_numpy(gains.ravel()).cuda()
    sig = np.stack([orc.noise(B * NB, 400 + i, np.float32) for i in range(I)])
    want = np.zeros((O, B * NB), dtype=np.float64)
    for o in range(O):
        for i in range(I):
            d = int(delays[o, i])
            want[o, d:] += gains[o, i] * sig[i, : B * NB - d]
    for T in (1, 4):
        conv = gpu.Convolver(gpu.UPOLS, np.float32, gpu.MATRIX, max_blocks=T)
        conv.set_stream(torch.cuda.current_stream())
        conv.impulse(ir, B)
        got = np.zeros((O, B * NB), dtype=np.float32)
        for pos in range(0, NB, T):
            x = torch.from_numpy(np.ascontiguousarray(sig[:, pos * B : (pos + T) * B])).cuda()
            y = torch.empty((O, T * B), device="cuda")
            conv(x, out=y)
            torch.cuda.synchronize()
            got[:, pos * B : (pos + T) * B] = y.cpu().numpy()
        assert rel_l2(got, want) <= 1e-5, T
        conv.close()


def test_baseline_config4_slice_matches_oracle(gpu, orc):
    # BASELINE config 4's geometry on a slice the oracle finishes in seconds: 8 outputs x 64 inputs, B=256, 2^16-tap random IRs
    # (P=256, K=257). Every (o, i) pair is one reference convolver, summed per output (uniform_partitioned_convolver.hpp:48-65,
    # dense_filter.hpp:31-35): streaming, time-batched direct form and frame mode.
    O, I, B, L, NB = 8, 64, 256, 1 << 16, 16
    rng = np.random.default_rng(41)
    ir = rng.uniform(-1, 1, size=(O, I, L)).astype(np.float32)
    ir *= np.float32(1.0 / np.sqrt((ir.astype(np.float64) ** 2).sum(axis=2).max()))
    sig = np.stack([orc.noise(B * NB, 500 + i, np.float32) for i in range(I)])
    want = np.zeros((O, B * NB), dtype=np.float64)
    for o in range(O):
        want[o] = orc.convolve_blocks(0, orc.uniform_partition(ir[o], B), sig).astype(np.float64).sum(axis=0)
    for frame, T in ((0, 1), (0, 16), (8, 8)):
        conv = gpu.Convolver(gpu.UPOLS, np.float32, gpu.MATRIX, max_blocks=T, frame_blocks=frame)
        conv.impulse(ir, B)
        got = np.zeros((O, B * NB), dtype=np.float32)
        for pos in range(0, NB, T):
            got[:, pos * B : (pos + T) * B] = conv(np.ascontiguousarray(sig[:, pos * B : (pos + T) * B]))
        assert rel_l2(got, want) <= 1e-5, (frame, T, rel_l2(got, want))
        conv.close()


def test_upola_grouped_forward_with_several_inverse_ranges(gpu, orc):
    # the overlap-add tail belongs to a channel, not to a call: a step finished by SEVERAL inverse calls over disjoint channel ranges
    # (the grouped reduce-scatter shape) must leave every channel's tail right (it used to ping-pong per inverse call)
    import torch

    C, B, P, T, steps = 6, 64, 5, 3, 6
    ir, sig = make_case(orc, C, B * P - 4, B, T * steps)
    H = orc.uniform_partition(ir, B)
    want = orc.convolve_blocks(gpu.UPOLA, H, sig)
    conv = gpu.Convolver(gpu.UPOLA, np.float32, gpu.DIAGONAL, max_blocks=T)
    conv.set_stream(torch.cuda.current_stream())
    conv.filter(H)
    got = np.zeros_like(sig)
    for s in range(steps):
        x = torch.from_numpy(np.ascontiguousarray(sig[:, s * T * B : (s + 1) * T * B])).cuda()
        conv.forward_range(x, 0, 2, False)
        conv.forward_range(x, 2, 4, True)
        spectra = conv.spectra_tensor(T)
        y = torch.empty((C, T * B), device="cuda", dtype=torch.float32)
        for first, count in ((0, 1), (1, 3), (4, 2)):  # three inverse ranges per step, not aligned with the forward groups
            conv.inverse(spectra[first : first + count].contiguous(), y[first : first + count], first, count, T)
        torch.cuda.synchronize()
        got[:, s * T * B : (s + 1) * T * B] = y.cpu().numpy()
    assert rel_l2(got, want) <= 1e-5, rel_l2(got, want)
    # the contract of forward_range is enforced: ascending tiling ranges, one block count, final with the last range, no process() inside
    x = torch.zeros((C, T * B), device="cuda")
    conv.reset()
    with pytest.raises(RuntimeError, match="must start at"):
        conv.forward_range(x, 2, 4, True)
    conv.forward_range(x, 0, 2, False)
    with pytest.raises(RuntimeError, match="must start at"):
        conv.forward_range(x, 0, 2, False)
    with pytest.raises(RuntimeError, match="final"):
        conv.forward_range(x, 2, 4, False)
    with pytest.raises(RuntimeError, match="in progress"):
        conv(x, out=torch.empty_like(x))
    with pytest.raises(RuntimeError, match="blocks"):
        conv.forward_range(torch.zeros((C, B), device="cuda"), 2, 4, True)
    conv.reset()  # abandons the grouped call
    conv(x, out=torch.empty_like(x))
    conv.close()


@pytest.mark.parametrize("tag,real", [("f32", np.float32), ("f64", np.float64)])
def test_fft_convolve_matches_reference_golden_and_oracle(gpu, orc, golden, tag, real):
    # fft_convolver (convolution/fft_convolver.hpp:18-93), mode::full
    import torch

    tol = TOL[np.dtype(real).name]
    for n, m in ((2, 2), (7, 3), (100, 31), (513, 512)):
        x, h = golden[f"fft_convolve/{tag}/{n}_{m}/signal"], golden[f"fft_convolve/{tag}/{n}_{m}/patch"]
        got = gpu.fft_convolve(x, h)
        assert got.shape == (n + m - 1,)
        assert rel_l2(got, golden[f"fft_convolve/{tag}/{n}_{m}/out"]) <= 10 * tol, (n, m)
    # batched, device resident, a transform beyond the single-CTA range (2^17 points)
    n, m, batch = 70000, 40000, 3
    xs = np.stack([orc.noise(n, 50 + b, real) for b in range(batch)])
    hs = np.stack([orc.noise(m, 60 + b, real) for b in range(batch)])
    got = gpu.fft_convolve(torch.from_numpy(xs).cuda(), torch.from_numpy(hs).cuda()).cpu().numpy()
    for b in range(batch):
        assert rel_l2(got[b], orc.fft_convolve(xs[b], hs[b])) <= 10 * tol, b
    assert rel_l2(gpu.fft_convolve(np.ones(1, dtype=real), np.full(1, 3, dtype=real)), np.full(1, 3.0)) <= tol  # N = 1
    if real == np.float32:
        assert rel_l2(gpu.convolve(xs[0, :500], hs[0, :60], method="fft"), orc.direct_convolve(xs[0, :500], hs[0, :60], 559)) <= 1e-5


def test_normalize_impulse_matches_oracle(gpu, orc):
    # convolution/normalize_impulse_test.cpp: unit energy for the loudest channel, common factor for all
    ir = np.stack([orc.noise(4097, 21 + c, np.float32) * (c + 1) for c in range(3)])
    got = gpu.normalize_impulse(ir.copy())
    want = orc.normalize_impulse(ir)
    assert rel_l2(got, want) <= 2e-6  # the oracle accumulates the energy in float32 like the reference, the kernel in double
    assert abs(float((got[2].astype(np.float64) ** 2).sum()) - 1.0) < 1e-5
    zeros = np.zeros((2, 64), dtype=np.float32)
    assert np.array_equal(gpu.normalize_impulse(zeros.copy()), zeros)  # energy exactly 0 -> factor 1
