"""CPU: pins the oracle (oracle/neo_oracle.c) against the reference's own known-answer tests, against golden vectors
produced by the unmodified reference (tests/golden/neo_ref_golden.npz, oracle/make_golden.py) and, where the prebuilt
oracle/_ref library is present, against the reference side by side."""
import os

import numpy as np
import pytest

from conftest import ROOT, rel_l2

KINDS = ("upols", "upola", "split_upols", "split_upola", "upola_v2")


# ---- integers: bit-exact ---------------------------------------------------------------------------------------------
def test_bitrev_table_golden(orc, golden):
    for order in range(0, 11):
        assert np.array_equal(orc.bitrev_table(order), golden[f"bitrev/{order}"])
    # SURVEY 8a row a3: order 4
    assert orc.bitrev_table(4).tolist() == [0, 8, 4, 12, 2, 10, 6, 14, 1, 9, 5, 13, 3, 11, 7, 15]


def test_digitrev_golden(orc, golden):
    for key in [k for k in golden.files if k.startswith("digitrev/")]:
        _, radix, size = key.split("/")
        assert np.array_equal(orc.digitrev_perm(int(radix), int(size)), golden[key]), key
    # the reference's LUT quirk: the last entry stays 0 (digitrevorder.hpp:34)
    assert orc.digitrev_lut(4, 16)[-1] == 0 and orc.digitrev_lut(4, 16)[1] == 4


def test_fdl_index_sequence(orc, golden):
    # convolution/fdl_index_test.cpp:13-65, P = 3
    wp, pairs = orc.fdl_index_sequence(3, 6)
    assert wp.tolist() == [0, 1, 2, 0, 1, 2]
    assert pairs[0].tolist() == [[0, 0], [1, 2], [2, 1]]
    assert pairs[1].tolist() == [[0, 1], [1, 0], [2, 2]]
    assert pairs[2].tolist() == [[0, 2], [1, 1], [2, 0]]
    for parts in (1, 2, 3, 4, 7):
        wp, pairs = orc.fdl_index_sequence(parts, 2 * parts + 3)
        assert np.array_equal(wp, golden[f"fdl_index/{parts}/write_pos"])
        assert np.array_equal(pairs, golden[f"fdl_index/{parts}/pairs"])


def test_frame_counts_and_orders(orc, golden):
    # fft/stft_test.cpp:8-13
    assert orc.num_stft_frames(1024, 128, 0) == 8
    assert orc.num_stft_frames(1024, 256, 128) == 8
    for args, want in zip(golden["stft_frames/args"], golden["stft_frames/out"]):
        assert orc.num_stft_frames(*[int(a) for a in args]) == int(want)
    for n, want in zip(golden["next_order/args"], golden["next_order/out"]):
        assert orc.next_order(int(n)) == int(want)
    assert int(golden["fft_max_order"][0]) == 27
    assert int(golden["fft_status_28"][0]) != 0 and orc.fft_status(28) != 0  # ctor throws past max_order
    assert orc.fft_status(27) == 0


# ---- inputs -------------------------------------------------------------------------------------------------------------
def test_noise_matches_reference_generator(orc, golden):
    for seed in (1, 2, 11, 13):
        assert np.array_equal(orc.noise(96, seed, np.float32), golden[f"noise/f32/{seed}"])
        assert np.array_equal(orc.noise(96, seed, np.float64), golden[f"noise/f64/{seed}"])
    assert np.array_equal(orc.noise(48, 1, np.complex64), golden["noise/c64/1"])


def test_twiddle_luts(orc, golden):
    for size in (2, 4, 16, 256):
        for d, name in ((-1, "fwd"), (1, "bwd")):
            assert np.array_equal(orc.twiddle_lut(size, d, np.float32), golden[f"twiddle/f32/{size}/{name}"])
            assert np.array_equal(orc.twiddle_lut(size, d, np.float64), golden[f"twiddle/f64/{size}/{name}"])


# ---- known answers of the reference's own tests ----------------------------------------------------------------------------
def test_kat_c2c_1234(orc, golden):
    # fft/rfft_test.cpp:170-186: FFT([1,2,3,4]) = [10, -2+2i, -2, -2-2i]
    got = orc.fft(np.array([1, 2, 3, 4], dtype=np.complex64), -1)
    assert np.allclose(got, [10, -2 + 2j, -2, -2 - 2j], atol=1e-6)
    assert np.allclose(got, golden["kat/c2c_1234"], atol=0)


def test_kat_delta_all_ones(orc, golden):
    # fft/rfft_test.cpp:132-168, fft/dft_test.cpp:31-46
    for n in (2, 16, 128):
        x = np.zeros(n, dtype=np.complex128)
        x[0] = 1
        assert np.allclose(orc.fft(x, -1), np.ones(n))
        assert np.allclose(orc.fft(x, +1), np.ones(n))
    assert np.array_equal(orc.fft(np.eye(1, 16, 0, dtype=np.complex64)[0], -1), golden["kat/c2c_delta16"])


def test_dft_plan_bluestein_golden_and_identity(orc, golden):
    # dft_plan == fallback_dft_plan (fft/dft.hpp:28-30, fallback_dft_plan.hpp:24-96): any size
    for tag, cplx, tol in (("c64", np.complex64, 0.0), ("c128", np.complex128, 2e-15)):
        for n in (2, 3, 5, 12, 21, 100, 127, 128):
            x = golden[f"dft/{tag}/{n}/x"]
            for d, name in ((-1, "fwd"), (1, "bwd")):
                want = golden[f"dft/{tag}/{n}/{name}"]
                got = orc.dft(x, d)
                assert np.linalg.norm(got - want) <= tol * np.linalg.norm(want), (tag, n, name)
                k = np.arange(n)
                exact = np.exp(d * 2j * np.pi * np.outer(k, k) / n) @ x.astype(np.complex128)  # the naive dft() of fft/dft.hpp:34-55
                assert np.linalg.norm(want - exact) <= (1e-5 if cplx == np.complex64 else 1e-12) * np.linalg.norm(exact)
    # fft/dft_test.cpp:31-46 ("identity"): a unit impulse transforms to all ones, and back to size at index 0
    for n in (2, 3, 7, 100, 127):
        x = np.zeros(n, dtype=np.complex128)
        x[0] = 1
        X = orc.dft(x, -1)
        assert np.allclose(X.real, 1.0) and np.allclose(X.imag, 0.0, atol=1e-12)
        assert np.isclose(orc.dft(X, +1)[0].real, n)


def test_dct2_plan_golden_and_scipy_known_answer(orc, golden):
    # fallback_dct2_plan (fft/dct.hpp:24-68); known answer fft/dct_test.cpp:24-39 = scipy.fft.dct([1..8], type=2)
    want = [72.0, -25.76929209, 0.0, -2.6938192, 0.0, -0.80361161, 0.0, -0.20280929]
    assert np.allclose(orc.dct2(np.arange(1, 9, dtype=np.float64)), want, atol=1e-7)
    assert np.allclose(golden["kat/dct2_1to8"], want, atol=1e-7)
    for tag, real, tol in (("f32", np.float32, 0.0), ("f64", np.float64, 1e-15)):
        for order in (1, 3, 6, 10):
            x, out = golden[f"dct2/{tag}/{order}/x"], golden[f"dct2/{tag}/{order}/out"]
            got = orc.dct2(x)
            assert np.linalg.norm(got - out) <= tol * max(np.linalg.norm(out), 1e-30), (tag, order)
    assert float(orc.dct2(np.array([3.0], dtype=np.float32))[0]) == 6.0  # order 0: undefined in the reference, DCT-II of one sample here


STFT_CASES = ((256, 256, 128, 1), (128, 256, 0, 0), (100, 128, 30, 2), (64, 64, 48, 1), (256, 300, 17, 1))


def test_stft_plan_golden(orc, golden):
    # stft_plan (fft/stft.hpp:39-109): frames with overlap, zero padding to the transform size, hann / hamming / rectangular window
    for tag, tol in (("f32", 0.0), ("f64", 1e-15)):
        x = golden[f"stft/{tag}/x"]
        for frame, transform, overlap, win in STFT_CASES:
            want = golden[f"stft/{tag}/{frame}_{transform}_{overlap}_{win}"]
            got = orc.stft(x, frame, transform, overlap, win)
            assert got.shape == want.shape == (2, orc.num_stft_frames(1000, frame, overlap), (1 << (transform - 1).bit_length()) // 2 + 1)
            assert np.linalg.norm(got - want) <= tol * np.linalg.norm(want), (tag, frame, transform, overlap, win)
    # uniform_partition is the frame = B, transform = 2B, no overlap, rectangular special case (uniform_partition.hpp:13-26)
    x = golden["stft/f32/x"][:, :896]
    assert np.array_equal(orc.uniform_partition(x, 128), orc.stft(x, 128, 256, 0, 0))
    # against numpy for one case
    xx = golden["stft/f64/x"]
    w = 0.5 * (1 - np.cos(2 * np.pi * np.arange(256) / 255))
    want = np.stack([[np.fft.rfft(xx[c, f * 128 : f * 128 + 256] * w[: len(xx[c, f * 128 : f * 128 + 256])], 256) for f in range(7)] for c in range(2)])
    assert np.allclose(golden["stft/f64/256_256_128_1"][:, :7], want, atol=1e-10)


def test_fft_convolve_golden_and_direct(orc, golden):
    # fft_convolver (convolution/fft_convolver.hpp:18-93) against the compiled reference and against direct_convolve
    for tag, tol in (("f32", 0.0), ("f64", 1e-15)):
        for n, m in ((2, 2), (7, 3), (100, 31), (513, 512)):
            x, h = golden[f"fft_convolve/{tag}/{n}_{m}/signal"], golden[f"fft_convolve/{tag}/{n}_{m}/patch"]
            want = golden[f"fft_convolve/{tag}/{n}_{m}/out"]
            got = orc.fft_convolve(x, h)
            assert got.shape == (n + m - 1,)
            assert np.linalg.norm(got - want) <= tol * np.linalg.norm(want), (tag, n, m)
            direct = orc.direct_convolve(x, h, n + m - 1)
            assert np.linalg.norm(want - direct) <= (1e-5 if tag == "f32" else 1e-12) * np.linalg.norm(direct)


def test_randomised_shapes_against_numpy(orc):
    # property checks over randomised sizes (hypothesis): the restated plans agree with numpy's definitions
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=40, deadline=None)
    @given(n=st.integers(1, 300), seed=st.integers(0, 1000), direction=st.sampled_from([-1, 1]))
    def dft_any_size(n, seed, direction):
        x = orc.noise(n, seed, np.complex128)
        k = np.arange(n)
        exact = np.exp(direction * 2j * np.pi * np.outer(k, k) / n) @ x
        assert np.linalg.norm(orc.dft(x, direction) - exact) <= 1e-11 * max(np.linalg.norm(exact), 1e-30)

    @settings(max_examples=25, deadline=None)
    @given(frame=st.integers(2, 64), pad=st.integers(0, 40), overlap_frac=st.floats(0, 0.9), extra=st.integers(0, 200), win=st.sampled_from([0, 1, 2]))
    def stft_frames(frame, pad, overlap_frac, extra, win):
        transform, overlap, length = frame + pad, int(overlap_frac * (frame - 1)), frame + extra
        n = 1 << max(0, (transform - 1).bit_length())
        x = orc.noise(length, 3, np.float64)[None]
        S = orc.stft(x, frame, transform, overlap, win)[0]
        i = np.arange(n)
        w = np.ones(n) if win == 0 else 0.5 * (1 - np.cos(2 * np.pi * i / (n - 1))) if win == 1 else 0.54 - 0.46 * np.cos(2 * np.pi * i / (n - 1))
        for f in range(S.shape[0]):
            seg = x[0, f * (frame - overlap) : f * (frame - overlap) + frame]
            buf = np.zeros(n)
            buf[: len(seg)] = seg
            assert np.allclose(S[f], np.fft.rfft(buf * w), atol=1e-10)

    @settings(max_examples=25, deadline=None)
    @given(n=st.integers(1, 200), m=st.integers(1, 200))
    def fft_convolve_full(n, m):
        x, h = orc.noise(n, 1, np.float64), orc.noise(m, 2, np.float64)
        assert np.allclose(orc.fft_convolve(x, h), np.convolve(x, h), atol=1e-11)

    dft_any_size()
    stft_frames()
    fft_convolve_full()


def test_kat_dct2_through_fft(orc):
    # fft/dct_test.cpp:23-39 pins fft_plan at N=8 through the DCT-II of [1..8] against scipy's values.
    # DCT-II via one N-point c2c (Makhoul): v = even samples then reversed odd samples, X = 2 Re(W4N^k FFT(v))
    x = np.arange(1, 9, dtype=np.float64)
    v = np.concatenate([x[0::2], x[1::2][::-1]]).astype(np.complex128)
    V = orc.fft(v, -1)
    k = np.arange(8)
    dct = 2 * np.real(np.exp(-1j * np.pi * k / 16) * V)
    want = [72.0, -25.76929209, 0.0, -2.6938192, 0.0, -0.80361161, 0.0, -0.20280929]
    assert np.allclose(dct, want, atol=1e-6)


def test_kat_multiply_add(orc, golden):
    # algorithm/multiply_add_test.cpp:52-95: (1+2i)(3+4i)+(5+6i) = 0+16i, sizes 2/33/128
    for n in (2, 33, 128):
        x, y, z = (np.full(n, v, dtype=np.complex64) for v in (1 + 2j, 3 + 4j, 5 + 6j))
        assert np.array_equal(orc.multiply_add(x, y, z), np.full(n, 16j, dtype=np.complex64))
    assert np.array_equal(golden["kat/multiply_add"], np.full(33, 16j, dtype=np.complex64))


# ---- transforms vs golden ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag,real,cplx,tol", [("f32", np.float32, np.complex64, 0.0), ("f64", np.float64, np.complex128, 4e-16)])
def test_transforms_match_reference_golden(orc, golden, tag, real, cplx, tol):
    # f32: bit-exact. f64: the reference build contracts a*b+c into FMA (-march=x86-64-v3), the oracle does not.
    for order in (1, 2, 3, 4, 5, 8, 10, 11):
        n = 1 << order
        x = orc.noise(n, 1, cplx)
        assert rel_l2(orc.fft(x, -1), golden[f"c2c/{tag}/{order}/fwd"]) <= tol
        assert rel_l2(orc.fft(x, +1), golden[f"c2c/{tag}/{order}/bwd"]) <= tol
        xr = orc.noise(n, 2, real)
        spec = orc.rfft(xr)
        assert rel_l2(spec, golden[f"r2c/{tag}/{order}"]) <= tol
        assert rel_l2(orc.irfft(golden[f"r2c/{tag}/{order}"], n), golden[f"c2r/{tag}/{order}"]) <= tol
    junk = orc.noise(64, 5, cplx)
    assert rel_l2(orc.irfft(junk[:33], 64), golden[f"c2r_junk/{tag}/half"]) <= tol
    assert rel_l2(orc.irfft(junk, 64), golden[f"c2r_junk/{tag}/full"]) <= tol
    # c2r ignores Im X[0], Im X[N/2] and everything past N/2 (fallback_rfft_plan.hpp:44-54)
    assert np.array_equal(golden[f"c2r_junk/{tag}/half"], golden[f"c2r_junk/{tag}/full"])


def test_split_complex_plan_is_the_same_transform(orc, golden):
    # fallback_split_fft_plan (SoA planes, backward by swapping the planes) computes what fft_plan computes: the oracle's c2c
    # stands for both; golden planes come from the reference's split plan itself
    for tag, cplx, tol in (("f32", np.complex64, 3e-7), ("f64", np.complex128, 1e-15)):
        for order in (1, 4, 8, 11):
            x = orc.noise(1 << order, 1, cplx)
            for d, name in ((-1, "fwd"), (1, "bwd")):
                planes = golden[f"split/{tag}/{order}/{name}"]
                assert rel_l2(orc.fft(x, d), planes[0] + 1j * planes[1]) <= tol, (tag, order, name)


def test_transforms_against_numpy(orc):
    for order in (1, 3, 6, 9, 12):
        n = 1 << order
        x = orc.noise(n, 1, np.complex128)
        assert rel_l2(orc.fft(x, -1), np.fft.fft(x)) < 1e-14
        assert rel_l2(orc.fft(x, +1), np.fft.ifft(x) * n) < 1e-14
        xr = orc.noise(n, 2, np.float64)
        assert rel_l2(orc.rfft(xr), np.fft.rfft(xr)) < 1e-14
        assert rel_l2(orc.irfft(np.fft.rfft(xr), n), xr * n) < 1e-14  # unnormalised round trip gains N
    # rfft(a), rfft(b) == deinterleave(fft(a + ib)) (fft/rfft_test.cpp:80-126)
    a, b = orc.noise(256, 3, np.float64), orc.noise(256, 4, np.float64)
    z = orc.fft(a + 1j * b, -1)
    zc = np.conj(np.roll(z[::-1], 1))
    assert np.allclose(orc.rfft(a), ((z + zc) / 2)[:129]) and np.allclose(orc.rfft(b), ((z - zc) / 2j)[:129])


# ---- filter preparation + convolvers vs golden ---------------------------------------------------------------------------------
@pytest.mark.parametrize("tag,tol", [("f32", 0.0), ("f64", 1e-15)])
def test_partition_and_convolvers_match_reference_golden(orc, golden, tag, tol):
    B, L, NB = (int(v) for v in golden["conv/block"])
    ir, sig, H = golden[f"conv/{tag}/ir"], golden[f"conv/{tag}/signal"], golden[f"conv/{tag}/H"]
    assert H.shape == (2, -(-L // B), B + 1)  # convolution/uniform_partition_test.cpp:8-38: [C][ceil(L/B)][B+1]
    assert rel_l2(orc.uniform_partition(ir, B), H) <= tol
    for kind, name in enumerate(KINDS):
        # split_* keep SoA planes; same arithmetic order, so the oracle (one AoS implementation) must match both
        tol_k = max(tol, 2e-7) if name.startswith("split") else tol
        assert rel_l2(orc.convolve_blocks(kind, H, sig), golden[f"conv/{tag}/{name}"]) <= tol_k, name
    assert rel_l2(orc.convolve_blocks(4, H, sig, chunk=96), golden[f"conv/{tag}/upola_v2_chunk96"]) <= tol


def test_sparse_filter_csr_and_sparse_convolvers_golden(orc, golden):
    # csr_matrix(partitions, predicate) (container/csr_matrix.hpp:64-98): index containers BIT-EXACT; sparse_upols / sparse_upola
    # (sparse_convolver.hpp:14-22) bit-identical to the compiled reference in float
    thr = float(golden["sparse/threshold"][0])
    H, sig = golden["conv/f32/H"], golden["conv/f32/signal"]
    rows, cols, vals = orc.csr_build(H[0], thr)
    assert np.array_equal(rows, golden["sparse/csr_rows"]) and np.array_equal(cols, golden["sparse/csr_cols"])
    assert np.array_equal(vals, golden["sparse/csr_vals"])
    assert 0 < rows[-1] < H[0].size  # the predicate drops something and keeps something
    for kind, name in ((5, "upols"), (6, "upola")):
        got = orc.convolve_blocks_sparse(kind, H, sig, thr)
        assert np.array_equal(got, golden[f"sparse/{name}"]), name
        # multiply_add over the stored elements only (algorithm/multiply_add.hpp:306-324) = the dense sum with the others zeroed
        Hz = np.where((np.abs(H.real) > thr) | (np.abs(H.imag) > thr), H, 0).astype(np.complex64)
        assert np.array_equal(got, orc.convolve_blocks(kind - 5, Hz, sig))


def test_compressed_fdl_rows_golden_and_known_answer(orc, golden):
    # compressed_fdl::insert + operator[] (compressed_fdl.hpp:26-48, compressed_accessor.hpp:27-45): the restatement reads back what
    # the compiled reference reads back, bit for bit; tolerances of compressed_fdl_test.cpp:24-29 on its known-answer row
    for bits, tol in ((8, 0.005), (16, 0.0001)):
        for name in ("kat", "noise"):
            x = golden[f"cfdl/{name}_in"]
            got = orc.compressed_fdl_roundtrip(x, bits)
            assert np.array_equal(got, golden[f"cfdl/{bits}/{name}_out"]), (bits, name)
            if name == "kat":
                assert np.abs((got - x).view(np.float32)).max() <= tol  # per part, as the reference's WithinAbs checks
        q = orc.compress_row(golden["cfdl/kat_in"], bits)
        top = 127 if bits == 8 else 32767
        assert q[3, 1] == top and q[7, 1] == -top and q[0, 0] == 0 and q[2, 0] == (64 if bits == 8 else 16384)  # lround: half away from zero
        # the stored integers are what the read-back values say they are
        assert np.array_equal(np.rint(golden[f"cfdl/{bits}/noise_out"].view(np.float32).astype(np.float64) * top).astype(np.int16).reshape(-1, 2),
                              orc.compress_row(golden["cfdl/noise_in"], bits))


def test_uniform_partition_shapes(orc):
    # convolution/uniform_partition_test.cpp:8-38
    for L in (4096, 4095):
        H = orc.uniform_partition(np.zeros((2, L), dtype=np.float32), 128)
        assert H.shape == (2, 32, 129)


def test_upols_equals_direct_convolution(orc):
    # the gap SURVEY section 4 names: non-trivial IR vs direct convolution
    B, L, NB = 128, 1000, 24
    ir = orc.normalize_impulse(orc.noise(L, 11, np.float32)[None, :])
    sig = orc.noise(B * NB, 13, np.float32)[None, :]
    H = orc.uniform_partition(ir, B)
    want = orc.direct_convolve(sig[0], ir[0], B * NB)
    for kind in (0, 1, 4):
        assert rel_l2(orc.convolve_blocks(kind, H, sig)[0], want) < 2e-6


def test_identity_filter_passes_signal(orc):
    # convolution/uniform_partitioned_convolver_test.cpp:35-75: partition 0 all-ones, 3 partitions, 20 blocks
    for B in (128, 256):
        H = np.zeros((1, 3, B + 1), dtype=np.complex64)
        H[0, 0, :] = 1
        sig = orc.noise(B * 20, 7, np.float32)[None, :]
        for kind in range(5):
            assert np.allclose(orc.convolve_blocks(kind, H, sig), sig, atol=1e-5)


def test_overlap_policies_identity(golden):
    # convolution/overlap_test.cpp:21-64 through the reference itself
    assert np.allclose(golden["overlap/save"], golden["overlap/signal"], atol=1e-5)
    assert np.allclose(golden["overlap/add"], golden["overlap/signal"], atol=1e-5)


# ---- side by side with the compiled reference: its stored outputs, and the library itself when it travelled ---------------------------
def test_oracle_vs_compiled_reference(orc, ref):
    # tests/golden/neo_ref_side_by_side.npz holds the inputs and the compiled reference's outputs (oracle/make_golden_side_by_side.py);
    # the oracle must reproduce them bit for bit, and so must the reference library where it is present
    from oracle.make_golden_side_by_side import side_by_side

    want = np.load(os.path.join(ROOT, "tests", "golden", "neo_ref_side_by_side.npz"))
    for name, chk in [("oracle", orc)] + ([("reference", ref)] if ref is not None else []):
        got = side_by_side(chk, orc.noise)
        assert sorted(got) == sorted(want.files), name
        for key in want.files:
            assert np.array_equal(got[key], want[key]), (name, key)
