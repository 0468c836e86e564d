"""GPU: parity of the CUDA FFT plans with the oracle (= the reference's fallback plans) through the C ABI.
Tolerances are north_star's: relative L2 <= 1e-5 (float32), <= 1e-12 (float64)."""
import numpy as np
import pytest

from conftest import TOL, rel_l2

pytestmark = pytest.mark.gpu

CASES = [(np.float32, np.complex64), (np.float64, np.complex128)]


@pytest.mark.parametrize("real,cplx", CASES)
def test_c2c_matches_oracle_every_order(gpu, orc, real, cplx):
    tol = TOL[np.dtype(real).name]
    for order in range(0, 15):  # order 0 is the identity (the reference itself is undefined there, see oracle dit2_v3)
        n = 1 << order
        batch = 5 if order < 12 else 2
        x = np.stack([orc.noise(n, 1 + b, cplx) for b in range(batch)])
        plan = gpu.FFTPlan(order, cplx)
        assert plan.size() == n and plan.order() == order
        for direction in (gpu.FORWARD, gpu.BACKWARD):
            got = plan(x.copy(), direction)
            assert rel_l2(got, orc.fft(x, direction)) <= tol, (order, direction)
        out = np.zeros_like(x)
        plan(x, gpu.FORWARD, out=out)  # out-of-place overload (fft/fft.hpp:63-71)
        assert rel_l2(out, orc.fft(x, -1)) <= tol
        plan.close()


@pytest.mark.parametrize("real,cplx", CASES)
def test_rfft_irfft_match_oracle_every_order(gpu, orc, real, cplx):
    tol = TOL[np.dtype(real).name]
    for order in range(1, 16):
        n = 1 << order
        batch = 5 if order < 12 else 2
        x = np.stack([orc.noise(n, 2 + b, real) for b in range(batch)])
        plan = gpu.RFFTPlan(order, real)
        want = orc.rfft(x)
        spec = plan.rfft(x)
        assert spec.shape == (batch, n // 2 + 1)
        assert rel_l2(spec, want) <= tol, order
        assert rel_l2(plan.irfft(want), orc.irfft(want, n)) <= tol, order
        plan.close()


@pytest.mark.parametrize("order,batch", [(13, 701), (14, 333), (14, 1201), (15, 301), (15, 610), (16, 151)])
def test_long_rfft_many_rows(gpu, orc, order, batch):
    # N = 2^13 / 2^14 (512-thread CTAs, two per SM): more rows than one wave of CTAs, odd and even rows (spectrum rows of N/2+1 bins
    # alternate between 16-byte aligned and not), and N-long spectrum rows on the way back.
    n = 1 << order
    x = np.stack([orc.noise(n, 2 + (b % 5), np.float32) * np.float32(1 + b % 3) for b in range(batch)])
    base = orc.rfft(x[:15])
    plan = gpu.RFFTPlan(order, np.float32)
    spec = plan.rfft(x)
    for b in range(batch):  # rows repeat with period 15 (5 seeds x 3 gains): every row is checked against the oracle
        assert rel_l2(spec[b], base[b % 15]) <= 1e-5, (order, b)
    back = plan.irfft(spec)
    assert rel_l2(back[:15], orc.irfft(base, n)) <= 1e-5
    assert rel_l2(back, x * np.float32(n)) <= 1e-5
    wide = np.zeros((batch, n), dtype=np.complex64)  # callers may hand N-long rows (overlap_save.hpp:57,107)
    wide[:, : n // 2 + 1] = spec
    assert np.array_equal(plan.irfft(wide), back)
    plan.close()


def test_golden_vectors_from_the_reference(gpu, golden):
    for tag, real, cplx in (("f32", np.float32, np.complex64), ("f64", np.float64, np.complex128)):
        tol = TOL[np.dtype(real).name]
        for order in (1, 2, 3, 4, 5, 8, 10, 11):
            n = 1 << order
            from oracle import pyoracle

            x = pyoracle.oracle().noise(n, 1, cplx)
            plan = gpu.FFTPlan(order, cplx)
            assert rel_l2(plan(x.copy(), -1), golden[f"c2c/{tag}/{order}/fwd"]) <= tol
            assert rel_l2(plan(x.copy(), +1), golden[f"c2c/{tag}/{order}/bwd"]) <= tol
            plan.close()
            rp = gpu.RFFTPlan(order, real)
            xr = pyoracle.oracle().noise(n, 2, real)
            assert rel_l2(rp.rfft(xr[None, :])[0], golden[f"r2c/{tag}/{order}"]) <= tol
            assert rel_l2(rp.irfft(golden[f"r2c/{tag}/{order}"][None, :].copy())[0], golden[f"c2r/{tag}/{order}"]) <= tol
            rp.close()
        # c2r semantics on junk spectra: Im X[0] / Im X[N/2] ignored, N-long rows accepted
        rp = gpu.RFFTPlan(6, real)
        junk = pyoracle.oracle().noise(64, 5, cplx)
        assert rel_l2(rp.irfft(junk[None, :33].copy())[0], golden[f"c2r_junk/{tag}/half"]) <= tol
        assert rel_l2(rp.irfft(junk[None, :].copy())[0], golden[f"c2r_junk/{tag}/full"]) <= tol
        rp.close()


def test_known_answers(gpu):
    # fft/rfft_test.cpp:170-186
    plan = gpu.FFTPlan(2, np.complex64)
    got = plan(np.array([1, 2, 3, 4], dtype=np.complex64), gpu.FORWARD)
    assert np.allclose(got, [10, -2 + 2j, -2, -2 - 2j], atol=1e-6)
    # delta -> all ones, both directions (rfft_test.cpp:132-168, dft_test.cpp:31-46; extra/python/test/test.py:12-19)
    for order in (1, 2, 5, 9, 12):
        for cplx in (np.complex64, np.complex128):
            x = np.zeros(1 << order, dtype=cplx)
            x[0] = 1
            p = gpu.FFTPlan(order, cplx)
            assert np.allclose(p(x.copy(), gpu.FORWARD), 1) and np.allclose(p(x.copy(), gpu.BACKWARD), 1)
            y = p(p(x.copy(), gpu.FORWARD), gpu.BACKWARD) / x.size
            assert np.allclose(y, x, atol=1e-6)
            p.close()
    # DCT-II of [1..8] through the c2c plan (fft/dct_test.cpp:23-39)
    x = np.arange(1, 9, dtype=np.float64)
    v = np.concatenate([x[0::2], x[1::2][::-1]]).astype(np.complex128)
    p = gpu.FFTPlan(3, np.complex128)
    V = p(v, gpu.FORWARD)
    dct = 2 * np.real(np.exp(-1j * np.pi * np.arange(8) / 16) * V)
    assert np.allclose(dct, [72.0, -25.76929209, 0.0, -2.6938192, 0.0, -0.80361161, 0.0, -0.20280929], atol=1e-6)


def test_plan_contract(gpu):
    # fft_test.cpp:53-130: size/order, throw past max_size, round trips in place / out of place / strided view
    assert gpu.FFTPlan.max_order() == 27 and gpu.FFTPlan.max_size() == 1 << 27
    with pytest.raises(RuntimeError):
        gpu.FFTPlan(gpu.next_order(gpu.FFTPlan.max_size() + 1))
    from oracle import pyoracle

    orc = pyoracle.oracle()
    for order in range(2, 15):
        for cplx, atol in ((np.complex64, 1e-5), (np.complex128, 1e-9)):  # algorithm/allclose.hpp:36-40
            n = 1 << order
            x = orc.noise(n, 99, cplx)
            p = gpu.FFTPlan(order, cplx)
            y = p(p(x.copy(), gpu.FORWARD), gpu.BACKWARD) / n
            assert np.allclose(y, x, atol=atol)
            mat = np.zeros((n, 2), dtype=cplx)  # stride-2 column view of a layout_left matrix (fft_test.cpp:114-128)
            mat[:, 1] = x
            p.strided(mat[:, 1], gpu.FORWARD)
            assert rel_l2(mat[:, 1], orc.fft(x, -1)) <= TOL[np.dtype(cplx).name]
            assert np.all(mat[:, 0] == 0)
            p.close()


def test_rfft_deinterleave_relation(gpu, orc):
    # fft/rfft_test.cpp:80-126: rfft(a), rfft(b) == deinterleave(fft(a + ib))
    for order in (4, 9, 13):
        n = 1 << order
        a, b = orc.noise(n, 3, np.float32), orc.noise(n, 4, np.float32)
        z = gpu.FFTPlan(order, np.complex64)((a + 1j * b).astype(np.complex64), gpu.FORWARD).astype(np.complex128)
        zc = np.conj(np.roll(z[::-1], 1))
        rp = gpu.RFFTPlan(order, np.float32)
        assert rel_l2(rp.rfft(a[None])[0], ((z + zc) / 2)[: n // 2 + 1]) < 1e-5
        assert rel_l2(rp.rfft(b[None])[0], ((z - zc) / 2j)[: n // 2 + 1]) < 1e-5


def test_large_and_ragged_batches(gpu, orc):
    # batch not a multiple of the transforms-per-CTA packing, and > 65535 transforms
    for order, batch in ((3, 7), (5, 33), (7, 70001)):
        n = 1 << order
        x = orc.noise(n * batch, 5, np.float32).reshape(batch, n)
        rp = gpu.RFFTPlan(order, np.float32)
        spec = rp.rfft(x)
        ref = np.fft.rfft(x.astype(np.float64), axis=1)
        assert rel_l2(spec, ref) < 1e-6
        assert rel_l2(rp.irfft(spec), x.astype(np.float64) * n) < 1e-6
        rp.close()


@pytest.mark.parametrize("order", [16, 18, 20])
def test_long_transforms_four_step(gpu, orc, order):
    # beyond the oracle's comfortable range for exhaustive checks: one oracle comparison + size-independent properties
    n = 1 << order
    x = orc.noise(n, 7, np.complex64)
    p = gpu.FFTPlan(order, np.complex64)
    X = p(x.copy(), gpu.FORWARD)
    assert rel_l2(X, orc.fft(x, -1)) <= 1e-5
    assert rel_l2(p(X.copy(), gpu.BACKWARD) / n, x) <= 1e-5          # round trip
    assert abs(np.vdot(X, X).real / n - np.vdot(x, x).real) / np.vdot(x, x).real < 1e-5  # Parseval
    y = orc.noise(n, 8, np.complex64)
    lin = p((2 * x + 3j * y).astype(np.complex64), gpu.FORWARD)
    assert rel_l2(lin, 2 * X.astype(np.complex128) + 3j * p(y.copy(), gpu.FORWARD).astype(np.complex128)) <= 1e-5
    p.close()
    xr = orc.noise(n, 9, np.float32)
    rp = gpu.RFFTPlan(order, np.float32)
    S = rp.rfft(xr[None])
    assert rel_l2(S[0], orc.rfft(xr)) <= 1e-5
    assert rel_l2(rp.irfft(S)[0] / n, xr) <= 1e-5
    rp.close()


@pytest.mark.parametrize("order", [14, 15, 16])
def test_long_rfft_device_rows_aligned_and_at_8_bytes(gpu, orc, order):
    # float N = 2^14 .. 2^16 has two forms, chosen by the alignment of the real rows: the wide kernels (fft_wide.cuh) need 16 bytes, rows
    # that are only 8-byte aligned take the cta_fft kernels (one 8192-point CTA, one 1024-thread CTA, two 2^14-point CTAs). Real rows
    # are read and written as complex pairs, so an offset of two floats is the smallest one a device array may have.
    import torch

    n, batch = 1 << order, 3
    x = np.stack([orc.noise(n, 40 + b, np.float32) for b in range(batch)])
    want = orc.rfft(x)
    plan = gpu.RFFTPlan(order, np.float32)
    plan.set_stream(torch.cuda.current_stream())
    spec = torch.from_numpy(want.astype(np.complex64)).cuda()
    for offset in (0, 2):
        rows = torch.empty(batch * n + offset, device="cuda")[offset:].view(batch, n)
        back = torch.empty(batch * n + offset, device="cuda")[offset:].view(batch, n)
        assert rows.data_ptr() % 16 == back.data_ptr() % 16 == 4 * offset
        rows.copy_(torch.from_numpy(x))
        got = plan.rfft(rows)
        plan.irfft(spec, out=back)
        torch.cuda.synchronize()
        assert rel_l2(got.cpu().numpy(), want) <= 1e-5, (order, offset)
        assert rel_l2(back.cpu().numpy(), orc.irfft(want, n)) <= 1e-5, (order, offset)
    plan.close()


@pytest.mark.parametrize("real,cplx", CASES)
def test_dft_plan_any_size_matches_oracle(gpu, orc, golden, real, cplx):
    # dft_plan == fallback_dft_plan (Bluestein, fft/fallback/fallback_dft_plan.hpp:24-96): the reference tests sizes 2..128/512
    # (fft/dft_test.cpp:24-26); here a spread of primes, composites and powers of two, batched, both directions
    tol = TOL[np.dtype(real).name]
    tag = "c64" if cplx == np.complex64 else "c128"
    for n in (2, 3, 5, 12, 21, 100, 127, 128):
        plan = gpu.DFTPlan(n, cplx)
        x = golden[f"dft/{tag}/{n}/x"]
        assert rel_l2(plan(x.copy(), gpu.FORWARD), golden[f"dft/{tag}/{n}/fwd"]) <= tol, n
        assert rel_l2(plan(x.copy(), gpu.BACKWARD), golden[f"dft/{tag}/{n}/bwd"]) <= tol, n
        plan.close()
    for n in (1, 7, 96, 255, 257, 1000, 4095, 4096, 4097, 10007):  # 4095 is the last padded size in the fused single-CTA form (float)
        batch = 3 if n < 5000 else 2
        x = np.stack([orc.noise(n, 5 + b, cplx) for b in range(batch)])
        plan = gpu.DFTPlan(n, cplx)
        assert plan.size() == n
        for direction in (gpu.FORWARD, gpu.BACKWARD):
            assert rel_l2(plan(x.copy(), direction), orc.dft(x, direction)) <= tol, (n, direction)
        out = np.zeros_like(x)
        plan(x, gpu.FORWARD, out=out)
        assert rel_l2(out, orc.dft(x, -1)) <= tol
        back = plan(out.copy(), gpu.BACKWARD)  # fft/dft_test.cpp:49-66: round trip gains a factor of size
        assert rel_l2(back / n, x) <= 10 * tol
        plan.close()
    # fft/dft_test.cpp:31-46: a unit impulse transforms to all ones
    for n in (2, 21, 127):
        x = np.zeros(n, dtype=cplx)
        x[0] = 1
        plan = gpu.DFTPlan(n, cplx)
        assert np.allclose(plan(x, gpu.FORWARD), np.ones(n), atol=1e-5 if real == np.float32 else 1e-12)
        plan.close()
    with pytest.raises(RuntimeError):
        gpu.DFTPlan(0, cplx)


@pytest.mark.parametrize("real", [np.float32, np.float64])
def test_dct2_plan_matches_oracle_and_scipy_known_answer(gpu, orc, golden, real):
    # fallback_dct2_plan (fft/dct.hpp:24-68); dct_test.cpp:24-39: scipy.fft.dct([1..8], type=2)
    tol = TOL[np.dtype(real).name]
    tag = "f32" if real == np.float32 else "f64"
    plan = gpu.DCT2Plan(3, real)
    assert plan.order() == 3 and plan.size() == 8
    got = plan(np.arange(1, 9, dtype=real))
    assert np.allclose(got, [72.0, -25.76929209, 0.0, -2.6938192, 0.0, -0.80361161, 0.0, -0.20280929], atol=2e-5 if real == np.float32 else 1e-7)
    plan.close()
    for order in (1, 3, 6, 10):
        plan = gpu.DCT2Plan(order, real)
        assert rel_l2(plan(golden[f"dct2/{tag}/{order}/x"].copy()), golden[f"dct2/{tag}/{order}/out"]) <= tol, order
        plan.close()
    for order in (0, 2, 5, 9, 12, 13, 14, 16):  # 14 and 16 leave the single-CTA range (float): pre / transform / post kernels
        n = 1 << order
        x = np.stack([orc.noise(n, 60 + b, real) for b in range(3 if order < 14 else 2)])
        plan = gpu.DCT2Plan(order, real)
        want = orc.dct2(x)
        assert rel_l2(plan(x.copy()), want) <= tol, order
        out = np.zeros_like(x)
        plan(x, out=out)
        assert rel_l2(out, want) <= tol
        plan.close()


@pytest.mark.parametrize("tag,real", [("f32", np.float32), ("f64", np.float64)])
def test_stft_matches_reference_golden_and_oracle(gpu, orc, golden, tag, real):
    # stft_plan (fft/stft.hpp:39-109): overlap, zero padding, hann / hamming / rectangular windows, ragged last frame
    import torch

    tol = TOL[np.dtype(real).name]
    kinds = {0: "rectangular", 1: "hann", 2: "hamming"}
    x = golden[f"stft/{tag}/x"]
    for frame, transform, overlap, win in ((256, 256, 128, 1), (128, 256, 0, 0), (100, 128, 30, 2), (64, 64, 48, 1), (256, 300, 17, 1)):
        want = golden[f"stft/{tag}/{frame}_{transform}_{overlap}_{win}"]
        got = gpu.stft(x, frame, transform, overlap, kinds[win])
        assert got.shape == want.shape
        assert rel_l2(got, want) <= tol, (frame, transform, overlap, win)
        assert gpu.num_stft_frames(x.shape[1], frame, overlap) == want.shape[1]
    # defaults of stft_plan(transform_size): frame = transform, half overlap, hann (stft.hpp:43-49; stft_test.cpp:33)
    assert rel_l2(gpu.stft(x, 256), golden[f"stft/{tag}/256_256_128_1"]) <= tol
    # larger, device-resident, many channels: oracle side by side
    xs = np.stack([orc.noise(20000, 30 + c, real) for c in range(5)])
    want = orc.stft(xs, 2048, 4096, 1536, 1)
    got = gpu.stft(torch.from_numpy(xs).cuda(), 2048, 4096, 1536, "hann")
    assert rel_l2(got.cpu().numpy(), want) <= tol
    # uniform_partition is the rectangular, no-overlap, transform = 2 * frame case
    head = np.ascontiguousarray(xs[:, :16384])
    assert rel_l2(gpu.stft(head, 1024, 2048, 0, "rectangular"), orc.uniform_partition(head, 1024)) <= tol
    with pytest.raises(RuntimeError):
        gpu.stft(x, 64, 64, 64)  # overlap must be smaller than the frame
    with pytest.raises(RuntimeError):
        gpu.stft(np.ascontiguousarray(x[:, :32]), 64)  # signal shorter than one frame


def test_dft_plan_device_buffers(gpu, orc):
    import torch

    n, batch = 1500, 64
    x = np.stack([orc.noise(n, 9 + b, np.complex64) for b in range(4)])
    xs = np.tile(x, (batch // 4, 1))
    plan = gpu.DFTPlan(n, np.complex64)
    plan.set_stream(torch.cuda.current_stream())
    dx = torch.from_numpy(xs).cuda()
    dy = torch.empty_like(dx)
    plan(dx, gpu.FORWARD, out=dy)
    torch.cuda.synchronize()
    want = orc.dft(x, -1)
    assert rel_l2(dy.cpu().numpy()[:4], want) <= 1e-5 and rel_l2(dy.cpu().numpy()[-4:], want) <= 1e-5
    plan.close()


def test_long_transform_f64(gpu, orc):
    order = 15
    x = orc.noise(1 << order, 7, np.complex128)
    p = gpu.FFTPlan(order, np.complex128)
    assert rel_l2(p(x.copy(), gpu.FORWARD), orc.fft(x, -1)) <= 1e-12
    xr = orc.noise(1 << order, 9, np.float64)
    rp = gpu.RFFTPlan(order, np.float64)
    S = rp.rfft(xr[None])
    assert rel_l2(S[0], orc.rfft(xr)) <= 1e-12
    assert rel_l2(rp.irfft(S)[0], orc.irfft(orc.rfft(xr), 1 << order)) <= 1e-12


def test_device_buffers_and_streams(gpu, orc):
    import torch

    x = np.stack([orc.noise(4096, 2 + b, np.float32) for b in range(16)])
    rp = gpu.RFFTPlan(12, np.float32)
    rp.set_stream(torch.cuda.current_stream())
    dx = torch.from_numpy(x).cuda()
    dspec = rp.rfft(dx)
    torch.cuda.synchronize()
    assert rel_l2(dspec.cpu().numpy(), orc.rfft(x)) <= 1e-5
    back = rp.irfft(dspec)
    torch.cuda.synchronize()
    assert rel_l2(back.cpu().numpy() / 4096, x) <= 1e-5


def test_python_front_end(gpu):
    # extra/python/test/test.py:12-19
    for n in (4, 64, 4096):
        for dt in (np.complex64, np.complex128):
            x = np.zeros(n, dtype=dt)
            x[0] = 1
            y = gpu.ifft(gpu.fft(x))
            assert y.shape == (n,) and np.allclose(y, x, atol=1e-6)
    with pytest.raises(RuntimeError):
        gpu.fft(np.zeros(12, dtype=np.complex64))  # non power of two (main.cpp:137-139)


@pytest.mark.parametrize("order", [10, 13, 16])
def test_baseline_config2_full_batch_properties(gpu, order):
    # BASELINE config 2 at its full size (batch = 2^29/N, 2 GiB in): size-independent properties on the device --
    # unnormalised round trip gains N, Parseval with the Hermitian weights, DC bin = row sum
    import torch

    n = 1 << order
    batch = (1 << 29) // n
    gen = torch.Generator(device="cuda").manual_seed(2)
    x = torch.rand((batch, n), device="cuda", generator=gen) * 2 - 1
    plan = gpu.RFFTPlan(order, "float32")
    plan.set_stream(torch.cuda.current_stream())
    spec = plan.rfft(x)
    back = plan.irfft(spec)
    torch.cuda.synchronize()
    err = (back / n - x).double().norm() / x.double().norm()
    assert float(err) <= 1e-5
    power = spec.abs().double().square()
    weights = torch.full((n // 2 + 1,), 2.0, device="cuda", dtype=torch.float64)
    weights[0] = weights[-1] = 1.0
    lhs = (power * weights).sum(dim=1) / n
    rhs = x.double().square().sum(dim=1)
    assert float(((lhs - rhs).abs() / rhs).max()) < 1e-5
    assert float((spec[:, 0].real.double() - x.double().sum(dim=1)).abs().max()) < 1e-2
    assert float(spec[:, 0].imag.abs().max()) == 0.0 and float(spec[:, -1].imag.abs().max()) == 0.0
    plan.close()


def test_split_complex_plan(gpu, orc, golden):
    # neo::fft::split_fft_plan (fft/split_fft_test.cpp:23-73: round trips in place / copy) + parity with the reference's planes
    import torch

    for tag, real, cplx in (("f32", np.float32, np.complex64), ("f64", np.float64, np.complex128)):
        tol = TOL[np.dtype(real).name]
        for order in (1, 4, 8, 11):
            x = orc.noise(1 << order, 1, cplx)
            plan = gpu.FFTPlan(order, cplx)
            for d, name in ((gpu.FORWARD, "fwd"), (gpu.BACKWARD, "bwd")):
                re, im = plan.split(np.ascontiguousarray(x.real), np.ascontiguousarray(x.imag), d)
                want = golden[f"split/{tag}/{order}/{name}"]
                assert rel_l2(re + 1j * im, want[0] + 1j * want[1]) <= tol, (tag, order, name)
            re, im = plan.split(np.ascontiguousarray(x.real), np.ascontiguousarray(x.imag), gpu.FORWARD)
            re, im = plan.split(re, im, gpu.BACKWARD)
            assert rel_l2((re + 1j * im) / x.size, x) <= tol
            plan.close()
    # batched planes on the device, and a size beyond one CTA (interleaved scratch path)
    for order, batch in ((10, 64), (15, 3)):
        x = np.stack([orc.noise(1 << order, 5 + b, np.complex64) for b in range(batch)])
        plan = gpu.FFTPlan(order, np.complex64)
        plan.set_stream(torch.cuda.current_stream())
        re, im = torch.from_numpy(np.ascontiguousarray(x.real)).cuda(), torch.from_numpy(np.ascontiguousarray(x.imag)).cuda()
        plan.split(re, im, gpu.FORWARD)
        torch.cuda.synchronize()
        got = re.cpu().numpy() + 1j * im.cpu().numpy()
        assert rel_l2(got, orc.fft(x, -1)) <= 1e-5, order
        plan.close()
