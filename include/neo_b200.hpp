// neo_b200.hpp -- C++ facade over the C ABI (neo_b200.h) that satisfies the reference's plan / convolver duck types, so the
// B200 backend can sit behind neo's compile-time aliases exactly like its IPP / MKL / vDSP backends do
// (src/neo/fft/fft.hpp:36-52, src/neo/fft/rfft.hpp:15-23, src/neo/convolution/dense_convolver.hpp:20-25; see INTEGRATION.md).
//
// The classes are templates over "any rank-1 / rank-2 view with the mdspan interface" (data_handle(), extent(i), stride(i)):
// Kokkos::mdspan (what neo uses), std::mdspan and cuda::std::mdspan all qualify, and so does the tiny span in the tests.
// Contiguous views go straight to the library; strided ones are staged through a contiguous buffer, the pattern of
// src/neo/fft/backend/ipp.hpp:150-158. Construction failures throw std::runtime_error like c2c_dit2_plan.hpp:98-104.
//
// Host code only: no CUDA headers are needed to compile against this file.
#pragma once

#include "neo_b200.h"

#include <cmath>
#include <complex>
#include <cstddef>
#include <cstdint>
#include <algorithm>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

namespace neo::b200 {

namespace detail {

template<typename Float>
inline constexpr int dtype_of = std::is_same_v<Float, double> ? NEO_B200_F64 : NEO_B200_F32;

inline auto check(int status) -> void
{
    if (status != NEO_B200_OK) { throw std::runtime_error{std::string{"neo_b200: "} + neo_b200_last_error()}; }
}

// neo::fft::direction is `enum struct direction : int { forward = -1, backward = 1 }` (fft/direction.hpp:8-12); any enum or
// integer with those values is accepted so that this header does not depend on neo's.
template<typename Direction>
constexpr auto direction_value(Direction dir) noexcept -> int
{
    return static_cast<int>(dir) < 0 ? NEO_B200_FORWARD : NEO_B200_BACKWARD;
}

template<typename Complex>
using real_of = typename Complex::value_type;

template<typename View>
using element_of = std::remove_cv_t<typename View::element_type>;

template<typename View>
auto is_contiguous(View const& v) noexcept -> bool
{
    return v.extent(0) <= 1 || v.stride(0) == 1;
}

}  // namespace detail

/// neo::fft::from_order_tag look-alike (fft/order.hpp:17-25); any tag type is accepted by the constructors.
struct from_order_tag
{
    explicit from_order_tag() = default;
};
inline constexpr auto from_order = from_order_tag{};

namespace detail {
/// hann_window (math/windowing.hpp:27-41), evaluated in double and rounded by the caller
struct hann
{
    auto operator()(std::size_t index, std::size_t size) const noexcept -> double
    {
        return 0.5 * (1.0 - std::cos(2.0 * 3.14159265358979323846 * static_cast<double>(index) / static_cast<double>(size - 1)));
    }
};
}  // namespace detail

/// Drop-in for neo::fft::fft_plan<Complex> (fft/reference/c2c_dit2_plan.hpp:22-104): in-place `plan(x, dir)`, unnormalised,
/// plus the optional out-of-place overload that fft/fft.hpp:63-71 looks for. Complex = std::complex<T> or
/// neo::scalar_complex<T> (both interleaved [re, im]).
template<typename Complex>
struct fft_plan
{
    using value_type = Complex;
    using size_type  = std::size_t;
    using real_type  = detail::real_of<Complex>;

    template<typename Tag>
    fft_plan(Tag /*from_order*/, size_type order)
    {
        detail::check(neo_b200_fft_plan_create(&_plan, order, detail::dtype_of<real_type>));
    }

    fft_plan(fft_plan const&)                    = delete;
    auto operator=(fft_plan const&) -> fft_plan& = delete;
    fft_plan(fft_plan&& other) noexcept : _plan{std::exchange(other._plan, nullptr)}, _staging{std::move(other._staging)} {}
    auto operator=(fft_plan&& other) noexcept -> fft_plan&
    {
        std::swap(_plan, other._plan);
        std::swap(_staging, other._staging);
        return *this;
    }
    ~fft_plan() { neo_b200_fft_plan_destroy(_plan); }

    [[nodiscard]] static constexpr auto max_order() noexcept -> size_type { return 27; }  // c2c_dit2_plan.hpp:59-62
    [[nodiscard]] static constexpr auto max_size() noexcept -> size_type { return size_type(1) << max_order(); }

    [[nodiscard]] auto order() const noexcept -> size_type { return neo_b200_fft_plan_order(_plan); }
    [[nodiscard]] auto size() const noexcept -> size_type { return neo_b200_fft_plan_size(_plan); }

    template<typename Vec, typename Direction>
    auto operator()(Vec x, Direction dir) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Vec>, Complex>);
        auto const d = detail::direction_value(dir);
        if (detail::is_contiguous(x)) {
            detail::check(neo_b200_fft_exec(_plan, x.data_handle(), x.data_handle(), 1, d, NEO_B200_HOST));
        } else {
            auto const s = static_cast<std::ptrdiff_t>(x.stride(0));
            detail::check(neo_b200_fft_exec_strided(_plan, x.data_handle(), s, x.data_handle(), s, d));
        }
    }

    template<typename InVec, typename OutVec, typename Direction>
    auto operator()(InVec in, OutVec out, Direction dir) -> void
    {
        auto const d = detail::direction_value(dir);
        if (detail::is_contiguous(in) && detail::is_contiguous(out)) {
            detail::check(neo_b200_fft_exec(_plan, in.data_handle(), out.data_handle(), 1, d, NEO_B200_HOST));
        } else {
            detail::check(neo_b200_fft_exec_strided(_plan, in.data_handle(), static_cast<std::ptrdiff_t>(in.stride(0)),
                                                    out.data_handle(), static_cast<std::ptrdiff_t>(out.stride(0)), d));
        }
    }

    /// batched extension: `batch` contiguous transforms [batch][size()], host or device memory
    auto batched(Complex const* in, Complex* out, size_type batch, int direction, int memspace = NEO_B200_HOST) -> void
    {
        detail::check(neo_b200_fft_exec(_plan, in, out, batch, direction, memspace));
    }

private:
    neo_b200_fft_plan* _plan{nullptr};
    std::vector<Complex> _staging;
};

/// Drop-in for neo::fft::dft_plan<Complex> == fallback_dft_plan (fft/dft.hpp:28-30, fft/fallback/fallback_dft_plan.hpp:24-96):
/// complex transform of ANY size (Bluestein), `explicit Plan(size)`, in-place `plan(x, dir)`, unnormalised both ways.
template<typename Complex>
struct dft_plan
{
    using value_type = Complex;
    using size_type  = std::size_t;
    using real_type  = detail::real_of<Complex>;

    explicit dft_plan(size_type size) { detail::check(neo_b200_dft_plan_create(&_plan, size, detail::dtype_of<real_type>)); }

    dft_plan(dft_plan const&)                    = delete;
    auto operator=(dft_plan const&) -> dft_plan& = delete;
    dft_plan(dft_plan&& other) noexcept : _plan{std::exchange(other._plan, nullptr)} {}
    auto operator=(dft_plan&& other) noexcept -> dft_plan&
    {
        std::swap(_plan, other._plan);
        return *this;
    }
    ~dft_plan() { neo_b200_dft_plan_destroy(_plan); }

    [[nodiscard]] auto size() const noexcept -> size_type { return neo_b200_dft_plan_size(_plan); }

    template<typename Vec, typename Direction>
    auto operator()(Vec x, Direction dir) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Vec>, Complex>);
        auto const d = detail::direction_value(dir);
        if (detail::is_contiguous(x)) {
            detail::check(neo_b200_dft_exec(_plan, x.data_handle(), x.data_handle(), 1, d, NEO_B200_HOST));
        } else {  // strided view: staged like backend/ipp.hpp:150-158
            auto const n = static_cast<size_type>(x.extent(0));
            _staging.resize(n);
            for (size_type i = 0; i < n; ++i) { _staging[i] = x[i]; }
            detail::check(neo_b200_dft_exec(_plan, _staging.data(), _staging.data(), 1, d, NEO_B200_HOST));
            for (size_type i = 0; i < n; ++i) { x[i] = _staging[i]; }
        }
    }

    /// batched extension: `batch` contiguous transforms [batch][size()], host or device memory
    auto batched(Complex const* in, Complex* out, size_type batch, int direction, int memspace = NEO_B200_HOST) -> void
    {
        detail::check(neo_b200_dft_exec(_plan, in, out, batch, direction, memspace));
    }

private:
    neo_b200_dft_plan* _plan{nullptr};
    std::vector<Complex> _staging;
};

/// neo::fft::stft_plan<Float> (fft/stft.hpp:39-109) on the device. The reference returns an owning rank-3 mdarray; this facade stays
/// container-agnostic: `frames(len)`, `bins()`, then `operator()(x, channels, len, out)` fills out [channels][frames][bins].
/// INTEGRATION.md shows the three-line wrapper that gives neo::fft::stft_plan::operator() back its signature.
template<typename Float>
struct stft_plan
{
    using size_type    = std::size_t;
    using complex_type = std::complex<Float>;

    /// stft_plan(transform_size) (stft.hpp:43-49): frame = transform, half overlap, hann window
    explicit stft_plan(size_type transform_size) : stft_plan(transform_size, transform_size, transform_size / 2) {}

    /// window(index, size) as in stft_options::window; default hann_window (math/windowing.hpp:27-41)
    template<typename Window = detail::hann>
    stft_plan(size_type frame_size, size_type transform_size, size_type overlap_size, Window window = {})
        : _frame{frame_size}, _transform{transform_size}, _overlap{overlap_size}
    {
        auto n = size_type(1);
        while (n < transform_size) { n *= 2; }
        _window.resize(n);
        for (size_type i = 0; i < n; ++i) { _window[i] = static_cast<Float>(window(i, n)); }  // fill_window, windowing.hpp:61-67
    }

    [[nodiscard]] auto bins() const noexcept -> size_type { return _window.size() / 2 + 1; }
    [[nodiscard]] auto frames(size_type signal_size) const noexcept -> size_type
    {
        return neo_b200_num_stft_frames(signal_size, _frame, _overlap);
    }

    auto operator()(Float const* x, size_type channels, size_type len, complex_type* out, int memspace = NEO_B200_HOST) -> void
    {
        if (memspace != NEO_B200_HOST) { throw std::invalid_argument{"stft_plan: the window lives in host memory; use neo_b200_stft directly"}; }
        detail::check(neo_b200_stft(x, channels, len, _frame, _transform, _overlap, _window.data(), out, detail::dtype_of<Float>, memspace));
    }

private:
    size_type _frame, _transform, _overlap;
    std::vector<Float> _window;
};

/// Drop-in for neo::fft::fallback_dct2_plan<Float> (fft/dct.hpp:24-68): `Plan{from_order, order}`, in-place `plan(x)`.
template<typename Float>
struct dct2_plan
{
    using value_type = Float;
    using size_type  = std::size_t;

    template<typename Tag>
    dct2_plan(Tag /*from_order*/, size_type order)
    {
        detail::check(neo_b200_dct2_plan_create(&_plan, order, detail::dtype_of<Float>));
    }

    dct2_plan(dct2_plan const&)                    = delete;
    auto operator=(dct2_plan const&) -> dct2_plan& = delete;
    dct2_plan(dct2_plan&& other) noexcept : _plan{std::exchange(other._plan, nullptr)} {}
    auto operator=(dct2_plan&& other) noexcept -> dct2_plan&
    {
        std::swap(_plan, other._plan);
        return *this;
    }
    ~dct2_plan() { neo_b200_dct2_plan_destroy(_plan); }

    [[nodiscard]] auto order() const noexcept -> size_type { return neo_b200_dct2_plan_order(_plan); }
    [[nodiscard]] auto size() const noexcept -> size_type { return neo_b200_dct2_plan_size(_plan); }

    template<typename Vec>
    auto operator()(Vec x) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Vec>, Float>);
        if (detail::is_contiguous(x)) {
            detail::check(neo_b200_dct2_exec(_plan, x.data_handle(), x.data_handle(), 1, NEO_B200_HOST));
        } else {
            auto const n = static_cast<size_type>(x.extent(0));
            _staging.resize(n);
            for (size_type i = 0; i < n; ++i) { _staging[i] = x[i]; }
            detail::check(neo_b200_dct2_exec(_plan, _staging.data(), _staging.data(), 1, NEO_B200_HOST));
            for (size_type i = 0; i < n; ++i) { x[i] = _staging[i]; }
        }
    }

    /// batched extension: `batch` contiguous rows [batch][size()], host or device memory
    auto batched(Float const* in, Float* out, size_type batch, int memspace = NEO_B200_HOST) -> void
    {
        detail::check(neo_b200_dct2_exec(_plan, in, out, batch, memspace));
    }

private:
    neo_b200_dct2_plan* _plan{nullptr};
    std::vector<Float> _staging;
};

/// Drop-in for neo::fft::split_fft_plan<Float> (fft/fallback/fallback_split_fft_plan.hpp:16-137): operates on any aggregate with
/// `.real` / `.imag` rank-1 views (neo::split_complex, complex/split_complex.hpp:10).
template<typename Float>
struct split_fft_plan
{
    using value_type = Float;
    using size_type  = std::size_t;

    template<typename Tag>
    split_fft_plan(Tag /*from_order*/, size_type order)
    {
        detail::check(neo_b200_fft_plan_create(&_plan, order, detail::dtype_of<Float>));
    }
    split_fft_plan(split_fft_plan const&)                    = delete;
    auto operator=(split_fft_plan const&) -> split_fft_plan& = delete;
    split_fft_plan(split_fft_plan&& other) noexcept : _plan{std::exchange(other._plan, nullptr)} {}
    ~split_fft_plan() { neo_b200_fft_plan_destroy(_plan); }

    [[nodiscard]] auto order() const noexcept -> size_type { return neo_b200_fft_plan_order(_plan); }
    [[nodiscard]] auto size() const noexcept -> size_type { return neo_b200_fft_plan_size(_plan); }

    template<typename Split, typename Direction>
    auto operator()(Split x, Direction dir) -> void
    {
        (*this)(x, x, dir);
    }

    template<typename SplitIn, typename SplitOut, typename Direction>
    auto operator()(SplitIn in, SplitOut out, Direction dir) -> void
    {
        auto const n = size();
        auto gather  = [n](auto view, std::vector<Float>& tmp) -> Float const* {
            if (detail::is_contiguous(view)) { return view.data_handle(); }
            tmp.resize(n);
            for (size_type i = 0; i < n; ++i) { tmp[i] = view[i]; }
            return tmp.data();
        };
        Float const* re = gather(in.real, _re_in);
        Float const* im = gather(in.imag, _im_in);
        bool const direct = detail::is_contiguous(out.real) && detail::is_contiguous(out.imag);
        _re_out.resize(direct ? 0 : n);
        _im_out.resize(direct ? 0 : n);
        Float* ro = direct ? out.real.data_handle() : _re_out.data();
        Float* io = direct ? out.imag.data_handle() : _im_out.data();
        detail::check(neo_b200_fft_exec_split(_plan, re, im, ro, io, 1, detail::direction_value(dir), NEO_B200_HOST));
        if (!direct) {
            for (size_type i = 0; i < n; ++i) {
                out.real[i] = _re_out[i];
                out.imag[i] = _im_out[i];
            }
        }
    }

private:
    neo_b200_fft_plan* _plan{nullptr};
    std::vector<Float> _re_in, _im_in, _re_out, _im_out;
};

/// Drop-in for neo::fft::rfft_plan<Float, Complex> (fft/fallback/fallback_rfft_plan.hpp:15-61): two call operators told apart
/// by element type, real -> complex (N/2+1 bins written) and complex -> real (unnormalised).
template<typename Float, typename Complex = std::complex<Float>>
struct rfft_plan
{
    using real_type    = Float;
    using complex_type = Complex;
    using size_type    = std::size_t;

    template<typename Tag>
    rfft_plan(Tag /*from_order*/, size_type order)
    {
        detail::check(neo_b200_rfft_plan_create(&_plan, order, detail::dtype_of<Float>));
    }

    rfft_plan(rfft_plan const&)                    = delete;
    auto operator=(rfft_plan const&) -> rfft_plan& = delete;
    rfft_plan(rfft_plan&& other) noexcept
        : _plan{std::exchange(other._plan, nullptr)}
        , _real{std::move(other._real)}
        , _cplx{std::move(other._cplx)}
    {}
    auto operator=(rfft_plan&& other) noexcept -> rfft_plan&
    {
        std::swap(_plan, other._plan);
        std::swap(_real, other._real);
        std::swap(_cplx, other._cplx);
        return *this;
    }
    ~rfft_plan() { neo_b200_rfft_plan_destroy(_plan); }

    [[nodiscard]] auto order() const noexcept -> size_type { return neo_b200_rfft_plan_order(_plan); }
    [[nodiscard]] auto size() const noexcept -> size_type { return neo_b200_rfft_plan_size(_plan); }

    template<typename InVec, typename OutVec>
        requires(std::is_same_v<detail::element_of<InVec>, Float> && std::is_same_v<detail::element_of<OutVec>, Complex>)
    auto operator()(InVec in, OutVec out) -> void
    {
        auto const n    = size();
        auto const bins = n / 2 + 1;
        Float const* src = in.data_handle();
        if (!detail::is_contiguous(in)) {
            _real.resize(n);
            for (size_type i = 0; i < n; ++i) { _real[i] = in[i]; }
            src = _real.data();
        }
        if (detail::is_contiguous(out)) {
            detail::check(neo_b200_rfft_exec(_plan, src, out.data_handle(), 1, NEO_B200_HOST));
        } else {
            _cplx.resize(bins);
            detail::check(neo_b200_rfft_exec(_plan, src, _cplx.data(), 1, NEO_B200_HOST));
            for (size_type i = 0; i < bins; ++i) { out[i] = _cplx[i]; }
        }
    }

    template<typename InVec, typename OutVec>
        requires(std::is_same_v<detail::element_of<InVec>, Complex> && std::is_same_v<detail::element_of<OutVec>, Float>)
    auto operator()(InVec in, OutVec out) -> void
    {
        auto const n    = size();
        auto const bins = n / 2 + 1;
        Complex const* src = in.data_handle();
        auto row          = static_cast<size_type>(in.extent(0));  // callers may hand N bins (overlap_save.hpp:57,107)
        if (!detail::is_contiguous(in)) {
            _cplx.resize(bins);
            for (size_type i = 0; i < bins; ++i) { _cplx[i] = in[i]; }
            src = _cplx.data();
            row = bins;
        }
        if (detail::is_contiguous(out)) {
            detail::check(neo_b200_irfft_exec(_plan, src, row, out.data_handle(), 1, NEO_B200_HOST));
        } else {
            _real.resize(n);
            detail::check(neo_b200_irfft_exec(_plan, src, row, _real.data(), 1, NEO_B200_HOST));
            for (size_type i = 0; i < n; ++i) { out[i] = _real[i]; }
        }
    }

    /// batched extensions: [batch][N] reals <-> [batch][N/2+1] complex, host or device memory
    auto rfft_batched(Float const* in, Complex* out, size_type batch, int memspace = NEO_B200_HOST) -> void
    {
        detail::check(neo_b200_rfft_exec(_plan, in, out, batch, memspace));
    }
    auto irfft_batched(Complex const* in, size_type row_len, Float* out, size_type batch, int memspace = NEO_B200_HOST) -> void
    {
        detail::check(neo_b200_irfft_exec(_plan, in, row_len, out, batch, memspace));
    }

private:
    neo_b200_rfft_plan* _plan{nullptr};
    std::vector<Float> _real;
    std::vector<Complex> _cplx;
};

/// neo::convolution::uniform_partition (convolution/uniform_partition.hpp:13-26): ir[C][L] -> [C][P][B+1] into `out`
template<typename Float>
inline auto uniform_partition(Float const* ir, std::size_t channels, std::size_t taps, std::size_t block, std::complex<Float>* out)
    -> std::size_t
{
    detail::check(neo_b200_uniform_partition(ir, channels, taps, block, out, detail::dtype_of<Float>, NEO_B200_HOST));
    return neo_b200_num_partitions(taps, block);
}

/// A bank of partitioned convolvers: what one GPU handle really is. `filter` takes H[outputs][P][B+1]
/// (or [outputs][inputs][P][B+1] for the matrix topology); `process` runs T blocks for every channel.
template<typename Float, int Kind>
struct convolver_bank
{
    using real_type    = Float;
    using complex_type = std::complex<Float>;
    using size_type    = std::size_t;

    convolver_bank() = default;
    convolver_bank(convolver_bank const&)                    = delete;
    auto operator=(convolver_bank const&) -> convolver_bank& = delete;
    convolver_bank(convolver_bank&& other) noexcept : _conv{std::exchange(other._conv, nullptr)}, _cfg{other._cfg} {}
    auto operator=(convolver_bank&& other) noexcept -> convolver_bank&
    {
        std::swap(_conv, other._conv);
        std::swap(_cfg, other._cfg);
        return *this;
    }
    ~convolver_bank() { neo_b200_conv_destroy(_conv); }

    auto filter(complex_type const* h, size_type outputs, size_type inputs, size_type partitions, size_type bins, int topology,
                size_type max_blocks = 1, int memspace = NEO_B200_HOST, size_type frame_blocks = 0) -> void
    {
        neo_b200_conv_destroy(std::exchange(_conv, nullptr));
        _cfg            = neo_b200_conv_config{};
        _cfg.kind       = Kind;
        _cfg.dtype      = detail::dtype_of<Float>;
        _cfg.topology   = topology;
        _cfg.outputs    = outputs;
        _cfg.inputs     = inputs;
        _cfg.block      = bins - 1;
        _cfg.partitions = partitions;
        _cfg.max_blocks = frame_blocks != 0 ? frame_blocks : max_blocks;
        _cfg.frame_blocks = frame_blocks;  // T > 0: calls of exactly T blocks, second overlap-save level along block time
        detail::check(neo_b200_conv_create(&_conv, &_cfg));
        detail::check(neo_b200_conv_set_filter(_conv, h, memspace));
    }

    /// diagonal bank with sparse filters: the CSR matrices of neo::csr_matrix (csr_matrix.hpp:64-98), see neo_b200_conv_set_filter_csr
    auto filter_csr(complex_type const* values, std::uint64_t const* cols, std::uint64_t const* row_ptr, std::uint64_t const* filter_base,
                    size_type outputs, size_type partitions, size_type bins, size_type max_blocks = 1) -> void
    {
        neo_b200_conv_destroy(std::exchange(_conv, nullptr));
        _cfg            = neo_b200_conv_config{};
        _cfg.kind       = Kind;
        _cfg.dtype      = detail::dtype_of<Float>;
        _cfg.topology   = NEO_B200_DIAGONAL;
        _cfg.outputs    = outputs;
        _cfg.inputs     = outputs;
        _cfg.block      = bins - 1;
        _cfg.partitions = partitions;
        _cfg.max_blocks = max_blocks;
        detail::check(neo_b200_conv_create(&_conv, &_cfg));
        detail::check(neo_b200_conv_set_filter_csr(_conv, values, cols, row_ptr, filter_base));
    }

    auto process(Float const* in, Float* out, size_type blocks, int memspace = NEO_B200_HOST) -> void
    {
        detail::check(neo_b200_conv_process(_conv, in, out, blocks, memspace));
    }

    /// a second filter next to the current one, in filter()'s layout (stage_filter) or as impulse responses [outputs][(inputs)][taps]
    /// (stage_impulse, zero-padded when shorter); no output or state changes. `crossfade(fade, delay)` then fades to it linearly over
    /// `fade` samples from `delay` samples after the last one delivered, keeping the delay line, and returns the fade's first sample
    /// (neo_b200_conv_stage_filter / _stage_impulse / _crossfade; overlap-save banks)
    auto stage_filter(complex_type const* h, int memspace = NEO_B200_HOST) -> void { detail::check(neo_b200_conv_stage_filter(_conv, h, memspace)); }
    auto stage_impulse(Float const* ir, size_type taps, int memspace = NEO_B200_HOST) -> void
    {
        detail::check(neo_b200_conv_stage_impulse(_conv, ir, taps, memspace));
    }
    auto crossfade(size_type fade, size_type delay = 0) -> size_type
    {
        size_type start = 0;
        detail::check(neo_b200_conv_crossfade(_conv, delay, fade, &start));
        return start;
    }

    [[nodiscard]] auto block_size() const noexcept -> size_type { return _cfg.block; }
    [[nodiscard]] auto partitions() const noexcept -> size_type { return _cfg.partitions; }
    [[nodiscard]] auto device_bytes() const noexcept -> size_type { return neo_b200_conv_device_bytes(_conv); }
    [[nodiscard]] auto handle() const noexcept -> neo_b200_conv* { return _conv; }

private:
    neo_b200_conv* _conv{nullptr};
    neo_b200_conv_config _cfg{};
};

/// The same bank spread over several GPUs of one box (neo_b200_bank_*): what a host that builds one convolver per channel on N
/// threads (extra/cli/src/convolver.cpp:37-40) does with N devices instead. `layout` = {channel groups, partition shards}; channels
/// (matrix topology: outputs) and inputs must be multiples of the number of devices. `impulse` takes the impulse responses of the
/// WHOLE bank ([channels][taps] or [outputs][inputs][taps], host memory) and hands every device its group's rows; `process` takes
/// whole [inputs][T*B] / [outputs][T*B] host arrays; `submit` + `wait` keep up to three calls in flight (pinned memory recommended).
template<typename Float, int Kind>
struct multi_gpu_bank
{
    using size_type = std::size_t;

    multi_gpu_bank() = default;
    multi_gpu_bank(multi_gpu_bank const&)                    = delete;
    auto operator=(multi_gpu_bank const&) -> multi_gpu_bank& = delete;
    ~multi_gpu_bank() { neo_b200_bank_destroy(_bank); }

    auto create(std::vector<int> const& devices, neo_b200_bank_layout layout, int topology, size_type outputs, size_type inputs,
                size_type block, size_type partitions, size_type max_blocks = 1, size_type frame_blocks = 0) -> void
    {
        neo_b200_bank_destroy(std::exchange(_bank, nullptr));
        _cfg              = neo_b200_conv_config{};
        _cfg.kind         = Kind;
        _cfg.dtype        = detail::dtype_of<Float>;
        _cfg.topology     = topology;
        _cfg.outputs      = outputs;
        _cfg.inputs       = topology == NEO_B200_DIAGONAL ? outputs : inputs;
        _cfg.block        = block;
        _cfg.partitions   = partitions;
        _cfg.max_blocks   = frame_blocks != 0 ? frame_blocks : max_blocks;
        _cfg.frame_blocks = frame_blocks;
        detail::check(neo_b200_bank_create(&_bank, &_cfg, &layout, devices.data(), devices.size()));
        _ranks.resize(devices.size());
        for (size_type l = 0; l < _ranks.size(); ++l) { detail::check(neo_b200_bank_local_rank(_bank, l, &_ranks[l])); }
    }

    /// `convolver.filter(uniform_partition(ir, block))` for every convolver of the bank, partitioned on the devices
    auto impulse(Float const* ir, size_type taps) -> void
    {
        size_type const row = (_cfg.topology == NEO_B200_MATRIX ? _cfg.inputs : 1) * taps;  // reals per output / channel
        auto ptrs           = std::vector<void const*>(_ranks.size());
        for (size_type l = 0; l < _ranks.size(); ++l) { ptrs[l] = ir + _ranks[l].group_first * row; }
        detail::check(neo_b200_bank_set_impulse(_bank, ptrs.data(), taps, NEO_B200_HOST));
    }

    auto submit(Float const* in, Float* out, size_type blocks) -> void
    {
        size_type const pitch = blocks * _cfg.block;
        auto ins              = std::vector<void const*>(_ranks.size());
        auto outs             = std::vector<void*>(_ranks.size());
        for (size_type l = 0; l < _ranks.size(); ++l) {
            ins[l]  = in + _ranks[l].in_first * pitch;
            outs[l] = out + _ranks[l].out_first * pitch;
        }
        detail::check(neo_b200_bank_submit(_bank, ins.data(), outs.data(), blocks, NEO_B200_HOST));
    }
    auto wait() -> void { detail::check(neo_b200_bank_wait(_bank)); }
    auto process(Float const* in, Float* out, size_type blocks) -> void
    {
        submit(in, out, blocks);
        for (int i = 0; i < 3; ++i) { wait(); }
    }
    auto reset() -> void { detail::check(neo_b200_bank_reset(_bank)); }

    [[nodiscard]] auto ranks() const noexcept -> std::vector<neo_b200_bank_rank_info> const& { return _ranks; }
    [[nodiscard]] auto handle() const noexcept -> neo_b200_bank* { return _bank; }

private:
    neo_b200_bank* _bank{nullptr};
    neo_b200_conv_config _cfg{};
    std::vector<neo_b200_bank_rank_info> _ranks;
};

/// Drop-in for neo::convolution::fft_convolver<Float> (convolution/fft_convolver.hpp:18-93): `fft_convolver{signal_size, patch_size}`,
/// `convolver(signal, patch, output)` with output_size() = signal_size + patch_size - 1 (mode::full).
template<typename Float>
struct fft_convolver
{
    using size_type = std::size_t;

    fft_convolver(size_type signal_size, size_type patch_size) : _signal{signal_size}, _patch{patch_size}
    {
        detail::check(neo_b200_fft_convolver_create(&_conv, signal_size, patch_size, detail::dtype_of<Float>));
    }
    fft_convolver(fft_convolver const&)                    = delete;
    auto operator=(fft_convolver const&) -> fft_convolver& = delete;
    ~fft_convolver() { neo_b200_fft_convolver_destroy(_conv); }

    [[nodiscard]] auto signal_size() const noexcept -> size_type { return _signal; }
    [[nodiscard]] auto patch_size() const noexcept -> size_type { return _patch; }
    [[nodiscard]] auto output_size() const noexcept -> size_type { return neo_b200_fft_convolver_output_size(_conv); }

    template<typename Signal, typename Patch, typename Output>
    auto operator()(Signal signal, Patch patch, Output output) -> void
    {
        _a.resize(_signal);
        _b.resize(_patch);
        _c.resize(output_size());
        for (size_type i = 0; i < _signal; ++i) { _a[i] = static_cast<Float>(signal[i]); }
        for (size_type i = 0; i < _patch; ++i) { _b[i] = static_cast<Float>(patch[i]); }
        detail::check(neo_b200_fft_convolver_exec(_conv, _a.data(), _b.data(), _c.data(), 1, NEO_B200_HOST));
        for (size_type i = 0; i < _c.size(); ++i) { output[i] = _c[i]; }
    }

    /// batched extension: [batch][signal_size] x [batch][patch_size] -> [batch][output_size()], host or device memory
    auto batched(Float const* signal, Float const* patch, Float* out, size_type batch, int memspace = NEO_B200_HOST) -> void
    {
        detail::check(neo_b200_fft_convolver_exec(_conv, signal, patch, out, batch, memspace));
    }

private:
    neo_b200_fft_convolver* _conv{nullptr};
    size_type _signal, _patch;
    std::vector<Float> _a, _b, _c;
};

/// Drop-in for neo::convolution::upols_convolver<Complex> / upola_convolver<Complex>
/// (convolution/uniform_partitioned_convolver.hpp:14-65): default constructible, `filter(H[P][K])` deep-copies the
/// partitions and resets all state, `operator()(block[B])` processes one block in place. One instance = one channel, as in
/// extra/cli/src/convolver.cpp:37-50; use convolver_bank to run many channels per call.
template<typename Complex, int Kind>
struct uniform_partitioned_convolver
{
    using value_type = Complex;
    using real_type  = detail::real_of<Complex>;

    uniform_partitioned_convolver() = default;

    /// `filter(H)` for the dense aliases; `filter(H, sparsity)` for the sparse ones (sparse_filter.hpp:25-28): `sparsity(row, col,
    /// value)` decides which bins the reference stores in its CSR matrix. The same three containers are built here, element for
    /// element as csr_matrix's constructor does (csr_matrix.hpp:64-98), and handed to the device, which keeps only the stored
    /// elements and multiplies only them (algorithm/multiply_add.hpp:306-324).
    template<typename Mat, typename... Args>
    auto filter(Mat h, Args... args) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Mat>, Complex>);
        auto const parts = static_cast<std::size_t>(h.extent(0));
        auto const bins  = static_cast<std::size_t>(h.extent(1));
        auto const* ptr  = reinterpret_cast<std::complex<real_type> const*>(h.data_handle());
        constexpr bool has_predicate = sizeof...(Args) == 1 && (std::is_invocable_r_v<bool, Args, std::size_t, std::size_t, Complex> && ...);
        if constexpr (has_predicate) {
            _csr_rows.assign(parts + 1, 0);
            _csr_cols.clear();
            _copy.clear();
            for (std::size_t p = 0; p < parts; ++p) {
                _csr_rows[p] = _csr_cols.size();
                for (std::size_t k = 0; k < bins; ++k) {
                    auto const v = h(p, k);
                    if ((static_cast<bool>(args(p, k, v)) && ...)) {
                        _copy.emplace_back(v.real(), v.imag());
                        _csr_cols.push_back(k);
                    }
                }
            }
            _csr_rows[parts]          = _csr_cols.size();
            std::uint64_t const fb[2] = {0, _csr_cols.size()};
            _bank.filter_csr(_copy.data(), _csr_cols.data(), _csr_rows.data(), fb, 1, parts, bins);
            return;
        }
        if (h.stride(1) != 1 || static_cast<std::size_t>(h.stride(0)) != bins) {
            _copy.resize(parts * bins);
            for (std::size_t p = 0; p < parts; ++p) {
                for (std::size_t k = 0; k < bins; ++k) {
                    auto const v        = h(p, k);
                    _copy[p * bins + k] = std::complex<real_type>{v.real(), v.imag()};
                }
            }
            ptr = _copy.data();
        }
        _bank.filter(ptr, 1, 1, parts, bins, NEO_B200_DIAGONAL);
    }

    /// switches to `h` (the H[P][B+1] view filter() takes, same P and B) with a linear crossfade of `fade` samples from the next sample
    /// on, keeping the delay line; returns the index of the fade's first sample, counted from the last filter() call. Overlap-save
    /// only: an overlap-add convolver's carried tail belongs to its filter. Throws while an earlier crossfade has not ended.
    template<typename Mat>
    auto crossfade_to(Mat h, std::size_t fade) -> std::size_t
    {
        static_assert(Kind == NEO_B200_UPOLS, "crossfade_to: overlap-save convolvers only (upols_convolver)");
        static_assert(std::is_same_v<detail::element_of<Mat>, Complex>);
        auto const parts = static_cast<std::size_t>(h.extent(0));
        auto const bins  = static_cast<std::size_t>(h.extent(1));
        if (_bank.handle() == nullptr) { throw std::invalid_argument{"neo::b200::uniform_partitioned_convolver: filter() has not been called"}; }
        if (parts != _bank.partitions() || bins != _bank.block_size() + 1) {
            throw std::invalid_argument{"neo::b200::uniform_partitioned_convolver: crossfade_to() needs the shape filter() was given"};
        }
        _copy.resize(parts * bins);
        for (std::size_t p = 0; p < parts; ++p) {
            for (std::size_t k = 0; k < bins; ++k) {
                auto const v        = h(p, k);
                _copy[p * bins + k] = std::complex<real_type>{v.real(), v.imag()};
            }
        }
        _bank.stage_filter(_copy.data());
        return _bank.crossfade(fade);
    }

    /// the CSR containers of the last sparse filter() call (row_container, column_container: csr_matrix.hpp:46-48) and what the
    /// device holds for this convolver
    [[nodiscard]] auto csr_row_container() const noexcept -> std::vector<std::uint64_t> const& { return _csr_rows; }
    [[nodiscard]] auto csr_column_container() const noexcept -> std::vector<std::uint64_t> const& { return _csr_cols; }
    [[nodiscard]] auto device_bytes() const noexcept -> std::size_t { return _bank.device_bytes(); }

    template<typename Vec>
    auto operator()(Vec block) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Vec>, real_type>);
        auto const n = static_cast<std::size_t>(block.extent(0));
        // the reference asserts the extent (uniform_partitioned_convolver.hpp:50); here a wrong extent would make the device copy
        // run past the caller's buffer, so it is an error in release builds too
        if (_bank.handle() == nullptr) { throw std::invalid_argument{"neo::b200::uniform_partitioned_convolver: filter() has not been called"}; }
        if (n != _bank.block_size()) {
            throw std::invalid_argument{"neo::b200::uniform_partitioned_convolver: block extent differs from the filter's block size"};
        }
        if (detail::is_contiguous(block)) {
            _bank.process(block.data_handle(), block.data_handle(), 1);
        } else {
            _tmp.resize(n);
            for (std::size_t i = 0; i < n; ++i) { _tmp[i] = block[i]; }
            _bank.process(_tmp.data(), _tmp.data(), 1);
            for (std::size_t i = 0; i < n; ++i) { block[i] = _tmp[i]; }
        }
    }

private:
    convolver_bank<real_type, Kind> _bank;
    std::vector<std::uint64_t> _csr_rows, _csr_cols;
    std::vector<std::complex<real_type>> _copy;
    std::vector<real_type> _tmp;
};

template<typename Complex>
using upols_convolver = uniform_partitioned_convolver<Complex, NEO_B200_UPOLS>;
template<typename Complex>
using upola_convolver = uniform_partitioned_convolver<Complex, NEO_B200_UPOLA>;

/// upols_convolver<Complex>'s duck type (`filter(H[P][K])`, `operator()(block[B])` in place) at one block of latency for long impulse
/// responses: the first partitions run per block, later stretches in frame mode on side streams (neo_b200_lowlat_*, non-uniform
/// partitioning). Same results up to rounding. One instance = one channel; `frame_blocks` = the level frame sizes, empty = the
/// library default. `process(samples)` takes any number of samples >= 1 in place and returns each output in the call that delivers
/// its input (neo_b200_lowlat_process_samples): what a plugin host's varying buffer size needs, with no FIFO in front.
/// `crossfade_to(H, fade)` swaps in a new impulse response mid-stream with a linear crossfade of `fade` samples and keeps the reverb
/// tail of everything played so far (neo_b200_lowlat_stage_filter + neo_b200_lowlat_crossfade).
template<typename Complex>
struct low_latency_convolver
{
    using value_type = Complex;
    using real_type  = detail::real_of<Complex>;

    low_latency_convolver() = default;
    explicit low_latency_convolver(std::vector<std::size_t> frame_blocks) : _frame_blocks(std::move(frame_blocks)) {}
    low_latency_convolver(low_latency_convolver const&)                    = delete;
    auto operator=(low_latency_convolver const&) -> low_latency_convolver& = delete;
    ~low_latency_convolver() { neo_b200_lowlat_destroy(_conv); }

    template<typename Mat>
    auto filter(Mat h) -> void
    {
        auto const parts = static_cast<std::size_t>(h.extent(0));
        auto const bins  = static_cast<std::size_t>(h.extent(1));
        copy_filter(h);
        neo_b200_lowlat_config cfg{detail::dtype_of<real_type>, 1, bins - 1, parts, _frame_blocks.size(), {0, 0, 0, 0}};
        for (std::size_t i = 0; i < _frame_blocks.size() && i < 4; ++i) { cfg.frame_blocks[i] = _frame_blocks[i]; }
        neo_b200_lowlat_destroy(_conv);
        _conv = nullptr;
        detail::check(neo_b200_lowlat_create(&_conv, &cfg));
        detail::check(neo_b200_lowlat_set_filter(_conv, _copy.data(), NEO_B200_HOST));
        _block = bins - 1;
        _parts = parts;
    }

    /// switches to `h` (the H[P][B+1] view filter() takes, same P and B) with a linear crossfade of `fade` samples, keeping every delay
    /// line; returns the index of the fade's first sample, counted from the last filter() call. Throws while an earlier crossfade has
    /// not ended (DESIGN §4.7: the fade starts one to two of the largest level's frames after the call).
    template<typename Mat>
    auto crossfade_to(Mat h, std::size_t fade) -> std::size_t
    {
        if (_conv == nullptr) { throw std::invalid_argument{"neo::b200::low_latency_convolver: filter() has not been called"}; }
        if (static_cast<std::size_t>(h.extent(0)) != _parts || static_cast<std::size_t>(h.extent(1)) != _block + 1) {
            throw std::invalid_argument{"neo::b200::low_latency_convolver: crossfade_to() needs the shape filter() was given"};
        }
        copy_filter(h);
        detail::check(neo_b200_lowlat_stage_filter(_conv, _copy.data(), NEO_B200_HOST));
        std::size_t start = 0;
        detail::check(neo_b200_lowlat_crossfade(_conv, fade, &start));
        return start;
    }

    template<typename Vec>
    auto operator()(Vec block) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Vec>, real_type>);
        auto const n = static_cast<std::size_t>(block.extent(0));
        if (_conv == nullptr) { throw std::invalid_argument{"neo::b200::low_latency_convolver: filter() has not been called"}; }
        if (n != _block) { throw std::invalid_argument{"neo::b200::low_latency_convolver: block extent differs from the filter's block size"}; }
        if (detail::is_contiguous(block)) {
            detail::check(neo_b200_lowlat_process(_conv, block.data_handle(), block.data_handle(), 1, NEO_B200_HOST));
        } else {
            _tmp.resize(n);
            for (std::size_t i = 0; i < n; ++i) { _tmp[i] = block[i]; }
            detail::check(neo_b200_lowlat_process(_conv, _tmp.data(), _tmp.data(), 1, NEO_B200_HOST));
            for (std::size_t i = 0; i < n; ++i) { block[i] = _tmp[i]; }
        }
    }

    template<typename Vec>
    auto process(Vec samples) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Vec>, real_type>);
        auto const n = static_cast<std::size_t>(samples.extent(0));
        if (_conv == nullptr) { throw std::invalid_argument{"neo::b200::low_latency_convolver: filter() has not been called"}; }
        if (n == 0) { throw std::invalid_argument{"neo::b200::low_latency_convolver: process() needs at least one sample"}; }
        if (detail::is_contiguous(samples)) {
            detail::check(neo_b200_lowlat_process_samples(_conv, samples.data_handle(), samples.data_handle(), n, NEO_B200_HOST));
        } else {
            _tmp.resize(n);
            for (std::size_t i = 0; i < n; ++i) { _tmp[i] = samples[i]; }
            detail::check(neo_b200_lowlat_process_samples(_conv, _tmp.data(), _tmp.data(), n, NEO_B200_HOST));
            for (std::size_t i = 0; i < n; ++i) { samples[i] = _tmp[i]; }
        }
    }

    [[nodiscard]] auto device_bytes() const noexcept -> std::size_t { return _conv == nullptr ? 0 : neo_b200_lowlat_device_bytes(_conv); }

private:
    template<typename Mat>
    auto copy_filter(Mat h) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Mat>, Complex>);
        auto const parts = static_cast<std::size_t>(h.extent(0));
        auto const bins  = static_cast<std::size_t>(h.extent(1));
        _copy.resize(parts * bins);
        for (std::size_t p = 0; p < parts; ++p) {
            for (std::size_t k = 0; k < bins; ++k) {
                auto const v        = h(p, k);
                _copy[p * bins + k] = std::complex<real_type>{v.real(), v.imag()};
            }
        }
    }

    neo_b200_lowlat* _conv{nullptr};
    std::vector<std::size_t> _frame_blocks;
    std::size_t _block{0}, _parts{0};
    std::vector<std::complex<real_type>> _copy;
    std::vector<real_type> _tmp;
};

/// Drop-in for neo::convolution::overlap_add_convolver / upola_convolver_v2 (convolution/overlap_add_convolver.hpp:21-136,
/// dense_convolver.hpp:28): `operator()(inout)` takes ANY number of samples >= one block (:74 asserts that).
///   - Calls of whole blocks on a clean window -- what its test and benchmark use (uniform_partitioned_convolver_test.cpp:40,
///     benchmark/convolution.cpp:58) -- run the block loop of :85 on the device, up to 32 blocks per launch.
///   - A call that ends inside a block follows the reference chunk by chunk (:85-132), including its peculiarity: the window is
///     transformed as it stands, and after a partial chunk it holds the previous inverse transform's OUTPUT (:114-115 write the result
///     back into the window), so the next chunk of the same block transforms output samples next to the new input. Window, overlap
///     and input position live here, as in the reference object; each chunk is one neo_b200_conv_process_window call. Once a call
///     has ended inside a block the object stays on this chunk path.
template<typename Complex>
struct overlap_add_convolver
{
    using value_type = Complex;
    using real_type  = detail::real_of<Complex>;
    using size_type  = std::size_t;

    overlap_add_convolver() = default;

    template<typename Mat>
    auto filter(Mat h) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Mat>, Complex>);
        auto const parts = static_cast<size_type>(h.extent(0));
        auto const bins  = static_cast<size_type>(h.extent(1));
        _copy.resize(parts * bins);
        for (size_type p = 0; p < parts; ++p) {
            for (size_type k = 0; k < bins; ++k) {
                auto const v        = h(p, k);
                _copy[p * bins + k] = {v.real(), v.imag()};
            }
        }
        _block = bins - 1;
        _bank.filter(_copy.data(), 1, 1, parts, bins, NEO_B200_DIAGONAL, max_blocks_per_launch);
        _window.assign(2 * _block, real_type{});   // overlap_add_convolver.hpp:61-63: zero-initialised
        _overlap.assign(_block, real_type{});
        _y.assign(2 * _block, real_type{});
        _input_pos  = 0;
        _chunk_path = false;
    }

    template<typename Vec>
    auto operator()(Vec inout) -> void
    {
        static_assert(std::is_same_v<detail::element_of<Vec>, real_type>);
        auto const n = static_cast<size_type>(inout.extent(0));
        if (_block == 0) { throw std::invalid_argument{"neo::b200::overlap_add_convolver: filter() has not been called"}; }
        if (n < _block) { throw std::invalid_argument{"neo::b200::overlap_add_convolver: call shorter than one block"}; }  // :74
        _tmp.resize(n);
        for (size_type i = 0; i < n; ++i) { _tmp[i] = inout[i]; }
        if (!_chunk_path && n % _block == 0) {
            for (size_type done = 0; done < n / _block;) {
                auto const blocks = std::min(max_blocks_per_launch, n / _block - done);
                _bank.process(_tmp.data() + done * _block, _tmp.data() + done * _block, blocks);
                done += blocks;
            }
        } else {
            if (!_chunk_path) {  // the overlap so far lives in the handle (overlap_add.hpp:106); from here on it lives in this object
                detail::check(neo_b200_conv_tail(_bank.handle(), _overlap.data(), NEO_B200_HOST));
                _chunk_path = true;
            }
            chunks(_tmp.data(), n);
        }
        for (size_type i = 0; i < n; ++i) { inout[i] = _tmp[i]; }
    }

private:
    // overlap_add_convolver.hpp:85-132, one device call per chunk
    auto chunks(real_type* inout, size_type num_samples) -> void
    {
        size_type done = 0;
        while (done < num_samples) {
            auto const todo = std::min(num_samples - done, _block - _input_pos);
            std::copy_n(inout + done, todo, _window.begin() + static_cast<std::ptrdiff_t>(_input_pos));                        // :91
            bool const completes = _input_pos + todo == _block;
            detail::check(neo_b200_conv_process_window(_bank.handle(), _window.data(), _y.data(), completes ? 1 : 0, NEO_B200_HOST));  // :92-115
            _window = _y;  // :114-115: the window now holds the scaled inverse transform
            for (size_type i = 0; i < todo; ++i) { inout[done + i] = _window[_input_pos + i] + _overlap[_input_pos + i]; }    // :117-118
            _input_pos += todo;
            if (_input_pos == _block) {                                                                                         // :122-131
                _input_pos = 0;
                std::copy_n(_window.begin() + static_cast<std::ptrdiff_t>(_block), _block, _overlap.begin());
                std::fill(_window.begin(), _window.end(), real_type{});
            }
            done += todo;
        }
    }

    static constexpr size_type max_blocks_per_launch = 32;
    convolver_bank<real_type, NEO_B200_UPOLA> _bank;
    std::vector<std::complex<real_type>> _copy;
    std::vector<real_type> _tmp, _window, _overlap, _y;
    size_type _block{0};
    size_type _input_pos{0};
    bool _chunk_path{false};
};

template<typename Complex>
using upola_convolver_v2 = overlap_add_convolver<Complex>;

/// neo::convolution::split_upols_convolver / split_upola_convolver (dense_convolver.hpp:32-41) differ from the dense aliases only
/// in how the reference lays its FDL and filter out in host memory (split re/im planes for its SIMD loops); interface and results
/// are the same (golden vectors: tests/test_conv_gpu.py), and the device layout is this library's own either way.
/// neo::convolution::compressed_fdl<FloatComplex, IntComplex> (compressed_fdl.hpp:17-52) with the rows on the device as int8 / int16
/// complex. `insert(row, index)` as there; `operator[](index)` returns the row as the reference's compressed_accessor would read it
/// (a materialised copy instead of a lazily converting view); `raw(index)` the stored integers.
template<typename FloatComplex, typename IntComplex>
struct compressed_fdl
{
    using value_type      = FloatComplex;
    using compressed_type = IntComplex;
    using real_type       = typename FloatComplex::value_type;
    using int_type        = typename IntComplex::value_type;
    static_assert(sizeof(int_type) == 1 || sizeof(int_type) == 2, "int8 or int16 parts");

    compressed_fdl() = default;
    compressed_fdl(std::size_t rows, std::size_t cols) : _rows{rows}, _cols{cols}
    {
        detail::check(neo_b200_compressed_fdl_create(&_fdl, rows, cols, detail::dtype_of<real_type>, int(8 * sizeof(int_type))));
    }
    /// the reference's constructor takes `stdex::dextents<size_t, 2>` (compressed_fdl.hpp:24)
    template<typename Extents, typename = decltype(std::declval<Extents const&>().extent(0))>
    explicit compressed_fdl(Extents const& e) : compressed_fdl{static_cast<std::size_t>(e.extent(0)), static_cast<std::size_t>(e.extent(1))}
    {}
    compressed_fdl(compressed_fdl const&)                    = delete;
    auto operator=(compressed_fdl const&) -> compressed_fdl& = delete;
    compressed_fdl(compressed_fdl&& o) noexcept : _fdl{std::exchange(o._fdl, nullptr)}, _rows{o._rows}, _cols{o._cols} {}
    auto operator=(compressed_fdl&& o) noexcept -> compressed_fdl&
    {
        if (this != &o) {
            neo_b200_compressed_fdl_destroy(_fdl);
            _fdl  = std::exchange(o._fdl, nullptr);
            _rows = o._rows;
            _cols = o._cols;
        }
        return *this;
    }
    ~compressed_fdl() { neo_b200_compressed_fdl_destroy(_fdl); }

    template<typename Vec>
    auto insert(Vec input, std::size_t index) -> void
    {
        auto row = std::vector<std::complex<real_type>>(_cols);
        for (std::size_t i = 0; i < _cols && i < static_cast<std::size_t>(input.extent(0)); ++i) { row[i] = {input[i].real(), input[i].imag()}; }
        detail::check(neo_b200_compressed_fdl_insert(_fdl, row.data(), index, NEO_B200_HOST));
    }
    [[nodiscard]] auto operator[](std::size_t index) const -> std::vector<FloatComplex>
    {
        auto row = std::vector<std::complex<real_type>>(_cols);
        detail::check(neo_b200_compressed_fdl_row(_fdl, index, row.data(), NEO_B200_HOST));
        auto out = std::vector<FloatComplex>(_cols);
        for (std::size_t i = 0; i < _cols; ++i) { out[i] = FloatComplex{row[i].real(), row[i].imag()}; }
        return out;
    }
    [[nodiscard]] auto raw(std::size_t index) const -> std::vector<int_type>
    {
        auto out = std::vector<int_type>(2 * _cols);
        detail::check(neo_b200_compressed_fdl_raw(_fdl, index, out.data()));
        return out;
    }

private:
    neo_b200_compressed_fdl* _fdl{nullptr};
    std::size_t _rows{0}, _cols{0};
};

/// neo::convolution::sparse_upols_convolver / sparse_upola_convolver (sparse_convolver.hpp:14-22): `filter(H, sparsity)` builds the
/// reference's CSR matrix on the host and the device keeps only its stored elements (neo_b200_conv_set_filter_csr).
template<typename Complex>
using sparse_upols_convolver = upols_convolver<Complex>;
template<typename Complex>
using sparse_upola_convolver = upola_convolver<Complex>;

template<typename Complex>
using split_upols_convolver = upols_convolver<Complex>;
template<typename Complex>
using split_upola_convolver = upola_convolver<Complex>;

}  // namespace neo::b200
