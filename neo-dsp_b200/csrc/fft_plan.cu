// fft_plan.cu -- C ABI of the c2c and r2c/c2r plans (include/neo_b200.h), the drop-in for
// neo::fft::fft_plan (src/neo/fft/reference/c2c_dit2_plan.hpp:22-104) and
// neo::fft::rfft_plan (src/neo/fft/fallback/fallback_rfft_plan.hpp:15-61).
#include "fft_kernels.cuh"
#include "fft_large.cuh"
#include "fft_split.cuh"
#include "fft_wide.cuh"

#include <cmath>
#include <memory>

namespace neo_b200 {

std::atomic<std::uint64_t>& launch_counter()
{
    static std::atomic<std::uint64_t> counter{0};
    return counter;
}

int require_device()
{
    int count             = 0;
    cudaError_t const err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(NEO_B200_ERR_CUDA, "no CUDA device available (%s); this backend has no CPU fallback",
                    err == cudaSuccess ? "device count is 0" : cudaGetErrorString(err));
    }
    return NEO_B200_OK;
}

namespace {

constexpr size_t k_max_order = 27;  // c2c_dit2_plan::max_order(), c2c_dit2_plan.hpp:59-62

template<typename T>
struct c2c_engine
{
    int order;
    fft_tables<T> tables;        // single-CTA path (order-point plan) or split path (max_cta-point plan)
    device_buffer w_big;         // split path: exp(-2 pi i n / 2^order), n < 2^max_cta
    device_buffer scratch;       // split path, in-place calls
    large_fft<T> large;          // four-step path above the split range
    bool use_large{false};
    int split{0};                // 2 or 4 CTAs per transform (fft_split.cuh)

    int init(int order_, cudaStream_t stream)
    {
        order          = order_;
        constexpr int c = max_cta_logm<T>();
        split          = order == c + 1 ? 2 : order == c + 2 ? 4 : 0;
        use_large      = order > c + 2;
        if (use_large) { return large.init(order, stream); }
        if (split != 0) {
            NEO_TRY(tables.build(c, false, stream));
            size_t const m2 = size_t(1) << c;
            std::vector<cx<T>> w(m2);
            for (size_t n = 0; n < m2; ++n) {
                double const a = -2.0 * 3.14159265358979323846264338327950288 * double(n) / std::ldexp(1.0, order);
                w[n]           = mk<T>(T(std::cos(a)), T(std::sin(a)));
            }
            NEO_TRY(w_big.reserve(m2 * sizeof(cx<T>)));
            NEO_CUDA_TRY(cudaMemcpyAsync(w_big.ptr, w.data(), m2 * sizeof(cx<T>), cudaMemcpyHostToDevice, stream));
            NEO_CUDA_TRY(cudaStreamSynchronize(stream));
            return NEO_B200_OK;
        }
        return tables.build(order, false, stream);
    }

    int exec_split(cx<T> const* in, cx<T>* out, size_t batch, int direction, cudaStream_t stream)
    {
        constexpr int c = max_cta_logm<T>();
        auto const* wb  = w_big.template as<cx<T>>();
        if (in != out) {
            return split == 2 ? launch_c2c_split<T, c, 2>(in, out, tables.tw(), wb, batch, direction, stream)
                              : launch_c2c_split<T, c, 4>(in, out, tables.tw(), wb, batch, direction, stream);
        }
        // in place: the CTAs of one transform read all of it and write interleaved bins -> go through a scratch chunk
        size_t const bytes = (size_t(1) << order) * sizeof(cx<T>);
        size_t const chunk = std::max<size_t>(1, std::min(batch, (size_t(64) << 20) / bytes));
        NEO_TRY(scratch.reserve(chunk * bytes));
        for (size_t first = 0; first < batch; first += chunk) {
            size_t const n  = std::min(chunk, batch - first);
            cx<T>* const s  = scratch.template as<cx<T>>();
            cx<T>* const io = out + (first << order);
            NEO_TRY(split == 2 ? launch_c2c_split<T, c, 2>(io, s, tables.tw(), wb, n, direction, stream)
                               : launch_c2c_split<T, c, 4>(io, s, tables.tw(), wb, n, direction, stream));
            NEO_CUDA_TRY(cudaMemcpyAsync(io, s, n * bytes, cudaMemcpyDeviceToDevice, stream));
        }
        return NEO_B200_OK;
    }

    int exec(cx<T> const* in, cx<T>* out, size_t batch, int direction, cudaStream_t stream)
    {
        if (use_large) { return large.exec(in, out, batch, direction, stream); }
        if (split != 0) { return exec_split(in, out, batch, direction, stream); }
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_DISPATCH_LOGM(T, order, {
            if constexpr (LOGM <= max_cta_logm<T>()) {
                status = direction < 0 ? launch_c2c<T, LOGM, -1>(in, out, tables.tw(), batch, stream)
                                       : launch_c2c<T, LOGM, +1>(in, out, tables.tw(), batch, stream);
            }
        });
        if (status == NEO_B200_ERR_UNSUPPORTED) { return fail(status, "c2c order %d not supported", order); }
        return status;
    }

    // split-complex (SoA) data, [batch][size] planes; single-CTA sizes run fused, longer ones through an interleaved scratch
    int exec_planes(T const* re_in, T const* im_in, T* re_out, T* im_out, size_t batch, int direction, cudaStream_t stream)
    {
        size_t const n = size_t(1) << order;
        if (!use_large && split == 0) {
            int status = NEO_B200_ERR_UNSUPPORTED;
            c2c_split_io<T> const io{re_in, im_in, re_out, im_out, n};
            NEO_DISPATCH_LOGM(T, order, {
                if constexpr (LOGM <= max_cta_logm<T>()) {
                    status = direction < 0 ? launch_c2c_io<T, LOGM, -1>(io, tables.tw(), batch, stream)
                                           : launch_c2c_io<T, LOGM, +1>(io, tables.tw(), batch, stream);
                }
            });
            return status;
        }
        size_t const chunk = std::max<size_t>(1, std::min(batch, (size_t(256) << 20) / (n * sizeof(cx<T>))));
        NEO_TRY(planes.reserve(2 * chunk * n * sizeof(cx<T>)));
        cx<T>* const a = planes.template as<cx<T>>();
        cx<T>* const b = a + chunk * n;
        for (size_t first = 0; first < batch; first += chunk) {
            size_t const cnt   = std::min(chunk, batch - first);
            size_t const elems = cnt * n;
            unsigned const grid = static_cast<unsigned>((elems + 255) / 256);
            split_to_interleaved_kernel<T><<<grid, 256, 0, stream>>>(re_in + first * n, im_in + first * n, a, elems);
            NEO_TRY(check_launch("split_to_interleaved_kernel"));
            NEO_TRY(exec(a, b, cnt, direction, stream));
            interleaved_to_split_kernel<T><<<grid, 256, 0, stream>>>(b, re_out + first * n, im_out + first * n, elems);
            NEO_TRY(check_launch("interleaved_to_split_kernel"));
        }
        return NEO_B200_OK;
    }

    device_buffer planes;
};

// dft_plan: any size n through Bluestein's chirp-z (fft/fallback/fallback_dft_plan.hpp:24-96), m = 2^next_order(2n+1)
template<typename T>
struct dft_engine
{
    size_t n{0}, m{0};
    int order{0};
    c2c_engine<T> fft;
    device_buffer chirp[2];  // w of the forward / backward direction, [n]
    device_buffer bhat[2];   // forward transform of b (b[0] = w[0], b[i] = b[m-i] = conj(w[i])), [m], per direction
    device_buffer work;      // [batch][m], grow-only

    int init(size_t size, cudaStream_t stream)
    {
        n     = size;
        order = 0;
        while ((size_t(1) << order) < 2 * n + 1) { ++order; }  // fallback_dft_plan.hpp:88-91
        if (size_t(order) > k_max_order) { return fail(NEO_B200_ERR_UNSUPPORTED, "dft size %zu needs a transform of order %d", size, order); }
        m = size_t(1) << order;
        NEO_TRY(fft.init(order, stream));
        std::vector<cx<T>> w(n), b(m);
        for (int d = 0; d < 2; ++d) {
            double const coef = (d == 0 ? -1.0 : 1.0) * 3.14159265358979323846264338327950288 / double(n);
            for (size_t i = 0; i < n; ++i) {
                // (i*i) % (2n) without overflow for any size that fits the plan
                unsigned __int128 const sq = static_cast<unsigned __int128>(i) * i;
                double const a             = double(static_cast<size_t>(sq % (2 * n))) * coef;
                w[i]                       = mk<T>(T(std::cos(a)), T(std::sin(a)));
            }
            std::fill(b.begin(), b.end(), mk<T>(T(0), T(0)));
            b[0] = w[0];  // as the reference does (:59); w[0] = 1 either way
            for (size_t i = 1; i < n; ++i) { b[i] = b[m - i] = mk<T>(w[i].x, -w[i].y); }
            NEO_TRY(chirp[d].reserve(n * sizeof(cx<T>)));
            NEO_TRY(bhat[d].reserve(m * sizeof(cx<T>)));
            NEO_CUDA_TRY(cudaMemcpyAsync(chirp[d].ptr, w.data(), n * sizeof(cx<T>), cudaMemcpyHostToDevice, stream));
            NEO_CUDA_TRY(cudaMemcpyAsync(bhat[d].ptr, b.data(), m * sizeof(cx<T>), cudaMemcpyHostToDevice, stream));
            NEO_TRY(fft.exec(bhat[d].template as<cx<T>>(), bhat[d].template as<cx<T>>(), 1, -1, stream));
            NEO_CUDA_TRY(cudaStreamSynchronize(stream));  // host vectors are reused
        }
        return NEO_B200_OK;
    }

    int exec(cx<T> const* in, cx<T>* out, size_t batch, int direction, cudaStream_t stream)
    {
        if (batch == 0) { return NEO_B200_OK; }
        int const d      = direction < 0 ? 0 : 1;
        auto const* w    = chirp[d].template as<cx<T>>();
        auto const* bh   = bhat[d].template as<cx<T>>();
        T const scale    = T(1) / T(m);
        // the padded transforms are walked in chunks of about 256 MB of work space
        size_t const chunk = std::max<size_t>(1, std::min(batch, (size_t(256) << 20) / (m * sizeof(cx<T>))));
        NEO_TRY(work.reserve(chunk * m * sizeof(cx<T>)));
        cx<T>* const a = work.template as<cx<T>>();
        for (size_t first = 0; first < batch; first += chunk) {
            size_t const cnt = std::min(chunk, batch - first);
            cx<T> const* x   = in + first * n;
            cx<T>* y         = out + first * n;
            if (order <= max_cta_logm<T>()) {
                // two launches: chirp multiply and zero padding ride on the forward transform's loads, the filter product on its
                // stores; scaling, the second chirp multiply and the cut to n points on the backward transform's stores
                int status = NEO_B200_ERR_UNSUPPORTED;
                bluestein_fwd_io<T> const fio{x, a, w, bh, n, m};
                bluestein_bwd_io<T> const bio{a, y, w, n, m, scale};
                NEO_DISPATCH_LOGM(T, order, {
                    if constexpr (LOGM <= max_cta_logm<T>()) {
                        status = launch_c2c_io<T, LOGM, -1>(fio, fft.tables.tw(), cnt, stream);
                        if (status == NEO_B200_OK) { status = launch_c2c_io<T, LOGM, +1>(bio, fft.tables.tw(), cnt, stream); }
                    }
                });
                if (status != NEO_B200_OK) { return status; }
            } else {
                size_t const padded = cnt * m, kept = cnt * n;
                bluestein_pre_kernel<T><<<unsigned((padded + 255) / 256), 256, 0, stream>>>(x, a, w, n, m, padded);
                NEO_TRY(check_launch("bluestein_pre_kernel"));
                NEO_TRY(fft.exec(a, a, cnt, -1, stream));
                bluestein_mul_kernel<T><<<unsigned((padded + 255) / 256), 256, 0, stream>>>(a, bh, m, padded);
                NEO_TRY(check_launch("bluestein_mul_kernel"));
                NEO_TRY(fft.exec(a, a, cnt, +1, stream));
                bluestein_post_kernel<T><<<unsigned((kept + 255) / 256), 256, 0, stream>>>(a, y, w, n, m, scale, kept);
                NEO_TRY(check_launch("bluestein_post_kernel"));
            }
        }
        return NEO_B200_OK;
    }
};

// fallback_dct2_plan (fft/dct.hpp:24-68): unnormalised type-2 DCT of 2^order reals
template<typename T>
struct dct2_engine
{
    int order{0};
    size_t n{1};
    c2c_engine<T> fft;
    device_buffer scale;  // 2 exp(-i pi k / (2n)), k < n
    device_buffer work;   // beyond the single-CTA range: [batch][n] complex, grow-only; in-place calls of the fused form: [batch][n] reals

    int init(int order_, cudaStream_t stream)
    {
        order = order_;
        n     = size_t(1) << order;
        NEO_TRY(fft.init(order, stream));
        std::vector<cx<T>> s(n);
        for (size_t k = 0; k < n; ++k) {
            double const a = -3.14159265358979323846264338327950288 * double(k) / (2.0 * double(n));
            s[k]           = mk<T>(T(2.0 * std::cos(a)), T(2.0 * std::sin(a)));
        }
        NEO_TRY(scale.reserve(n * sizeof(cx<T>)));
        NEO_CUDA_TRY(cudaMemcpyAsync(scale.ptr, s.data(), n * sizeof(cx<T>), cudaMemcpyHostToDevice, stream));
        NEO_CUDA_TRY(cudaStreamSynchronize(stream));
        return NEO_B200_OK;
    }

    int exec(T const* in, T* out, size_t batch, cudaStream_t stream)
    {
        if (batch == 0) { return NEO_B200_OK; }
        auto const* sc = scale.template as<cx<T>>();
        if (order <= max_cta_logm<T>()) {
            // one launch. In place is fine: a row is read completely, by the threads that later write it, before the transform's
            // first barrier (a one-thread transform has no barrier and no second reader)
            int status = NEO_B200_ERR_UNSUPPORTED;
            dct2_io<T> const io{in, out, sc, n};
            NEO_DISPATCH_LOGM(T, order, {
                if constexpr (LOGM <= max_cta_logm<T>()) { status = launch_c2c_io<T, LOGM, -1>(io, fft.tables.tw(), batch, stream); }
            });
            return status;
        }
        size_t const chunk = std::max<size_t>(1, std::min(batch, (size_t(256) << 20) / (n * sizeof(cx<T>))));
        NEO_TRY(work.reserve(chunk * n * sizeof(cx<T>)));
        cx<T>* const a = work.template as<cx<T>>();
        for (size_t first = 0; first < batch; first += chunk) {
            size_t const cnt = std::min(chunk, batch - first), total = cnt * n;
            dct2_pre_kernel<T><<<unsigned((total + 255) / 256), 256, 0, stream>>>(in + first * n, a, n, total);
            NEO_TRY(check_launch("dct2_pre_kernel"));
            NEO_TRY(fft.exec(a, a, cnt, -1, stream));
            dct2_post_kernel<T><<<unsigned((total + 255) / 256), 256, 0, stream>>>(a, out + first * n, sc, n, total);
            NEO_TRY(check_launch("dct2_post_kernel"));
        }
        return NEO_B200_OK;
    }
};

template<typename T>
struct rfft_engine
{
    int order;                   // real size N = 2^order, complex half size M = N/2
    fft_tables<T> tables;        // one-CTA path: M-point plan; two-CTA path: M/2-point plan
    device_buffer w_n;           // two-CTA path: exp(-2 pi i k / N), k < M/2
    bool use_split{false};       // two CTAs per transform (fft_split.cuh)
    bool use_big_cta{false};     // float32, M = 2^14: one 1024-thread CTA per transform (139 KB exchange tile)
    bool use_wide{false};        // float32, N = 2^14..2^16: 32 points per thread, three stages, Hermitian split in registers (fft_wide.cuh)
    wide_tables<13, 4, 5> wide13;
    wide_tables<14, 5, 5> wide14;
    wide_split_tables<14, 5, 5> wide15s;  // N = 2^16: two CTAs of 2^14 points per transform
    bool use_two_pass{false};    // half-size complex transform into a chunked scratch + Hermitian split pass (split_pass_kernel)
    c2c_engine<T> half;          // two-pass path: the half-size complex transform (four-CTA split or four-step)
    twiddle2<T> w2m;             // two-pass path: exp(-2 pi i k / N)
    device_buffer zbuf;

    // the half size that runs as two CTAs of half that size each: double the first one past a CTA; float the one after it, since
    // M = 2^14 fits one 1024-thread CTA (use_big_cta)
    static constexpr int k_split = max_cta_logm<T>() + (sizeof(T) == 4 ? 2 : 1);

    int init(int order_, cudaStream_t stream)
    {
        order = order_;
        if (order == 0) { return NEO_B200_OK; }
        int const logm = order - 1;
        if constexpr (sizeof(T) == 4) {
            if (order >= 14 && order <= 16) {
                use_wide = true;
                NEO_TRY(order == 14 ? wide13.build(stream) : order == 15 ? wide14.build(stream) : wide15s.build(stream));
                // no return: the 16-points-per-thread path below stays initialised for arrays that are not 16-byte aligned
            }
            if (logm == 14) {
                use_big_cta = true;
                return tables.build(logm, true, stream);
            }
        }
        use_split    = logm == k_split;
        use_two_pass = logm > k_split;
        if (use_two_pass) {
            NEO_TRY(half.init(logm, stream));
            return w2m.build(order, stream);
        }
        if (use_split) {
            NEO_TRY(tables.build(logm - 1, true, stream));
            auto const wn = make_split_twiddles<T>(logm);  // exp(-i pi k / M) = exp(-2 pi i k / N); first M/2 entries used
            size_t const bytes = (wn.size() / 2) * sizeof(cx<T>);
            NEO_TRY(w_n.reserve(bytes));
            NEO_CUDA_TRY(cudaMemcpyAsync(w_n.ptr, wn.data(), bytes, cudaMemcpyHostToDevice, stream));
            NEO_CUDA_TRY(cudaStreamSynchronize(stream));
            return NEO_B200_OK;
        }
        return tables.build(logm, true, stream);
    }

    // chunks keep the intermediate spectrum L2-resident between the two passes: 48 MB behind the four-CTA split c2c, 32 MB behind
    // the four-step (fft_large.cuh), which walks its own scratch in 32 MB chunks as well
    size_t two_pass_chunk(size_t batch) const
    {
        size_t const bytes = (size_t(1) << (order - 1)) * sizeof(cx<T>);
        size_t const mb    = half.use_large ? 32 : 48;
        return std::max<size_t>(1, std::min(batch, (mb << 20) / bytes));
    }

    int forward_two_pass(T const* in, cx<T>* out, size_t batch, cudaStream_t stream)
    {
        size_t const m     = size_t(1) << (order - 1);
        size_t const chunk = two_pass_chunk(batch);
        NEO_TRY(zbuf.reserve(chunk * m * sizeof(cx<T>)));
        cx<T>* const z = zbuf.template as<cx<T>>();
        for (size_t first = 0; first < batch; first += chunk) {
            size_t const cnt = std::min(chunk, batch - first);
            NEO_TRY(half.exec(reinterpret_cast<cx<T> const*>(in) + first * m, z, cnt, -1, stream));
            dim3 const grid(static_cast<unsigned>((m + 255) / 256), static_cast<unsigned>(cnt));
            split_pass_kernel<T, -1><<<grid, 256, 0, stream>>>(z, m, out + first * (m + 1), m + 1, w2m.view(), m);
            NEO_TRY(check_launch("split_pass_kernel"));
        }
        return NEO_B200_OK;
    }

    int backward_two_pass(cx<T> const* in, size_t row_len, T* out, size_t batch, cudaStream_t stream)
    {
        size_t const m     = size_t(1) << (order - 1);
        size_t const chunk = two_pass_chunk(batch);
        NEO_TRY(zbuf.reserve(chunk * m * sizeof(cx<T>)));
        cx<T>* const z = zbuf.template as<cx<T>>();
        for (size_t first = 0; first < batch; first += chunk) {
            size_t const cnt = std::min(chunk, batch - first);
            dim3 const grid(static_cast<unsigned>((m + 255) / 256), static_cast<unsigned>(cnt));
            split_pass_kernel<T, +1><<<grid, 256, 0, stream>>>(in + first * row_len, row_len, z, m, w2m.view(), m);
            NEO_TRY(check_launch("split_pass_kernel"));
            NEO_TRY(half.exec(z, reinterpret_cast<cx<T>*>(out) + first * m, cnt, +1, stream));
        }
        return NEO_B200_OK;
    }

    int forward(T const* in, cx<T>* out, size_t batch, cudaStream_t stream)
    {
        if (order == 0) {
            size_one_r2c_kernel<T><<<static_cast<unsigned>((batch + 255) / 256), 256, 0, stream>>>(in, out, batch);
            return check_launch("size_one_r2c_kernel");
        }
        if constexpr (sizeof(T) == 4) {
            // the wide kernels need 16-byte aligned rows; the others take any 8-byte aligned array
            if (use_wide && wide_aligned(in)) {
                if (order == 16) { return launch_r2c_wide_split(wide15s, in, out, batch, stream); }
                return order == 14 ? launch_r2c_wide(wide13, in, out, batch, stream) : launch_r2c_wide(wide14, in, out, batch, stream);
            }
            if (use_big_cta) { return launch_r2c<T, 14>(r2c_plain_io<T, 14>{in, out}, tables.tw(), tables.rtw(), batch, stream); }
        }
        if (use_two_pass) { return forward_two_pass(in, out, batch, stream); }
        if (use_split) { return launch_r2c_split2<T, k_split - 1>(in, out, tables.tw(), tables.rtw(), batch, stream); }
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_DISPATCH_LOGM(T, order - 1, {
            if constexpr (LOGM <= max_cta_logm<T>()) {
                status = launch_r2c<T, LOGM>(r2c_plain_io<T, LOGM>{in, out}, tables.tw(), tables.rtw(), batch, stream);
            }
        });
        if (status == NEO_B200_ERR_UNSUPPORTED) { return fail(status, "rfft order %d not supported", order); }
        return status;
    }

    int backward(cx<T> const* in, size_t row_len, T* out, size_t batch, cudaStream_t stream)
    {
        if (order == 0) {
            size_one_c2r_kernel<T><<<static_cast<unsigned>((batch + 255) / 256), 256, 0, stream>>>(in, row_len, out, batch);
            return check_launch("size_one_c2r_kernel");
        }
        if constexpr (sizeof(T) == 4) {
            // the wide kernels need 16-byte aligned rows; the others take any 8-byte aligned array
            if (use_wide && wide_aligned(out)) {
                if (order == 16) { return launch_c2r_wide_split(wide15s, in, row_len, out, batch, stream); }
                return order == 14 ? launch_c2r_wide(wide13, in, row_len, out, batch, stream)
                                   : launch_c2r_wide(wide14, in, row_len, out, batch, stream);
            }
            if (use_big_cta) {
                return launch_c2r<T, 14>(c2r_plain_io<T, 14>{in, out, row_len}, tables.tw(), tables.rtw(), batch, stream);
            }
        }
        if (use_two_pass) { return backward_two_pass(in, row_len, out, batch, stream); }
        if (use_split) {
            return launch_c2r_split2<T, k_split - 1>(in, row_len, out, tables.tw(), tables.rtw(), w_n.template as<cx<T>>(), batch, stream);
        }
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_DISPATCH_LOGM(T, order - 1, {
            if constexpr (LOGM <= max_cta_logm<T>()) {
                status = launch_c2r<T, LOGM>(c2r_plain_io<T, LOGM>{in, out, row_len}, tables.tw(), tables.rtw(), batch, stream);
            }
        });
        if (status == NEO_B200_ERR_UNSUPPORTED) { return fail(status, "irfft order %d not supported", order); }
        return status;
    }
};

}  // namespace
}  // namespace neo_b200

using namespace neo_b200;

struct neo_b200_fft_plan
{
    size_t order;
    int dtype;
    int device;
    stream_ref stream;
    c2c_engine<float> f32;
    c2c_engine<double> f64;
    device_buffer staging_in, staging_out;
};

struct neo_b200_rfft_plan
{
    size_t order;
    int dtype;
    int device;
    stream_ref stream;
    rfft_engine<float> f32;
    rfft_engine<double> f64;
    device_buffer staging_in, staging_out;
};

// fft_convolver (convolution/fft_convolver.hpp:18-93): rows of [batch][len] reals -> [2*batch][n] zero padded (signal rows, then patch rows)
template<typename T>
__global__ void __launch_bounds__(256) fftconv_pad_kernel(T const* __restrict__ signal, size_t sig_len, T const* __restrict__ patch,
                                                          size_t patch_len, T* __restrict__ padded, size_t n, size_t batch)
{
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= 2 * batch * n) { return; }
    size_t const row = i / n, j = i - row * n;
    padded[i] = row < batch ? (j < sig_len ? signal[row * sig_len + j] : T(0)) : (j < patch_len ? patch[(row - batch) * patch_len + j] : T(0));
}

template<typename T>
__global__ void __launch_bounds__(256) fftconv_mul_kernel(cx<T>* __restrict__ spec, size_t half)
{
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= half) { return; }
    spec[i] = cmul(spec[i], spec[half + i]);  // multiply(signal_spectrum, patch_spectrum, signal_spectrum), fft_convolver.hpp:52
}

template<typename T>
__global__ void __launch_bounds__(256) fftconv_cut_kernel(T const* __restrict__ full, size_t n, T* __restrict__ out, size_t out_len,
                                                          T scale, size_t batch)
{
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= batch * out_len) { return; }
    size_t const row = i / out_len, j = i - row * out_len;
    out[i]           = full[row * n + j] * scale;  // scale(1/N) + copy of the first output_size() samples, :69-71
}

struct neo_b200_fft_convolver
{
    size_t signal_size, patch_size, order;
    int dtype;
    int device;
    stream_ref stream;
    rfft_engine<float> f32;
    rfft_engine<double> f64;
    device_buffer padded, spectra, full, staging_a, staging_b, staging_out;

    template<typename T>
    int run(rfft_engine<T>& eng, T const* signal, T const* patch, T* out, size_t batch)
    {
        cudaStream_t const s = stream.stream;
        size_t const n = size_t(1) << order, bins = n / 2 + 1, out_len = signal_size + patch_size - 1;
        NEO_TRY(padded.reserve(2 * batch * n * sizeof(T)));
        NEO_TRY(spectra.reserve(2 * batch * bins * sizeof(cx<T>)));
        NEO_TRY(full.reserve(batch * n * sizeof(T)));
        size_t const total = 2 * batch * n;
        fftconv_pad_kernel<T><<<unsigned((total + 255) / 256), 256, 0, s>>>(signal, signal_size, patch, patch_size, padded.template as<T>(), n, batch);
        NEO_TRY(check_launch("fftconv_pad_kernel"));
        NEO_TRY(eng.forward(padded.template as<T>(), spectra.template as<cx<T>>(), 2 * batch, s));
        size_t const half = batch * bins;
        fftconv_mul_kernel<T><<<unsigned((half + 255) / 256), 256, 0, s>>>(spectra.template as<cx<T>>(), half);
        NEO_TRY(check_launch("fftconv_mul_kernel"));
        NEO_TRY(eng.backward(spectra.template as<cx<T>>(), bins, full.template as<T>(), batch, s));
        size_t const kept = batch * out_len;
        fftconv_cut_kernel<T><<<unsigned((kept + 255) / 256), 256, 0, s>>>(full.template as<T>(), n, out, out_len, T(1) / T(n), batch);
        return check_launch("fftconv_cut_kernel");
    }
};

struct neo_b200_dct2_plan
{
    size_t order;
    int dtype;
    int device;
    stream_ref stream;
    dct2_engine<float> f32;
    dct2_engine<double> f64;
    device_buffer staging;
};

struct neo_b200_dft_plan
{
    size_t size;
    int dtype;
    int device;
    stream_ref stream;
    dft_engine<float> f32;
    dft_engine<double> f64;
    device_buffer staging_in, staging_out;
};

extern "C" {

const char* neo_b200_last_error(void) { return last_error_slot().c_str(); }

const char* neo_b200_version(void) { return "neo_b200 0.1 (sm_100a)"; }

int neo_b200_device_count(void)
{
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return count;
}

int neo_b200_set_device(int device)
{
    NEO_CUDA_TRY(cudaSetDevice(device));
    return NEO_B200_OK;
}

int neo_b200_kernel_launches(uint64_t* count)
{
    if (count == nullptr) { return fail(NEO_B200_ERR_INVALID, "count is null"); }
    *count = launch_counter().load();
    return NEO_B200_OK;
}

size_t neo_b200_fft_max_order(void) { return k_max_order; }

size_t neo_b200_next_order(size_t size)
{
    size_t order = 0;
    while ((size_t(1) << order) < size) { ++order; }
    return order;
}

// ---- c2c ---------------------------------------------------------------------------------------------------------------
int neo_b200_fft_plan_create(neo_b200_fft_plan** plan, size_t order, int dtype)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    *plan = nullptr;
    if (dtype != NEO_B200_F32 && dtype != NEO_B200_F64) { return fail(NEO_B200_ERR_INVALID, "bad dtype %d", dtype); }
    // same contract as c2c_dit2_plan::check_order (c2c_dit2_plan.hpp:98-104)
    if (order > k_max_order) { return fail(NEO_B200_ERR_UNSUPPORTED, "neo_b200: unsupported order '%zu'", order); }
    NEO_TRY(require_device());
    auto p    = std::unique_ptr<neo_b200_fft_plan>(new (std::nothrow) neo_b200_fft_plan{});
    if (!p) { return fail(NEO_B200_ERR_ALLOC, "out of host memory"); }
    p->order = order;
    p->dtype = dtype;
    NEO_CUDA_TRY(cudaGetDevice(&p->device));
    NEO_TRY(p->stream.create());
    if (dtype == NEO_B200_F32) { NEO_TRY(p->f32.init(static_cast<int>(order), p->stream.stream)); }
    else { NEO_TRY(p->f64.init(static_cast<int>(order), p->stream.stream)); }
    *plan = p.release();
    return NEO_B200_OK;
}

void neo_b200_fft_plan_destroy(neo_b200_fft_plan* plan)
{
    if (plan == nullptr) { return; }
    cudaStreamSynchronize(plan->stream.stream);
    delete plan;
}

size_t neo_b200_fft_plan_order(neo_b200_fft_plan const* plan) { return plan != nullptr ? plan->order : 0; }
size_t neo_b200_fft_plan_size(neo_b200_fft_plan const* plan) { return plan != nullptr ? size_t(1) << plan->order : 0; }

int neo_b200_fft_plan_set_stream(neo_b200_fft_plan* plan, void* cuda_stream)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    plan->stream.adopt(cuda_stream);
    return NEO_B200_OK;
}

int neo_b200_fft_plan_synchronize(neo_b200_fft_plan* plan)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    NEO_CUDA_TRY(cudaStreamSynchronize(plan->stream.stream));
    return NEO_B200_OK;
}

static int fft_exec_device(neo_b200_fft_plan* plan, void const* in, void* out, size_t batch, int direction)
{
    if (plan->dtype == NEO_B200_F32) {
        return plan->f32.exec(static_cast<float2 const*>(in), static_cast<float2*>(out), batch, direction, plan->stream.stream);
    }
    return plan->f64.exec(static_cast<double2 const*>(in), static_cast<double2*>(out), batch, direction, plan->stream.stream);
}

int neo_b200_fft_exec(neo_b200_fft_plan* plan, void const* in, void* out, size_t batch, int direction, int memspace)
{
    if (plan == nullptr || in == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (direction != NEO_B200_FORWARD && direction != NEO_B200_BACKWARD) {
        return fail(NEO_B200_ERR_INVALID, "direction must be -1 (forward) or +1 (backward)");
    }
    if (batch == 0) { return NEO_B200_OK; }
    NEO_CUDA_TRY(cudaSetDevice(plan->device));
    if (memspace == NEO_B200_DEVICE) { return fft_exec_device(plan, in, out, batch, direction); }

    // HOST: stage through device memory in chunks, synchronous semantics like the reference
    size_t const row   = (size_t(1) << plan->order) * 2 * elem_size(plan->dtype);
    size_t const chunk = std::max<size_t>(1, std::min(batch, (size_t(256) << 20) / row));
    NEO_TRY(plan->staging_in.reserve(chunk * row));
    cudaStream_t const s = plan->stream.stream;
    for (size_t first = 0; first < batch; first += chunk) {
        size_t const n = std::min(chunk, batch - first);
        NEO_CUDA_TRY(cudaMemcpyAsync(plan->staging_in.ptr, static_cast<char const*>(in) + first * row, n * row, cudaMemcpyHostToDevice, s));
        NEO_TRY(fft_exec_device(plan, plan->staging_in.ptr, plan->staging_in.ptr, n, direction));
        NEO_CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(out) + first * row, plan->staging_in.ptr, n * row, cudaMemcpyDeviceToHost, s));
    }
    NEO_CUDA_TRY(cudaStreamSynchronize(s));
    return NEO_B200_OK;
}

// ---- fft_convolver (convolution/fft_convolver.hpp:18-93) ------------------------------------------------------------------------------
int neo_b200_fft_convolver_create(neo_b200_fft_convolver** conv, size_t signal_size, size_t patch_size, int dtype)
{
    if (conv == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    *conv = nullptr;
    if (dtype != NEO_B200_F32 && dtype != NEO_B200_F64) { return fail(NEO_B200_ERR_INVALID, "bad dtype %d", dtype); }
    if (signal_size == 0 || patch_size == 0) { return fail(NEO_B200_ERR_INVALID, "signal and patch sizes must be > 0"); }
    size_t const order = neo_b200_next_order(signal_size + patch_size - 1);  // fft_convolver.hpp:76
    if (order > k_max_order) { return fail(NEO_B200_ERR_UNSUPPORTED, "neo_b200: unsupported order '%zu'", order); }
    NEO_TRY(require_device());
    auto p = std::unique_ptr<neo_b200_fft_convolver>(new (std::nothrow) neo_b200_fft_convolver{});
    if (!p) { return fail(NEO_B200_ERR_ALLOC, "out of host memory"); }
    p->signal_size = signal_size;
    p->patch_size  = patch_size;
    p->order       = order;
    p->dtype       = dtype;
    NEO_CUDA_TRY(cudaGetDevice(&p->device));
    NEO_TRY(p->stream.create());
    if (dtype == NEO_B200_F32) { NEO_TRY(p->f32.init(int(order), p->stream.stream)); }
    else { NEO_TRY(p->f64.init(int(order), p->stream.stream)); }
    *conv = p.release();
    return NEO_B200_OK;
}

void neo_b200_fft_convolver_destroy(neo_b200_fft_convolver* conv)
{
    if (conv == nullptr) { return; }
    cudaStreamSynchronize(conv->stream.stream);
    delete conv;
}

size_t neo_b200_fft_convolver_output_size(neo_b200_fft_convolver const* conv)
{
    return conv != nullptr ? conv->signal_size + conv->patch_size - 1 : 0;  // output_size<mode::full>, convolution/mode.hpp:24-29
}

int neo_b200_fft_convolver_exec(neo_b200_fft_convolver* conv, void const* signal, void const* patch, void* out, size_t batch, int memspace)
{
    if (conv == nullptr || signal == nullptr || patch == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (batch == 0) { return NEO_B200_OK; }
    NEO_CUDA_TRY(cudaSetDevice(conv->device));
    cudaStream_t const s = conv->stream.stream;
    size_t const es = elem_size(conv->dtype), out_len = conv->signal_size + conv->patch_size - 1;
    void const* ds = signal;
    void const* dp = patch;
    void* dout     = out;
    if (memspace == NEO_B200_HOST) {
        NEO_TRY(conv->staging_a.reserve(batch * conv->signal_size * es));
        NEO_TRY(conv->staging_b.reserve(batch * conv->patch_size * es));
        NEO_TRY(conv->staging_out.reserve(batch * out_len * es));
        NEO_CUDA_TRY(cudaMemcpyAsync(conv->staging_a.ptr, signal, batch * conv->signal_size * es, cudaMemcpyHostToDevice, s));
        NEO_CUDA_TRY(cudaMemcpyAsync(conv->staging_b.ptr, patch, batch * conv->patch_size * es, cudaMemcpyHostToDevice, s));
        ds   = conv->staging_a.ptr;
        dp   = conv->staging_b.ptr;
        dout = conv->staging_out.ptr;
    }
    if (conv->dtype == NEO_B200_F32) {
        NEO_TRY(conv->run(conv->f32, static_cast<float const*>(ds), static_cast<float const*>(dp), static_cast<float*>(dout), batch));
    } else {
        NEO_TRY(conv->run(conv->f64, static_cast<double const*>(ds), static_cast<double const*>(dp), static_cast<double*>(dout), batch));
    }
    if (memspace == NEO_B200_HOST) {
        NEO_CUDA_TRY(cudaMemcpyAsync(out, dout, batch * out_len * es, cudaMemcpyDeviceToHost, s));
        NEO_CUDA_TRY(cudaStreamSynchronize(s));
    }
    return NEO_B200_OK;
}

// ---- dct2 plan (fft/dct.hpp:24-68) ---------------------------------------------------------------------------------------------------
int neo_b200_dct2_plan_create(neo_b200_dct2_plan** plan, size_t order, int dtype)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    *plan = nullptr;
    if (dtype != NEO_B200_F32 && dtype != NEO_B200_F64) { return fail(NEO_B200_ERR_INVALID, "bad dtype %d", dtype); }
    if (order > k_max_order) { return fail(NEO_B200_ERR_UNSUPPORTED, "neo_b200: unsupported order '%zu'", order); }
    NEO_TRY(require_device());
    auto p = std::unique_ptr<neo_b200_dct2_plan>(new (std::nothrow) neo_b200_dct2_plan{});
    if (!p) { return fail(NEO_B200_ERR_ALLOC, "out of host memory"); }
    p->order = order;
    p->dtype = dtype;
    NEO_CUDA_TRY(cudaGetDevice(&p->device));
    NEO_TRY(p->stream.create());
    if (dtype == NEO_B200_F32) { NEO_TRY(p->f32.init(int(order), p->stream.stream)); }
    else { NEO_TRY(p->f64.init(int(order), p->stream.stream)); }
    *plan = p.release();
    return NEO_B200_OK;
}

void neo_b200_dct2_plan_destroy(neo_b200_dct2_plan* plan)
{
    if (plan == nullptr) { return; }
    cudaStreamSynchronize(plan->stream.stream);
    delete plan;
}

size_t neo_b200_dct2_plan_order(neo_b200_dct2_plan const* plan) { return plan != nullptr ? plan->order : 0; }
size_t neo_b200_dct2_plan_size(neo_b200_dct2_plan const* plan) { return plan != nullptr ? size_t(1) << plan->order : 0; }

int neo_b200_dct2_plan_set_stream(neo_b200_dct2_plan* plan, void* cuda_stream)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    plan->stream.adopt(cuda_stream);
    return NEO_B200_OK;
}

int neo_b200_dct2_exec(neo_b200_dct2_plan* plan, void const* in, void* out, size_t batch, int memspace)
{
    if (plan == nullptr || in == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (batch == 0) { return NEO_B200_OK; }
    NEO_CUDA_TRY(cudaSetDevice(plan->device));
    cudaStream_t const s = plan->stream.stream;
    auto run = [&](void const* i, void* o, size_t n) {
        if (plan->dtype == NEO_B200_F32) { return plan->f32.exec(static_cast<float const*>(i), static_cast<float*>(o), n, s); }
        return plan->f64.exec(static_cast<double const*>(i), static_cast<double*>(o), n, s);
    };
    if (memspace == NEO_B200_DEVICE) { return run(in, out, batch); }
    size_t const row   = (size_t(1) << plan->order) * elem_size(plan->dtype);
    size_t const chunk = std::max<size_t>(1, std::min(batch, (size_t(128) << 20) / row));
    NEO_TRY(plan->staging.reserve(chunk * row));
    for (size_t first = 0; first < batch; first += chunk) {
        size_t const n = std::min(chunk, batch - first);
        NEO_CUDA_TRY(cudaMemcpyAsync(plan->staging.ptr, static_cast<char const*>(in) + first * row, n * row, cudaMemcpyHostToDevice, s));
        NEO_TRY(run(plan->staging.ptr, plan->staging.ptr, n));
        NEO_CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(out) + first * row, plan->staging.ptr, n * row, cudaMemcpyDeviceToHost, s));
    }
    NEO_CUDA_TRY(cudaStreamSynchronize(s));
    return NEO_B200_OK;
}

// ---- dft_plan: any size (Bluestein) ------------------------------------------------------------------------------------------------
int neo_b200_dft_plan_create(neo_b200_dft_plan** plan, size_t size, int dtype)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    *plan = nullptr;
    if (dtype != NEO_B200_F32 && dtype != NEO_B200_F64) { return fail(NEO_B200_ERR_INVALID, "bad dtype %d", dtype); }
    if (size == 0) { return fail(NEO_B200_ERR_INVALID, "dft size must be > 0"); }
    if (size > (size_t(1) << (k_max_order - 1))) { return fail(NEO_B200_ERR_UNSUPPORTED, "neo_b200: unsupported dft size '%zu'", size); }
    NEO_TRY(require_device());
    auto p = std::unique_ptr<neo_b200_dft_plan>(new (std::nothrow) neo_b200_dft_plan{});
    if (!p) { return fail(NEO_B200_ERR_ALLOC, "out of host memory"); }
    p->size  = size;
    p->dtype = dtype;
    NEO_CUDA_TRY(cudaGetDevice(&p->device));
    NEO_TRY(p->stream.create());
    if (dtype == NEO_B200_F32) { NEO_TRY(p->f32.init(size, p->stream.stream)); }
    else { NEO_TRY(p->f64.init(size, p->stream.stream)); }
    *plan = p.release();
    return NEO_B200_OK;
}

void neo_b200_dft_plan_destroy(neo_b200_dft_plan* plan)
{
    if (plan == nullptr) { return; }
    cudaStreamSynchronize(plan->stream.stream);
    delete plan;
}

size_t neo_b200_dft_plan_size(neo_b200_dft_plan const* plan) { return plan != nullptr ? plan->size : 0; }

int neo_b200_dft_plan_set_stream(neo_b200_dft_plan* plan, void* cuda_stream)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    plan->stream.adopt(cuda_stream);
    return NEO_B200_OK;
}

int neo_b200_dft_exec(neo_b200_dft_plan* plan, void const* in, void* out, size_t batch, int direction, int memspace)
{
    if (plan == nullptr || in == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (direction != NEO_B200_FORWARD && direction != NEO_B200_BACKWARD) {
        return fail(NEO_B200_ERR_INVALID, "direction must be -1 (forward) or +1 (backward)");
    }
    if (batch == 0) { return NEO_B200_OK; }
    NEO_CUDA_TRY(cudaSetDevice(plan->device));
    cudaStream_t const s = plan->stream.stream;
    auto run = [&](void const* i, void* o, size_t n) {
        if (plan->dtype == NEO_B200_F32) { return plan->f32.exec(static_cast<float2 const*>(i), static_cast<float2*>(o), n, direction, s); }
        return plan->f64.exec(static_cast<double2 const*>(i), static_cast<double2*>(o), n, direction, s);
    };
    if (memspace == NEO_B200_DEVICE) { return run(in, out, batch); }
    size_t const row   = plan->size * 2 * elem_size(plan->dtype);
    size_t const chunk = std::max<size_t>(1, std::min(batch, (size_t(128) << 20) / row));
    NEO_TRY(plan->staging_in.reserve(chunk * row));
    for (size_t first = 0; first < batch; first += chunk) {
        size_t const n = std::min(chunk, batch - first);
        NEO_CUDA_TRY(cudaMemcpyAsync(plan->staging_in.ptr, static_cast<char const*>(in) + first * row, n * row, cudaMemcpyHostToDevice, s));
        NEO_TRY(run(plan->staging_in.ptr, plan->staging_in.ptr, n));
        NEO_CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(out) + first * row, plan->staging_in.ptr, n * row, cudaMemcpyDeviceToHost, s));
    }
    NEO_CUDA_TRY(cudaStreamSynchronize(s));
    return NEO_B200_OK;
}

int neo_b200_fft_exec_split(neo_b200_fft_plan* plan, void const* re_in, void const* im_in, void* re_out, void* im_out, size_t batch,
                            int direction, int memspace)
{
    if (plan == nullptr || re_in == nullptr || im_in == nullptr || re_out == nullptr || im_out == nullptr) {
        return fail(NEO_B200_ERR_INVALID, "null argument");
    }
    if (direction != NEO_B200_FORWARD && direction != NEO_B200_BACKWARD) {
        return fail(NEO_B200_ERR_INVALID, "direction must be -1 (forward) or +1 (backward)");
    }
    if (batch == 0) { return NEO_B200_OK; }
    NEO_CUDA_TRY(cudaSetDevice(plan->device));
    cudaStream_t const s = plan->stream.stream;
    auto run = [&](void const* ri, void const* ii, void* ro, void* io, size_t n) {
        if (plan->dtype == NEO_B200_F32) {
            return plan->f32.exec_planes(static_cast<float const*>(ri), static_cast<float const*>(ii), static_cast<float*>(ro),
                                         static_cast<float*>(io), n, direction, s);
        }
        return plan->f64.exec_planes(static_cast<double const*>(ri), static_cast<double const*>(ii), static_cast<double*>(ro),
                                     static_cast<double*>(io), n, direction, s);
    };
    if (memspace == NEO_B200_DEVICE) { return run(re_in, im_in, re_out, im_out, batch); }

    size_t const row   = (size_t(1) << plan->order) * elem_size(plan->dtype);
    size_t const chunk = std::max<size_t>(1, std::min(batch, (size_t(128) << 20) / row));
    NEO_TRY(plan->staging_in.reserve(2 * chunk * row));
    char* const dre = static_cast<char*>(plan->staging_in.ptr);
    char* const dim = dre + chunk * row;
    for (size_t first = 0; first < batch; first += chunk) {
        size_t const n = std::min(chunk, batch - first);
        NEO_CUDA_TRY(cudaMemcpyAsync(dre, static_cast<char const*>(re_in) + first * row, n * row, cudaMemcpyHostToDevice, s));
        NEO_CUDA_TRY(cudaMemcpyAsync(dim, static_cast<char const*>(im_in) + first * row, n * row, cudaMemcpyHostToDevice, s));
        NEO_TRY(run(dre, dim, dre, dim, n));
        NEO_CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(re_out) + first * row, dre, n * row, cudaMemcpyDeviceToHost, s));
        NEO_CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(im_out) + first * row, dim, n * row, cudaMemcpyDeviceToHost, s));
    }
    NEO_CUDA_TRY(cudaStreamSynchronize(s));
    return NEO_B200_OK;
}

int neo_b200_fft_exec_strided(
    neo_b200_fft_plan* plan, void const* in, ptrdiff_t in_stride, void* out, ptrdiff_t out_stride, int direction)
{
    if (plan == nullptr || in == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    NEO_CUDA_TRY(cudaSetDevice(plan->device));
    size_t const n    = size_t(1) << plan->order;
    size_t const elem = 2 * elem_size(plan->dtype);
    NEO_TRY(plan->staging_in.reserve(n * elem));
    cudaStream_t const s = plan->stream.stream;
    // strided gather / scatter with 2-D copies: n rows of one complex element, pitch = stride
    if (in_stride < 1 || out_stride < 1) { return fail(NEO_B200_ERR_INVALID, "strides must be positive"); }
    NEO_CUDA_TRY(cudaMemcpy2DAsync(plan->staging_in.ptr, elem, in, size_t(in_stride) * elem, elem, n, cudaMemcpyHostToDevice, s));
    NEO_TRY(fft_exec_device(plan, plan->staging_in.ptr, plan->staging_in.ptr, 1, direction));
    NEO_CUDA_TRY(cudaMemcpy2DAsync(out, size_t(out_stride) * elem, plan->staging_in.ptr, elem, elem, n, cudaMemcpyDeviceToHost, s));
    NEO_CUDA_TRY(cudaStreamSynchronize(s));
    return NEO_B200_OK;
}

// ---- rfft ----------------------------------------------------------------------------------------------------------------
int neo_b200_rfft_plan_create(neo_b200_rfft_plan** plan, size_t order, int dtype)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    *plan = nullptr;
    if (dtype != NEO_B200_F32 && dtype != NEO_B200_F64) { return fail(NEO_B200_ERR_INVALID, "bad dtype %d", dtype); }
    // fallback_rfft_plan owns an fft_plan of the same order (fallback_rfft_plan.hpp:58), so the same limit applies
    if (order > k_max_order) { return fail(NEO_B200_ERR_UNSUPPORTED, "neo_b200: unsupported order '%zu'", order); }
    NEO_TRY(require_device());
    auto p = std::unique_ptr<neo_b200_rfft_plan>(new (std::nothrow) neo_b200_rfft_plan{});
    if (!p) { return fail(NEO_B200_ERR_ALLOC, "out of host memory"); }
    p->order = order;
    p->dtype = dtype;
    NEO_CUDA_TRY(cudaGetDevice(&p->device));
    NEO_TRY(p->stream.create());
    if (dtype == NEO_B200_F32) { NEO_TRY(p->f32.init(static_cast<int>(order), p->stream.stream)); }
    else { NEO_TRY(p->f64.init(static_cast<int>(order), p->stream.stream)); }
    *plan = p.release();
    return NEO_B200_OK;
}

void neo_b200_rfft_plan_destroy(neo_b200_rfft_plan* plan)
{
    if (plan == nullptr) { return; }
    cudaStreamSynchronize(plan->stream.stream);
    delete plan;
}

size_t neo_b200_rfft_plan_order(neo_b200_rfft_plan const* plan) { return plan != nullptr ? plan->order : 0; }
size_t neo_b200_rfft_plan_size(neo_b200_rfft_plan const* plan) { return plan != nullptr ? size_t(1) << plan->order : 0; }

int neo_b200_rfft_plan_set_stream(neo_b200_rfft_plan* plan, void* cuda_stream)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    plan->stream.adopt(cuda_stream);
    return NEO_B200_OK;
}

int neo_b200_rfft_plan_synchronize(neo_b200_rfft_plan* plan)
{
    if (plan == nullptr) { return fail(NEO_B200_ERR_INVALID, "plan is null"); }
    NEO_CUDA_TRY(cudaStreamSynchronize(plan->stream.stream));
    return NEO_B200_OK;
}

static int rfft_device(neo_b200_rfft_plan* plan, void const* in, void* out, size_t batch)
{
    cudaStream_t const s = plan->stream.stream;
    if (plan->dtype == NEO_B200_F32) { return plan->f32.forward(static_cast<float const*>(in), static_cast<float2*>(out), batch, s); }
    return plan->f64.forward(static_cast<double const*>(in), static_cast<double2*>(out), batch, s);
}

static int irfft_device(neo_b200_rfft_plan* plan, void const* in, size_t row_len, void* out, size_t batch)
{
    cudaStream_t const s = plan->stream.stream;
    if (plan->dtype == NEO_B200_F32) {
        return plan->f32.backward(static_cast<float2 const*>(in), row_len, static_cast<float*>(out), batch, s);
    }
    return plan->f64.backward(static_cast<double2 const*>(in), row_len, static_cast<double*>(out), batch, s);
}

int neo_b200_rfft_exec(neo_b200_rfft_plan* plan, void const* in, void* out, size_t batch, int memspace)
{
    if (plan == nullptr || in == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (batch == 0) { return NEO_B200_OK; }
    NEO_CUDA_TRY(cudaSetDevice(plan->device));
    if (memspace == NEO_B200_DEVICE) { return rfft_device(plan, in, out, batch); }

    size_t const n       = size_t(1) << plan->order;
    size_t const in_row  = n * elem_size(plan->dtype);
    size_t const out_row = (n / 2 + 1) * 2 * elem_size(plan->dtype);
    size_t const chunk   = std::max<size_t>(1, std::min(batch, (size_t(256) << 20) / in_row));
    NEO_TRY(plan->staging_in.reserve(chunk * in_row));
    NEO_TRY(plan->staging_out.reserve(chunk * out_row));
    cudaStream_t const s = plan->stream.stream;
    for (size_t first = 0; first < batch; first += chunk) {
        size_t const cnt = std::min(chunk, batch - first);
        NEO_CUDA_TRY(cudaMemcpyAsync(plan->staging_in.ptr, static_cast<char const*>(in) + first * in_row, cnt * in_row, cudaMemcpyHostToDevice, s));
        NEO_TRY(rfft_device(plan, plan->staging_in.ptr, plan->staging_out.ptr, cnt));
        NEO_CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(out) + first * out_row, plan->staging_out.ptr, cnt * out_row, cudaMemcpyDeviceToHost, s));
    }
    NEO_CUDA_TRY(cudaStreamSynchronize(s));
    return NEO_B200_OK;
}

int neo_b200_irfft_exec(neo_b200_rfft_plan* plan, void const* in, size_t in_row_len, void* out, size_t batch, int memspace)
{
    if (plan == nullptr || in == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    size_t const n = size_t(1) << plan->order;
    if (in_row_len < n / 2 + 1) { return fail(NEO_B200_ERR_INVALID, "irfft needs at least N/2+1 = %zu bins per row, got %zu", n / 2 + 1, in_row_len); }
    if (batch == 0) { return NEO_B200_OK; }
    NEO_CUDA_TRY(cudaSetDevice(plan->device));
    if (memspace == NEO_B200_DEVICE) { return irfft_device(plan, in, in_row_len, out, batch); }

    size_t const in_row  = in_row_len * 2 * elem_size(plan->dtype);
    size_t const out_row = n * elem_size(plan->dtype);
    size_t const chunk   = std::max<size_t>(1, std::min(batch, (size_t(256) << 20) / in_row));
    NEO_TRY(plan->staging_in.reserve(chunk * in_row));
    NEO_TRY(plan->staging_out.reserve(chunk * out_row));
    cudaStream_t const s = plan->stream.stream;
    for (size_t first = 0; first < batch; first += chunk) {
        size_t const cnt = std::min(chunk, batch - first);
        NEO_CUDA_TRY(cudaMemcpyAsync(plan->staging_in.ptr, static_cast<char const*>(in) + first * in_row, cnt * in_row, cudaMemcpyHostToDevice, s));
        NEO_TRY(irfft_device(plan, plan->staging_in.ptr, in_row_len, plan->staging_out.ptr, cnt));
        NEO_CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(out) + first * out_row, plan->staging_out.ptr, cnt * out_row, cudaMemcpyDeviceToHost, s));
    }
    NEO_CUDA_TRY(cudaStreamSynchronize(s));
    return NEO_B200_OK;
}

}  // extern "C"
