// fft_large.cuh -- transforms too long for one CTA (more than 2^13 complex float / 2^12 complex double points).
//
// Bailey four-step over global memory, N = N1*N2, n = n1*N2 + n2, k = k1 + N1*k2:
//   (1) column pass : N2 strided FFTs of length N1 (<= 2^10), 16 adjacent columns per CTA so that every global access is
//                     a full 128-byte segment, fused with the W_N^(k1*n2) twiddle;
//   (2) row pass    : N1 contiguous FFTs of length N2 (single-CTA kernel, or this scheme again when N2 is itself too long);
//   (3) transpose   : [N1][N2] -> [N2][N1] through shared-memory tiles.
// The batch is walked in chunks whose scratch copy fits the 126 MB L2, so passes (2),(3) read what the previous pass
// just wrote from L2 instead of HBM. The reference covers these sizes with the same radix-2 loop as the small ones
// (c2c_dit2_plan.hpp:59-62: max_order 27); this keeps the same API range.
#pragma once

#include "fft_kernels.cuh"

#include <algorithm>
#include <memory>

namespace neo_b200 {

// W_N^j = hi[j >> lo_bits] * lo[j & mask]: two short tables instead of an N-entry LUT (N up to 2^28)
template<typename T>
struct twiddle2_view
{
    cx<T> const* hi;
    cx<T> const* lo;
    int lo_bits;

    template<int DIR>
    __device__ __forceinline__ cx<T> get(size_t j) const
    {
        cx<T> const w = cmul(__ldg(hi + (j >> lo_bits)), __ldg(lo + (j & ((size_t(1) << lo_bits) - 1))));
        return DIR < 0 ? w : cconj(w);
    }
};

template<typename T>
struct twiddle2
{
    device_buffer hi, lo;
    int lo_bits{0};

    // tables for W_N, N = 2^logn, forward sign
    int build(int logn, cudaStream_t stream)
    {
        lo_bits             = (logn + 1) / 2;
        size_t const n_lo   = size_t(1) << lo_bits;
        size_t const n_hi   = size_t(1) << (logn - lo_bits);
        double const two_pi = 2.0 * 3.14159265358979323846264338327950288;
        double const n      = std::ldexp(1.0, logn);
        std::vector<cx<T>> h(n_hi), l(n_lo);
        for (size_t i = 0; i < n_hi; ++i) {
            double const a = -two_pi * (double(i) * double(n_lo)) / n;
            h[i]           = mk<T>(T(std::cos(a)), T(std::sin(a)));
        }
        for (size_t i = 0; i < n_lo; ++i) {
            double const a = -two_pi * double(i) / n;
            l[i]           = mk<T>(T(std::cos(a)), T(std::sin(a)));
        }
        NEO_TRY(hi.reserve(n_hi * sizeof(cx<T>)));
        NEO_TRY(lo.reserve(n_lo * sizeof(cx<T>)));
        NEO_CUDA_TRY(cudaMemcpyAsync(hi.ptr, h.data(), n_hi * sizeof(cx<T>), cudaMemcpyHostToDevice, stream));
        NEO_CUDA_TRY(cudaMemcpyAsync(lo.ptr, l.data(), n_lo * sizeof(cx<T>), cudaMemcpyHostToDevice, stream));
        NEO_CUDA_TRY(cudaStreamSynchronize(stream));
        return NEO_B200_OK;
    }

    twiddle2_view<T> view() const { return {hi.template as<cx<T>>(), lo.template as<cx<T>>(), lo_bits}; }
};

// ---- (1) column pass -------------------------------------------------------------------------------------------------
template<typename T, int LOGL>
struct col_cfg
{
    using F                      = cta_fft<T, LOGL, -1>;
    static constexpr int E       = F::E;
    static constexpr int TN      = F::TN;
    static constexpr int L       = F::M;
    static constexpr int G0      = 128 / int(sizeof(cx<T>));             // columns that fill one 128-byte segment
    static constexpr int G       = (128 / TN) > G0 ? (128 / TN) : G0;  // adjacent columns per CTA
    static constexpr int THREADS = TN * G;
    static constexpr size_t SMEM = size_t(G) * F::TILE * sizeof(cx<T>);
};

// data: [batch][L][cols]; FFT along the L axis of every column, then *= W_(L*cols)^(k1 * col)
template<typename T, int LOGL, int DIR>
__global__ void __launch_bounds__(col_cfg<T, LOGL>::THREADS)
    col_pass_kernel(cx<T> const* in, cx<T>* out, cx<T> const* __restrict__ tw, twiddle2_view<T> big, size_t cols)
{
    using cfg = col_cfg<T, LOGL>;
    using F   = cta_fft<T, LOGL, DIR>;
    using C   = cx<T>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int const g      = threadIdx.x % cfg::G;
    int const t      = threadIdx.x / cfg::G;
    C* sm            = reinterpret_cast<C*>(smem_raw) + g * F::TILE;
    size_t const col = size_t(blockIdx.x) * cfg::G + g;  // cols is a multiple of G (power of two >= 2^10)
    size_t const mat = size_t(blockIdx.y) * cfg::L * cols;

    C v[cfg::E];
#pragma unroll
    for (int e = 0; e < cfg::E; ++e) { v[e] = in[mat + size_t(t + e * cfg::TN) * cols + col]; }
    F::run(v, sm, tw, t);
#pragma unroll
    for (int e = 0; e < cfg::E; ++e) {
        size_t const k1 = size_t(t + e * cfg::TN);
        out[mat + k1 * cols + col] = cmul(v[e], big.template get<DIR>(k1 * col));
    }
}

// ---- (3) transpose [rows][cols] -> [cols][rows] per batch entry -------------------------------------------------------------
template<typename T>
__global__ void __launch_bounds__(256) transpose_kernel(cx<T> const* __restrict__ in, cx<T>* __restrict__ out, size_t rows, size_t cols)
{
    __shared__ cx<T> tile[32][33];
    size_t const mat = size_t(blockIdx.z) * rows * cols;
    size_t const c0  = size_t(blockIdx.x) * 32;
    size_t const r0  = size_t(blockIdx.y) * 32;
    int const tx     = threadIdx.x % 32;
    int const ty     = threadIdx.x / 32;  // 0..7
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
        size_t const r = r0 + ty + i, c = c0 + tx;
        if (r < rows && c < cols) { tile[ty + i][tx] = in[mat + r * cols + c]; }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
        size_t const c = c0 + ty + i, r = r0 + tx;
        if (r < rows && c < cols) { out[mat + c * rows + r] = tile[tx][ty + i]; }
    }
}

template<typename T>
int launch_transpose(cx<T> const* in, cx<T>* out, size_t batch, size_t rows, size_t cols, cudaStream_t stream)
{
    // gridDim.z <= 65535: walk the batch in slabs
    for (size_t first = 0; first < batch; first += 65535) {
        size_t const n = std::min<size_t>(65535, batch - first);
        dim3 const grid(static_cast<unsigned>((cols + 31) / 32), static_cast<unsigned>((rows + 31) / 32), static_cast<unsigned>(n));
        transpose_kernel<T><<<grid, 256, 0, stream>>>(in + first * rows * cols, out + first * rows * cols, rows, cols);
        NEO_TRY(check_launch("transpose_kernel"));
    }
    return NEO_B200_OK;
}

// ---- the recursive plan --------------------------------------------------------------------------------------------------
template<typename T>
struct large_fft
{
    static constexpr int k_max_col = 10;  // column FFTs: 2^10 points * 16 columns = 1024 threads

    int logn{0};
    int log1{0}, log2{0};               // N = 2^log1 (columns pass) * 2^log2 (rows)
    fft_tables<T> col_tables;           // stage twiddles of the column FFT
    fft_tables<T> row_tables;           // stage twiddles of the row FFT (when it fits one CTA)
    twiddle2<T> big;                    // W_N
    std::unique_ptr<large_fft<T>> rows; // rows too long for one CTA
    device_buffer scratch;

    int init(int logn_, cudaStream_t stream)
    {
        logn = logn_;
        log2 = std::min(max_cta_logm<T>(), logn - 1);
        log1 = logn - log2;
        if (log1 > k_max_col) {
            log1 = k_max_col;
            log2 = logn - log1;
        }
        NEO_TRY(col_tables.build(log1, false, stream));
        NEO_TRY(big.build(logn, stream));
        if (log2 > max_cta_logm<T>()) {
            rows = std::make_unique<large_fft<T>>();
            NEO_TRY(rows->init(log2, stream));
        } else {
            NEO_TRY(row_tables.build(log2, false, stream));
        }
        return NEO_B200_OK;
    }

    template<int DIR>
    int col_pass(cx<T> const* in, cx<T>* out, size_t batch, cudaStream_t stream)
    {
        int status        = NEO_B200_ERR_UNSUPPORTED;
        size_t const cols = size_t(1) << log2;
        NEO_DISPATCH_LOGM(T, log1, {
            if constexpr (LOGM >= 1 && LOGM <= k_max_col) {
                using cfg   = col_cfg<T, LOGM>;
                auto kernel = col_pass_kernel<T, LOGM, DIR>;
                NEO_TRY(enable_smem(kernel, cfg::SMEM));
                for (size_t first = 0; first < batch; first += 65535) {
                    size_t const n = std::min<size_t>(65535, batch - first);
                    dim3 const grid(static_cast<unsigned>(cols / cfg::G), static_cast<unsigned>(n));
                    size_t const off = first << logn;
                    kernel<<<grid, cfg::THREADS, cfg::SMEM, stream>>>(in + off, out + off, col_tables.tw(), big.view(), cols);
                    NEO_TRY(check_launch("col_pass_kernel"));
                }
                status = NEO_B200_OK;
            }
        });
        if (status != NEO_B200_OK) { return fail(status, "column pass of 2^%d points not supported", log1); }
        return status;
    }

    int row_pass(cx<T>* data, size_t nrows, int direction, cudaStream_t stream)
    {
        if (rows) { return rows->exec(data, data, nrows, direction, stream); }
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_DISPATCH_LOGM(T, log2, {
            if constexpr (LOGM <= max_cta_logm<T>()) {
                status = direction < 0 ? launch_c2c<T, LOGM, -1>(data, data, row_tables.tw(), nrows, stream)
                                       : launch_c2c<T, LOGM, +1>(data, data, row_tables.tw(), nrows, stream);
            }
        });
        return status;
    }

    // [batch][N] contiguous; in == out allowed
    int exec(cx<T> const* in, cx<T>* out, size_t batch, int direction, cudaStream_t stream)
    {
        size_t const n     = size_t(1) << logn;
        size_t const bytes = n * sizeof(cx<T>);
        // chunk so that the scratch copy stays L2-resident between the passes (at least one transform)
        size_t const chunk = std::max<size_t>(1, std::min(batch, (size_t(32) << 20) / bytes));
        NEO_TRY(scratch.reserve(chunk * bytes));
        cx<T>* const s = scratch.template as<cx<T>>();
        for (size_t first = 0; first < batch; first += chunk) {
            size_t const cnt = std::min(chunk, batch - first);
            if (direction < 0) { NEO_TRY(col_pass<-1>(in + first * n, s, cnt, stream)); }
            else { NEO_TRY(col_pass<+1>(in + first * n, s, cnt, stream)); }
            NEO_TRY(row_pass(s, cnt << log1, direction, stream));
            NEO_TRY(launch_transpose<T>(s, out + first * n, cnt, size_t(1) << log1, size_t(1) << log2, stream));
        }
        return NEO_B200_OK;
    }
};

// ---- real transforms past the one- and two-CTA forms: half-size complex FFT + split pass over global memory (rfft_engine) -------
template<typename T, int DIR>
__global__ void __launch_bounds__(256) split_pass_kernel(cx<T> const* __restrict__ in, size_t in_row, cx<T>* __restrict__ out, size_t out_row,
                                                         twiddle2_view<T> w2m, size_t m)
{
    // DIR < 0: in = Z[batch][M]   -> out = X[batch][M+1]   (r2c post-pass)
    // DIR > 0: in = X[batch][>=M+1] -> out = Z[batch][M]   (c2r pre-pass)
    size_t const b = blockIdx.y;
    size_t const k = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    cx<T> const* src = in + b * in_row;
    cx<T>* dst       = out + b * out_row;
    if (k >= m) { return; }
    if (k == 0) {
        if constexpr (DIR < 0) {
            cx<T> const z = src[0];
            dst[0]        = mk<T>(z.x + z.y, T(0));
            dst[m]        = mk<T>(z.x - z.y, T(0));
        } else {
            T const a0 = src[0].x, am = src[m].x;
            dst[0]     = mk<T>(a0 + am, a0 - am);
        }
        return;
    }
    cx<T> const a = src[k];
    cx<T> const p = src[m - k];
    cx<T> const w = w2m.template get<-1>(k);
    dst[k]        = DIR < 0 ? r2c_post(a, p, w) : c2r_pre(a, p, w);
}

// N = 1 (rfft_engine): the spectrum is the sample, and back
template<typename T>
__global__ void size_one_r2c_kernel(T const* in, cx<T>* out, size_t batch)
{
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < batch) { out[i] = mk<T>(in[i], T(0)); }
}

template<typename T>
__global__ void size_one_c2r_kernel(cx<T> const* in, size_t row_len, T* out, size_t batch)
{
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < batch) { out[i] = in[i * row_len].x; }
}

}  // namespace neo_b200
