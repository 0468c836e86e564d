// conv_kernels.cuh -- device side of the uniformly partitioned convolver bank.
//
// Reference per block and channel (src/neo/convolution/uniform_partitioned_convolver.hpp:48-65, overlap_save.hpp:85-112):
//   slide window, rfft(2B), FDL insert, clear accumulator, P x multiply_add(fdl[s], H[(w+P-s)%P]), irfft, scale, keep last B.
// Here, per call of T blocks over a bank of channels, three kernels:
//   r2c_kernel<conv_r2c_io>   window assembly + r2c + FDL insert fused        (K3, K5, K6 of SURVEY 2a)
//   fdl_mac_*                 the spectral multiply-accumulate                 (K7, K8)
//   c2r_kernel<conv_c2r_io>   partial-sum gather + c2r + 1/N scale + discard   (K4, K9, K10)
//
// HBM layout. Every spectrum row is B = N/2 complex elements: bin 0 carries (Re X[0], Re X[B]) because both are real.
// FDL and filter rows are cut into tiles of W elements (1 KB) and stored tile-major, so that the rows one CTA walks
// (one tile column of one channel) are contiguous and a pipeline stage is ONE bulk copy:
//   fdl    [inputs][B/W][R][W]             ring of spectra, R = partition_end + max_blocks - 1 slots, slot(n) = n mod R
//   filter [outputs*sources][B/W][Pl][W]   Pl local partitions, sources = 1 (diagonal) or inputs (matrix)
//   acc    [S][outputs][T][B]              S partial planes (split over partitions so small banks still fill the GPU)
#pragma once

#include "fft_kernels.cuh"

namespace neo_b200 {

// fdl_index (src/neo/convolution/fdl_index.hpp:28-31): the filter row paired with FDL row `segment` when the newest
// spectrum sits in row `write_pos` of a P-row ring. The MAC kernels pair rows by age = (write_pos - segment) mod P,
// which is this value; neo_b200_fdl_index_sequence evaluates the same function on the device.
__host__ __device__ __forceinline__ unsigned fdl_filter_index(unsigned write_pos, unsigned segment, unsigned parts)
{
    return (write_pos + parts - segment) % parts;
}

// complex elements per 1 KB tile
template<typename T>
__host__ __device__ constexpr int tile_width()
{
    return 1024 / int(sizeof(cx<T>));
}

// element offset of (chan, row, k) in a tile-major array with `rows` rows per channel
__host__ __device__ __forceinline__ size_t tiled_offset(size_t chan, int nt, int logw, size_t rows, size_t row, int k)
{
    return (((chan * nt + size_t(k >> logw)) * rows + row) << logw) + size_t(k & ((1 << logw) - 1));
}

struct mac_geom
{
    int m;             // complex elements per row (= B)
    int logw;          // log2 of the tile width W = min(B, tile_width)
    int nt;            // tiles per row = B / W
    int ring;          // R
    int parts;         // Pl, partitions held by this handle
    int age0;          // age of the first local partition (= partition_begin)
    int sources;       // FDL channels summed per output
    int diagonal;      // 1: source channel = output channel
    int wp;            // ring slot of the first block of this launch
    int blocks;        // T of the whole call (row stride of acc)
    int tau0;          // first block of this launch inside the call
    int splits;        // S
    int out0;          // first output channel of this launch (blockIdx.y is relative to it)
    int packed_edge;   // 1: element 0 of a row is the packed pair (Re X[0], Re X[B]); 0: an ordinary complex bin (frame level)
    size_t acc_plane;  // elements per partial plane
    unsigned* tickets; // one counter per (blockIdx.x, output row of the grid): which split CTA finishes last
};

// Small banks split the partition loop over gridDim.z CTAs, each leaving a partial plane. The LAST of them to finish (ticket
// counter) folds the planes into plane 0 in plane order -- deterministic, no float atomics, and the c2r kernel reads one plane.
// Every thread of the CTA must call it; `mine` says whether this thread owns elements; they sit at acc[first + r*stride].
template<typename V>
__device__ __forceinline__ void fold_split_planes(V* acc, size_t plane, int splits, bool mine, size_t first, int rows, size_t stride,
                                                   unsigned* ticket)
{
    if (splits <= 1) { return; }
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned const t = atomicAdd(ticket, 1U);
        is_last          = (t == unsigned(splits) - 1U);
        if (is_last) { *ticket = 0U; }  // ready for the next launch
    }
    __syncthreads();
    if (!is_last || !mine) { return; }
    __threadfence();
    for (int r = 0; r < rows; ++r) {
        V* const p0 = acc + first + size_t(r) * stride;
        V s         = __ldcg(p0);
        for (int p = 1; p < splits; ++p) {
            V const v = __ldcg(p0 + size_t(p) * plane);
            s.x += v.x;
            s.y += v.y;
            if constexpr (sizeof(V) == 16 && sizeof(s.x) == 4) {
                s.z += v.z;
                s.w += v.w;
            }
        }
        *p0 = s;
    }
}

// ---- T = 1: pure stream. Every filter and FDL element is used exactly once -> HBM roofline. -------------------------------
// thread = VEC adjacent bins (16 bytes), 8 rows in flight per thread.
template<typename T>
struct mac_vec;
template<>
struct mac_vec<float>
{
    using type               = float4;
    static constexpr int VEC = 2;
    static __device__ __forceinline__ void cfma(float4& a, float4 const x, float4 const h)
    {
        a.x = fmaf(x.x, h.x, a.x);
        a.x = fmaf(-x.y, h.y, a.x);
        a.y = fmaf(x.x, h.y, a.y);
        a.y = fmaf(x.y, h.x, a.y);
        a.z = fmaf(x.z, h.z, a.z);
        a.z = fmaf(-x.w, h.w, a.z);
        a.w = fmaf(x.z, h.w, a.w);
        a.w = fmaf(x.w, h.z, a.w);
    }
    // packed bin 0 = (Re X0, Re XB): two independent real products
    static __device__ __forceinline__ void cfma_edge(float4& a, float4 const x, float4 const h)
    {
        a.x = fmaf(x.x, h.x, a.x);
        a.y = fmaf(x.y, h.y, a.y);
        a.z = fmaf(x.z, h.z, a.z);
        a.z = fmaf(-x.w, h.w, a.z);
        a.w = fmaf(x.z, h.w, a.w);
        a.w = fmaf(x.w, h.z, a.w);
    }
    static __device__ __forceinline__ float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
};
template<>
struct mac_vec<double>
{
    using type               = double2;
    static constexpr int VEC = 1;
    static __device__ __forceinline__ void cfma(double2& a, double2 const x, double2 const h)
    {
        a.x = ::fma(x.x, h.x, a.x);
        a.x = ::fma(-x.y, h.y, a.x);
        a.y = ::fma(x.x, h.y, a.y);
        a.y = ::fma(x.y, h.x, a.y);
    }
    static __device__ __forceinline__ void cfma_edge(double2& a, double2 const x, double2 const h)
    {
        a.x = ::fma(x.x, h.x, a.x);
        a.y = ::fma(x.y, h.y, a.y);
    }
    static __device__ __forceinline__ double2 zero() { return make_double2(0.0, 0.0); }
};

template<typename V>
__device__ __forceinline__ V ld_stream(V const* p)
{
    return __ldcs(p);  // read-once data: evict-first
}

constexpr int k_mac_threads = 128;
constexpr int k_mac_unroll  = 8;

// OT outputs per thread: in the matrix topology the same FDL row feeds every output, so it is loaded once per OT filter rows.
template<typename T, int OT>
__global__ void __launch_bounds__(k_mac_threads)
    fdl_mac_stream_kernel(cx<T> const* __restrict__ fdl, cx<T> const* __restrict__ filter, cx<T>* __restrict__ acc, mac_geom g)
{
    using MV           = mac_vec<T>;
    using V            = typename MV::type;
    constexpr int UNR  = OT == 1 ? k_mac_unroll : 4;
    int const col      = blockIdx.x * k_mac_threads + threadIdx.x;  // in units of V
    int const out0     = blockIdx.y * OT + g.out0;
    int const split    = blockIdx.z;
    int const row_vec  = g.m / MV::VEC;
    bool const mine    = col < row_vec;

    int const total = g.sources * g.parts;  // virtual partitions of one output
    int const v0    = int((long long)total * split / g.splits);
    int const v1    = mine ? int((long long)total * (split + 1) / g.splits) : v0;

    V a[OT];
#pragma unroll
    for (int o = 0; o < OT; ++o) { a[o] = MV::zero(); }
    bool const edge = (col == 0) && g.packed_edge != 0;  // this thread owns the packed bin 0

    // tile-major addressing in units of V (VEC elements)
    int const k0       = col * MV::VEC;
    int const tile     = k0 >> g.logw;
    int const tile_vec = (1 << g.logw) / MV::VEC;
    int const within   = (k0 & ((1 << g.logw) - 1)) / MV::VEC;
    V const* const fbase = reinterpret_cast<V const*>(filter) + within;
    V const* const xbase = reinterpret_cast<V const*>(fdl) + within;
    size_t const ostride = size_t(g.sources) * g.nt * g.parts * tile_vec;  // V elements between consecutive outputs' filters

    for (int v = v0; v < v1; v += UNR) {
        V x[UNR], h[UNR][OT];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            int const vp = v + u;
            if (vp < v1) {
                int const src = vp / g.parts;
                int const p   = vp - src * g.parts;
                int slot      = g.wp - g.age0 - p;
                slot          = slot % g.ring;
                slot += slot < 0 ? g.ring : 0;
                int const ch         = g.diagonal ? out0 : src;
                V const* const hrow = fbase + (((size_t(out0) * g.sources + src) * g.nt + tile) * g.parts + p) * tile_vec;
#pragma unroll
                for (int o = 0; o < OT; ++o) { h[u][o] = ld_stream(hrow + o * ostride); }
                x[u] = OT == 1 ? ld_stream(xbase + ((size_t(ch) * g.nt + tile) * g.ring + slot) * tile_vec)
                               : xbase[((size_t(ch) * g.nt + tile) * g.ring + slot) * tile_vec];
            } else {
#pragma unroll
                for (int o = 0; o < OT; ++o) { h[u][o] = MV::zero(); }
                x[u] = MV::zero();
            }
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
#pragma unroll
            for (int o = 0; o < OT; ++o) {
                if (edge) { MV::cfma_edge(a[o], x[u], h[u][o]); }
                else { MV::cfma(a[o], x[u], h[u][o]); }
            }
        }
    }
    size_t const first = (size_t(out0) * g.blocks + g.tau0) * row_vec + col;
    if (mine) {
#pragma unroll
        for (int o = 0; o < OT; ++o) {
            reinterpret_cast<V*>(acc)[size_t(split) * (g.acc_plane / MV::VEC) + first + size_t(o) * g.blocks * row_vec] = a[o];
        }
    }
    fold_split_planes(reinterpret_cast<V*>(acc), g.acc_plane / MV::VEC, g.splits, mine, first, OT, size_t(g.blocks) * row_vec,
                      g.tickets + (size_t(blockIdx.y) * gridDim.x + blockIdx.x));
}

// ---- T = TB > 1: Toeplitz form. acc[tau] += H[p] * X(tau - age0 - p); each H[p] is reused TB times from registers and
// each spectrum up to TB times, so bytes per block drop ~TB-fold until FP32 FMA throughput binds. thread = one bin. ------------
template<typename T, int TB>
__global__ void __launch_bounds__(k_mac_threads)
    fdl_mac_toeplitz_kernel(cx<T> const* __restrict__ fdl, cx<T> const* __restrict__ filter, cx<T>* __restrict__ acc, mac_geom g)
{
    using C         = cx<T>;
    int const k     = blockIdx.x * k_mac_threads + threadIdx.x;
    int const out   = blockIdx.y + g.out0;
    int const split = blockIdx.z;
    bool const mine = k < g.m;
    bool const edge = (k == 0);

    int const chunks_per_src = (g.parts + TB - 1) / TB;
    int const total          = g.sources * chunks_per_src;
    int const c0             = int((long long)total * split / g.splits);
    int const c1             = mine ? int((long long)total * (split + 1) / g.splits) : c0;

    C a[TB];
#pragma unroll
    for (int i = 0; i < TB; ++i) { a[i] = mk<T>(0, 0); }

    C win[2 * TB - 1];
    int prev_src = -1;
    int slot_lo  = 0;  // ring slot of win[0]
    size_t xbase = 0;

    for (int c = c0; c < c1; ++c) {
        int const src = c / chunks_per_src;
        int const p0  = (c - src * chunks_per_src) * TB;
        if (src != prev_src) {
            // fresh window: pretend a previous chunk at p0 - TB left its lower TB-1 entries behind
            int const ch = g.diagonal ? out : src;
            xbase        = tiled_offset(size_t(ch), g.nt, g.logw, size_t(g.ring), 0, k);
            int base     = g.wp - g.age0 - p0 + 1;  // d of win[0] of that virtual previous chunk: -(age0 + p0 - TB) - (TB-1)
            base         = base % g.ring;
            base += base < 0 ? g.ring : 0;
            slot_lo = base;
            int s   = base;
#pragma unroll
            for (int i = 0; i < TB - 1; ++i) {
                win[i] = fdl[xbase + (size_t(s) << g.logw)];
                s      = (s + 1 == g.ring) ? 0 : s + 1;
            }
            prev_src = src;
        }
        // shift: entries [0, TB-1) become [TB, 2TB-1); then load TB older spectra below them
#pragma unroll
        for (int i = TB - 2; i >= 0; --i) { win[i + TB] = win[i]; }
        slot_lo -= TB;
        slot_lo += slot_lo < 0 ? g.ring : 0;
        {
            int s = slot_lo;
#pragma unroll
            for (int i = 0; i < TB; ++i) {
                win[i] = fdl[xbase + (size_t(s) << g.logw)];
                s      = (s + 1 == g.ring) ? 0 : s + 1;
            }
        }
        C const* hrow = filter + tiled_offset(size_t(out) * g.sources + src, g.nt, g.logw, size_t(g.parts), size_t(p0), k);
#pragma unroll
        for (int pp = 0; pp < TB; ++pp) {
            if (p0 + pp < g.parts) {
                C const h = __ldcs(hrow + (size_t(pp) << g.logw));
#pragma unroll
                for (int tau = 0; tau < TB; ++tau) {
                    C const x = win[tau - pp + TB - 1];
                    if (edge) {
                        a[tau].x = fma(x.x, h.x, a[tau].x);
                        a[tau].y = fma(x.y, h.y, a[tau].y);
                    } else {
                        a[tau].x = fma(x.x, h.x, a[tau].x);
                        a[tau].x = fma(-x.y, h.y, a[tau].x);
                        a[tau].y = fma(x.x, h.y, a[tau].y);
                        a[tau].y = fma(x.y, h.x, a[tau].y);
                    }
                }
            }
        }
    }
    size_t const first = (size_t(out) * g.blocks + g.tau0) * g.m + k;
    if (mine) {
        C* dst = acc + size_t(split) * g.acc_plane + first;
#pragma unroll
        for (int tau = 0; tau < TB; ++tau) { dst[size_t(tau) * g.m] = a[tau]; }
    }
    fold_split_planes(acc, g.acc_plane, g.splits, mine, first, TB, size_t(g.m), g.tickets + (size_t(blockIdx.y) * gridDim.x + blockIdx.x));
}

// ---- the same Toeplitz MAC for float32 rows of at least one full tile, fed by TMA -------------------------------------------------
// CTA = 128 threads = one tile column (128 bins, 1 KB per row) of one output. The partition loop advances CH rows per
// pipeline stage; thanks to the tile-major layout the CH filter rows are one contiguous CH KB block and so are the CH FDL
// rows (two blocks where the ring wraps), fetched with cp.async.bulk into shared memory and signalled through an mbarrier.
// STAGES-1 stages are in flight while the FMAs of the current one issue: the loads never sit in registers, so the kernel
// is bound by FP32 issue (TB large) or HBM (TB small) instead of load latency.
namespace tma {

__device__ __forceinline__ unsigned smem_addr(void const* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(void* bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

__device__ __forceinline__ void mbar_expect_tx(void* bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(void* bar, unsigned parity)
{
    unsigned ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_addr(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}

__device__ __forceinline__ void mbar_wait(void* bar, unsigned parity)
{
    while (!mbar_try_wait(bar, parity)) {}
}

// global -> shared bulk copy (TMA, SASS UBLKCP); bytes and both addresses are multiples of 16
__device__ __forceinline__ void bulk_g2s(void* dst, void const* src, unsigned bytes, void* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}

}  // namespace tma

template<int TB, int CH, int STAGES>
struct mac_tma_cfg
{
    static constexpr int W         = 128;                       // bins per CTA = one float2 tile
    static constexpr int WARPS     = 4;
    static constexpr int STAGE_EL  = 2 * CH * W;                // float2 elements per stage: CH filter rows + CH FDL rows
    static constexpr size_t SMEM   = size_t(STAGES) * STAGE_EL * sizeof(float2) + STAGES * (sizeof(unsigned long long) + sizeof(int));
};

// RAGGED: the partition count is not a multiple of CH, the last chunk of every source is predicated.
template<int TB, int CH, int STAGES, bool RAGGED>
__global__ void __launch_bounds__(128)
    fdl_mac_tma_kernel(float2 const* __restrict__ fdl, float2 const* __restrict__ filter, float2* __restrict__ acc, mac_geom g)
{
    using cfg = mac_tma_cfg<TB, CH, STAGES>;
    constexpr int W = cfg::W;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* const stage_mem        = reinterpret_cast<float2*>(smem_raw);
    unsigned long long* const full = reinterpret_cast<unsigned long long*>(smem_raw + size_t(STAGES) * cfg::STAGE_EL * sizeof(float2));
    int* const done                = reinterpret_cast<int*>(full + STAGES);  // warps finished with the stage

    int const tid   = threadIdx.x;
    int const lane  = tid & 31;
    int const tile  = blockIdx.x;
    int const out   = blockIdx.y + g.out0;
    int const split = blockIdx.z;
    bool const edge = (tile == 0 && tid == 0);  // packed bin 0: (Re X0, Re XB) are two real products

    int const chunks_per_src = (g.parts + CH - 1) / CH;
    int const total          = g.sources * chunks_per_src;
    int const c0             = int((long long)total * split / g.splits);
    int const c1             = int((long long)total * (split + 1) / g.splits);

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            tma::mbar_init(&full[s], 1);
            done[s] = 0;
        }
        tma::fence_mbar_init();
    }
    __syncthreads();

    // fill stage (c - c0) % STAGES with chunk c: one bulk copy of filter rows, one (two at the ring wrap) of FDL rows
    auto issue = [&](int c) {
        int const src   = c / chunks_per_src;
        int const p0    = (c - src * chunks_per_src) * CH;
        int const ch    = g.diagonal ? out : src;
        int const st    = (c - c0) % STAGES;
        float2* const h = stage_mem + size_t(st) * cfg::STAGE_EL;
        float2* const x = h + CH * W;
        int const hrows = RAGGED ? min(CH, g.parts - p0) : CH;
        // FDL rows: the CH spectra just older than the previous chunk's, ascending ring slots starting at `lo`
        int lo = g.wp - g.age0 - p0 - CH + 1;
        lo %= g.ring;
        lo += lo < 0 ? g.ring : 0;
        int const first = min(CH, g.ring - lo);
        tma::mbar_expect_tx(&full[st], unsigned((hrows + CH) * W * sizeof(float2)));
        tma::bulk_g2s(h, filter + ((((size_t(out) * g.sources + src) * g.nt + tile) * g.parts + p0) << 7), unsigned(hrows * W * sizeof(float2)),
                      &full[st]);
        float2 const* const xrows = fdl + (((size_t(ch) * g.nt + tile) * g.ring) << 7);
        tma::bulk_g2s(x, xrows + (size_t(lo) << 7), unsigned(first * W * sizeof(float2)), &full[st]);
        if (first < CH) { tma::bulk_g2s(x + first * W, xrows, unsigned((CH - first) * W * sizeof(float2)), &full[st]); }
    };

    if (tid == 0) {
        for (int c = c0; c < c1 && c < c0 + STAGES; ++c) { issue(c); }
    }

    float2 a[TB];
#pragma unroll
    for (int i = 0; i < TB; ++i) { a[i] = make_float2(0.f, 0.f); }
    float2 win[TB + CH - 1];  // win[i] = X(d0 + i), d0 = -(age0 + p0) - CH + 1 for the chunk being consumed

    int src = c0 / chunks_per_src;
    int p0  = (c0 - src * chunks_per_src) * CH;
    bool fresh = true;
    int st = 0;
    unsigned parity = 0;

    for (int c = c0; c < c1; ++c) {
        if (fresh) {
            // the TB-1 spectra newer than X(-(age0+p0)), straight from global memory (once per source)
            int const ch = g.diagonal ? out : src;
            float2 const* const xcol = fdl + (((size_t(ch) * g.nt + tile) * g.ring) << 7) + tid;
            int s = g.wp - g.age0 - p0 + 1;
            s %= g.ring;
            s += s < 0 ? g.ring : 0;
#pragma unroll
            for (int i = 0; i < TB - 1; ++i) {
                win[i] = xcol[size_t(s) << 7];
                s      = (s + 1 == g.ring) ? 0 : s + 1;
            }
            fresh = false;
        }
#pragma unroll
        for (int i = TB - 2; i >= 0; --i) { win[i + CH] = win[i]; }

        tma::mbar_wait(&full[st], parity);
        float2 const* const h = stage_mem + size_t(st) * cfg::STAGE_EL + tid;
        float2 const* const x = h + CH * W;
        float2 hreg[CH];
#pragma unroll
        for (int i = 0; i < CH; ++i) {
            win[i]  = x[i * W];
            hreg[i] = h[i * W];
        }

        // the stage now lives in registers: release it BEFORE the FMAs so the refill flies during this chunk's compute.
        // No CTA barrier: the last of the four warps to get here re-arms the mbarrier and issues the bulk copies.
        __syncwarp();
        if (lane == 0) {
            __threadfence_block();
            int const before = atomicAdd(&done[st], 1);
            if (before == cfg::WARPS - 1) {
                done[st] = 0;
                if (c + STAGES < c1) { issue(c + STAGES); }
            }
        }
        __syncwarp();

        if (!edge) {
#pragma unroll
            for (int pp = 0; pp < CH; ++pp) {
                if (!RAGGED || p0 + pp < g.parts) {
                    float2 const hv = hreg[pp];
#pragma unroll
                    for (int tau = 0; tau < TB; ++tau) {
                        float2 const xv = win[tau - pp + CH - 1];
                        a[tau].x = fmaf(xv.x, hv.x, a[tau].x);
                        a[tau].x = fmaf(-xv.y, hv.y, a[tau].x);
                        a[tau].y = fmaf(xv.x, hv.y, a[tau].y);
                        a[tau].y = fmaf(xv.y, hv.x, a[tau].y);
                    }
                }
            }
        } else {
#pragma unroll
            for (int pp = 0; pp < CH; ++pp) {
                if (!RAGGED || p0 + pp < g.parts) {
                    float2 const hv = hreg[pp];
#pragma unroll
                    for (int tau = 0; tau < TB; ++tau) {
                        float2 const xv = win[tau - pp + CH - 1];
                        a[tau].x = fmaf(xv.x, hv.x, a[tau].x);
                        a[tau].y = fmaf(xv.y, hv.y, a[tau].y);
                    }
                }
            }
        }

        p0 += CH;
        if (p0 >= g.parts) {
            p0 = 0;
            ++src;
            fresh = true;
        }
        if (++st == STAGES) {
            st = 0;
            parity ^= 1U;
        }
    }

    size_t const first = (size_t(out) * g.blocks + g.tau0) * g.m + tile * W + tid;
    float2* dst        = acc + size_t(split) * g.acc_plane + first;
#pragma unroll
    for (int tau = 0; tau < TB; ++tau) { dst[size_t(tau) * g.m] = a[tau]; }
    fold_split_planes(acc, g.acc_plane, g.splits, true, first, TB, size_t(g.m), g.tickets + (size_t(blockIdx.y) * gridDim.x + blockIdx.x));
}

// ---- forward side: window assembly + r2c + FDL insert ---------------------------------------------------------------------------
// ROWS: the destination rows are plain [slot][B] rows (frame mode's two-frame buffer) instead of 1 KB tiles
template<typename T, int LOGM, bool ROWS = false>
struct conv_r2c_io
{
    using C = cx<T>;
    T const* in;       // [inputs][in_stride] reals, block tau at offset tau*B
    size_t in_stride;  // reals between channels
    T const* prev;     // [inputs][B] last block of the previous call (overlap-save)
    T* prev_next;      // [inputs][B] receives the last block of THIS call (ping-pong partner of `prev`)
    C* fdl;
    int ring, wp, blocks;
    int overlap_add;   // 0: window = [previous block | block]   1: window = [block | zeros]  (overlap_add.hpp:88-90)
    int logw, nt;      // tile-major FDL layout
    size_t chan0;      // `in` row 0 is input channel chan0 (channel groups of a pipelined host call)

    struct row_state
    {
        C const* lo;
        C const* hi;
        C* dst;        // element (tile 0, slot, 0); tiles are ring << logw apart
        C* keep;       // non-null for the last block of the call: where its samples are saved as the next half-window
    };
    __device__ __forceinline__ row_state open(size_t b) const
    {
        constexpr size_t B = size_t(1) << LOGM;
        size_t const rel   = b / blocks;
        size_t const ch    = chan0 + rel;
        int const tau      = int(b - rel * blocks);
        T const* cur       = in + rel * in_stride + size_t(tau) * B;
        int slot           = wp + tau;
        slot -= slot >= ring ? ring : 0;
        C* dst = fdl + tiled_offset(ch, nt, logw, size_t(ring), size_t(slot), 0);
        if (overlap_add) { return {reinterpret_cast<C const*>(cur), nullptr, dst, nullptr}; }
        T const* before = tau == 0 ? prev + ch * B : cur - B;
        // slide_window_left + append (overlap_save.hpp:94-95): the newest block is next call's left half
        C* const save = tau == blocks - 1 ? reinterpret_cast<C*>(prev_next + ch * B) : nullptr;
        return {reinterpret_cast<C const*>(before), reinterpret_cast<C const*>(cur), dst, save};
    }
    __device__ __forceinline__ void keep(row_state const& r, int j, C z) const
    {
        constexpr int H = (1 << LOGM) / 2;
        if (r.keep != nullptr && j >= H) { r.keep[j - H] = z; }
    }
    __device__ __forceinline__ C load(row_state const& r, int j) const
    {
        constexpr int H = (1 << LOGM) / 2;  // complex pairs per block
        if (j < H) { return r.lo[j]; }
        return r.hi != nullptr ? r.hi[j - H] : mk<T>(0, 0);
    }
    __device__ __forceinline__ void store(row_state const& r, int k, C x) const
    {
        if constexpr (ROWS) { r.dst[k] = x; }
        else { r.dst[((size_t(k >> logw) * ring) << logw) + (k & ((1 << logw) - 1))] = x; }
    }
    __device__ __forceinline__ void store_edges(row_state const& r, T dc, T nyq) const { r.dst[0] = mk<T>(dc, nyq); }
};

// neo::convolution::overlap_add_convolver (overlap_add_convolver.hpp:85-132) transforms its real window AS IT STANDS: after a call
// that ended inside a block the window holds the previous inverse transform's output with the new samples written over part of it.
// rows: [channels][2B] reals; the spectrum replaces delay-line row `wp` (the reference re-inserts into _current_segment, :94).
template<typename T, int LOGM>
struct window_r2c_io : conv_r2c_io<T, LOGM>
{
    using base = conv_r2c_io<T, LOGM>;
    using C    = cx<T>;
    using typename base::row_state;
    __device__ __forceinline__ row_state open(size_t b) const
    {
        constexpr int H    = (1 << LOGM) / 2;
        C const* const lo  = reinterpret_cast<C const*>(this->in + b * this->in_stride);
        return {lo, lo + H, this->fdl + tiled_offset(this->chan0 + b, this->nt, this->logw, size_t(this->ring), size_t(this->wp), 0), nullptr};
    }
};

// ---- inverse side: partial-plane gather + c2r + scale + overlap-save discard -------------------------------------------------
template<typename T, int LOGM>
struct conv_c2r_io
{
    using C = cx<T>;
    C const* acc;       // [count][blocks][B], row 0 = first output channel handled (partial planes are folded by the MAC kernel)
    int blocks;
    T* out;             // overlap-save: [count][out_stride] reals;  overlap-add: scratch [count][blocks][2B]
    size_t out_stride;
    T scale;            // 1 / (2B)  (overlap_save.hpp:108)
    int overlap_add;

    struct row_state
    {
        C const* src;
        C* dst;
    };
    __device__ __forceinline__ row_state open(size_t b) const
    {
        constexpr size_t B = size_t(1) << LOGM;
        size_t const ch    = b / blocks;
        size_t const tau   = b - ch * blocks;
        C const* src       = acc + (ch * blocks + tau) * B;
        T* dst             = overlap_add ? out + (ch * blocks + tau) * 2 * B : out + ch * out_stride + tau * B;
        return {src, reinterpret_cast<C*>(dst)};
    }
    __device__ __forceinline__ C load(row_state const& r, int k) const
    {
        return r.src[k];  // plain loads: the kernel batches all of a thread's points before the first use
    }
    __device__ __forceinline__ C load_edges(row_state const& r) const { return load(r, 0); }
    __device__ __forceinline__ void store(row_state const& r, int j, C z) const
    {
        constexpr int H = (1 << LOGM) / 2;
        z.x *= scale;
        z.y *= scale;
        if (overlap_add) {
            r.dst[j] = z;  // all 2B samples; combined with the saved tail afterwards
        } else if (j >= H) {
            r.dst[j - H] = z;  // keep samples [B, 2B) (overlap_save.hpp:111)
        }
    }
    // the wide kernel's 128-bit stores: samples z0, z1 = complex pairs j, j + 1 of the lower / upper half of the real row
    template<bool HI>
    __device__ __forceinline__ void store_pair(row_state const& r, int j, C z0, C z1) const
    {
        static_assert(sizeof(T) == 4, "float rows");
        constexpr int H = (1 << LOGM) / 2;
        float4 const v  = make_float4(z0.x * scale, z0.y * scale, z1.x * scale, z1.y * scale);
        if (overlap_add) { *reinterpret_cast<float4*>(r.dst + j + (HI ? H : 0)) = v; }
        else if (HI) { *reinterpret_cast<float4*>(r.dst + j) = v; }
    }
};

// ---- crossfade between two filters (neo_b200_conv_crossfade, neo_b200_lowlat_crossfade): out = y_A before `start`,
// y_A + g (y_B - y_A) with g = (t - start) / len inside, y_B after. One formula for both convolvers.
struct conv_fade
{
    unsigned long long t0;          // absolute sample index of block position 0 (of the row's first block)
    unsigned long long start, len;  // the fade covers samples [start, start + len)
};

template<typename T>
__device__ __forceinline__ T conv_blend(T ya, T yb, unsigned long long t, conv_fade const& f)
{
    if (t < f.start) { return ya; }
    if (t - f.start >= f.len) { return yb; }
    T const g = T(double(t - f.start) / double(f.len));
    return ya + g * (yb - ya);
}

// the A side of a bank call inside a crossfade: conv_c2r_io's overlap-save store (no overlap-add: its tail depends on the filter), each
// kept sample blended with the B side's output at the same place of `yb` ([count][out_stride] reals, laid out as `out`). Sample j of
// block tau of a row is absolute sample fade.t0 + tau B + j.
template<typename T, int LOGM>
struct conv_c2r_fade_io
{
    using C = cx<T>;
    C const* acc;  // [count][blocks][B]
    int blocks;
    T* out;
    size_t out_stride;
    T scale;
    T const* yb;
    conv_fade fade;

    struct row_state
    {
        C const* src;
        C* dst;
        C const* yb;
        unsigned long long t;  // absolute index of the block's first sample
    };
    __device__ __forceinline__ row_state open(size_t b) const
    {
        constexpr size_t B = size_t(1) << LOGM;
        size_t const ch    = b / blocks;
        size_t const tau   = b - ch * blocks;
        size_t const off   = ch * out_stride + tau * B;
        return {acc + (ch * blocks + tau) * B, reinterpret_cast<C*>(out + off), reinterpret_cast<C const*>(yb + off), fade.t0 + tau * B};
    }
    __device__ __forceinline__ C load(row_state const& r, int k) const { return r.src[k]; }
    __device__ __forceinline__ C load_edges(row_state const& r) const { return load(r, 0); }
    __device__ __forceinline__ void store(row_state const& r, int j, C z) const
    {
        constexpr int H = (1 << LOGM) / 2;
        if (j >= H) {
            C const b                  = r.yb[j - H];
            unsigned long long const t = r.t + 2ULL * unsigned(j - H);
            r.dst[j - H]               = mk<T>(conv_blend(z.x * scale, b.x, t, fade), conv_blend(z.y * scale, b.y, t + 1, fade));
        }
    }
    // the wide kernel's 128-bit stores; the four samples of a float4 are blended one by one
    template<bool HI>
    __device__ __forceinline__ void store_pair(row_state const& r, int j, C z0, C z1) const
    {
        static_assert(sizeof(T) == 4, "float rows");
        if constexpr (HI) {
            float4 const b             = *reinterpret_cast<float4 const*>(r.yb + j);
            unsigned long long const t = r.t + 2ULL * unsigned(j);
            *reinterpret_cast<float4*>(r.dst + j) = make_float4(conv_blend(z0.x * scale, b.x, t, fade), conv_blend(z0.y * scale, b.y, t + 1, fade),
                                                                conv_blend(z1.x * scale, b.z, t + 2, fade), conv_blend(z1.y * scale, b.w, t + 3, fade));
        }
    }
};

// ---- inverse side of a partition-sharded bank whose shards sit in peer-mapped memory: the cross-device reduction of the partial
// spectra is fused into the loads of the c2r kernel. src[j] is the partial-spectra buffer of partition shard j (this device's own
// buffer or a peer's, read over NVLink through the mapped pointer), all with the same [count][blocks][B] layout; they are summed in
// shard order, so every device would produce the same bits for the same channel.
constexpr int k_bank_max_shards = 8;

// NSRC > 0: the number of shards is a compile-time constant (two, the common split: no predicated loads or adds in the instruction
// stream -- the run-time form issues all k_bank_max_shards of them, 40 % more instructions at two shards); NSRC = 0: `nsrc` at run time
template<typename T, int LOGM, int NSRC = 0>
struct conv_c2r_sum_io
{
    using C = cx<T>;
    C const* src[k_bank_max_shards];
    int nsrc;
    int blocks;
    T* out;
    size_t out_stride;
    T scale;
    int overlap_add;

    struct row_state
    {
        size_t off;
        C* dst;
    };
    __device__ __forceinline__ row_state open(size_t b) const
    {
        constexpr size_t B = size_t(1) << LOGM;
        size_t const ch    = b / blocks;
        size_t const tau   = b - ch * blocks;
        T* dst             = overlap_add ? out + (ch * blocks + tau) * 2 * B : out + ch * out_stride + tau * B;
        return {(ch * blocks + tau) * B, reinterpret_cast<C*>(dst)};
    }
    __device__ __forceinline__ C load(row_state const& r, int k) const
    {
        if constexpr (NSRC > 0) {
            C p[NSRC];
#pragma unroll
            for (int j = 0; j < NSRC; ++j) { p[j] = src[j][r.off + k]; }
            C v = p[0];
#pragma unroll
            for (int j = 1; j < NSRC; ++j) {
                v.x += p[j].x;
                v.y += p[j].y;
            }
            return v;
        } else {
            // fully unrolled with a uniform predicate: the source pointers stay in registers / constant bank (a run-time indexed
            // pointer array would be copied to local memory) and the loads of all sources are in flight together
            C p[k_bank_max_shards];
#pragma unroll
            for (int j = 0; j < k_bank_max_shards; ++j) { p[j] = j < nsrc ? src[j][r.off + k] : mk<T>(T(0), T(0)); }
            C v = p[0];
#pragma unroll
            for (int j = 1; j < k_bank_max_shards; ++j) {
                if (j < nsrc) {
                    v.x += p[j].x;
                    v.y += p[j].y;
                }
            }
            return v;
        }
    }
    __device__ __forceinline__ C load_edges(row_state const& r) const { return load(r, 0); }
    __device__ __forceinline__ void store(row_state const& r, int j, C z) const
    {
        constexpr int H = (1 << LOGM) / 2;
        z.x *= scale;
        z.y *= scale;
        if (overlap_add) {
            r.dst[j] = z;
        } else if (j >= H) {
            r.dst[j - H] = z;
        }
    }
    // the wide kernel's 128-bit stores: samples z0, z1 = complex pairs j, j + 1 of the lower / upper half of the real row
    template<bool HI>
    __device__ __forceinline__ void store_pair(row_state const& r, int j, C z0, C z1) const
    {
        static_assert(sizeof(T) == 4, "float rows");
        constexpr int H = (1 << LOGM) / 2;
        float4 const v  = make_float4(z0.x * scale, z0.y * scale, z1.x * scale, z1.y * scale);
        if (overlap_add) { *reinterpret_cast<float4*>(r.dst + j + (HI ? H : 0)) = v; }
        else if (HI) { *reinterpret_cast<float4*>(r.dst + j) = v; }
    }
};

// overlap-add epilogue (overlap_add.hpp:103-106): out = y[0..B) + tail, tail' = y[B..2B) of the last block.
// One thread walks all blocks of one sample position of one channel, so the tail is read and rewritten IN PLACE by the same
// thread: the tail state belongs to a channel, and a step may be finished by several calls over disjoint channel ranges
// (neo_b200_conv_inverse) without any per-call ping-pong.
template<typename T>
__global__ void __launch_bounds__(256)
    ola_combine_kernel(T const* __restrict__ y, T* __restrict__ tail, T* __restrict__ out, size_t out_stride, int block, int blocks, size_t first)
{
    size_t const ch = blockIdx.y;
    int const i     = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= block) { return; }
    T const* yrow = y + ch * size_t(blocks) * 2 * size_t(block) + i;
    T* const dst  = out + ch * out_stride + i;
    T* const keep = tail + (first + ch) * size_t(block) + i;
    T before      = *keep;
#pragma unroll 4
    for (int tau = 0; tau < blocks; ++tau) {
        T const lo = yrow[size_t(tau) * 2 * block];
        T const hi = yrow[size_t(tau) * 2 * block + block];
        dst[size_t(tau) * block] = lo + before;
        before                   = hi;
    }
    *keep = before;
}

// ---- filter preparation ----------------------------------------------------------------------------------------------------------
// uniform_partition (convolution/uniform_partition.hpp:13-26 -> fft/stft.hpp:78-96): frame p of filter f, zero padded to 2B
template<typename T, int LOGM>
struct partition_r2c_io
{
    using C = cx<T>;
    T const* ir;         // [filters][taps]
    size_t taps;
    int part0, parts;    // partitions [part0, part0 + parts) are produced
    C* out;
    int packed;          // 1: convolver layout [f][B/W][parts][W] (bin 0 packed), 0: reference layout [f][parts][B+1]
    int logw, nt;

    struct row_state
    {
        T const* src;
        long count;
        C* dst;
    };
    __device__ __forceinline__ row_state open(size_t b) const
    {
        constexpr size_t B = size_t(1) << LOGM;
        size_t const f     = b / parts;
        size_t const p     = part0 + (b - f * parts);
        long const left    = long(taps) - long(p * B);
        long const count   = left < long(B) ? left : long(B);
        C* dst = packed ? out + tiled_offset(f, nt, logw, size_t(parts), b - f * parts, 0) : out + b * (B + 1);
        return {ir + f * taps + p * B, count, dst};
    }
    __device__ __forceinline__ C load(row_state const& r, int j) const
    {
        long const i = 2L * j;
        return mk<T>(i < r.count ? r.src[i] : T(0), i + 1 < r.count ? r.src[i + 1] : T(0));
    }
    __device__ __forceinline__ void keep(row_state const&, int, C) const {}
    __device__ __forceinline__ void store(row_state const& r, int k, C x) const
    {
        if (packed) { r.dst[((size_t(k >> logw) * parts) << logw) + (k & ((1 << logw) - 1))] = x; }
        else { r.dst[k] = x; }
    }
    __device__ __forceinline__ void store_edges(row_state const& r, T dc, T nyq) const
    {
        if (packed) {
            r.dst[0] = mk<T>(dc, nyq);
        } else {
            r.dst[0]         = mk<T>(dc, T(0));
            r.dst[1 << LOGM] = mk<T>(nyq, T(0));
        }
    }
};

// stft_plan (fft/stft.hpp:70-99): frame f of channel c = x[c][f*hop .. f*hop + frame) (clipped at the end of the signal), zero padded to
// the transform size 2M, times the window (null = rectangular); out [C][frames][M+1]
template<typename T, int LOGM>
struct stft_r2c_io
{
    using C = cx<T>;
    T const* x;          // [channels][len]
    size_t len;
    size_t frame, hop;   // hop = frame - overlap
    size_t frames;
    T const* window;     // [2M] or null
    C* out;

    struct row_state
    {
        T const* src;
        long count;
        C* dst;
    };
    __device__ __forceinline__ row_state open(size_t b) const
    {
        constexpr size_t M = size_t(1) << LOGM;
        size_t const c     = b / frames;
        size_t const f     = b - c * frames;
        size_t const first = f * hop;
        size_t const left  = len - first;
        return {x + c * len + first, long(left < frame ? left : frame), out + b * (M + 1)};
    }
    __device__ __forceinline__ C load(row_state const& r, int j) const
    {
        long const i = 2L * j;
        T a = i < r.count ? r.src[i] : T(0);
        T b = i + 1 < r.count ? r.src[i + 1] : T(0);
        if (window != nullptr) {
            a *= window[i];
            b *= window[i + 1];
        }
        return mk<T>(a, b);
    }
    __device__ __forceinline__ void keep(row_state const&, int, C) const {}
    __device__ __forceinline__ void store(row_state const& r, int k, C v) const { r.dst[k] = v; }
    __device__ __forceinline__ void store_edges(row_state const& r, T dc, T nyq) const
    {
        r.dst[0]         = mk<T>(dc, T(0));
        r.dst[1 << LOGM] = mk<T>(nyq, T(0));
    }
};

// ---- sparse filters (neo::convolution::sparse_filter, sparse_filter.hpp:16-38; CSR multiply_add, algorithm/multiply_add.hpp:306-324)
// The reference keeps each channel's partitions as a CSR matrix (rows = partitions, columns = bins) and touches only the stored
// elements. A GPU wants the bins of a warp side by side, so the device layout is a BITMAP form of the same matrix: the row of B packed
// bins is cut into segments of 32 bins; per (filter, segment, partition) one word of presence bits and the offset of the segment's
// stored values, which lie packed in (segment, partition, bin) order -- the order one warp walks them in:
//     meta [filters][nseg][parts]  uint2 {mask, offset into the filter's run of values}
//     vals [filters' runs]         complex, fbase[f] = first value of filter f
// One CTA = one segment of one channel, its four warps taking 32-partition chunks in turn: a warp reads 32 partitions' meta words in
// one coalesced load, hands them round by shuffle, SKIPS what is empty (no filter bytes, no delay-line bytes), and otherwise
// gathers the stored values (a contiguous run) and the delay-line row segment. Bytes per block and channel: 8 P nseg of meta + 8 nnz + the delay-line segments touched,
// against 16 P B for the dense stream. Stored elements give the reference's sum, dropped ones add nothing; the four warps' partial
// sums are added in a fixed order. Diagonal topology, T = 1 per launch, packed bin 0 = (Re X[0], Re X[B]).
template<typename T>
__global__ void __launch_bounds__(128)
    fdl_mac_sparse_kernel(cx<T> const* __restrict__ fdl, uint2 const* __restrict__ meta, cx<T> const* __restrict__ vals,
                          unsigned long long const* __restrict__ fbase, cx<T>* __restrict__ acc, mac_geom g, int nseg)
{
    using C             = cx<T>;
    constexpr int U     = 8;  // partitions gathered together
    constexpr int WARPS = 4;  // warps of a CTA share one segment: they take the 32-partition chunks in turn (a bank of few channels
                              // would otherwise leave most warp slots empty and every warp a long dependent walk)
    int const lane   = int(threadIdx.x) & 31;
    int const warp   = int(threadIdx.x) >> 5;
    int const seg    = blockIdx.x;
    int const out    = blockIdx.y + g.out0;
    int const k      = seg * 32 + lane;
    bool const mine  = k < g.m;
    bool const edge  = k == 0 && g.packed_edge != 0;
    unsigned const below = (1U << lane) - 1U;
    uint2 const* const mrow = meta + (size_t(out) * nseg + seg) * g.parts;
    C const* const vrow     = vals + fbase[out];
    size_t const xbase      = tiled_offset(size_t(out), g.nt, g.logw, size_t(g.ring), 0, mine ? k : 0);

    C a = mk<T>(T(0), T(0));
    for (int p0 = 32 * warp; p0 < g.parts; p0 += 32 * WARPS) {
        uint2 const word = p0 + lane < g.parts ? mrow[p0 + lane] : make_uint2(0U, 0U);
        int sbase        = (g.wp - g.age0 - p0) % g.ring;  // ring slot of partition p0; the following ones lie below it
        sbase += sbase < 0 ? g.ring : 0;
        // the partitions of this chunk that store anything in this segment, U at a time. The body is branch-free (every lane loads:
        // a lane without a stored bin re-reads the segment's first value and multiplies by zero; a turn with fewer than U partitions
        // left repeats the last one with an empty mask), so all 2 U loads of a turn are in flight together -- with a branch per
        // partition the walk was one dependent load after the other (ncu: 80 % of the stall samples on the gathers' addresses)
        unsigned todo = __ballot_sync(0xffffffffU, word.x != 0U);
        while (todo != 0U) {
            C h[U], x[U];
            int j = 0;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                bool const live = todo != 0U;
                j               = live ? __ffs(int(todo)) - 1 : j;
                todo &= todo - 1U;  // 0 stays 0
                unsigned const mask = live ? __shfl_sync(0xffffffffU, word.x, j) : 0U;
                unsigned const off  = __shfl_sync(0xffffffffU, word.y, j);
                bool const on       = ((mask >> lane) & 1U) != 0U;
                int slot            = sbase - j;
                slot += slot < 0 ? g.ring : 0;
                C const hv = vrow[off + (on ? __popc(mask & below) : 0)];
                x[u]       = fdl[xbase + (size_t(slot) << g.logw)];
                h[u]       = on ? hv : mk<T>(T(0), T(0));
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (edge) {
                    a.x = fma(x[u].x, h[u].x, a.x);
                    a.y = fma(x[u].y, h[u].y, a.y);
                } else {
                    a.x = fma(x[u].x, h[u].x, a.x);
                    a.x = fma(-x[u].y, h[u].y, a.x);
                    a.y = fma(x[u].x, h[u].y, a.y);
                    a.y = fma(x[u].y, h[u].x, a.y);
                }
            }
        }
    }
    // the warps' partial sums, added in warp order (deterministic)
    __shared__ C partial[WARPS][32];
    partial[warp][lane] = a;
    __syncthreads();
    if (warp == 0 && mine) {
#pragma unroll
        for (int w = 1; w < WARPS; ++w) {
            a.x += partial[w][lane].x;
            a.y += partial[w][lane].y;
        }
        acc[(size_t(out) * g.blocks + g.tau0) * g.m + k] = a;
    }
}

// reference layout H[f][P][B+1] -> convolver layout [f][parts][B] for partitions [part0, part0+parts)
template<typename T>
__global__ void __launch_bounds__(256)
    pack_filter_kernel(cx<T> const* __restrict__ h, cx<T>* __restrict__ packed, size_t src_parts, int part0, int parts, int block,
                       size_t row0, int logw, int nt)
{
    size_t const row = row0 + blockIdx.y;  // f * parts + p
    int const k      = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= block) { return; }
    size_t const f   = row / parts;
    size_t const p   = part0 + (row - f * parts);
    cx<T> const* src = h + (f * src_parts + p) * (size_t(block) + 1);
    cx<T> v          = src[k];
    if (k == 0) { v.y = src[block].x; }
    packed[tiled_offset(f, nt, logw, size_t(parts), row - f * parts, k)] = v;
}

// normalize_impulse step 1: energy[c] = sum_i ir[c][i]^2, one CTA per channel, double accumulation
template<typename T>
__global__ void __launch_bounds__(256) channel_energy_kernel(T const* __restrict__ ir, size_t taps, double* __restrict__ energy)
{
    __shared__ double partial[256];
    T const* row = ir + size_t(blockIdx.x) * taps;
    double acc   = 0.0;
    for (size_t i = threadIdx.x; i < taps; i += blockDim.x) {
        double const v = double(row[i]);
        acc += v * v;
    }
    partial[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (int(threadIdx.x) < s) { partial[threadIdx.x] += partial[threadIdx.x + s]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { energy[blockIdx.x] = partial[0]; }
}

// step 2: factor = min_c (energy == 0 ? 1 : 1/sqrt(energy)) (normalize_impulse.hpp:24-31), applied to every sample
template<typename T>
__global__ void __launch_bounds__(256) scale_by_min_factor_kernel(T* __restrict__ ir, size_t total, double const* __restrict__ energy, unsigned channels)
{
    double factor = 0.0;
    for (unsigned c = 0; c < channels; ++c) {
        double const f = energy[c] == 0.0 ? 1.0 : rsqrt(energy[c]);
        factor         = (c == 0 || f < factor) ? f : factor;
    }
    T const scale = T(factor);
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) { ir[i] = ir[i] * scale; }
}

// ---- compressed delay line (neo::convolution::compressed_fdl, compressed_fdl.hpp:17-52): rows stored as int8 / int16 complex ----
// insert (:36-48): q = (int_type) lround(val * (float) max); read through compressed_accessor (compressed_accessor.hpp:27-45):
// (Float) q * (Float(1) / Float(max)). One thread per real or imaginary part; the device stores exactly the reference's integers.
template<typename T, typename I>
__global__ void __launch_bounds__(256) compress_parts_kernel(T const* __restrict__ in, I* __restrict__ out, size_t n)
{
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) { return; }
    constexpr float max_val = sizeof(I) == 1 ? 127.0F : 32767.0F;
    long long q;
    if constexpr (sizeof(T) == 4) { q = llroundf(in[i] * max_val); }
    else { q = llround(in[i] * double(max_val)); }
    out[i] = static_cast<I>(q);
}

template<typename T, typename I>
__global__ void __launch_bounds__(256) decompress_parts_kernel(I const* __restrict__ in, T* __restrict__ out, size_t n)
{
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) { return; }
    constexpr T inv_scale = T(1) / T(sizeof(I) == 1 ? 127 : 32767);
    out[i]                = static_cast<T>(in[i]) * inv_scale;
}

__global__ void fdl_index_kernel(unsigned parts, unsigned calls, unsigned* write_pos, unsigned* pairs);
__global__ void bitrev_table_kernel(unsigned order, unsigned* out);

}  // namespace neo_b200
