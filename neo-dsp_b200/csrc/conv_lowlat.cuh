// conv_lowlat.cuh -- device side of the one-block-latency convolver (neo_b200_lowlat_*, include/neo_b200.h).
//
// Non-uniform partitioning (Gardner 1995, Garcia 2002): partitions [0, 2*T_1) -- the "head" -- run in the direct form one block at a
// time; longer stretches [2*T_i, 2*T_{i+1}) run in frame mode (conv_frame.cuh) with frame_blocks = T_i on side streams, a whole frame
// period ahead of the block that needs them. Per block the head kernel below does, for every channel in ONE launch:
//   window [previous block | block] -> 2B-point r2c -> delay-line insert -> MAC over the head partitions on the thread's own bins ->
//   Hermitian pre-pass -> c2r -> 1/2B, keep the last B samples -> + each level's partial output (level order) -> store,
// and saves the block as the next left half-window and into the levels' input ring.
//
// Layouts (shared with conv_engine, whose head-range handle owns filter, delay line and half-window buffers):
//   fdl    [C][B/W][R][W]    ring of head spectra, R = 2*T_1 rows, bin 0 packed as (Re X[0], Re X[B])
//   filter [C][B/W][Ph][W]   head partitions, same packing
#pragma once

#include "conv_kernels.cuh"

namespace neo_b200 {

constexpr int k_lowlat_max_levels = 4;

template<typename T>
struct lowlat_levels
{
    int count;
    T const* plane[k_lowlat_max_levels];   // level i's partial output of THIS block, channel 0
    size_t stride[k_lowlat_max_levels];    // reals between channels of a plane
};

template<typename T>
struct lowlat_head_args
{
    T const* in;  // block of channel c at in + c * in_stride
    size_t in_stride;
    T* out;
    size_t out_stride;
    T const* prev;       // [C][B] previous block (left half-window)
    T* prev_next;        // [C][B] receives this block
    T* in_ring;          // this block's slot of the levels' input ring, channel 0
    size_t ring_stride;  // reals between channels of the input ring
    cx<T>* fdl;
    cx<T> const* filter;
    int ring, wp, parts, logw;
    size_t channels;
    lowlat_levels<T> levels;
};

// register budget: the MAC keeps E accumulators next to the transform's E points. 128 registers leave no spills (-Xptxas -v) except
// for double at 2^10 and 2^11 points (100 bytes spilled at 128, 4 at 168), which get the whole 255
template<typename T, int LOGM>
constexpr int lowlat_min_ctas()
{
    int const regs = sizeof(T) == 8 && LOGM >= 10 ? 255 : 128;
    int const n    = 65536 / (regs * fft_cfg<T, LOGM>::THREADS);
    return n > 0 ? n : 1;
}

template<typename C>
__device__ __forceinline__ void lowlat_cfma(C& a, C x, C h)
{
    a.x = fma(x.x, h.x, a.x);
    a.x = fma(-x.y, h.y, a.x);
    a.y = fma(x.x, h.y, a.y);
    a.y = fma(x.y, h.x, a.y);
}

// bin 0 = (Re X[0], Re X[B]): two independent real products
template<typename C>
__device__ __forceinline__ void lowlat_cfma_edge(C& a, C x, C h)
{
    a.x = fma(x.x, h.x, a.x);
    a.y = fma(x.y, h.y, a.y);
}

// element k of a tile-major row
__device__ __forceinline__ size_t lowlat_tiled(int ring_rows, int logw, int k)
{
    return ((size_t(k >> logw) * size_t(ring_rows)) << logw) + size_t(k & ((1 << logw) - 1));
}

// One CTA holds G channels (fft_cfg); thread t owns the Hermitian pairs (k, M-k), k = t + e*TN for e < E/2 -- the same bins in the
// r2c post-pass, the MAC and the c2r pre-pass, so the accumulators never leave registers. Thread 0's pair e = 0 is (packed bin 0,
// bin M/2).
template<typename T, int LOGM>
__global__ void __launch_bounds__(fft_cfg<T, LOGM>::THREADS, lowlat_min_ctas<T, LOGM>())
    lowlat_head_kernel(lowlat_head_args<T> a, cx<T> const* __restrict__ tw, cx<T> const* __restrict__ rtw)
{
    using cfg = fft_cfg<T, LOGM>;
    using C   = cx<T>;
    constexpr int M = cfg::M, E = cfg::E, TN = cfg::TN, HALF = E / 2;
    static_assert(E >= 4, "pairs need at least four points per thread");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C* sm = reinterpret_cast<C*>(smem_raw) + (threadIdx.x / TN) * cfg::TILE;

    int const t      = threadIdx.x % TN;
    size_t const ch  = size_t(blockIdx.x) * cfg::G + threadIdx.x / TN;
    bool const live  = ch < a.channels;
    size_t const row = live ? ch : 0;

    // 1. window [previous block | this block]: points e < E/2 are the left half, the rest this block (H = M/2 = HALF * TN pairs)
    C const* lo = reinterpret_cast<C const*>(a.prev + row * M);
    C const* hi = reinterpret_cast<C const*>(a.in + row * a.in_stride);
    C v[E];
#pragma unroll
    for (int e = 0; e < E; ++e) { v[e] = !live ? mk<T>(0, 0) : e < HALF ? lo[t + e * TN] : hi[t + (e - HALF) * TN]; }
    // 9. this block is the next left half-window and the levels' input (both buffers are distinct from in / out)
    if (live) {
        C* const keep = reinterpret_cast<C*>(a.prev_next + row * M);
        C* const ring = reinterpret_cast<C*>(a.in_ring + row * a.ring_stride);
#pragma unroll
        for (int e = HALF; e < E; ++e) {
            keep[t + (e - HALF) * TN] = v[e];
            ring[t + (e - HALF) * TN] = v[e];
        }
    }

    // 2. r2c
    cta_fft<T, LOGM, -1>::run(v, sm, tw, t);
#pragma unroll
    for (int e = 0; e < E; ++e) { sm[t + e * TN] = v[e]; }  // unpadded, as r2c_kernel's Hermitian exchange
    __syncthreads();
    C xk[HALF], xm[HALF];
#pragma unroll
    for (int e = 0; e < HALF; ++e) {
        int const k = t + e * TN;
        if (k == 0) {
            xk[e] = mk<T>(v[e].x + v[e].y, v[e].x - v[e].y);
            xm[e] = cconj(v[HALF]);  // the self-paired bin M/2 is thread 0's point HALF
        } else {
            r2c_post_pair(v[e], sm[M - k], __ldg(rtw + k), xk[e], xm[e]);
        }
    }
    __syncthreads();  // the tile is reused by the c2r pre-pass

    // 3. delay-line insert into slot wp; 4. MAC over the head partitions, partition 0 from registers, fixed partition order
    C* const x_row       = a.fdl + tiled_offset(row, M >> a.logw, a.logw, size_t(a.ring), 0, 0);
    C const* const h_row = a.filter + tiled_offset(row, M >> a.logw, a.logw, size_t(a.parts), 0, 0);
    C ak[HALF], am[HALF];
#pragma unroll
    for (int e = 0; e < HALF; ++e) {
        int const k  = t + e * TN;
        int const km = k == 0 ? M / 2 : M - k;
        if (live) {
            x_row[lowlat_tiled(a.ring, a.logw, k) + (size_t(a.wp) << a.logw)]  = xk[e];
            x_row[lowlat_tiled(a.ring, a.logw, km) + (size_t(a.wp) << a.logw)] = xm[e];
        }
        C const hk = h_row[lowlat_tiled(a.parts, a.logw, k)];
        C const hm = h_row[lowlat_tiled(a.parts, a.logw, km)];
        ak[e] = am[e] = mk<T>(0, 0);
        if (k == 0) { lowlat_cfma_edge(ak[e], xk[e], hk); }
        else { lowlat_cfma(ak[e], xk[e], hk); }
        lowlat_cfma(am[e], xm[e], hm);
    }
    int slot = a.wp;
    for (int p = 1; p < a.parts; ++p) {
        slot = slot == 0 ? a.ring - 1 : slot - 1;  // the spectrum of p blocks ago
        C const* const xr = x_row + (size_t(slot) << a.logw);
        C const* const hr = h_row + (size_t(p) << a.logw);
        C xs[HALF], xms[HALF], hs[HALF], hms[HALF];
#pragma unroll
        for (int e = 0; e < HALF; ++e) {  // all loads of the partition in flight before the first FMA
            int const k  = t + e * TN;
            int const km = k == 0 ? M / 2 : M - k;
            xs[e]        = xr[lowlat_tiled(a.ring, a.logw, k)];
            xms[e]       = xr[lowlat_tiled(a.ring, a.logw, km)];
            hs[e]        = __ldg(hr + lowlat_tiled(a.parts, a.logw, k));
            hms[e]       = __ldg(hr + lowlat_tiled(a.parts, a.logw, km));
        }
#pragma unroll
        for (int e = 0; e < HALF; ++e) {
            if (e == 0 && t == 0) { lowlat_cfma_edge(ak[e], xs[e], hs[e]); }
            else { lowlat_cfma(ak[e], xs[e], hs[e]); }
            lowlat_cfma(am[e], xms[e], hms[e]);
        }
    }

    // 5. Hermitian pre-pass (as c2r_kernel) and c2r
#pragma unroll
    for (int e = 0; e < HALF; ++e) {
        int const k = t + e * TN;
        if (k == 0) {
            v[e]    = mk<T>(ak[e].x + ak[e].y, ak[e].x - ak[e].y);
            v[HALF] = mk<T>(T(2) * am[e].x, T(-2) * am[e].y);
        } else {
            C zmk;
            c2r_pre_pair(ak[e], am[e], __ldg(rtw + k), v[e], zmk);
            sm[M - k] = zmk;
        }
    }
    __syncthreads();
#pragma unroll
    for (int e = HALF; e < E; ++e) {
        if (!(e == HALF && t == 0)) { v[e] = sm[t + e * TN]; }
    }
    __syncthreads();
    cta_fft<T, LOGM, +1>::run(v, sm, tw, t);

    // 6.-8. scale, keep samples [B, 2B), add the levels in level order, store
    if (live) {
        T const scale = T(1) / T(2 * M);
        C* const dst  = reinterpret_cast<C*>(a.out + row * a.out_stride);
#pragma unroll
        for (int e = HALF; e < E; ++e) {
            int const j = t + (e - HALF) * TN;
            C y         = mk<T>(v[e].x * scale, v[e].y * scale);
#pragma unroll
            for (int i = 0; i < k_lowlat_max_levels; ++i) {
                if (i < a.levels.count) {
                    C const l = reinterpret_cast<C const*>(a.levels.plane[i] + row * a.levels.stride[i])[j];
                    y.x += l.x;
                    y.y += l.y;
                }
            }
            dst[j] = y;
        }
    }
}

// the unfused form's tail: out = head + levels (level order), and the block into the levels' input ring. grid (ceil(B/256), C)
template<typename T>
__global__ void __launch_bounds__(256) lowlat_combine_kernel(T const* __restrict__ head, int block, T const* in, size_t in_stride, T* out,
                                                             size_t out_stride, T* __restrict__ in_ring, size_t ring_stride,
                                                             lowlat_levels<T> levels)
{
    size_t const ch = blockIdx.y;
    int const i     = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= block) { return; }
    in_ring[ch * ring_stride + i] = in[ch * in_stride + i];  // read before the store below: in == out is allowed
    T y = head[ch * size_t(block) + i];
#pragma unroll
    for (int l = 0; l < k_lowlat_max_levels; ++l) {
        if (l < levels.count) { y += levels.plane[l][ch * levels.stride[l] + i]; }
    }
    out[ch * out_stride + i] = y;
}

}  // namespace neo_b200
