// fft_wide.cuh -- long real transforms (float32, N = 2^14 .. 2^16) with 32 complex points per thread.
//
// Same contract as r2c_kernel / c2r_kernel (fallback_rfft_plan.hpp:28-55: half-size complex transform + Hermitian split), different
// shape. The 16-points-per-thread cta_fft needs 4 shared-memory exchanges for a 2^13-point row (three stages + the Hermitian
// partner exchange): 64 bytes of shared-memory traffic and ~89 instructions per complex point, which is issue-bound BELOW the HBM
// roofline (DESIGN 4.1). Here a row of M = R1*R2*16 points goes through exactly THREE register stages and TWO exchanges:
//
//   forward   n = n' + (M/R1) n1,  n' = a + 16 a2,   k = k1 + R1 k2 + (M/16) k3
//     S1  butterfly n'      : DFT_R1 over n1, times W_M^(n' k1)               -> tile (k1, a2, a)     [thread: 32/R1 adjacent n']
//     S2  butterfly (k1, a) : DFT_R2 over a2, times W_(16 R2)^(a k2)          -> tile (k1, k2, a)     [in place: no barrier between
//                                                                                                      its loads and its stores]
//     S3  butterfly j = k1 + R1 k2 : DFT_16 over a                            -> Z[j + J k3], J = M/16
//   A thread owns stage-3 butterflies j and J - j: Z[j + J k3] and its Hermitian partner Z[M - (j + J k3)] = Z[(J - j) + J (15 - k3)]
//   are then both in ITS registers, so the real-transform split needs no exchange at all (thread 0 owns the two self-paired
//   butterflies 0 and J/2). The backward transform is the transposed flow (Hermitian pre-pass in registers, S3', S2' in place, S1').
//
// Tile: row (k1, x) = 16 complex values = 128 bytes, its eight 16-byte chunks XOR-swizzled by k1 & 7. Every access is conflict-free
// (tools/wide_fft_model.py replays the index math and the bank pattern): S1 stores / S1' loads are 128-bit and unit stride, S2 moves
// one row per half-warp, S3 reads its rows with 128-bit loads whose 8 lanes per wavefront hit 8 different chunks.
// Global side: the real row moves as 128-bit accesses (two adjacent complex points per thread), the spectrum as coalesced 64-bit
// accesses ascending (k) and descending (M - k).
#pragma once

#include "fft_kernels.cuh"

#include <algorithm>
#include <type_traits>

namespace neo_b200 {

template<int I, int N, class F>
__device__ __forceinline__ void static_for(F&& f)
{
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        static_for<I + 1, N>(f);
    }
}

// bulk-copy (TMA) plumbing of the prefetching kernels: one mbarrier, one global -> shared bulk copy per row
namespace wtma {
__device__ __forceinline__ unsigned saddr(void const* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void init(void* bar, unsigned arrivals)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(saddr(bar)), "r"(arrivals) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// the tile was last touched through the generic proxy (LDS / STS); order those accesses before the bulk copy's writes
__device__ __forceinline__ void fetch(void* dst, void const* src, unsigned bytes, void* bar)
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(saddr(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(saddr(dst)), "l"(src),
                 "r"(bytes), "r"(saddr(bar))
                 : "memory");
}
__device__ __forceinline__ void wait(void* bar, unsigned parity)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "WAIT_%=:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                 "@!p bra WAIT_%=;\n"
                 "}\n" ::"r"(saddr(bar)),
                 "r"(parity)
                 : "memory");
}
}  // namespace wtma

// cos / sin of 2 pi e / 64 as compile-time constants
__host__ __device__ constexpr double wide_cos64_quarter(int e)
{
    constexpr double q[17] = {1.0,
                              0.9951847266721969,
                              0.9807852804032304,
                              0.9569403357322088,
                              0.9238795325112867,
                              0.881921264348355,
                              0.8314696123025452,
                              0.773010453362737,
                              0.7071067811865476,
                              0.6343932841636455,
                              0.5555702330196023,
                              0.4713967368259978,
                              0.38268343236508984,
                              0.29028467725446233,
                              0.19509032201612833,
                              0.09801714032956077,
                              0.0};
    return q[e];
}
__host__ __device__ constexpr double wide_cos64(int e)
{
    e = ((e % 64) + 64) % 64;
    if (e <= 16) { return wide_cos64_quarter(e); }
    if (e <= 32) { return -wide_cos64_quarter(32 - e); }
    if (e <= 48) { return -wide_cos64_quarter(e - 32); }
    return wide_cos64_quarter(64 - e);
}
__host__ __device__ constexpr double wide_sin64(int e) { return wide_cos64(e - 16); }
__host__ __device__ constexpr double wide_sqrt(double x)
{
    double y = x > 1.0 ? x : 1.0;  // Newton from above
    for (int i = 0; i < 64; ++i) { y = 0.5 * (y + x / y); }
    return x <= 0.0 ? 0.0 : y;
}

// multiply by exp(DIR * 2 pi i EXP / 64), EXP known at compile time
template<int EXP, int DIR>
__device__ __forceinline__ float2 mul_w64(float2 a)
{
    constexpr int e = ((EXP % 64) + 64) % 64;
    if constexpr (e == 0) {
        return a;
    } else if constexpr (e == 16) {
        return rot90<DIR>(a);
    } else if constexpr (e == 32) {
        return make_float2(-a.x, -a.y);
    } else if constexpr (e == 48) {
        return rot90<-DIR>(a);
    } else {
        constexpr float wr = float(wide_cos64(e));
        constexpr float wi = float(DIR < 0 ? -wide_sin64(e) : wide_sin64(e));
        return make_float2(a.x * wr - a.y * wi, a.x * wi + a.y * wr);
    }
}

// exp(-2 pi i EXP / 64) as a value
template<int EXP>
__device__ __forceinline__ float2 w64_const()
{
    return make_float2(float(wide_cos64(EXP)), float(-wide_sin64(EXP)));
}

// exp(-2 pi i EXP / 128), EXP odd: half-angle of the table above
template<int EXP>
__device__ __forceinline__ float2 w128_const()
{
    static_assert(EXP >= 0 && EXP < 64, "first half turn");
    // cos(x/2), sin(x/2) from cos x, 0 <= x/2 < pi/2 ... pi: EXP < 32 -> first quadrant, else second
    constexpr double c  = wide_cos64(EXP);  // cos(2 pi EXP / 64) = cos of twice the wanted angle
    constexpr double ch = EXP < 32 ? wide_sqrt((1.0 + c) * 0.5) : -wide_sqrt((1.0 + c) * 0.5);
    constexpr double sh = wide_sqrt((1.0 - c) * 0.5);
    return make_float2(float(ch), float(-sh));
}

// 32-point DFT in registers: 4 x 8 (n = 8 n1 + n2, k = k1 + 4 k2)
template<int DIR>
struct dft32
{
    static __device__ __forceinline__ void run(float2* u)
    {
        float2 a[8][4];
#pragma unroll
        for (int n2 = 0; n2 < 8; ++n2) {
#pragma unroll
            for (int n1 = 0; n1 < 4; ++n1) { a[n2][n1] = u[8 * n1 + n2]; }
            dft<4, DIR>::run(a[n2]);
        }
        static_for<1, 8>([&](auto n2) {
            static_for<1, 4>([&](auto k1) {
                constexpr int N2 = decltype(n2)::value, K1 = decltype(k1)::value;
                a[N2][K1] = mul_w64<2 * N2 * K1, DIR>(a[N2][K1]);
            });
        });
#pragma unroll
        for (int k1 = 0; k1 < 4; ++k1) {
            float2 b[8];
#pragma unroll
            for (int n2 = 0; n2 < 8; ++n2) { b[n2] = a[n2][k1]; }
            dft<8, DIR>::run(b);
#pragma unroll
            for (int k2 = 0; k2 < 8; ++k2) { u[k1 + 4 * k2] = b[k2]; }
        }
    }
};

// the same butterfly under the name cta_fft looks up (float only): lets cta_fft run with 32 points per thread
template<int DIR>
struct dft<32, DIR>
{
    static __device__ __forceinline__ void run(float2* u) { dft32<DIR>::run(u); }
};

template<int R, int DIR>
struct wdft
{
    static __device__ __forceinline__ void run(float2* u)
    {
        if constexpr (R == 32) { dft32<DIR>::run(u); }
        else { dft<R, DIR>::run(u); }
    }
};

template<int LOGM, int LOGR1, int LOGR2>
struct wide_cfg
{
    static_assert(LOGR1 + LOGR2 + 4 == LOGM, "three stages, the last one radix 16");
    static_assert(LOGR1 >= 3 && LOGR1 <= 5 && LOGR2 >= 3 && LOGR2 <= 5, "radix 8, 16 or 32");
    static constexpr int M       = 1 << LOGM;
    static constexpr int R1      = 1 << LOGR1;
    static constexpr int R2      = 1 << LOGR2;
    static constexpr int NT      = M / 32;   // threads per transform
    static constexpr int S1      = M / R1;   // stage-1 butterflies = input stride of n1
    static constexpr int J       = M / 16;   // stage-3 butterflies
    static constexpr int BF1     = 32 / R1;  // stage-1 butterflies per thread
    static constexpr int BF2     = 32 / R2;
    static constexpr int LOGP    = LOGR1 > 4 ? LOGR1 : 4;  // rows of the power-of-two twiddle table
    static constexpr int XS      = S1 > J ? S1 : J;        // its row length
    static constexpr size_t SMEM    = size_t(M) * sizeof(float2);              // the tile
    // prefetching kernels: tile + staging buffer + the stage-2 twiddle table, 7/4 of the tile in total. The staging buffer holds the
    // first ST elements of the next row (a whole number of stage-1 input segments / stage-3 rows), the table sits behind it
    static constexpr int TB_FWD     = R2 * 16;   // W_(16 R2)^(a k2)
    static constexpr int TB_BWD     = R1 * R2;   // W_(R1 R2)^(a2 k1)
    static constexpr int ST_FWD     = 3 * M / 4 - TB_FWD;
    static constexpr int ST_BWD     = 3 * M / 4 - TB_BWD;
    static constexpr size_t SMEM_PF = SMEM + size_t(3 * M / 4) * sizeof(float2);
    static_assert(ST_FWD % S1 == 0 && ST_BWD % J == 0, "staging boundary between two stage-1 inputs / two stage-3 rows");
    static_assert(NT % 32 == 0, "whole warps");
};

// twiddles w[q] = W^(q x), q < R: the powers of two come from the table (row log2 q, stride xs), the rest are products
template<int R, class Load>
__device__ __forceinline__ void wide_twiddles(float2 (&w)[R], Load&& load)
{
#pragma unroll
    for (int q = 1; q < R; ++q) {
        int const hi = 1 << (31 - __clz(q));
        if (q == hi) { w[q] = load(31 - __clz(q)); }
        else { w[q] = cmul(w[hi], w[q - hi]); }
    }
}

// Hermitian split of a thread's two stage-3 butterflies (za: butterfly jA, zb: butterfly jB), results straight to the spectrum row.
// t > 0: jA = t, jB = J - t, Z[t + J k3] pairs with zb[15 - k3], twiddle W_2M^(t + J k3) = W_2M^t * exp(-2 pi i k3 / 32).
// t = 0: butterflies 0 and J/2 pair within themselves.
template<int M, class Store, class Edges>
__device__ __forceinline__ void wide_r2c_post(float2 const (&za)[16], float2 const (&zb)[16], int t, float2 wt, Store&& store, Edges&& edges)
{
    constexpr int J = M / 16;
    if (t != 0) {
        static_for<0, 16>([&](auto k3c) {
            constexpr int k3 = decltype(k3c)::value;
            float2 xk, xmk;
            r2c_post_pair(za[k3], zb[15 - k3], cmul(wt, w64_const<2 * k3>()), xk, xmk);
            int const k = t + J * k3;
            store(k, xk);
            store(M - k, xmk);
        });
    } else {
        edges(za[0].x + za[0].y, za[0].x - za[0].y);  // X[0], X[M]: both real
        store(M / 2, cconj(za[8]));
        static_for<1, 8>([&](auto k3c) {
            constexpr int k3 = decltype(k3c)::value;
            float2 xk, xmk;
            r2c_post_pair(za[k3], za[16 - k3], w64_const<2 * k3>(), xk, xmk);
            store(J * k3, xk);
            store(M - J * k3, xmk);
        });
        static_for<0, 8>([&](auto k3c) {
            constexpr int k3 = decltype(k3c)::value;
            float2 xk, xmk;
            r2c_post_pair(zb[k3], zb[15 - k3], w64_const<1 + 2 * k3>(), xk, xmk);
            store(J / 2 + J * k3, xk);
            store(M - J / 2 - J * k3, xmk);
        });
    }
}

// the reverse: xa[k3] = X[jA + J k3], xb[k3] = X[jB + J k3] (and Re X[M] for thread 0) -> Z of both butterflies, in place
template<int M>
__device__ __forceinline__ void wide_c2r_pre(float2 (&xa)[16], float2 (&xb)[16], int t, float2 wt, float nyq)
{
    if (t != 0) {
        static_for<0, 16>([&](auto k3c) {
            constexpr int k3 = decltype(k3c)::value;
            float2 zk, zmk;
            c2r_pre_pair(xa[k3], xb[15 - k3], cmul(wt, w64_const<2 * k3>()), zk, zmk);
            xa[k3]      = zk;
            xb[15 - k3] = zmk;
        });
    } else {
        float const dc = xa[0].x;
        xa[0]          = make_float2(dc + nyq, dc - nyq);
        xa[8]          = make_float2(2.0F * xa[8].x, -2.0F * xa[8].y);
        static_for<1, 8>([&](auto k3c) {
            constexpr int k3 = decltype(k3c)::value;
            float2 zk, zmk;
            c2r_pre_pair(xa[k3], xa[16 - k3], w64_const<2 * k3>(), zk, zmk);
            xa[k3]      = zk;
            xa[16 - k3] = zmk;
        });
        static_for<0, 8>([&](auto k3c) {
            constexpr int k3 = decltype(k3c)::value;
            float2 zk, zmk;
            c2r_pre_pair(xb[k3], xb[15 - k3], w64_const<1 + 2 * k3>(), zk, zmk);
            xb[k3]      = zk;
            xb[15 - k3] = zmk;
        });
    }
}

// ---- the three stages over one CTA's tile. DIR = -1: forward (S1, S2, S3), +1: backward (S3', S2', S1') ----------------------------
template<int LOGM, int LOGR1, int LOGR2>
struct wide_fft
{
    using cfg = wide_cfg<LOGM, LOGR1, LOGR2>;
    static constexpr int M = cfg::M, R1 = cfg::R1, R2 = cfg::R2, NT = cfg::NT, S1 = cfg::S1, J = cfg::J, BF1 = cfg::BF1, BF2 = cfg::BF2,
                         XS = cfg::XS;

    // stage 2 / 2': DFT_R2 along x of tile (k1, x, a), in place. tb: forward [R2][16] = W_(16 R2)^(a k2); backward [R1][R2] =
    // W_(R1 R2)^(a2 k1) (applied conjugated)
    // TB_SHARED: tb points into shared memory (the persistent kernels copy the table once per CTA)
    template<int DIR, bool TB_SHARED = false>
    static __device__ __forceinline__ void stage2(float2* sm, float2 const* __restrict__ tb, int t)
    {
        auto const tw = [&](int i) { return TB_SHARED ? tb[i] : __ldg(tb + i); };
#pragma unroll
        for (int m = 0; m < BF2; ++m) {
            int const beta = t + NT * m;
            int const a = beta & 15, k1 = beta >> 4;
            float2* const p = sm + k1 * (R2 * 16) + ((((a >> 1) ^ (k1 & 7)) << 1) | (a & 1));
            float2 u[R2];
#pragma unroll
            for (int x = 0; x < R2; ++x) { u[x] = p[x * 16]; }
            wdft<R2, DIR>::run(u);
            if constexpr (DIR < 0) {
#pragma unroll
                for (int k2 = 1; k2 < R2; ++k2) { u[k2] = cmul(u[k2], tw(k2 * 16 + a)); }
            } else {
#pragma unroll
                for (int a2 = 1; a2 < R2; ++a2) { u[a2] = cmulc(u[a2], tw(k1 * R2 + a2)); }
            }
#pragma unroll
            for (int x = 0; x < R2; ++x) { p[x * 16] = u[x]; }
        }
    }

    // rows of a stage-3 butterfly: 8 chunks of two values
    static __device__ __forceinline__ int row_chunk0(int j) { return ((j & (R1 - 1)) * R2 + (j >> LOGR1)) * 8; }

    static __device__ __forceinline__ void load_row(float4 const* sm4, int j, float2 (&v)[16])
    {
        int const base = row_chunk0(j), key = j & 7;  // k1 & 7 = j & 7 (R1 >= 8)
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            float4 const q = sm4[base + (c ^ key)];
            v[2 * c]       = make_float2(q.x, q.y);
            v[2 * c + 1]   = make_float2(q.z, q.w);
        }
    }

    static __device__ __forceinline__ void store_row(float4* sm4, int j, float2 const (&v)[16])
    {
        int const base = row_chunk0(j), key = j & 7;
#pragma unroll
        for (int c = 0; c < 8; ++c) { sm4[base + (c ^ key)] = make_float4(v[2 * c].x, v[2 * c].y, v[2 * c + 1].x, v[2 * c + 1].y); }
    }
};

// in: [batch][2M] reals (16-byte aligned), out: [batch][M+1] complex. ta: [LOGP][XS] W_M^(2^p x); tb: [R2][16]; rtw: W_2M^k, k < J/2
// Persistent CTAs, and no warp ever waits on DRAM: the NEXT row travels into shared memory by bulk copies (TMA) while this row is
// transformed. Its first three quarters go into a staging buffer behind the tile as soon as stage 1 has taken this row's inputs
// (a whole row time ahead: at the SM's fair share of the HBM bandwidth a row needs about that long); the last quarter goes into the
// tile itself, which is idle from the stage-3 loads on. Both copies signal one mbarrier (two arrivals per phase).
template<int M, int ST>  // ST: complex elements of a row kept in the staging buffer; the rest sits at the tile's start
struct wide_stage
{
    static constexpr unsigned EARLY = unsigned(ST) * 8U, LATE = unsigned(M - ST) * 8U;
    float2* tile;
    float2* stage;
    __device__ __forceinline__ void fetch_early(float2 const* row, void* bar) const { wtma::fetch(stage, row, EARLY, bar); }
    __device__ __forceinline__ void fetch_late(float2 const* row, void* bar) const { wtma::fetch(tile, row + ST, LATE, bar); }
    // element e of the staged row; REGION known at compile time wherever the caller's index is
    template<bool IN_TILE>
    __device__ __forceinline__ float2 const* at(int e) const
    {
        return IN_TILE ? tile + (e - ST) : stage + e;
    }
    __device__ __forceinline__ float2 get(int e) const { return e < ST ? stage[e] : tile[e - ST]; }
};

template<int LOGM, int LOGR1, int LOGR2, int MINCTAS>
__global__ void __launch_bounds__(wide_cfg<LOGM, LOGR1, LOGR2>::NT, MINCTAS)
    r2c_wide_kernel(float const* __restrict__ in, float2* __restrict__ out, float2 const* __restrict__ ta, float2 const* __restrict__ tb,
                    float2 const* __restrict__ rtw, size_t batch)
{
    using W   = wide_fft<LOGM, LOGR1, LOGR2>;
    using cfg = wide_cfg<LOGM, LOGR1, LOGR2>;
    constexpr int M = cfg::M, R1 = cfg::R1, R2 = cfg::R2, NT = cfg::NT, S1 = cfg::S1, J = cfg::J, BF1 = cfg::BF1, XS = cfg::XS;
    extern __shared__ __align__(128) unsigned char wide_smem_raw[];
    float2* const sm  = reinterpret_cast<float2*>(wide_smem_raw);
    float4* const sm4 = reinterpret_cast<float4*>(wide_smem_raw);
    int const t       = threadIdx.x;
    __shared__ __align__(8) unsigned long long bar;
    unsigned parity = 0;
    using stage_t = wide_stage<M, cfg::ST_FWD>;
    stage_t const st{sm, sm + M};
    float2* const tbs = sm + M + cfg::ST_FWD;  // stage-2 twiddles in shared memory
    auto const zrow = [&](size_t row) { return reinterpret_cast<float2 const*>(in) + row * size_t(M); };
    static_assert(BF1 == 2 || BF1 == 1, "one pass over the staged row");
    for (int i = t; i < cfg::TB_FWD; i += NT) { tbs[i] = __ldg(tb + i); }
    if (t == 0) {
        wtma::init(&bar, 2);
        if (blockIdx.x < batch) {
            st.fetch_early(zrow(blockIdx.x), &bar);
            st.fetch_late(zrow(blockIdx.x), &bar);
        }
    }
    __syncthreads();

    for (size_t b = blockIdx.x; b < batch; b += gridDim.x) {
        bool const more = b + gridDim.x < batch;
        // ---- stage 1
        if constexpr (BF1 >= 2) {
#pragma unroll
            for (int m = 0; m < BF1 / 2; ++m) {
                int const n = 2 * t + 2 * NT * m;  // this thread's butterflies n and n + 1
                float2 ua[R1], ub[R1];
                wtma::wait(&bar, parity);
                parity ^= 1U;
                static_for<0, R1>([&](auto n1c) {
                    constexpr int n1 = decltype(n1c)::value;
                    float4 const q = *reinterpret_cast<float4 const*>(st.template at<(n1 * S1 >= cfg::ST_FWD)>(n + n1 * S1));
                    ua[n1]         = make_float2(q.x, q.y);
                    ub[n1]         = make_float2(q.z, q.w);
                });
                __syncthreads();  // every thread has its inputs: staging buffer and tile may be overwritten
                if (t == 0 && more) { st.fetch_early(zrow(b + gridDim.x), &bar); }
                wdft<R1, -1>::run(ua);
                wdft<R1, -1>::run(ub);
                {
                    float4 const* const ta4 = reinterpret_cast<float4 const*>(ta) + (n >> 1);
                    float2 wa[R1], wb[R1];
#pragma unroll
                    for (int q = 1; q < R1; ++q) {
                        int const hi = 1 << (31 - __clz(q));
                        if (q == hi) {
                            float4 const w4 = __ldg(ta4 + (31 - __clz(q)) * (XS / 2));
                            wa[q]           = make_float2(w4.x, w4.y);
                            wb[q]           = make_float2(w4.z, w4.w);
                        } else {
                            wa[q] = cmul(wa[hi], wa[q - hi]);
                            wb[q] = cmul(wb[hi], wb[q - hi]);
                        }
                        ua[q] = cmul(ua[q], wa[q]);
                        ub[q] = cmul(ub[q], wb[q]);
                    }
                }
                int const a2 = n >> 4, ah = (n & 15) >> 1;
#pragma unroll
                for (int k1 = 0; k1 < R1; ++k1) {
                    sm4[(k1 * R2 + a2) * 8 + (ah ^ (k1 & 7))] = make_float4(ua[k1].x, ua[k1].y, ub[k1].x, ub[k1].y);
                }
            }
        } else {
            int const n = t;
            float2 u[R1];
            wtma::wait(&bar, parity);
            parity ^= 1U;
            static_for<0, R1>([&](auto n1c) {
                constexpr int n1 = decltype(n1c)::value;
                u[n1]            = *st.template at<(n1 * S1 >= cfg::ST_FWD)>(n + n1 * S1);
            });
            __syncthreads();
            if (t == 0 && more) { st.fetch_early(zrow(b + gridDim.x), &bar); }
            wdft<R1, -1>::run(u);
            {
                float2 w[R1];
#pragma unroll
                for (int q = 1; q < R1; ++q) {
                    int const hi = 1 << (31 - __clz(q));
                    if (q == hi) { w[q] = __ldg(ta + (31 - __clz(q)) * XS + n); }
                    else { w[q] = cmul(w[hi], w[q - hi]); }
                    u[q] = cmul(u[q], w[q]);
                }
            }
            int const a = n & 15, a2 = n >> 4;
#pragma unroll
            for (int k1 = 0; k1 < R1; ++k1) { sm[(k1 * R2 + a2) * 16 + ((((a >> 1) ^ (k1 & 7)) << 1) | (a & 1))] = u[k1]; }
        }
        __syncthreads();
        // ---- stage 2, in place
        W::template stage2<-1, true>(sm, tbs, t);
        __syncthreads();
        // ---- stage 3 + Hermitian split in registers
        {
            int const ja = t, jb = t == 0 ? J / 2 : J - t;
            float2 const wt = __ldg(rtw + t);
            float2 za[16], zb[16];
            W::load_row(sm4, ja, za);
            W::load_row(sm4, jb, zb);
            __syncthreads();  // the tile is free for the next row
            if (t == 0 && more) { st.fetch_late(zrow(b + gridDim.x), &bar); }
            dft<16, -1>::run(za);
            dft<16, -1>::run(zb);
            float2* const row = out + b * (size_t(M) + 1);
            wide_r2c_post<M>(za, zb, t, wt, [&](int k, float2 x) { row[k] = x; },
                             [&](float dc, float nyq) {
                                 row[0] = make_float2(dc, 0.0F);
                                 row[M] = make_float2(nyq, 0.0F);
                             });
        }
    }
}

// in: [batch][row_len] complex (first M+1 used), out: [batch][2M] reals (16-byte aligned), unnormalised. tb: [R1][R2]
// Persistent CTAs fed by bulk copies as in r2c_wide_kernel. A spectrum row of M+1 bins starts on an 8-byte boundary only, so the bulk copies take the M bins from
// the row's first 16-byte boundary on (bins lo .. lo+M-1, lo = 0 or 1) and thread 0 fetches the one bin left out (X[M] or X[0]).
template<int LOGM, int LOGR1, int LOGR2, int MINCTAS>
__global__ void __launch_bounds__(wide_cfg<LOGM, LOGR1, LOGR2>::NT, MINCTAS)
    c2r_wide_kernel(float2 const* __restrict__ in, size_t row_len, float* __restrict__ out, float2 const* __restrict__ ta,
                    float2 const* __restrict__ tb, float2 const* __restrict__ rtw, size_t batch)
{
    using W   = wide_fft<LOGM, LOGR1, LOGR2>;
    using cfg = wide_cfg<LOGM, LOGR1, LOGR2>;
    constexpr int M = cfg::M, R1 = cfg::R1, R2 = cfg::R2, NT = cfg::NT, S1 = cfg::S1, J = cfg::J, BF1 = cfg::BF1, XS = cfg::XS;
    extern __shared__ __align__(128) unsigned char wide_smem_raw[];
    float2* const sm  = reinterpret_cast<float2*>(wide_smem_raw);
    float4* const sm4 = reinterpret_cast<float4*>(wide_smem_raw);
    int const t       = threadIdx.x;
    __shared__ __align__(8) unsigned long long bar;
    unsigned parity = 0;
    using stage_t = wide_stage<M, cfg::ST_BWD>;
    stage_t const st{sm, sm + M};
    float2* const tbs = sm + M + cfg::ST_BWD;
    constexpr int K3T = cfg::ST_BWD / J;  // stage-3 inputs k3 >= K3T sit in the tile, the others in the staging buffer
    // first bin of row `row` that sits on a 16-byte boundary
    auto const xrow = [&](size_t row) {
        float2 const* const x = in + row * row_len;
        return x + ((reinterpret_cast<std::uintptr_t>(x) >> 3) & 1U);
    };
    for (int i = t; i < cfg::TB_BWD; i += NT) { tbs[i] = __ldg(tb + i); }
    if (t == 0) {
        wtma::init(&bar, 2);
        if (blockIdx.x < batch) {
            st.fetch_early(xrow(blockIdx.x), &bar);
            st.fetch_late(xrow(blockIdx.x), &bar);
        }
    }
    __syncthreads();

    for (size_t b = blockIdx.x; b < batch; b += gridDim.x) {
        bool const more = b + gridDim.x < batch;
        // ---- Hermitian pre-pass in registers + stage 3'
        {
            float2 const* const x = in + b * row_len;
            int const ja = t, jb = t == 0 ? J / 2 : J - t;
            float2 const wt = __ldg(rtw + t);
            float2 za[16], zb[16];
            float nyq = 0.0F;
            int const lo = int(xrow(b) - x);
            float2 edge  = make_float2(0.0F, 0.0F);
            if (t == 0) { edge = x[lo ? 0 : M]; }
            wtma::wait(&bar, parity);
            parity ^= 1U;
            // bin k sits at staged element k - lo. For t > 0 both ja + J k3 - lo and jb + J k3 - lo stay inside [J k3, J (k3 + 1)),
            // so the region follows from k3 alone (the staging boundary is K3T J)
            if (t != 0) {
                static_for<0, 16>([&](auto k3c) {
                    constexpr int k3 = decltype(k3c)::value;
                    za[k3]           = *st.template at<(k3 >= K3T)>(ja + J * k3 - lo);
                    zb[k3]           = *st.template at<(k3 >= K3T)>(jb + J * k3 - lo);
                });
            } else {
#pragma unroll
                for (int k3 = 1; k3 < 16; ++k3) { za[k3] = st.get(J * k3 - lo); }
#pragma unroll
                for (int k3 = 0; k3 < 16; ++k3) { zb[k3] = st.get(J / 2 + J * k3 - lo); }
                za[0] = lo ? edge : st.get(0);
                nyq   = lo ? st.get(M - 1).x : edge.x;
            }
            __syncthreads();  // every thread has its inputs: staging buffer and tile may be overwritten
            if (t == 0 && more) { st.fetch_early(xrow(b + gridDim.x), &bar); }
            wide_c2r_pre<M>(za, zb, t, wt, nyq);
            dft<16, +1>::run(za);
            dft<16, +1>::run(zb);
            {
                float2 w[16];
                wide_twiddles(w, [&](int p) { return __ldg(ta + p * XS + ja); });
#pragma unroll
                for (int a = 1; a < 16; ++a) { za[a] = cmulc(za[a], w[a]); }
                wide_twiddles(w, [&](int p) { return __ldg(ta + p * XS + jb); });
#pragma unroll
                for (int a = 1; a < 16; ++a) { zb[a] = cmulc(zb[a], w[a]); }
            }
            W::store_row(sm4, ja, za);
            W::store_row(sm4, jb, zb);
        }
        __syncthreads();
        // ---- stage 2', in place
        W::template stage2<+1, true>(sm, tbs, t);
        __syncthreads();
        // ---- stage 1'
        if constexpr (BF1 >= 2) {
#pragma unroll
            for (int m = 0; m < BF1 / 2; ++m) {
                int const n  = 2 * t + 2 * NT * m;
                int const a2 = n >> 4, ah = (n & 15) >> 1;
                float2 ua[R1], ub[R1];
#pragma unroll
                for (int k1 = 0; k1 < R1; ++k1) {
                    float4 const q = sm4[(k1 * R2 + a2) * 8 + (ah ^ (k1 & 7))];
                    ua[k1]         = make_float2(q.x, q.y);
                    ub[k1]         = make_float2(q.z, q.w);
                }
                if (m == BF1 / 2 - 1) {
                    __syncthreads();  // the tile is free for the next row
                    if (t == 0 && more) { st.fetch_late(xrow(b + gridDim.x), &bar); }
                }
                wdft<R1, +1>::run(ua);
                wdft<R1, +1>::run(ub);
                float4* const dst = reinterpret_cast<float4*>(out + b * (2 * size_t(M))) + (n >> 1);
#pragma unroll
                for (int b2 = 0; b2 < R1; ++b2) { __stcs(dst + b2 * (S1 / 2), make_float4(ua[b2].x, ua[b2].y, ub[b2].x, ub[b2].y)); }
            }
        } else {
            int const n = t, a = n & 15, a2 = n >> 4;
            float2 u[R1];
#pragma unroll
            for (int k1 = 0; k1 < R1; ++k1) { u[k1] = sm[(k1 * R2 + a2) * 16 + ((((a >> 1) ^ (k1 & 7)) << 1) | (a & 1))]; }
            __syncthreads();
            if (t == 0 && more) { st.fetch_late(xrow(b + gridDim.x), &bar); }
            wdft<R1, +1>::run(u);
            float2* const dst = reinterpret_cast<float2*>(out + b * (2 * size_t(M))) + n;
#pragma unroll
            for (int b2 = 0; b2 < R1; ++b2) { __stcs(dst + b2 * S1, u[b2]); }
        }
    }
}

// ---- N = 4 M2 real points as TWO CTAs per transform (the half-size complex transform of M = 2 M2 points is one decimation-in-
// frequency step too long for one tile): CTA r = 0, 1 forms y_r[n] = (z[n] + (-1)^r z[n + M2]) W_M^(r n) on the fly and its M2-point
// wide transform yields the bins of parity r. Both CTAs of a row run side by side (adjacent block indices), so the second read of
// every line is an L2 hit. Each CTA still needs the WHOLE row (2 M2 complex = twice the tile): the first half travels into the tile
// (late bulk copy), the first three quarters of the second half into the staging buffer (early bulk copy), the rest comes by
// ordinary loads issued before the wait.
//   forward:  Z[r + 2 k2] pairs with Z[M - r - 2 k2] = sub-bin M2 - r - k2: r = 0 as in r2c_wide_kernel, r = 1 rows j and J-1-j (no
//             self-paired rows); twiddle W_2M^(r + 2 k2) = W_2M^r * W_2M2^k2.
//   backward: the Hermitian pre-pass pairs X[k] with X[M - k] BEFORE the parity split, so both parities use rows j and J - j:
//             X[k2], X[M-k2], X[M2-k2], X[M2+k2] give Z at those four bins and from them y_r[k2] and y_r[M2-k2].
template<int LOGM2, int LOGR1, int LOGR2>
__global__ void __launch_bounds__(wide_cfg<LOGM2, LOGR1, LOGR2>::NT, 1)
    r2c_wide_split_kernel(float const* __restrict__ in, float2* __restrict__ out, float2 const* __restrict__ ta, float2 const* __restrict__ tb,
                          float2 const* __restrict__ rtw, float2 const* __restrict__ w_m, float2 w_2m1, size_t batch)
{
    using W   = wide_fft<LOGM2, LOGR1, LOGR2>;
    using cfg = wide_cfg<LOGM2, LOGR1, LOGR2>;
    constexpr int M2 = cfg::M, M = 2 * M2, R1 = cfg::R1, R2 = cfg::R2, S1 = cfg::S1, J = cfg::J, XS = cfg::XS;
    static_assert(cfg::BF1 == 1 && R1 == 32, "one radix-32 butterfly per thread in stage 1");
    constexpr int ST = cfg::ST_FWD;      // staged part of the second half
    constexpr int NG = (M2 - ST) / S1;   // inputs per thread that come by ordinary loads
    extern __shared__ __align__(128) unsigned char wide_smem_raw[];
    float2* const sm  = reinterpret_cast<float2*>(wide_smem_raw);
    float4* const sm4 = reinterpret_cast<float4*>(wide_smem_raw);
    float2* const stg = sm + M2;
    float2* const tbs = stg + ST;  // stage-2 twiddles
    int const t       = threadIdx.x;
    int const r       = blockIdx.x & 1;
    __shared__ __align__(8) unsigned long long bar;
    unsigned parity = 0;
    size_t const units = 2 * batch;  // (row, parity), parity fastest: gridDim.x is even, so a CTA keeps its parity
    auto const zrow = [&](size_t unit) { return reinterpret_cast<float2 const*>(in) + (unit >> 1) * size_t(M); };
    for (int i = t; i < cfg::TB_FWD; i += cfg::NT) { tbs[i] = __ldg(tb + i); }
    if (t == 0) {
        wtma::init(&bar, 2);
        if (blockIdx.x < units) {
            wtma::fetch(stg, zrow(blockIdx.x) + M2, unsigned(ST) * 8U, &bar);
            wtma::fetch(sm, zrow(blockIdx.x), unsigned(M2) * 8U, &bar);
        }
    }
    __syncthreads();
    float2 const w_in = r ? __ldg(w_m + t) : make_float2(1.0F, 0.0F);  // W_M^n', n' = t

    for (size_t unit = blockIdx.x; unit < units; unit += gridDim.x) {
        bool const more = unit + gridDim.x < units;
        // ---- stage 1 on y_r
        {
            int const n = t;
            float2 u[R1], g[NG];
            float2 const* const z = zrow(unit);
#pragma unroll
            for (int i = 0; i < NG; ++i) { g[i] = __ldcs(z + M2 + ST + n + i * S1); }
            wtma::wait(&bar, parity);
            parity ^= 1U;
            static_for<0, R1>([&](auto n1c) {
                constexpr int n1 = decltype(n1c)::value;
                float2 const a   = sm[n + n1 * S1];
                float2 c;
                if constexpr (n1 * S1 < ST) { c = stg[n + n1 * S1]; }
                else { c = g[n1 - ST / S1]; }
                // W_M^(n' + S1 n1) = W_M^n' * exp(-2 pi i n1 / 64)
                u[n1] = r ? cmul(mul_w64<n1, -1>(csub(a, c)), w_in) : cadd(a, c);
            });
            __syncthreads();  // every thread has its inputs: staging buffer and tile may be overwritten
            if (t == 0 && more) { wtma::fetch(stg, zrow(unit + gridDim.x) + M2, unsigned(ST) * 8U, &bar); }
            wdft<R1, -1>::run(u);
            {
                float2 w[R1];
#pragma unroll
                for (int q = 1; q < R1; ++q) {
                    int const hi = 1 << (31 - __clz(q));
                    if (q == hi) { w[q] = __ldg(ta + (31 - __clz(q)) * XS + n); }
                    else { w[q] = cmul(w[hi], w[q - hi]); }
                    u[q] = cmul(u[q], w[q]);
                }
            }
            int const a = n & 15, a2 = n >> 4;
#pragma unroll
            for (int k1 = 0; k1 < R1; ++k1) { sm[(k1 * R2 + a2) * 16 + ((((a >> 1) ^ (k1 & 7)) << 1) | (a & 1))] = u[k1]; }
        }
        __syncthreads();
        W::template stage2<-1, true>(sm, tbs, t);
        __syncthreads();
        {
            int const ja = t, jb = r ? J - 1 - t : (t == 0 ? J / 2 : J - t);
            float2 wt = __ldg(rtw + t);
            float2 za[16], zb[16];
            W::load_row(sm4, ja, za);
            W::load_row(sm4, jb, zb);
            __syncthreads();  // the tile is free for the next unit
            if (t == 0 && more) { wtma::fetch(sm, zrow(unit + gridDim.x), unsigned(M2) * 8U, &bar); }
            dft<16, -1>::run(za);
            dft<16, -1>::run(zb);
            float2* const row = out + (unit >> 1) * (size_t(M) + 1);
            if (r == 0) {
                wide_r2c_post<M2>(za, zb, t, wt, [&](int k, float2 x) { row[2 * k] = x; },
                                  [&](float dc, float nyq) {
                                      row[0] = make_float2(dc, 0.0F);
                                      row[M] = make_float2(nyq, 0.0F);
                                  });
            } else {
                wt = cmul(wt, w_2m1);
                static_for<0, 16>([&](auto k3c) {
                    constexpr int k3 = decltype(k3c)::value;
                    float2 xk, xmk;
                    r2c_post_pair(za[k3], zb[15 - k3], cmul(wt, w64_const<2 * k3>()), xk, xmk);
                    int const k2 = t + J * k3;
                    row[1 + 2 * k2]     = xk;
                    row[M - 1 - 2 * k2] = xmk;
                });
            }
        }
    }
}

// in: [batch][row_len] complex (first 2 M2 + 1 used), out: [batch][4 M2] reals, unnormalised. w_m[k] = exp(-2 pi i k / M), k < J
template<int LOGM2, int LOGR1, int LOGR2>
__global__ void __launch_bounds__(wide_cfg<LOGM2, LOGR1, LOGR2>::NT, 1)
    c2r_wide_split_kernel(float2 const* __restrict__ in, size_t row_len, float* __restrict__ out, float2 const* __restrict__ ta,
                          float2 const* __restrict__ tb, float2 const* __restrict__ rtw, float2 const* __restrict__ w_m, size_t batch)
{
    using W   = wide_fft<LOGM2, LOGR1, LOGR2>;
    using cfg = wide_cfg<LOGM2, LOGR1, LOGR2>;
    constexpr int M2 = cfg::M, M = 2 * M2, R1 = cfg::R1, R2 = cfg::R2, S1 = cfg::S1, J = cfg::J, XS = cfg::XS;
    static_assert(cfg::BF1 == 1 && R1 == 32, "one radix-32 butterfly per thread in stage 1'");
    constexpr int ST  = cfg::ST_BWD;
    constexpr int K3T = ST / J;  // second-half bins with k3 >= K3T lie beyond the staged window
    extern __shared__ __align__(128) unsigned char wide_smem_raw[];
    float2* const sm  = reinterpret_cast<float2*>(wide_smem_raw);
    float4* const sm4 = reinterpret_cast<float4*>(wide_smem_raw);
    float2* const stg = sm + M2;
    float2* const tbs = stg + ST;
    int const t       = threadIdx.x;
    int const r       = blockIdx.x & 1;
    __shared__ __align__(8) unsigned long long bar;
    unsigned parity = 0;
    size_t const units = 2 * batch;
    for (int i = t; i < cfg::TB_BWD; i += cfg::NT) { tbs[i] = __ldg(tb + i); }
    // first bin of a unit's row that sits on a 16-byte boundary
    auto const xrow = [&](size_t unit) {
        float2 const* const x = in + (unit >> 1) * row_len;
        return x + ((reinterpret_cast<std::uintptr_t>(x) >> 3) & 1U);
    };
    if (t == 0) {
        wtma::init(&bar, 2);
        if (blockIdx.x < units) {
            wtma::fetch(stg, xrow(blockIdx.x) + M2, unsigned(ST) * 8U, &bar);
            wtma::fetch(sm, xrow(blockIdx.x), unsigned(M2) * 8U, &bar);
        }
    }
    __syncthreads();
    // the staged window holds bins lo .. lo + M2 + ST - 1 at tile[k - lo] (k - lo < M2) / stg[k - lo - M2]
    auto const staged = [&](int e) { return e < M2 ? sm[e] : stg[e - M2]; };

    for (size_t unit = blockIdx.x; unit < units; unit += gridDim.x) {
        bool const more = unit + gridDim.x < units;
        {
            float2 const* const x = in + (unit >> 1) * row_len;
            int const lo = int(xrow(unit) - x);
            int const ja = t, jb = t == 0 ? J / 2 : J - t;
            float2 const wt = __ldg(rtw + t);
            // xa[k3] = X[k2], xb[15-k3] = X[M2-k2], ya[k3] = X[M2+k2], yb[15-k3] = X[M-k2]   (k2 = ja + J k3; row jb = J - ja)
            float2 xa[16], xb[16], ya[16], yb[16];
            // ordinary loads first: the bins beyond the staged window (k - lo >= M2 + ST  <=>  k3 >= K3T of the second half)
            if (t != 0) {
#pragma unroll
                for (int k3 = K3T; k3 < 16; ++k3) {
                    ya[k3] = __ldcs(x + M2 + ja + J * k3);
                    yb[k3] = __ldcs(x + M2 + jb + J * k3);
                }
            }
            wtma::wait(&bar, parity);
            parity ^= 1U;
            if (t != 0) {
                static_for<0, 16>([&](auto k3c) {
                    constexpr int k3 = decltype(k3c)::value;
                    xa[k3]           = sm[ja + J * k3 - lo];
                    xb[k3]           = sm[jb + J * k3 - lo];
                    if constexpr (k3 < K3T) {
                        ya[k3] = stg[ja + J * k3 - lo];
                        yb[k3] = stg[jb + J * k3 - lo];
                    }
                });
            } else {
                // thread 0: rows 0 and J/2 of both halves; bins at the window's edges come by ordinary loads
                auto const bin = [&](int k) { return (k - lo >= 0 && k - lo < M2 + ST) ? staged(k - lo) : x[k]; };
#pragma unroll
                for (int k3 = 0; k3 < 16; ++k3) {
                    xa[k3] = bin(J * k3);
                    xb[k3] = bin(J / 2 + J * k3);
                    ya[k3] = bin(M2 + J * k3);
                    yb[k3] = bin(M2 + J / 2 + J * k3);
                }
            }
            float const nyq = t == 0 ? x[M].x : 0.0F;
            // Hermitian pre-pass on the FULL-size spectrum (M bins), twiddle W_2M^k -- before the barrier, so that 32 values per thread
            // are live across it, not 64
            float2 za[16], zb[16];
            if (t != 0) {
                static_for<0, 16>([&](auto k3c) {
                    constexpr int k3 = decltype(k3c)::value;
                    // k = k2 = ja + J k3:  W_2M^k2 = W_2M^ja * exp(-2 pi i k3 / 64)   (J / 2M = 1/64)
                    float2 const w = cmul(wt, w64_const<k3>());
                    float2 z_k, z_mk, z_m2mk, z_m2pk;
                    c2r_pre_pair(xa[k3], yb[15 - k3], w, z_k, z_mk);  // X[k2], X[M - k2]
                    // k = M2 - k2: W_2M^(M2 - k2) = -i conj(W_2M^k2)
                    float2 const wp = make_float2(-w.y, -w.x);
                    c2r_pre_pair(xb[15 - k3], ya[k3], wp, z_m2mk, z_m2pk);  // X[M2 - k2], X[M2 + k2]
                    if (r == 0) {
                        za[k3]      = cadd(z_k, z_m2pk);
                        zb[15 - k3] = cadd(z_m2mk, z_mk);
                    } else {
                        za[k3]      = csub(z_k, z_m2pk);
                        zb[15 - k3] = csub(z_m2mk, z_mk);
                    }
                });
            } else {
                // row 0: k2 = J k3. k3 = 0: Z[0] from the edges, Z[M2] = 2 conj(X[M2]); the other bins pair first half <-> second half
                float2 zf[16], zs[16];  // Z[k2] and Z[M2 + k2] along row 0
                zf[0] = make_float2(xa[0].x + nyq, xa[0].x - nyq);
                zs[0] = make_float2(2.0F * ya[0].x, -2.0F * ya[0].y);
                static_for<1, 16>([&](auto k3c) {
                    constexpr int k3 = decltype(k3c)::value;
                    // X[k2] and X[M - k2], M - k2 = M2 + J (16 - k3); twiddle W_2M^(J k3) = exp(-2 pi i k3 / 64)
                    float2 z_k, z_mk;
                    c2r_pre_pair(xa[k3], ya[16 - k3], w64_const<k3>(), z_k, z_mk);
                    zf[k3]      = z_k;
                    zs[16 - k3] = z_mk;
                });
                float2 zf2[16], zs2[16];  // along row J/2: k2 = J/2 + J k3, twiddle exp(-2 pi i (1 + 2 k3) / 128)
                static_for<0, 16>([&](auto k3c) {
                    constexpr int k3 = decltype(k3c)::value;
                    // X[k2] = xb[k3], X[M - k2] = X[M2 + J/2 + J (15 - k3)] = yb[15 - k3]
                    float2 const w = w128_const<1 + 2 * k3>();
                    float2 z_k, z_mk;
                    c2r_pre_pair(xb[k3], yb[15 - k3], w, z_k, z_mk);
                    zf2[k3]      = z_k;   // Z[k2]
                    zs2[15 - k3] = z_mk;  // Z[M - k2] = Z[M2 + (J/2 + J (15 - k3))]
                });
#pragma unroll
                for (int k3 = 0; k3 < 16; ++k3) {
                    za[k3] = r == 0 ? cadd(zf[k3], zs[k3]) : csub(zf[k3], zs[k3]);
                    zb[k3] = r == 0 ? cadd(zf2[k3], zs2[k3]) : csub(zf2[k3], zs2[k3]);
                }
            }
            __syncthreads();  // every thread has consumed its inputs: staging buffer and tile may be overwritten
            if (t == 0 && more) { wtma::fetch(stg, xrow(unit + gridDim.x) + M2, unsigned(ST) * 8U, &bar); }
            if (r != 0) {
                // times conj(W_M^k2), k2 = j + J k3:  W_M^j * exp(-2 pi i k3 / 32)
                float2 const wa = __ldg(w_m + ja), wb = __ldg(w_m + jb);
                static_for<0, 16>([&](auto k3c) {
                    constexpr int k3 = decltype(k3c)::value;
                    za[k3]           = cmulc(mul_w64<2 * k3, +1>(za[k3]), wa);
                    zb[k3]           = cmulc(mul_w64<2 * k3, +1>(zb[k3]), wb);
                });
            }
            dft<16, +1>::run(za);
            dft<16, +1>::run(zb);
            {
                float2 w[16];
                wide_twiddles(w, [&](int p) { return __ldg(ta + p * XS + ja); });
#pragma unroll
                for (int a = 1; a < 16; ++a) { za[a] = cmulc(za[a], w[a]); }
                wide_twiddles(w, [&](int p) { return __ldg(ta + p * XS + jb); });
#pragma unroll
                for (int a = 1; a < 16; ++a) { zb[a] = cmulc(zb[a], w[a]); }
            }
            W::store_row(sm4, ja, za);
            W::store_row(sm4, jb, zb);
        }
        __syncthreads();
        W::template stage2<+1, true>(sm, tbs, t);
        __syncthreads();
        {
            int const n = t, a = n & 15, a2 = n >> 4;
            float2 u[R1];
#pragma unroll
            for (int k1 = 0; k1 < R1; ++k1) { u[k1] = sm[(k1 * R2 + a2) * 16 + ((((a >> 1) ^ (k1 & 7)) << 1) | (a & 1))]; }
            __syncthreads();
            if (t == 0 && more) { wtma::fetch(sm, xrow(unit + gridDim.x), unsigned(M2) * 8U, &bar); }
            wdft<R1, +1>::run(u);
            // y_r's transform is z[r + 2 n]
            float2* const dst = reinterpret_cast<float2*>(out + (unit >> 1) * (2 * size_t(M))) + r + 2 * n;
#pragma unroll
            for (int b2 = 0; b2 < R1; ++b2) { __stcs(dst + 2 * b2 * S1, u[b2]); }
        }
    }
}

// ---- inverse transform with one WARP per transform (M = 1024: the convolver's 2048-point real transforms), load / store sides as
// policy objects like c2r_kernel. The three stages only need __syncwarp(): warps never wait for each other, so their load, butterfly
// and store phases drift apart and overlap. Policies provide (besides open / load of the narrow kernel) the 128-bit stores of the
// real side: store_pair<HI>(row, j, z0, z1) with j an even index inside the lower (HI = false) or upper half of the real row's
// complex pairs. MINB: resident CTAs per SM the kernel is compiled for (5: 96 registers).
template<int LOGM, int LOGR1, int LOGR2, int G, class IO, int MINB>
__global__ void __launch_bounds__(32 * G, MINB)
    c2r_wide_io_kernel(IO io, float2 const* __restrict__ ta, float2 const* __restrict__ tb, float2 const* __restrict__ rtw, size_t batch)
{
    using W   = wide_fft<LOGM, LOGR1, LOGR2>;
    using cfg = wide_cfg<LOGM, LOGR1, LOGR2>;
    constexpr int M = cfg::M, R1 = cfg::R1, R2 = cfg::R2, NT = cfg::NT, S1 = cfg::S1, J = cfg::J, BF1 = cfg::BF1, XS = cfg::XS, H = M / 2;
    static_assert(NT == 32 && BF1 >= 2, "one warp per transform, pairs of stage-1 butterflies");
    extern __shared__ __align__(128) unsigned char wide_smem_raw[];
    int const t    = threadIdx.x & 31;
    size_t const b = size_t(blockIdx.x) * G + (threadIdx.x >> 5);
    if (b >= batch) { return; }
    float2* const sm  = reinterpret_cast<float2*>(wide_smem_raw) + (threadIdx.x >> 5) * M;
    float4* const sm4 = reinterpret_cast<float4*>(sm);
    typename IO::row_state const row = io.open(b);
    {
        int const ja = t, jb = t == 0 ? J / 2 : J - t;
        float2 const wt = __ldg(rtw + t);
        float2 za[16], zb[16];
#pragma unroll
        for (int k3 = 0; k3 < 16; ++k3) { za[k3] = io.load(row, ja + J * k3); }  // thread 0, k3 = 0: the packed pair (Re X[0], Re X[M])
#pragma unroll
        for (int k3 = 0; k3 < 16; ++k3) { zb[k3] = io.load(row, jb + J * k3); }
        float const nyq = za[0].y;  // only thread 0 uses it
        wide_c2r_pre<M>(za, zb, t, wt, nyq);
        dft<16, +1>::run(za);
        dft<16, +1>::run(zb);
        {
            float2 w[16];
            wide_twiddles(w, [&](int p) { return __ldg(ta + p * XS + ja); });
#pragma unroll
            for (int a = 1; a < 16; ++a) { za[a] = cmulc(za[a], w[a]); }
            wide_twiddles(w, [&](int p) { return __ldg(ta + p * XS + jb); });
#pragma unroll
            for (int a = 1; a < 16; ++a) { zb[a] = cmulc(zb[a], w[a]); }
        }
        W::store_row(sm4, ja, za);
        W::store_row(sm4, jb, zb);
    }
    __syncwarp();
    W::template stage2<+1>(sm, tb, t);
    __syncwarp();
#pragma unroll
    for (int m = 0; m < BF1 / 2; ++m) {
        int const n  = 2 * t + 2 * NT * m;
        int const a2 = n >> 4, ah = (n & 15) >> 1;
        float2 ua[R1], ub[R1];
#pragma unroll
        for (int k1 = 0; k1 < R1; ++k1) {
            float4 const q = sm4[(k1 * R2 + a2) * 8 + (ah ^ (k1 & 7))];
            ua[k1]         = make_float2(q.x, q.y);
            ub[k1]         = make_float2(q.z, q.w);
        }
        wdft<R1, +1>::run(ua);
        wdft<R1, +1>::run(ub);
        static_for<0, R1>([&](auto b2c) {
            constexpr int b2 = decltype(b2c)::value;
            if constexpr (b2 < R1 / 2) { io.template store_pair<false>(row, n + S1 * b2, ua[b2], ub[b2]); }
            else { io.template store_pair<true>(row, n + S1 * b2 - H, ua[b2], ub[b2]); }
        });
    }
}

template<int LOGM, int LOGR1, int LOGR2, class IO>
int launch_c2r_wide_io(IO const& io, float2 const* ta, float2 const* tb, float2 const* rtw, size_t batch, cudaStream_t stream)
{
    using cfg       = wide_cfg<LOGM, LOGR1, LOGR2>;
    constexpr int G = 4;
    if (batch == 0) { return NEO_B200_OK; }
    auto kernel = c2r_wide_io_kernel<LOGM, LOGR1, LOGR2, G, IO, 5>;
    NEO_TRY(enable_smem(kernel, G * cfg::SMEM));
    kernel<<<unsigned((batch + G - 1) / G), 32 * G, G * cfg::SMEM, stream>>>(io, ta, tb, rtw, batch);
    return check_launch("c2r_wide_io_kernel");
}

// ---- tables + launchers --------------------------------------------------------------------------------------------------------------
template<int LOGM, int LOGR1, int LOGR2>
struct wide_tables
{
    using cfg = wide_cfg<LOGM, LOGR1, LOGR2>;
    device_buffer ta, tb_fwd, tb_bwd, rtw;

    int build(cudaStream_t stream)
    {
        constexpr double pi = 3.14159265358979323846264338327950288;
        constexpr int M = cfg::M, R1 = cfg::R1, R2 = cfg::R2, J = cfg::J, XS = cfg::XS, LOGP = cfg::LOGP;
        std::vector<float2> a(size_t(LOGP) * XS), f(size_t(R2) * 16), g(size_t(R1) * R2), r(J / 2 + 1);
        for (int p = 0; p < LOGP; ++p) {
            for (int x = 0; x < XS; ++x) {
                // exponent reduced mod M in integers before the angle is formed
                long const e   = (long(x) << p) & (M - 1);
                double const v = -2.0 * pi * double(e) / double(M);
                a[size_t(p) * XS + x] = make_float2(float(std::cos(v)), float(std::sin(v)));
            }
        }
        for (int k2 = 0; k2 < R2; ++k2) {
            for (int x = 0; x < 16; ++x) {
                double const v   = -2.0 * pi * double(x * k2) / double(16 * R2);
                f[k2 * 16 + x] = make_float2(float(std::cos(v)), float(std::sin(v)));
            }
        }
        for (int k1 = 0; k1 < R1; ++k1) {
            for (int a2 = 0; a2 < R2; ++a2) {
                double const v    = -2.0 * pi * double(k1 * a2) / double(R1 * R2);
                g[k1 * R2 + a2] = make_float2(float(std::cos(v)), float(std::sin(v)));
            }
        }
        for (int k = 0; k <= J / 2; ++k) {
            double const v = -pi * double(k) / double(M);
            r[k]           = make_float2(float(std::cos(v)), float(std::sin(v)));
        }
        auto upload = [&](device_buffer& dst, std::vector<float2> const& src) -> int {
            NEO_TRY(dst.reserve(src.size() * sizeof(float2)));
            NEO_CUDA_TRY(cudaMemcpyAsync(dst.ptr, src.data(), src.size() * sizeof(float2), cudaMemcpyHostToDevice, stream));
            return NEO_B200_OK;
        };
        NEO_TRY(upload(ta, a));
        NEO_TRY(upload(tb_fwd, f));
        NEO_TRY(upload(tb_bwd, g));
        NEO_TRY(upload(rtw, r));
        NEO_CUDA_TRY(cudaStreamSynchronize(stream));  // host vectors die here
        return NEO_B200_OK;
    }
};

inline bool wide_aligned(void const* p) { return (reinterpret_cast<std::uintptr_t>(p) & 15U) == 0; }

// resident CTAs per SM at 128 registers per thread
template<int LOGM, int LOGR1, int LOGR2>
constexpr int wide_min_ctas()
{
    int const by_regs = 512 / wide_cfg<LOGM, LOGR1, LOGR2>::NT;
    int const by_smem = int((228 * 1024) / (wide_cfg<LOGM, LOGR1, LOGR2>::SMEM_PF + 1024 + 64));
    int const n       = by_regs < by_smem ? by_regs : by_smem;
    return n > 0 ? n : 1;
}

inline unsigned wide_grid(size_t batch, int ctas_per_sm)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return unsigned(std::min<size_t>(batch, size_t(sms) * ctas_per_sm));
}

template<int LOGM, int LOGR1, int LOGR2>
int launch_r2c_wide(wide_tables<LOGM, LOGR1, LOGR2> const& tb, float const* in, float2* out, size_t batch, cudaStream_t stream)
{
    using cfg = wide_cfg<LOGM, LOGR1, LOGR2>;
    if (batch == 0) { return NEO_B200_OK; }
    constexpr int ctas = wide_min_ctas<LOGM, LOGR1, LOGR2>();
    auto kernel        = r2c_wide_kernel<LOGM, LOGR1, LOGR2, ctas>;
    NEO_TRY(enable_smem(kernel, cfg::SMEM_PF));
    kernel<<<wide_grid(batch, ctas), cfg::NT, cfg::SMEM_PF, stream>>>(in, out, tb.ta.template as<float2>(), tb.tb_fwd.template as<float2>(),
                                                                       tb.rtw.template as<float2>(), batch);
    return check_launch("r2c_wide_kernel");
}

template<int LOGM, int LOGR1, int LOGR2>
int launch_c2r_wide(wide_tables<LOGM, LOGR1, LOGR2> const& tb, float2 const* in, size_t row_len, float* out, size_t batch,
                    cudaStream_t stream)
{
    using cfg = wide_cfg<LOGM, LOGR1, LOGR2>;
    if (batch == 0) { return NEO_B200_OK; }
    constexpr int ctas = wide_min_ctas<LOGM, LOGR1, LOGR2>();
    auto kernel        = c2r_wide_kernel<LOGM, LOGR1, LOGR2, ctas>;
    NEO_TRY(enable_smem(kernel, cfg::SMEM_PF));
    kernel<<<wide_grid(batch, ctas), cfg::NT, cfg::SMEM_PF, stream>>>(in, row_len, out, tb.ta.template as<float2>(),
                                                                       tb.tb_bwd.template as<float2>(), tb.rtw.template as<float2>(), batch);
    return check_launch("c2r_wide_kernel");
}

// ---- split pair (N = 2^16): tables of the M2-point transform + the decimation step's twiddles ------------------------------------
template<int LOGM2, int LOGR1, int LOGR2>
struct wide_split_tables
{
    using cfg = wide_cfg<LOGM2, LOGR1, LOGR2>;
    wide_tables<LOGM2, LOGR1, LOGR2> sub;
    device_buffer w_m;       // exp(-2 pi i k / M), k < J   (M = 2 M2)
    device_buffer rtw_full;  // exp(-i pi k / M), k <= J/2: the real-transform twiddle of the FULL size
    float2 w_2m1{};          // exp(-i pi / M)

    int build(cudaStream_t stream)
    {
        constexpr double pi = 3.14159265358979323846264338327950288;
        constexpr int M = 2 * cfg::M, J = cfg::J;
        NEO_TRY(sub.build(stream));
        std::vector<float2> a(J), b(J / 2 + 1);
        for (int k = 0; k < J; ++k) {
            double const v = -2.0 * pi * double(k) / double(M);
            a[k]           = make_float2(float(std::cos(v)), float(std::sin(v)));
        }
        for (int k = 0; k <= J / 2; ++k) {
            double const v = -pi * double(k) / double(M);
            b[k]           = make_float2(float(std::cos(v)), float(std::sin(v)));
        }
        w_2m1 = make_float2(float(std::cos(-pi / double(M))), float(std::sin(-pi / double(M))));
        NEO_TRY(w_m.reserve(a.size() * sizeof(float2)));
        NEO_CUDA_TRY(cudaMemcpyAsync(w_m.ptr, a.data(), a.size() * sizeof(float2), cudaMemcpyHostToDevice, stream));
        NEO_TRY(rtw_full.reserve(b.size() * sizeof(float2)));
        NEO_CUDA_TRY(cudaMemcpyAsync(rtw_full.ptr, b.data(), b.size() * sizeof(float2), cudaMemcpyHostToDevice, stream));
        NEO_CUDA_TRY(cudaStreamSynchronize(stream));
        return NEO_B200_OK;
    }
};

inline unsigned wide_split_grid(size_t batch)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return unsigned(std::min<size_t>(2 * batch, size_t(sms) & ~size_t(1)));  // even: a CTA keeps its parity, the pair of a row runs together
}

template<int LOGM2, int LOGR1, int LOGR2>
int launch_r2c_wide_split(wide_split_tables<LOGM2, LOGR1, LOGR2> const& tb, float const* in, float2* out, size_t batch, cudaStream_t stream)
{
    using cfg = wide_cfg<LOGM2, LOGR1, LOGR2>;
    if (batch == 0) { return NEO_B200_OK; }
    auto kernel = r2c_wide_split_kernel<LOGM2, LOGR1, LOGR2>;
    NEO_TRY(enable_smem(kernel, cfg::SMEM_PF));
    kernel<<<wide_split_grid(batch), cfg::NT, cfg::SMEM_PF, stream>>>(in, out, tb.sub.ta.template as<float2>(),
                                                                      tb.sub.tb_fwd.template as<float2>(), tb.sub.rtw.template as<float2>(),
                                                                      tb.w_m.template as<float2>(), tb.w_2m1, batch);
    return check_launch("r2c_wide_split_kernel");
}

template<int LOGM2, int LOGR1, int LOGR2>
int launch_c2r_wide_split(wide_split_tables<LOGM2, LOGR1, LOGR2> const& tb, float2 const* in, size_t row_len, float* out, size_t batch,
                          cudaStream_t stream)
{
    using cfg = wide_cfg<LOGM2, LOGR1, LOGR2>;
    if (batch == 0) { return NEO_B200_OK; }
    auto kernel = c2r_wide_split_kernel<LOGM2, LOGR1, LOGR2>;
    NEO_TRY(enable_smem(kernel, cfg::SMEM_PF));
    kernel<<<wide_split_grid(batch), cfg::NT, cfg::SMEM_PF, stream>>>(in, row_len, out, tb.sub.ta.template as<float2>(),
                                                                      tb.sub.tb_bwd.template as<float2>(),
                                                                      tb.rtw_full.template as<float2>(), tb.w_m.template as<float2>(), batch);
    return check_launch("c2r_wide_split_kernel");
}

}  // namespace neo_b200
