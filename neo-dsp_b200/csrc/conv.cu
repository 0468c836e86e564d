// conv.cu -- C ABI of the partitioned convolver bank, uniform_partition and the index tables (include/neo_b200.h).
// Drop-in for neo::convolution::upols_convolver / upola_convolver
// (src/neo/convolution/uniform_partitioned_convolver.hpp:14-65, dense_convolver.hpp:20-25) and
// neo::convolution::uniform_partition (uniform_partition.hpp:13-26).
#include "conv_frame.cuh"
#include "conv_lowlat.cuh"
#include "fft_wide.cuh"

#include <algorithm>
#include <cstdlib>
#include <memory>
#include <thread>
#include <type_traits>
#include <vector>

namespace neo_b200 {

__global__ void fdl_index_kernel(unsigned parts, unsigned calls, unsigned* write_pos, unsigned* pairs)
{
    // one thread per (call, segment): the ring position advances by one per call (fdl_index.hpp:33-35)
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= size_t(parts) * calls) { return; }
    unsigned const call    = unsigned(i / parts);
    unsigned const segment = unsigned(i - size_t(call) * parts);
    unsigned const wp      = call % parts;
    if (segment == 0) { write_pos[call] = wp; }
    pairs[2 * i + 0] = segment;
    pairs[2 * i + 1] = fdl_filter_index(wp, segment, parts);
}

__global__ void bitrev_table_kernel(unsigned order, unsigned* out)
{
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= (size_t(1) << order)) { return; }
    out[i] = order == 0 ? 0U : (__brev(unsigned(i)) >> (32U - order));
}

// digitrevorder_plan<R>::make (fft/reference/digitrevorder.hpp:27-45) walks a carry chain; entry i is the base-R digit
// reversal of i for i < size-1 and 0 for the last entry. Applying the plan to iota (swap when i < lut[i]) yields the
// permutation below: perm[i] = digitrev(i), and position size-1 stays in place because its lut entry is 0.
__global__ void digitrev_perm_kernel(unsigned radix, unsigned digits, unsigned size, unsigned* out)
{
    size_t const i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= size) { return; }
    unsigned v = unsigned(i), r = 0;
    for (unsigned d = 0; d < digits; ++d) {
        r = r * radix + v % radix;
        v /= radix;
    }
    out[i] = r;
}

namespace {

template<typename T>
struct conv_engine
{
    neo_b200_conv_config cfg{};
    int logb{0};
    int m{0};           // B
    int parts{0};       // local partitions
    size_t age0{0};     // age (in blocks) of the first local partition as THIS handle sees its input: partition_begin, or 0 when the
                        // caller feeds the input already delayed by partition_begin blocks (config.input_delayed)
    int ring{0};
    int sources{1};
    int splits{1};
    int logw{0}, nt{1};  // tile-major row layout
    size_t filters{0};  // outputs * sources
    size_t write_pos{0};
    bool has_filter{false};

    fft_tables<T> tables;
    // float32, B = 1024 (the 2048-point real transforms of BASELINE config 5): one warp per transform, 32 points per thread, Hermitian
    // split in registers, 128-bit accesses on the real side (fft_wide.cuh). NEO_B200_CONV_NO_WIDE keeps the 16-points-per-thread kernels.
    // Measured (C5, frame mode T = 256, ms per step): c2r 0.668 -> 0.631 (15 % fewer instructions, 0.78 of HBM by its 12 bytes per sample);
    // r2c 0.682 -> 0.699 (14 % fewer instructions, but 16 instead of 32 resident warps leave its loads exposed), so the forward side
    // takes the wide kernel only with NEO_B200_CONV_WIDE_R2C.
    wide_tables<10, 3, 3> wide10;
    bool use_wide{false}, use_wide_r2c{false};
    // resident CTAs the wide kernels are compiled for (NEO_B200_CONV_WIDE_R2C / _C2R = 4, 5, 6 -> 128 / 96 / 80 registers). Measured (C5, frame
    // mode T = 256, ms per step, r2c / c2r): 4: 0.704 / 0.636, 5: 0.672 / 0.611, 6: 0.756 / 0.743 (spills), cta_fft r2c 0.689
    int wide_minb_r2c{5}, wide_minb_c2r{5};
    device_buffer filter, fdl, prev[2], tail, acc, acc_alt, ola_y, stage_in, stage_out, stage_filter, tickets;
    // sparse filters (set_filter_csr): bitmap form of the reference's CSR matrices (conv_kernels.cuh, fdl_mac_sparse_kernel); the
    // dense filter buffer is released while they are in place
    bool sparse{false};
    int nseg{1};
    device_buffer sp_meta, sp_vals, sp_base;
    // partition-sharded handles alternate between two partial-spectra buffers, so the reduction of call i (NCCL reads the buffer
    // neo_b200_conv_spectra returned) may still be running while call i+1 writes the other one
    int acc_cur{0}, acc_last{0};
    bool in_call{false};  // a forward_range call has started and its final range has not been seen yet
    size_t range_next{0}, range_blocks{0};  // ... the channel its next range must start at, and its block count
    cx<T>* acc_w() const { return (acc_cur != 0 ? acc_alt : acc).template as<cx<T>>(); }
    void* acc_r() const { return in_call ? static_cast<void*>(acc_w()) : (acc_last != 0 ? acc_alt : acc).ptr; }
    int prev_flip{0};  // prev[prev_flip] holds the last block of the previous call

    // second partition level along block time (conv_frame.cuh). frame == 0: direct form. In frame mode `fdl` is the two-frame
    // level-1 spectra buffer x1 (2T plain rows of B per channel, not tiled) and `filter` only lives while a filter is prepared.
    int frame{0}, logl{0}, tiles2{0}, ring2{0}, parts2{0}, splits2{1};
    size_t write_pos2{0};
    int x1_half{0};  // half of x1 the current call writes
    fft_tables<T> frame_tables;
    device_buffer frame_tw8;  // stage twiddles of the 8-points-per-thread variant of the long frame transforms
    device_buffer frame_tw32; // ... and of the 32-points-per-thread form (float, L = 512 / 1024)
    device_buffer fdl2, filter2, acc2, tickets2, nyq_acc;
    bool fused{false};  // bank with an unsplit partition loop: one kernel per frame step (frame_fused_kernel)
    // set by a multi-device bank before forward_mac (frame_fused_io::y1_owner): where the result rows of each owner's channels go
    cx<T>* push_dst[k_bank_max_shards] = {};
    int push_owners{0}, push_own_count{0};
    frame_knobs knobs;  // environment knobs as they stood when the handle was created

    // optional per-phase timing with CUDA events on the handle's stream (bench.py's roofline numbers)
    struct span
    {
        cudaEvent_t begin, end;
    };
    bool profiling{false};
    static constexpr int k_phases = 5;
    std::vector<span> spans[k_phases];  // 0 r2c + FDL insert, 1 MAC, 2 c2r, 3 frame transform forward, 4 frame transform inverse
    std::uint64_t mac_launches{0};

    // event pairs are recycled through `pool`: nothing is created inside a steady-state timed loop, nothing leaks when the caller
    // never reads, and whatever is left is destroyed with the engine
    std::vector<span> pool;
    double folded_ms[k_phases] = {0, 0, 0, 0, 0};
    static constexpr size_t k_max_open_spans = 4096;

    ~conv_engine()
    {
        for (auto& list : spans) {
            for (auto& s : list) { pool.push_back(s); }
        }
        for (auto& s : pool) {
            cudaEventDestroy(s.begin);
            cudaEventDestroy(s.end);
        }
    }

    int mark_begin(int phase, cudaStream_t stream)
    {
        if (!profiling) { return NEO_B200_OK; }
        if (spans[phase].size() >= k_max_open_spans) { NEO_TRY(fold_spans(stream)); }  // a caller that never reads: bounded memory
        span s{};
        if (!pool.empty()) {
            s = pool.back();
            pool.pop_back();
        } else {
            NEO_CUDA_TRY(cudaEventCreate(&s.begin));
            cudaError_t const err = cudaEventCreate(&s.end);
            if (err != cudaSuccess) {
                cudaEventDestroy(s.begin);
                return fail(NEO_B200_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(err));
            }
        }
        cudaError_t const err = cudaEventRecord(s.begin, stream);
        if (err != cudaSuccess) {
            pool.push_back(s);
            return fail(NEO_B200_ERR_CUDA, "cudaEventRecord: %s", cudaGetErrorString(err));
        }
        spans[phase].push_back(s);
        return NEO_B200_OK;
    }

    int mark_end(int phase, cudaStream_t stream)
    {
        if (!profiling) { return NEO_B200_OK; }
        NEO_CUDA_TRY(cudaEventRecord(spans[phase].back().end, stream));
        return NEO_B200_OK;
    }

    // accumulate every finished span into folded_ms and recycle its events
    int fold_spans(cudaStream_t stream)
    {
        NEO_CUDA_TRY(cudaStreamSynchronize(stream));
        for (int p = 0; p < k_phases; ++p) {
            for (auto& s : spans[p]) {
                float t = 0.f;
                if (cudaEventElapsedTime(&t, s.begin, s.end) == cudaSuccess) { folded_ms[p] += double(t); }
                pool.push_back(s);
            }
            spans[p].clear();
        }
        (void)cudaGetLastError();
        return NEO_B200_OK;
    }

    int read_profile(double* ms, std::uint64_t* launches, cudaStream_t stream)
    {
        NEO_TRY(fold_spans(stream));
        for (int p = 0; p < k_phases; ++p) {
            ms[p]        = folded_ms[p];
            folded_ms[p] = 0.0;
        }
        *launches    = mac_launches;
        mac_launches = 0;
        return NEO_B200_OK;
    }

    size_t device_bytes() const
    {
        return sp_meta.bytes + sp_vals.bytes + sp_base.bytes + filter.bytes + fdl.bytes + prev[0].bytes + prev[1].bytes + tail.bytes + acc.bytes + acc_alt.bytes + ola_y.bytes + stage_in.bytes
             + stage_out.bytes + stage_filter.bytes + fdl2.bytes + filter2.bytes + acc2.bytes + nyq_acc.bytes;
    }

    int init(neo_b200_conv_config const& c, cudaStream_t stream)
    {
        cfg     = c;
        m       = int(c.block);
        logb    = int(log2_exact(c.block));
        parts   = int(c.partition_end - c.partition_begin);
        frame   = int(c.frame_blocks);
        age0    = c.input_delayed != 0 ? 0 : c.partition_begin;
        ring    = frame > 0 ? 2 * frame : int(age0 + size_t(parts) + c.max_blocks - 1);
        sources = c.topology == NEO_B200_MATRIX ? int(c.inputs) : 1;
        filters = c.outputs * size_t(sources);
        logw    = std::min(logb, int(log2_exact(size_t(tile_width<T>()))));
        nt      = m >> logw;
        NEO_TRY(tables.build(logb, true, stream));
        if constexpr (sizeof(T) == 4) {
            use_wide = logb == 10 && std::getenv("NEO_B200_CONV_NO_WIDE") == nullptr;
            if (use_wide) { NEO_TRY(wide10.build(stream)); }
            use_wide_r2c = use_wide && std::getenv("NEO_B200_CONV_WIDE_R2C") != nullptr;
            if (char const* v = std::getenv("NEO_B200_CONV_WIDE_R2C")) { wide_minb_r2c = std::max(4, std::min(6, std::atoi(v))); }
            if (char const* v = std::getenv("NEO_B200_CONV_WIDE_C2R")) { wide_minb_c2r = std::max(4, std::min(6, std::atoi(v))); }
        }

        size_t const csz = sizeof(cx<T>);
        if (frame == 0) { NEO_TRY(filter.reserve(filters * parts * m * csz)); }
        NEO_TRY(fdl.reserve(c.inputs * size_t(ring) * m * csz));
        NEO_TRY(prev[0].reserve(c.inputs * m * sizeof(T)));
        NEO_TRY(prev[1].reserve(c.inputs * m * sizeof(T)));
        if (c.kind == NEO_B200_UPOLA) {
            NEO_TRY(tail.reserve(c.outputs * m * sizeof(T)));
            NEO_TRY(ola_y.reserve(c.outputs * c.max_blocks * 2 * m * sizeof(T)));
        }
        int sms = 148;
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        splits = frame > 0 ? 1 : pick_splits(sms, size_t(m), size_t(parts));
        NEO_TRY(acc.reserve(size_t(splits) * c.outputs * c.max_blocks * m * csz));
        if (!(c.partition_begin == 0 && c.partition_end == c.partitions)) { NEO_TRY(acc_alt.reserve(acc.bytes)); }
        // one ticket per MAC grid cell (x: at most B/128 column blocks, y: outputs); the last split CTA to finish resets it
        NEO_TRY(tickets.reserve(c.outputs * size_t(std::max(1, m / 128 + 1)) * sizeof(unsigned)));
        NEO_CUDA_TRY(cudaMemsetAsync(tickets.ptr, 0, tickets.bytes, stream));

        if (frame > 0) {
            int const len = 2 * frame;
            int const w   = 1 << logw;
            logl          = int(log2_exact(size_t(len)));
            tiles2        = nt * len + (len + w - 1) / w;
            ring2         = int((age0 + size_t(parts) + size_t(frame) - 1) / size_t(frame));
            parts2        = (parts + frame - 1) / frame;
            size_t const m2 = size_t(tiles2) << logw;
            splits2       = pick_splits(sms, m2, size_t(parts2));
            NEO_TRY(frame_tables.build(logl, false, stream));
            knobs = frame_knobs::from_env();
            if (knobs.wide_points(logl, sizeof(T) == 4)) {
                auto const tw = make_stage_twiddles<T>(logl, 5);
                NEO_TRY(frame_tw32.reserve(tw.size() * csz));
                NEO_CUDA_TRY(cudaMemcpyAsync(frame_tw32.ptr, tw.data(), tw.size() * csz, cudaMemcpyHostToDevice, stream));
                NEO_CUDA_TRY(cudaStreamSynchronize(stream));
            }
            if (knobs.eight_points(logl, sizeof(T) == 4)) {
                auto const tw = make_stage_twiddles<T>(logl, 3);
                NEO_TRY(frame_tw8.reserve(tw.size() * csz));
                NEO_CUDA_TRY(cudaMemcpyAsync(frame_tw8.ptr, tw.data(), tw.size() * csz, cudaMemcpyHostToDevice, stream));
                NEO_CUDA_TRY(cudaStreamSynchronize(stream));
            }
            NEO_TRY(filter2.reserve(filters * parts2 * m2 * csz));
            NEO_TRY(fdl2.reserve(c.inputs * size_t(ring2) * m2 * csz));
            fused = sources == 1 && splits2 == 1 && std::getenv("NEO_B200_FRAME_UNFUSED") == nullptr;
            if (fused) { NEO_TRY(nyq_acc.reserve(c.outputs * size_t(len) * csz)); }
            else { NEO_TRY(acc2.reserve(size_t(splits2) * c.outputs * m2 * csz)); }
            NEO_TRY(tickets2.reserve(c.outputs * (m2 / 128 + 1) * sizeof(unsigned)));
            NEO_CUDA_TRY(cudaMemsetAsync(tickets2.ptr, 0, tickets2.bytes, stream));
        }
        return clear_state(stream);
    }

    // split the partition loop when (bins x outputs) alone cannot fill the GPU: ~4 CTAs per SM wanted
    int pick_splits(int sms, size_t bins, size_t rows) const
    {
        size_t const ctas_xy = ((bins / mac_vec<T>::VEC + k_mac_threads - 1) / k_mac_threads) * cfg.outputs;
        size_t const work    = size_t(sources) * rows;
        size_t want          = (size_t(sms) * (sources > 1 ? 16 : 4) + ctas_xy - 1) / ctas_xy;
        want                 = std::min(want, std::max<size_t>(1, work / 8));
        return int(std::max<size_t>(1, std::min<size_t>(want, 64)));
    }

    int clear_state(cudaStream_t stream)
    {
        NEO_CUDA_TRY(cudaMemsetAsync(fdl.ptr, 0, fdl.bytes, stream));
        NEO_CUDA_TRY(cudaMemsetAsync(prev[0].ptr, 0, prev[0].bytes, stream));
        NEO_CUDA_TRY(cudaMemsetAsync(prev[1].ptr, 0, prev[1].bytes, stream));
        prev_flip = 0;
        if (tail.ptr != nullptr) { NEO_CUDA_TRY(cudaMemsetAsync(tail.ptr, 0, tail.bytes, stream)); }
        if (fdl2.ptr != nullptr) { NEO_CUDA_TRY(cudaMemsetAsync(fdl2.ptr, 0, fdl2.bytes, stream)); }
        write_pos  = 0;
        write_pos2 = 0;
        x1_half    = 0;
        in_call    = false;  // a reset in the middle of a grouped call abandons it
        range_next = range_blocks = 0;
        acc_cur = acc_last = 0;
        return NEO_B200_OK;
    }

    // frame mode: the level-1 filter exists only between begin_filter and finish_filter
    int begin_filter()
    {
        if (frame > 0 || filter.ptr == nullptr) { NEO_TRY(filter.reserve(filters * parts * m * sizeof(cx<T>))); }
        if (sparse) {  // a dense filter replaces the sparse one
            sparse = false;
            sp_meta.release();
            sp_vals.release();
            sp_base.release();
        }
        return NEO_B200_OK;
    }

    // `sparse_filter::filter(partitions, sparsity)` (sparse_filter.hpp:25-28) for every channel of a diagonal bank: the CSR matrices
    // exactly as neo::csr_matrix builds them (csr_matrix.hpp:64-98; rows = partitions, columns = the B+1 bins). Filter f owns entries
    // [filter_base[f], filter_base[f+1]) of values / cols; row_ptr[f * (P+1) + p] is relative to filter_base[f]. Host memory.
    int set_filter_csr(cx<T> const* values, std::uint64_t const* cols, std::uint64_t const* row_ptr, std::uint64_t const* filter_base,
                       cudaStream_t stream)
    {
        if (cfg.topology != NEO_B200_DIAGONAL || frame > 0 || cfg.partition_begin != 0 || cfg.partition_end != cfg.partitions) {
            return fail(NEO_B200_ERR_UNSUPPORTED, "sparse filters: diagonal topology, direct form (frame_blocks = 0), unsharded partitions");
        }
        size_t const P = size_t(parts), B = size_t(m);
        nseg           = int((B + 31) / 32);
        std::vector<uint2> meta(filters * size_t(nseg) * P, make_uint2(0U, 0U));
        std::vector<unsigned long long> base(filters + 1, 0ULL);
        std::vector<cx<T>> vals;
        for (size_t f = 0; f < filters; ++f) {
            std::uint64_t const* const rows = row_ptr + f * (P + 1);
            std::uint64_t const* const fc   = cols + filter_base[f];
            cx<T> const* const fv           = values + filter_base[f];
            uint2* const fm                 = meta.data() + f * size_t(nseg) * P;
            if (filter_base[f] + rows[P] != filter_base[f + 1]) { return fail(NEO_B200_ERR_INVALID, "CSR filter %zu: row_ptr and filter_base disagree", f); }
            // presence bits; column B (Nyquist) shares packed element 0 with column 0
            for (size_t p = 0; p < P; ++p) {
                if (rows[p] > rows[p + 1]) { return fail(NEO_B200_ERR_INVALID, "CSR filter %zu: row_ptr not ascending", f); }
                for (std::uint64_t i = rows[p]; i < rows[p + 1]; ++i) {
                    if (fc[i] > B) { return fail(NEO_B200_ERR_INVALID, "CSR filter %zu: column %llu out of range", f, static_cast<unsigned long long>(fc[i])); }
                    size_t const k = fc[i] == B ? 0 : size_t(fc[i]);
                    fm[(k >> 5) * P + p].x |= 1U << (k & 31U);
                }
            }
            // value offsets in (segment, partition) order, then the values themselves
            base[f]           = vals.size();
            std::uint64_t run = 0;
            for (size_t sgm = 0; sgm < size_t(nseg); ++sgm) {
                for (size_t p = 0; p < P; ++p) {
                    fm[sgm * P + p].y = unsigned(run);
                    run += std::uint64_t(__builtin_popcount(fm[sgm * P + p].x));
                }
            }
            if (run > 0xffffffffULL) { return fail(NEO_B200_ERR_UNSUPPORTED, "CSR filter %zu: more than 2^32 stored elements", f); }
            vals.resize(vals.size() + size_t(run), mk<T>(T(0), T(0)));
            cx<T>* const out = vals.data() + base[f];
            for (size_t p = 0; p < P; ++p) {
                for (std::uint64_t i = rows[p]; i < rows[p + 1]; ++i) {
                    size_t const k   = fc[i] == B ? 0 : size_t(fc[i]);
                    uint2 const w    = fm[(k >> 5) * P + p];
                    cx<T>& dst       = out[w.y + unsigned(__builtin_popcount(w.x & ((1U << (k & 31U)) - 1U)))];
                    if (fc[i] == B) { dst.y = fv[i].x; }        // packed element 0 = (Re H[0], Re H[B]), as pack_filter_kernel
                    else if (fc[i] == 0) { dst.x = fv[i].x; }
                    else { dst = fv[i]; }
                }
            }
        }
        base[filters] = vals.size();
        NEO_TRY(sp_meta.reserve(meta.size() * sizeof(uint2)));
        NEO_TRY(sp_vals.reserve(std::max<size_t>(1, vals.size()) * sizeof(cx<T>)));
        NEO_TRY(sp_base.reserve(base.size() * sizeof(unsigned long long)));
        NEO_CUDA_TRY(cudaMemcpyAsync(sp_meta.ptr, meta.data(), meta.size() * sizeof(uint2), cudaMemcpyHostToDevice, stream));
        if (!vals.empty()) { NEO_CUDA_TRY(cudaMemcpyAsync(sp_vals.ptr, vals.data(), vals.size() * sizeof(cx<T>), cudaMemcpyHostToDevice, stream)); }
        NEO_CUDA_TRY(cudaMemcpyAsync(sp_base.ptr, base.data(), base.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, stream));
        NEO_CUDA_TRY(cudaStreamSynchronize(stream));
        filter.release();  // the dense layout is not kept: the stored elements are all the filter bytes there are
        sparse = true;
        return finish_filter(stream);
    }

    int finish_filter(cudaStream_t stream)
    {
        if (frame > 0) {
            frame_geom const fg{logb, logw, nt, frame, tiles2};
            int status = NEO_B200_ERR_UNSUPPORTED;
            NEO_CUDA_TRY(cudaMemsetAsync(filter2.ptr, 0, filter2.bytes, stream));  // unused Nyquist-tile columns stay zero
            NEO_DISPATCH_LOGL(logl, {
                frame_filter_io<T, false> io{filter.template as<cx<T>>(), filter2.template as<cx<T>>(), fg, parts, parts2};
                status = launch_frame_fft<T, LOGL, -1>(io, frame_tables.tw(), (filters * size_t(parts2)) << logb, stream);
                if (status == NEO_B200_OK) {
                    frame_filter_io<T, true> nq{filter.template as<cx<T>>(), filter2.template as<cx<T>>(), fg, parts, parts2};
                    status = launch_frame_fft<T, LOGL, -1>(nq, frame_tables.tw(), filters * size_t(parts2), stream);
                }
            });
            if (status != NEO_B200_OK) { return status == NEO_B200_ERR_UNSUPPORTED ? fail(status, "frame of %d blocks not supported", frame) : status; }
            NEO_CUDA_TRY(cudaStreamSynchronize(stream));
            filter.release();
        }
        has_filter = true;
        return clear_state(stream);
    }

    // H in the reference layout [filters][P][B+1]; device pointer
    int pack_filter(cx<T> const* h_dev, size_t first_filter, size_t count, size_t src_parts, int part0, cudaStream_t stream)
    {
        size_t const rows = count * parts;
        for (size_t r0 = 0; r0 < rows; r0 += 65535) {  // gridDim.y <= 65535
            dim3 const grid(unsigned((m + 255) / 256), unsigned(std::min<size_t>(65535, rows - r0)));
            pack_filter_kernel<T><<<grid, 256, 0, stream>>>(h_dev, filter.template as<cx<T>>() + first_filter * parts * m, src_parts, part0,
                                                            parts, m, r0, logw, nt);
            NEO_TRY(check_launch("pack_filter_kernel"));
        }
        return NEO_B200_OK;
    }

    int set_filter(void const* h, int memspace, cudaStream_t stream)
    {
        size_t const p_total = cfg.partitions;
        size_t const k       = size_t(m) + 1;
        size_t const csz     = sizeof(cx<T>);
        NEO_TRY(begin_filter());
        if (memspace == NEO_B200_DEVICE) {
            NEO_TRY(pack_filter(static_cast<cx<T> const*>(h), 0, filters, p_total, int(cfg.partition_begin), stream));
        } else {
            // stage only this handle's partition range of each filter, a few hundred MB at a time
            size_t const row_bytes = size_t(parts) * k * csz;
            size_t const chunk     = std::max<size_t>(1, std::min(filters, (size_t(256) << 20) / row_bytes));
            NEO_TRY(stage_filter.reserve(chunk * row_bytes));
            char const* src = static_cast<char const*>(h) + cfg.partition_begin * k * csz;
            for (size_t f = 0; f < filters; f += chunk) {
                size_t const n = std::min(chunk, filters - f);
                NEO_CUDA_TRY(cudaMemcpy2DAsync(stage_filter.ptr, row_bytes, src + f * p_total * k * csz, p_total * k * csz, row_bytes, n,
                                               cudaMemcpyHostToDevice, stream));
                NEO_TRY(pack_filter(stage_filter.template as<cx<T>>(), f, n, size_t(parts), 0, stream));
                NEO_CUDA_TRY(cudaStreamSynchronize(stream));  // staging buffer is reused
            }
        }
        return finish_filter(stream);
    }

    int partition_into(T const* ir_dev, size_t taps, size_t first_filter, size_t count, cudaStream_t stream)
    {
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_DISPATCH_LOGM(T, logb, {
            if constexpr (LOGM >= 1 && LOGM <= max_cta_logm<T>()) {
                partition_r2c_io<T, LOGM> io{ir_dev, taps, int(cfg.partition_begin), parts,
                                             filter.template as<cx<T>>() + first_filter * parts * m, 1, logw, nt};
                status = launch_r2c<T, LOGM>(io, tables.tw(), tables.rtw(), count * parts, stream);
            }
        });
        return status;
    }

    int set_impulse(void const* ir, size_t taps, int memspace, cudaStream_t stream)
    {
        NEO_TRY(begin_filter());
        if (memspace == NEO_B200_DEVICE) {
            NEO_TRY(partition_into(static_cast<T const*>(ir), taps, 0, filters, stream));
        } else {
            size_t const row_bytes = taps * sizeof(T);
            size_t const chunk     = std::max<size_t>(1, std::min(filters, (size_t(256) << 20) / row_bytes));
            NEO_TRY(stage_filter.reserve(chunk * row_bytes));
            for (size_t f = 0; f < filters; f += chunk) {
                size_t const n = std::min(chunk, filters - f);
                NEO_CUDA_TRY(cudaMemcpyAsync(stage_filter.ptr, static_cast<char const*>(ir) + f * row_bytes, n * row_bytes,
                                             cudaMemcpyHostToDevice, stream));
                NEO_TRY(partition_into(stage_filter.template as<T>(), taps, f, n, stream));
                NEO_CUDA_TRY(cudaStreamSynchronize(stream));
            }
        }
        return finish_filter(stream);
    }

    // the wide kernels move the real rows with 128-bit accesses
    bool wide_rows_ok(void const* rows, size_t stride) const
    {
        return use_wide && (reinterpret_cast<std::uintptr_t>(rows) & 15U) == 0 && stride % 4 == 0;
    }

    template<int LOGM, class IO>
    int run_r2c(IO const& io, bool wide, size_t batch, cudaStream_t stream)
    {
        if constexpr (sizeof(T) == 4 && LOGM == 10) {
            if (wide) {
                return launch_r2c_wide_io<10, 3, 3>(io, wide10.ta.template as<float2>(), wide10.tb_fwd.template as<float2>(),
                                                    wide10.rtw.template as<float2>(), batch, stream, wide_minb_r2c);
            }
        }
        return launch_r2c<T, LOGM>(io, tables.tw(), tables.rtw(), batch, stream);
    }

    template<int LOGM, class IO>
    int run_c2r(IO const& io, bool wide, size_t batch, cudaStream_t stream)
    {
        if constexpr (sizeof(T) == 4 && LOGM == 10) {
            if (wide) {
                return launch_c2r_wide_io<10, 3, 3>(io, wide10.ta.template as<float2>(), wide10.tb_bwd.template as<float2>(),
                                                    wide10.rtw.template as<float2>(), batch, stream, wide_minb_c2r);
            }
        }
        return launch_c2r<T, LOGM>(io, tables.tw(), tables.rtw(), batch, stream);
    }

    // window + r2c + FDL insert for input channels [chan0, chan0 + nchan); `in` points at channel chan0's row
    int forward_r2c(T const* in, size_t in_stride, size_t blocks, size_t chan0, size_t nchan, cudaStream_t stream)
    {
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_TRY(mark_begin(0, stream));
        NEO_DISPATCH_LOGM(T, logb, {
            if constexpr (LOGM >= 1 && LOGM <= max_cta_logm<T>()) {
                if (frame > 0) {  // plain rows [2T][B] per channel, this call's half starts at row x1_half * T
                    conv_r2c_io<T, LOGM, true> io{in, in_stride, prev[prev_flip].template as<T>(), prev[prev_flip ^ 1].template as<T>(),
                                                  fdl.template as<cx<T>>(), ring, x1_half * frame, int(blocks),
                                                  cfg.kind == NEO_B200_UPOLA ? 1 : 0, logb, 1, chan0};
                    status = run_r2c<LOGM>(io, use_wide_r2c && wide_rows_ok(in, in_stride), nchan * blocks, stream);
                } else {
                    conv_r2c_io<T, LOGM> io{in, in_stride, prev[prev_flip].template as<T>(), prev[prev_flip ^ 1].template as<T>(),
                                            fdl.template as<cx<T>>(), ring, int(write_pos), int(blocks),
                                            cfg.kind == NEO_B200_UPOLA ? 1 : 0, logw, nt, chan0};
                    status = run_r2c<LOGM>(io, use_wide_r2c && wide_rows_ok(in, in_stride), nchan * blocks, stream);
                }
            }
        });
        if (status != NEO_B200_OK) { return status == NEO_B200_ERR_UNSUPPORTED ? fail(status, "block size %d not supported", m) : status; }
        NEO_TRY(mark_end(0, stream));
        return frame > 0 && !fused ? frame_forward(chan0, nchan, stream) : NEO_B200_OK;
    }

    // one chunk of neo::convolution::overlap_add_convolver (overlap_add_convolver.hpp:91-115): transform the windows [channels][2B] as
    // they stand into the newest delay-line row, MAC over all partitions, inverse transform, scale by 1/2B -> y [channels][2B].
    // commit: the chunk completed a block, the delay line advances (:122-131). Overlap-add, direct form.
    int window_step(T const* window, T* y, bool commit, cudaStream_t stream)
    {
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_DISPATCH_LOGM(T, logb, {
            if constexpr (LOGM >= 1 && LOGM <= max_cta_logm<T>()) {
                window_r2c_io<T, LOGM> io{};
                io.in          = window;
                io.in_stride   = 2 * size_t(m);
                io.prev        = nullptr;
                io.prev_next   = nullptr;
                io.fdl         = fdl.template as<cx<T>>();
                io.ring        = ring;
                io.wp          = int(write_pos);
                io.blocks      = 1;
                io.overlap_add = 0;
                io.logw        = logw;
                io.nt          = nt;
                io.chan0       = 0;
                status         = launch_r2c<T, LOGM>(io, tables.tw(), tables.rtw(), cfg.inputs, stream);
            }
        });
        if (status != NEO_B200_OK) { return status; }
        NEO_TRY(forward_mac(1, 0, cfg.outputs, stream));
        NEO_DISPATCH_LOGM(T, logb, {
            if constexpr (LOGM >= 1 && LOGM <= max_cta_logm<T>()) {
                conv_c2r_io<T, LOGM> io{acc_w(), 1, y, 2 * size_t(m), T(1) / T(2 * m), 1};
                status = launch_c2r<T, LOGM>(io, tables.tw(), tables.rtw(), cfg.outputs, stream);
            }
        });
        if (status != NEO_B200_OK) { return status; }
        if (commit) { advance(1); }
        return NEO_B200_OK;
    }

    // frame mode, bank: frame transform + ring insert + MAC + inverse frame transform in one kernel (Nyquist sequences first)
    int frame_fused_step(size_t out0, size_t nout, cudaStream_t stream)
    {
        frame_geom const fg{logb, logw, nt, frame, tiles2};
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_TRY(mark_begin(1, stream));
        NEO_DISPATCH_LOGL(logl, {
            frame_fused_io<T, true> nq{fdl.template as<cx<T>>(), fdl2.template as<cx<T>>(), filter2.template as<cx<T>>(),
                                       acc_w(), nyq_acc.template as<cx<T>>(), fg, x1_half, ring2, int(write_pos2),
                                       parts2, int(age0 / size_t(frame)), T(1) / T(2 * frame), out0, {}, 0, 0};
            status = launch_frame_fused<T, LOGL, true>(nq, frame_tables.tw(), frame_tw8.template as<cx<T>>(), frame_tw32.template as<cx<T>>(), nout, stream, knobs);
            if (status == NEO_B200_OK) {
                frame_fused_io<T, false> io{nq.x1, nq.fdl2, nq.filt2, nq.y1, nq.nyq_acc, fg, nq.new_half, nq.ring2, nq.slot,
                                            nq.parts2, nq.age0, nq.scale, out0, {}, push_owners, push_own_count};
                for (int o = 0; o < push_owners; ++o) { io.y1_owner[o] = push_dst[o]; }
                status = launch_frame_fused<T, LOGL, false>(io, frame_tables.tw(), frame_tw8.template as<cx<T>>(), frame_tw32.template as<cx<T>>(), nout << logb,
                                                           stream, knobs);
            }
        });
        if (status != NEO_B200_OK) { return status; }
        ++mac_launches;
        return mark_end(1, stream);
    }

    // frame mode: transform the spectra of (previous frame, this frame) along block time into ring slot write_pos2
    int frame_forward(size_t chan0, size_t nchan, cudaStream_t stream)
    {
        frame_geom const fg{logb, logw, nt, frame, tiles2};
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_TRY(mark_begin(3, stream));
        NEO_DISPATCH_LOGL(logl, {
            frame_fwd_io<T, false> io{fdl.template as<cx<T>>(), fdl2.template as<cx<T>>(), fg, x1_half, ring2, int(write_pos2), chan0};
            status = launch_frame_fft<T, LOGL, -1>(io, frame_tables.tw(), nchan << logb, stream, knobs);
            if (status == NEO_B200_OK) {
                frame_fwd_io<T, true> nq{fdl.template as<cx<T>>(), fdl2.template as<cx<T>>(), fg, x1_half, ring2, int(write_pos2), chan0};
                status = launch_frame_fft<T, LOGL, -1>(nq, frame_tables.tw(), nchan, stream);
            }
        });
        if (status != NEO_B200_OK) { return status; }
        return mark_end(3, stream);
    }

    // frame mode: Q streamed rows of L*B (+ Nyquist) bins, then back to the level-1 spectra of this frame's T blocks
    int frame_mac(size_t out0, size_t nout, cudaStream_t stream)
    {
        if (fused) { return frame_fused_step(out0, nout, stream); }
        size_t const m2 = size_t(tiles2) << logw;
        mac_geom g{};
        g.m           = int(m2);
        g.logw        = logw;
        g.nt          = tiles2;
        g.ring        = ring2;
        g.parts       = parts2;
        g.age0        = int(age0 / size_t(frame));
        g.sources     = sources;
        g.diagonal    = cfg.topology == NEO_B200_DIAGONAL ? 1 : 0;
        g.wp          = int(write_pos2);
        g.blocks      = 1;
        g.tau0        = 0;
        g.splits      = splits2;
        g.out0        = int(out0);
        g.packed_edge = 0;
        g.acc_plane   = cfg.outputs * m2;
        g.tickets     = tickets2.template as<unsigned>();
        NEO_TRY(mark_begin(1, stream));
        if (sources == 1 && splits2 == 1) {
            // bank: short row loops, several columns per thread (about 32 (filter, spectrum) pairs each)
            int const ncols   = std::max(1, std::min(16, 32 / parts2));
            size_t const cols = (m2 / mac_vec<T>::VEC + k_mac_threads - 1) / k_mac_threads;
            dim3 const grid(unsigned((cols + size_t(ncols) - 1) / size_t(ncols)), unsigned(nout));
            frame_mac_kernel<T><<<grid, k_mac_threads, 0, stream>>>(fdl2.template as<cx<T>>(), filter2.template as<cx<T>>(),
                                                                     acc2.template as<cx<T>>(), g, ncols);
            NEO_TRY(check_launch("frame_mac_kernel"));
        } else {
            NEO_TRY(launch_stream(fdl2.template as<cx<T>>(), filter2.template as<cx<T>>(), acc2.template as<cx<T>>(), g, nout, stream));
        }
        ++mac_launches;
        NEO_TRY(mark_end(1, stream));

        frame_geom const fg{logb, logw, nt, frame, tiles2};
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_TRY(mark_begin(4, stream));
        NEO_DISPATCH_LOGL(logl, {
            frame_inv_io<T> io{acc2.template as<cx<T>>(), acc_w(), fg, T(1) / T(2 * frame), out0};
            status = launch_frame_fft<T, LOGL, 1>(io, frame_tables.tw(), nout << logb, stream, knobs);
        });
        if (status != NEO_B200_OK) { return status; }
        return mark_end(4, stream);
    }

    // spectral MAC of outputs [out0, out0 + nout) for the `blocks` blocks just inserted
    int forward_mac(size_t blocks, size_t out0, size_t nout, cudaStream_t stream)
    {
        if (frame > 0) { return frame_mac(out0, nout, stream); }
        mac_geom g{};
        g.m         = m;
        g.logw      = logw;
        g.nt        = nt;
        g.ring      = ring;
        g.parts     = parts;
        g.age0      = int(age0);
        g.sources   = sources;
        g.diagonal  = cfg.topology == NEO_B200_DIAGONAL ? 1 : 0;
        g.blocks    = int(blocks);
        g.splits    = splits;
        g.out0      = int(out0);
        g.packed_edge = 1;
        g.acc_plane = cfg.outputs * blocks * size_t(m);
        g.tickets   = tickets.template as<unsigned>();

        size_t tau = 0;
        NEO_TRY(mark_begin(1, stream));
        if (sparse) {  // one launch per block: every stored element is used once, as in the streaming kernel
            dim3 const grid{unsigned(nseg), unsigned(nout), 1U};
            for (; tau < blocks; ++tau) {
                g.tau0 = int(tau);
                g.wp   = int((write_pos + tau) % size_t(ring));
                fdl_mac_sparse_kernel<T><<<grid, 128, 0, stream>>>(fdl.template as<cx<T>>(), sp_meta.template as<uint2>(), sp_vals.template as<cx<T>>(),
                                                                  sp_base.template as<unsigned long long>(), acc_w(), g, nseg);
                NEO_TRY(check_launch("fdl_mac_sparse_kernel"));
                ++mac_launches;
            }
        }
        while (tau < blocks) {
            size_t const left = blocks - tau;
            g.tau0            = int(tau);
            g.wp              = int((write_pos + tau) % size_t(ring));
            bool const tma    = sizeof(T) == 4 && m >= 128;  // float rows of whole 1 KB tiles: TMA-staged kernel
            int const tb      = left >= 32 && tma ? 32 : left >= 16 && sizeof(T) == 4 ? 16 : left >= 8 ? 8 : left >= 4 ? 4 : left >= 2 ? 2 : 1;
            NEO_TRY(launch_mac(tb, g, nout, stream));
            ++mac_launches;
            tau += size_t(tb);
        }
        return mark_end(1, stream);
    }

    // the ring position moves once per call, after every channel group has been inserted
    void advance(size_t blocks)
    {
        if (frame > 0) {
            write_pos2 = (write_pos2 + 1) % size_t(ring2);
            x1_half ^= 1;
        } else {
            write_pos = (write_pos + blocks) % size_t(ring);
        }
        prev_flip ^= 1;  // the r2c kernels saved this call's last block into the other half-window buffer
        in_call = false;
        if (acc_alt.ptr != nullptr) {
            acc_last = acc_cur;
            acc_cur ^= 1;
        }
    }

    int forward(T const* in, size_t in_stride, size_t blocks, cudaStream_t stream)
    {
        NEO_TRY(forward_r2c(in, in_stride, blocks, 0, cfg.inputs, stream));
        NEO_TRY(forward_mac(blocks, 0, cfg.outputs, stream));
        advance(blocks);
        return NEO_B200_OK;
    }

    int launch_mac(int tb, mac_geom const& g, size_t nout, cudaStream_t stream)
    {
        auto const* x = fdl.template as<cx<T>>();
        auto const* h = filter.template as<cx<T>>();
        auto* a       = acc_w();
        if (tb == 1) { return launch_stream(x, h, a, g, nout, stream); }
        if constexpr (sizeof(T) == 4) {
            if (m >= 128 && tb >= 8) {
                dim3 const tgrid{static_cast<unsigned>(nt), static_cast<unsigned>(nout), static_cast<unsigned>(splits)};
                // measured on B200 (C5): 16 rows per stage x 2 stages beats 8 x 3 at TB=16 (5072 vs 4650 channel-Msamples/s):
                // fewer window shifts and stage hand-overs per FMA; TB=32 has no registers left for 16-row stages
                if (tb == 32) { return launch_tma<32, 8, 3>(tgrid, x, h, a, g, stream); }
                if (tb == 16) { return launch_tma<16, 16, 2>(tgrid, x, h, a, g, stream); }
                return launch_tma<8, 8, 3>(tgrid, x, h, a, g, stream);
            }
        }
        dim3 const grid(unsigned((m + k_mac_threads - 1) / k_mac_threads), unsigned(nout), unsigned(splits));
        switch (tb) {
            case 2: fdl_mac_toeplitz_kernel<T, 2><<<grid, k_mac_threads, 0, stream>>>(x, h, a, g); break;
            case 4: fdl_mac_toeplitz_kernel<T, 4><<<grid, k_mac_threads, 0, stream>>>(x, h, a, g); break;
            case 8: fdl_mac_toeplitz_kernel<T, 8><<<grid, k_mac_threads, 0, stream>>>(x, h, a, g); break;
            default:
                if constexpr (sizeof(T) == 4) { fdl_mac_toeplitz_kernel<T, 16><<<grid, k_mac_threads, 0, stream>>>(x, h, a, g); }
                break;
        }
        return check_launch("fdl_mac_toeplitz_kernel");
    }

    int launch_stream(cx<T> const* x, cx<T> const* h, cx<T>* a, mac_geom const& g, size_t nout, cudaStream_t stream)
    {
        unsigned const gx = unsigned((g.m / mac_vec<T>::VEC + k_mac_threads - 1) / k_mac_threads);
        if (cfg.topology == NEO_B200_MATRIX && nout % 4 == 0) {
            // four outputs per thread share every FDL row they load
            dim3 const grid(gx, unsigned(nout / 4), unsigned(g.splits));
            fdl_mac_stream_kernel<T, 4><<<grid, k_mac_threads, 0, stream>>>(x, h, a, g);
        } else {
            dim3 const grid(gx, unsigned(nout), unsigned(g.splits));
            fdl_mac_stream_kernel<T, 1><<<grid, k_mac_threads, 0, stream>>>(x, h, a, g);
        }
        return check_launch("fdl_mac_stream_kernel");
    }

    template<int TB, int CH, int STAGES>
    int launch_tma(dim3 grid, float2 const* x, float2 const* h, float2* a, mac_geom const& g, cudaStream_t stream)
    {
        using tc = mac_tma_cfg<TB, CH, STAGES>;
        if (g.parts % CH == 0) {
            auto kernel = fdl_mac_tma_kernel<TB, CH, STAGES, false>;
            NEO_TRY(enable_smem(kernel, tc::SMEM));
            kernel<<<grid, 128, tc::SMEM, stream>>>(x, h, a, g);
        } else {
            auto kernel = fdl_mac_tma_kernel<TB, CH, STAGES, true>;
            NEO_TRY(enable_smem(kernel, tc::SMEM));
            kernel<<<grid, 128, tc::SMEM, stream>>>(x, h, a, g);
        }
        return check_launch("fdl_mac_tma_kernel");
    }

    // c2r + scale + overlap handling of spectra [count][blocks][B] (S partial planes `plane` apart) into out [count][out_stride]
    int inverse(cx<T> const* spectra, size_t /*plane*/, int /*nsplits*/, T* out, size_t out_stride, size_t first, size_t count,
                size_t blocks, cudaStream_t stream)
    {
        cx<T> const* one[1] = {spectra};
        return inverse_sum(one, 1, out, out_stride, first, count, blocks, stream);
    }

    // the same for the sum of `nsrc` partial spectra buffers (partition shards of a multi-device bank; peer-mapped pointers are
    // read over NVLink inside the c2r kernel: reduction and inverse transform are one pass)
    int inverse_sum(cx<T> const* const* srcs, int nsrc, T* out, size_t out_stride, size_t first, size_t count, size_t blocks,
                    cudaStream_t stream)
    {
        bool const ola = cfg.kind == NEO_B200_UPOLA;
        T* const dst   = ola ? ola_y.template as<T>() : out;
        int status     = NEO_B200_ERR_UNSUPPORTED;
        if (nsrc < 1 || nsrc > k_bank_max_shards) { return fail(NEO_B200_ERR_INVALID, "bad number of partial spectra %d", nsrc); }
        NEO_TRY(mark_begin(2, stream));
        NEO_DISPATCH_LOGM(T, logb, {
            if constexpr (LOGM >= 1 && LOGM <= max_cta_logm<T>()) {
                if (nsrc == 1) {
                    conv_c2r_io<T, LOGM> io{srcs[0], int(blocks), dst, out_stride, T(1) / T(2 * m), ola ? 1 : 0};
                    status = run_c2r<LOGM>(io, wide_rows_ok(dst, ola ? 4 : out_stride), count * blocks, stream);
                } else {
                    auto const run = [&](auto io) {
                        for (int j = 0; j < nsrc; ++j) { io.src[j] = srcs[j]; }
                        io.nsrc        = nsrc;
                        io.blocks      = int(blocks);
                        io.out         = dst;
                        io.out_stride  = out_stride;
                        io.scale       = T(1) / T(2 * m);
                        io.overlap_add = ola ? 1 : 0;
                        return run_c2r<LOGM>(io, wide_rows_ok(dst, ola ? 4 : out_stride), count * blocks, stream);
                    };
                    status = nsrc == 2 ? run(conv_c2r_sum_io<T, LOGM, 2>{}) : run(conv_c2r_sum_io<T, LOGM, 0>{});
                }
            }
        });
        if (status != NEO_B200_OK) { return status; }
        if (ola) {
            // the tail belongs to a channel and is updated in place: any number of inverse calls over disjoint channel ranges
            // may finish one step (overlap_add.hpp:103-106)
            dim3 const grid(unsigned((m + 255) / 256), unsigned(count));
            ola_combine_kernel<T><<<grid, 256, 0, stream>>>(ola_y.template as<T>(), tail.template as<T>(), out, out_stride, m, int(blocks), first);
            NEO_TRY(check_launch("ola_combine_kernel"));
        }
        NEO_TRY(mark_end(2, stream));
        return NEO_B200_OK;
    }
};

int validate(neo_b200_conv_config& c)
{
    if (c.kind != NEO_B200_UPOLS && c.kind != NEO_B200_UPOLA) { return fail(NEO_B200_ERR_INVALID, "bad kind %d", c.kind); }
    if (c.dtype != NEO_B200_F32 && c.dtype != NEO_B200_F64) { return fail(NEO_B200_ERR_INVALID, "bad dtype %d", c.dtype); }
    if (c.topology != NEO_B200_DIAGONAL && c.topology != NEO_B200_MATRIX) { return fail(NEO_B200_ERR_INVALID, "bad topology %d", c.topology); }
    if (c.outputs == 0) { return fail(NEO_B200_ERR_INVALID, "outputs must be > 0"); }
    if (c.topology == NEO_B200_DIAGONAL) {
        if (c.inputs == 0) { c.inputs = c.outputs; }
        if (c.inputs != c.outputs) { return fail(NEO_B200_ERR_INVALID, "diagonal topology needs inputs == outputs"); }
    } else if (c.inputs == 0) {
        return fail(NEO_B200_ERR_INVALID, "inputs must be > 0");
    }
    // overlap_save sizes its rfft as bit_ceil(2B-1) (overlap_save.hpp:53), uniform_partition as 2B (stft.hpp:104):
    // they agree only for power-of-two B, which is also what every reference test uses
    if (!is_pow2(c.block) || c.block < 2) { return fail(NEO_B200_ERR_INVALID, "block size must be a power of two >= 2, got %zu", c.block); }
    if (c.partitions == 0) { return fail(NEO_B200_ERR_INVALID, "partitions must be > 0"); }
    if (c.frame_blocks != 0) {
        if (!is_pow2(c.frame_blocks) || c.frame_blocks < 2 || c.frame_blocks > k_max_frame_blocks) {
            return fail(NEO_B200_ERR_INVALID, "frame_blocks must be a power of two in [2, %zu], got %zu", k_max_frame_blocks, c.frame_blocks);
        }
        if (c.max_blocks != 0 && c.max_blocks != c.frame_blocks) {
            return fail(NEO_B200_ERR_INVALID, "frame mode processes exactly frame_blocks=%zu blocks per call (max_blocks=%zu)", c.frame_blocks,
                        c.max_blocks);
        }
        c.max_blocks = c.frame_blocks;
    }
    if (c.max_blocks == 0) { c.max_blocks = 1; }
    if (c.partition_begin == 0 && c.partition_end == 0) { c.partition_end = c.partitions; }
    if (c.partition_begin >= c.partition_end || c.partition_end > c.partitions) {
        return fail(NEO_B200_ERR_INVALID, "bad partition range [%zu, %zu) of %zu", c.partition_begin, c.partition_end, c.partitions);
    }
    if (c.frame_blocks != 0 && c.partition_begin % c.frame_blocks != 0) {
        return fail(NEO_B200_ERR_INVALID, "frame mode: partition_begin=%zu must be a multiple of frame_blocks=%zu", c.partition_begin, c.frame_blocks);
    }
    if (c.partition_end + c.max_blocks > (size_t(1) << 30) || c.outputs > 65535) { return fail(NEO_B200_ERR_INVALID, "configuration too large"); }
    return NEO_B200_OK;
}

}  // namespace
}  // namespace neo_b200

using namespace neo_b200;

struct neo_b200_conv
{
    neo_b200_conv_config cfg;
    int device;
    stream_ref stream;
    conv_engine<float> f32;
    conv_engine<double> f64;
    bool sharded;

    // copy streams + events of the pipelined HOST path (created on first use)
    cudaStream_t s_in{nullptr}, s_out{nullptr};
    cudaEvent_t ev_start{nullptr};
    std::vector<cudaEvent_t> ev_in, ev_done;
    // pageable HOST buffers of long calls are staged through these pinned chunks (two per direction), so the DMA engines run at PCIe
    // speed and the copies overlap the kernels whatever memory the caller hands over
    pinned_buffer pin_in[2], pin_out[2];
    cudaEvent_t ev_h2d[2]{}, ev_d2h[2]{};

    int ensure_pipeline(size_t groups)
    {
        if (s_in == nullptr) {
            NEO_CUDA_TRY(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
            NEO_CUDA_TRY(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
            NEO_CUDA_TRY(cudaEventCreateWithFlags(&ev_start, cudaEventDisableTiming));
        }
        if (ev_h2d[0] == nullptr) {
            for (cudaEvent_t* ev : {&ev_h2d[0], &ev_h2d[1], &ev_d2h[0], &ev_d2h[1]}) {
                NEO_CUDA_TRY(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
            }
        }
        while (ev_in.size() < groups) {
            cudaEvent_t a, b;
            NEO_CUDA_TRY(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
            NEO_CUDA_TRY(cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
            ev_in.push_back(a);
            ev_done.push_back(b);
        }
        return NEO_B200_OK;
    }

    ~neo_b200_conv()
    {
        for (auto ev : ev_in) { cudaEventDestroy(ev); }
        for (auto ev : ev_done) { cudaEventDestroy(ev); }
        if (ev_start != nullptr) { cudaEventDestroy(ev_start); }
        for (cudaEvent_t ev : {ev_h2d[0], ev_h2d[1], ev_d2h[0], ev_d2h[1]}) {
            if (ev != nullptr) { cudaEventDestroy(ev); }
        }
        if (s_in != nullptr) { cudaStreamDestroy(s_in); }
        if (s_out != nullptr) { cudaStreamDestroy(s_out); }
    }
};

#include "conv_bank.cuh"

#define NEO_CONV_ENGINE(conv, CALL) ((conv)->cfg.dtype == NEO_B200_F32 ? (conv)->f32.CALL : (conv)->f64.CALL)

extern "C" {

int neo_b200_conv_create(neo_b200_conv** conv, neo_b200_conv_config const* config)
{
    if (conv == nullptr || config == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    *conv = nullptr;
    neo_b200_conv_config c = *config;
    NEO_TRY(validate(c));
    size_t const logb = log2_exact(c.block);
    if (int(logb) > (c.dtype == NEO_B200_F32 ? max_cta_logm<float>() : max_cta_logm<double>())) {
        return fail(NEO_B200_ERR_UNSUPPORTED, "block size %zu exceeds the single-CTA transform range", c.block);
    }
    NEO_TRY(require_device());
    auto p = std::unique_ptr<neo_b200_conv>(new (std::nothrow) neo_b200_conv{});
    if (!p) { return fail(NEO_B200_ERR_ALLOC, "out of host memory"); }
    p->cfg     = c;
    p->sharded = !(c.partition_begin == 0 && c.partition_end == c.partitions);
    NEO_CUDA_TRY(cudaGetDevice(&p->device));
    NEO_TRY(p->stream.create());
    NEO_TRY(NEO_CONV_ENGINE(p, init(c, p->stream.stream)));
    NEO_CUDA_TRY(cudaStreamSynchronize(p->stream.stream));
    *conv = p.release();
    return NEO_B200_OK;
}

void neo_b200_conv_destroy(neo_b200_conv* conv)
{
    if (conv == nullptr) { return; }
    cudaStreamSynchronize(conv->stream.stream);
    delete conv;
}

int neo_b200_conv_set_filter(neo_b200_conv* conv, void const* H, int memspace)
{
    if (conv == nullptr || H == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    NEO_CUDA_TRY(cudaSetDevice(conv->device));
    NEO_TRY(NEO_CONV_ENGINE(conv, set_filter(H, memspace, conv->stream.stream)));
    NEO_CUDA_TRY(cudaStreamSynchronize(conv->stream.stream));
    return NEO_B200_OK;
}

int neo_b200_conv_set_filter_csr(neo_b200_conv* conv, void const* values, uint64_t const* cols, uint64_t const* row_ptr, uint64_t const* filter_base)
{
    if (conv == nullptr || cols == nullptr || row_ptr == nullptr || filter_base == nullptr || (values == nullptr && filter_base[conv->cfg.outputs] != 0)) {
        return fail(NEO_B200_ERR_INVALID, "null argument");
    }
    NEO_CUDA_TRY(cudaSetDevice(conv->device));
    if (conv->cfg.dtype == NEO_B200_F32) {
        NEO_TRY(conv->f32.set_filter_csr(static_cast<float2 const*>(values), cols, row_ptr, filter_base, conv->stream.stream));
    } else {
        NEO_TRY(conv->f64.set_filter_csr(static_cast<double2 const*>(values), cols, row_ptr, filter_base, conv->stream.stream));
    }
    NEO_CUDA_TRY(cudaStreamSynchronize(conv->stream.stream));
    return NEO_B200_OK;
}

int neo_b200_conv_set_impulse(neo_b200_conv* conv, void const* ir, size_t taps, int memspace)
{
    if (conv == nullptr || ir == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    // stft would underflow L-B for L < B (fft/stft.hpp:24); the frame count must match the configured partitions
    if (taps < conv->cfg.block) { return fail(NEO_B200_ERR_INVALID, "impulse response shorter than one block"); }
    if (neo_b200_num_partitions(taps, conv->cfg.block) != conv->cfg.partitions) {
        return fail(NEO_B200_ERR_INVALID, "taps=%zu gives %zu partitions, handle was created for %zu", taps,
                    neo_b200_num_partitions(taps, conv->cfg.block), conv->cfg.partitions);
    }
    NEO_CUDA_TRY(cudaSetDevice(conv->device));
    NEO_TRY(NEO_CONV_ENGINE(conv, set_impulse(ir, taps, memspace, conv->stream.stream)));
    NEO_CUDA_TRY(cudaStreamSynchronize(conv->stream.stream));
    return NEO_B200_OK;
}

int neo_b200_conv_reset(neo_b200_conv* conv)
{
    if (conv == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    NEO_CUDA_TRY(cudaSetDevice(conv->device));
    return NEO_CONV_ENGINE(conv, clear_state(conv->stream.stream));
}

// true when the CUDA runtime knows the pointer as page-locked host memory (cudaMallocHost / cudaHostRegister / torch pin_memory)
static bool host_is_pinned(void const* p)
{
    cudaPointerAttributes attr{};
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}

// host memcpy with a few helper threads: one core moves ~10 GB/s, a PCIe 5 x16 link ~50 GB/s each way
static void parallel_copy(void* dst, void const* src, size_t bytes)
{
    size_t const min_piece = size_t(4) << 20;
    unsigned const hw      = std::max(1U, std::thread::hardware_concurrency());
    size_t const pieces    = std::min<size_t>({size_t(8), size_t(hw), bytes / min_piece});
    if (pieces <= 1) {
        std::memcpy(dst, src, bytes);
        return;
    }
    std::vector<std::thread> helpers;
    size_t const piece = ((bytes / pieces) + 4095) / 4096 * 4096;
    for (size_t i = 1; i < pieces; ++i) {
        size_t const off = i * piece;
        if (off >= bytes) { break; }
        size_t const len = std::min(piece, bytes - off);
        helpers.emplace_back([=] { std::memcpy(static_cast<char*>(dst) + off, static_cast<char const*>(src) + off, len); });
    }
    std::memcpy(dst, src, std::min(piece, bytes));
    for (auto& t : helpers) { t.join(); }
}

extern "C++" template<typename T>
int conv_process_impl(neo_b200_conv* conv, conv_engine<T>& e, void const* in, void* out, size_t blocks, int memspace)
{
    cudaStream_t const s = conv->stream.stream;
    size_t const stride  = blocks * e.m;
    size_t const plane   = conv->cfg.outputs * blocks * size_t(e.m);
    if (memspace == NEO_B200_DEVICE) {
        NEO_TRY(e.forward(static_cast<T const*>(in), stride, blocks, s));
        NEO_TRY(e.inverse(e.acc.template as<cx<T>>(), plane, 1, static_cast<T*>(out), stride, 0, conv->cfg.outputs, blocks, s));
        return NEO_B200_OK;
    }

    // HOST buffers. Channels of a diagonal bank are independent, so the call is cut into channel groups and pipelined over
    // three streams: H2D of group g+1 and D2H of group g-1 overlap the kernels of group g (both PCIe directions busy).
    size_t const chans = conv->cfg.outputs;
    NEO_TRY(e.stage_in.reserve(conv->cfg.inputs * stride * sizeof(T)));
    NEO_TRY(e.stage_out.reserve(chans * stride * sizeof(T)));
    T* const din  = e.stage_in.template as<T>();
    T* const dout = e.stage_out.template as<T>();
    size_t groups = 1;
    // worth it only when the copies are long enough to matter next to the kernels (several blocks per call)
    if (conv->cfg.topology == NEO_B200_DIAGONAL && blocks >= 4) {
        groups = chans >= 512 ? 4 : chans >= 128 ? 2 : 1;
        // long calls (frame mode): about 64 MB per group, so the un-overlapped first H2D and last D2H stay a small share
        size_t const by_bytes = chans * stride * sizeof(T) / (size_t(64) << 20);
        groups                = std::max(groups, std::min<size_t>({by_bytes, size_t(16), chans / 32}));
        groups                = std::max<size_t>(groups, 1);
    }
    if (char const* env = std::getenv("NEO_B200_HOST_GROUPS")) {  // tuning knob
        size_t const want = size_t(std::max(1, std::atoi(env)));
        if (conv->cfg.topology == NEO_B200_DIAGONAL && want <= chans) { groups = want; }
    }
    if (groups == 1) {
        NEO_CUDA_TRY(cudaMemcpyAsync(din, in, conv->cfg.inputs * stride * sizeof(T), cudaMemcpyHostToDevice, s));
        NEO_TRY(e.forward(din, stride, blocks, s));
        NEO_TRY(e.inverse(e.acc.template as<cx<T>>(), plane, 1, dout, stride, 0, chans, blocks, s));
        NEO_CUDA_TRY(cudaMemcpyAsync(out, dout, chans * stride * sizeof(T), cudaMemcpyDeviceToHost, s));
    } else {
        NEO_TRY(conv->ensure_pipeline(groups));
        NEO_CUDA_TRY(cudaEventRecord(conv->ev_start, s));
        NEO_CUDA_TRY(cudaStreamWaitEvent(conv->s_in, conv->ev_start, 0));   // previous work on the handle's stream is done first
        NEO_CUDA_TRY(cudaStreamWaitEvent(conv->s_out, conv->ev_start, 0));
        // Pinned caller memory is handed to the DMA engines as it is. Pageable memory (std::vector, numpy) would make every
        // cudaMemcpyAsync host-synchronous and slow, so it is staged: the calling thread (plus helpers) copies group g into a pinned
        // chunk while the device works on group g-1, and copies group g-2 out of its pinned chunk.
        bool const staged      = !host_is_pinned(in) || !host_is_pinned(out);
        size_t const max_group = ((chans + groups - 1) / groups) * stride * sizeof(T);
        if (staged) {
            for (int i = 0; i < 2; ++i) {
                NEO_TRY(conv->pin_in[i].reserve(max_group));
                NEO_TRY(conv->pin_out[i].reserve(max_group));
            }
        }
        auto const range = [&](size_t g, size_t* c0, size_t* n) {
            *c0 = g * chans / groups;
            *n  = (g + 1) * chans / groups - *c0;
        };
        auto const drain = [&](size_t g) -> int {  // staged: group g has arrived in its pinned chunk, hand it to the caller
            size_t c0, n;
            range(g, &c0, &n);
            NEO_CUDA_TRY(cudaEventSynchronize(conv->ev_d2h[g & 1]));
            parallel_copy(static_cast<T*>(out) + c0 * stride, conv->pin_out[g & 1].ptr, n * stride * sizeof(T));
            return NEO_B200_OK;
        };
        for (size_t g = 0; g < groups; ++g) {
            size_t c0, n;
            range(g, &c0, &n);
            void const* src = static_cast<T const*>(in) + c0 * stride;
            if (staged) {
                if (g >= 2) { NEO_CUDA_TRY(cudaEventSynchronize(conv->ev_h2d[g & 1])); }  // the chunk's previous copy has left
                parallel_copy(conv->pin_in[g & 1].ptr, src, n * stride * sizeof(T));
                src = conv->pin_in[g & 1].ptr;
            }
            NEO_CUDA_TRY(cudaMemcpyAsync(din + c0 * stride, src, n * stride * sizeof(T), cudaMemcpyHostToDevice, conv->s_in));
            if (staged) { NEO_CUDA_TRY(cudaEventRecord(conv->ev_h2d[g & 1], conv->s_in)); }
            NEO_CUDA_TRY(cudaEventRecord(conv->ev_in[g], conv->s_in));
            NEO_CUDA_TRY(cudaStreamWaitEvent(s, conv->ev_in[g], 0));
            NEO_TRY(e.forward_r2c(din + c0 * stride, stride, blocks, c0, n, s));
            NEO_TRY(e.forward_mac(blocks, c0, n, s));
            NEO_TRY(e.inverse(e.acc.template as<cx<T>>() + c0 * blocks * size_t(e.m), plane, 1, dout + c0 * stride, stride, c0, n,
                              blocks, s));
            NEO_CUDA_TRY(cudaEventRecord(conv->ev_done[g], s));
            NEO_CUDA_TRY(cudaStreamWaitEvent(conv->s_out, conv->ev_done[g], 0));
            if (staged && g >= 2) { NEO_TRY(drain(g - 2)); }  // frees pin_out[g & 1] for this group
            void* const dst = staged ? conv->pin_out[g & 1].ptr : static_cast<void*>(static_cast<T*>(out) + c0 * stride);
            NEO_CUDA_TRY(cudaMemcpyAsync(dst, dout + c0 * stride, n * stride * sizeof(T), cudaMemcpyDeviceToHost, conv->s_out));
            if (staged) { NEO_CUDA_TRY(cudaEventRecord(conv->ev_d2h[g & 1], conv->s_out)); }
        }
        e.advance(blocks);
        if (staged) {
            for (size_t g = groups >= 2 ? groups - 2 : 0; g < groups; ++g) { NEO_TRY(drain(g)); }
        }
        NEO_CUDA_TRY(cudaStreamSynchronize(conv->s_out));
    }
    NEO_CUDA_TRY(cudaStreamSynchronize(s));
    return NEO_B200_OK;
}

static int conv_check_call(neo_b200_conv* conv, size_t blocks, bool whole_bank = true)
{
    if (conv == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    bool const ready = conv->cfg.dtype == NEO_B200_F32 ? conv->f32.has_filter : conv->f64.has_filter;
    if (!ready) { return fail(NEO_B200_ERR_INVALID, "no filter set"); }
    bool const in_call = conv->cfg.dtype == NEO_B200_F32 ? conv->f32.in_call : conv->f64.in_call;
    if (whole_bank && in_call) {
        return fail(NEO_B200_ERR_INVALID, "a forward_range call is in progress: pass final != 0 with its last channel range (or reset) first");
    }
    if (blocks == 0 || blocks > conv->cfg.max_blocks) {
        return fail(NEO_B200_ERR_INVALID, "blocks=%zu outside [1, max_blocks=%zu]", blocks, conv->cfg.max_blocks);
    }
    if (conv->cfg.frame_blocks != 0 && blocks != conv->cfg.frame_blocks) {
        return fail(NEO_B200_ERR_INVALID, "frame mode: every call processes exactly frame_blocks=%zu blocks, got %zu", conv->cfg.frame_blocks, blocks);
    }
    NEO_CUDA_TRY(cudaSetDevice(conv->device));
    return NEO_B200_OK;
}

int neo_b200_conv_process(neo_b200_conv* conv, void const* in, void* out, size_t blocks, int memspace)
{
    NEO_TRY(conv_check_call(conv, blocks));
    if (in == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null buffer"); }
    if (conv->sharded) { return fail(NEO_B200_ERR_INVALID, "partition-sharded handle: use conv_forward / conv_inverse around the reduction"); }
    if (in == out && conv->cfg.topology != NEO_B200_DIAGONAL) { return fail(NEO_B200_ERR_INVALID, "in-place needs the diagonal topology"); }
    if (conv->cfg.dtype == NEO_B200_F32) { return conv_process_impl<float>(conv, conv->f32, in, out, blocks, memspace); }
    return conv_process_impl<double>(conv, conv->f64, in, out, blocks, memspace);
}

extern "C++" template<typename T>
int conv_forward_impl(neo_b200_conv* conv, conv_engine<T>& e, void const* in, size_t blocks, int memspace)
{
    cudaStream_t const s = conv->stream.stream;
    size_t const stride  = blocks * e.m;
    T const* din         = static_cast<T const*>(in);
    if (memspace == NEO_B200_HOST) {
        NEO_TRY(e.stage_in.reserve(conv->cfg.inputs * stride * sizeof(T)));
        NEO_CUDA_TRY(cudaMemcpyAsync(e.stage_in.ptr, in, conv->cfg.inputs * stride * sizeof(T), cudaMemcpyHostToDevice, s));
        din = e.stage_in.template as<T>();
    }
    return e.forward(din, stride, blocks, s);
}

int neo_b200_conv_forward(neo_b200_conv* conv, void const* in, size_t blocks, int memspace)
{
    NEO_TRY(conv_check_call(conv, blocks));
    if (in == nullptr) { return fail(NEO_B200_ERR_INVALID, "null buffer"); }
    if (conv->cfg.dtype == NEO_B200_F32) { return conv_forward_impl<float>(conv, conv->f32, in, blocks, memspace); }
    return conv_forward_impl<double>(conv, conv->f64, in, blocks, memspace);
}

extern "C++" template<typename T>
int conv_forward_range_impl(neo_b200_conv* conv, conv_engine<T>& e, void const* in, size_t blocks, size_t first, size_t count, int final)
{
    cudaStream_t const s = conv->stream.stream;
    size_t const stride  = blocks * e.m;
    // the ranges of one call tile the bank in ascending order, every channel exactly once, the same block count throughout
    if (!e.in_call) {
        e.range_next   = 0;
        e.range_blocks = blocks;
    }
    if (first != e.range_next) {
        return fail(NEO_B200_ERR_INVALID, "forward_range: channel range must start at %zu (ranges tile the bank in ascending order), got %zu",
                    e.range_next, first);
    }
    if (blocks != e.range_blocks) {
        return fail(NEO_B200_ERR_INVALID, "forward_range: blocks=%zu differs from the %zu of the call in progress", blocks, e.range_blocks);
    }
    if ((final != 0) != (first + count == conv->cfg.outputs)) {
        return fail(NEO_B200_ERR_INVALID, "forward_range: final must be set exactly with the range that ends at channel %zu", conv->cfg.outputs);
    }
    cudaPointerAttributes attr{};
    if (cudaPointerGetAttributes(&attr, in) != cudaSuccess || (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged)) {
        (void)cudaGetLastError();
        return fail(NEO_B200_ERR_INVALID, "forward_range needs DEVICE memory");
    }
    NEO_TRY(e.forward_r2c(static_cast<T const*>(in) + first * stride, stride, blocks, first, count, s));
    NEO_TRY(e.forward_mac(blocks, first, count, s));
    e.in_call    = true;
    e.range_next = first + count;
    if (final != 0) { e.advance(blocks); }
    return NEO_B200_OK;
}

int neo_b200_conv_forward_range(neo_b200_conv* conv, void const* in, size_t blocks, size_t first, size_t count, int final)
{
    NEO_TRY(conv_check_call(conv, blocks, false));
    if (in == nullptr) { return fail(NEO_B200_ERR_INVALID, "null buffer"); }
    if (conv->cfg.topology != NEO_B200_DIAGONAL) { return fail(NEO_B200_ERR_INVALID, "forward_range needs the diagonal topology"); }
    if (count == 0 || first + count > conv->cfg.outputs) { return fail(NEO_B200_ERR_INVALID, "bad channel range"); }
    if (conv->cfg.dtype == NEO_B200_F32) { return conv_forward_range_impl<float>(conv, conv->f32, in, blocks, first, count, final); }
    return conv_forward_range_impl<double>(conv, conv->f64, in, blocks, first, count, final);
}

int neo_b200_conv_spectra(neo_b200_conv* conv, void** device_ptr, size_t* bytes_per_output_block)
{
    if (conv == nullptr || device_ptr == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    *device_ptr = conv->cfg.dtype == NEO_B200_F32 ? conv->f32.acc_r() : conv->f64.acc_r();
    if (bytes_per_output_block != nullptr) { *bytes_per_output_block = conv->cfg.block * 2 * elem_size(conv->cfg.dtype); }
    return NEO_B200_OK;
}

extern "C++" template<typename T>
int conv_inverse_impl(neo_b200_conv* conv, conv_engine<T>& e, void const* spectra, void* out, size_t first, size_t count,
                             size_t blocks, int memspace)
{
    cudaStream_t const s = conv->stream.stream;
    size_t const stride  = blocks * e.m;
    T* dout              = static_cast<T*>(out);
    if (memspace == NEO_B200_HOST) {
        NEO_TRY(e.stage_out.reserve(count * stride * sizeof(T)));
        dout = e.stage_out.template as<T>();
    }
    NEO_TRY(e.inverse(static_cast<cx<T> const*>(spectra), 0, 1, dout, stride, first, count, blocks, s));
    if (memspace == NEO_B200_HOST) {
        NEO_CUDA_TRY(cudaMemcpyAsync(out, dout, count * stride * sizeof(T), cudaMemcpyDeviceToHost, s));
        NEO_CUDA_TRY(cudaStreamSynchronize(s));
    }
    return NEO_B200_OK;
}

int neo_b200_conv_inverse(neo_b200_conv* conv, void const* spectra_device, void* out, size_t first, size_t count, size_t blocks, int memspace)
{
    NEO_TRY(conv_check_call(conv, blocks, false));
    if (spectra_device == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null buffer"); }
    if (first + count > conv->cfg.outputs) { return fail(NEO_B200_ERR_INVALID, "output range [%zu, %zu) outside the bank", first, first + count); }
    if (count == 0) { return NEO_B200_OK; }
    if (conv->cfg.dtype == NEO_B200_F32) { return conv_inverse_impl<float>(conv, conv->f32, spectra_device, out, first, count, blocks, memspace); }
    return conv_inverse_impl<double>(conv, conv->f64, spectra_device, out, first, count, blocks, memspace);
}

extern "C++" template<typename T>
int conv_window_impl(neo_b200_conv* conv, conv_engine<T>& e, void const* window, void* y, int commit, int memspace)
{
    cudaStream_t const s = conv->stream.stream;
    size_t const bytes   = conv->cfg.outputs * 2 * size_t(e.m) * sizeof(T);
    T const* win         = static_cast<T const*>(window);
    T* out               = static_cast<T*>(y);
    if (memspace == NEO_B200_HOST) {
        NEO_TRY(e.stage_in.reserve(bytes));
        NEO_TRY(e.stage_out.reserve(bytes));
        NEO_CUDA_TRY(cudaMemcpyAsync(e.stage_in.ptr, window, bytes, cudaMemcpyHostToDevice, s));
        win = e.stage_in.template as<T>();
        out = e.stage_out.template as<T>();
    }
    NEO_TRY(e.window_step(win, out, commit != 0, s));
    if (memspace == NEO_B200_HOST) {
        NEO_CUDA_TRY(cudaMemcpyAsync(y, out, bytes, cudaMemcpyDeviceToHost, s));
        NEO_CUDA_TRY(cudaStreamSynchronize(s));
    }
    return NEO_B200_OK;
}

int neo_b200_conv_process_window(neo_b200_conv* conv, void const* window, void* y, int commit, int memspace)
{
    NEO_TRY(conv_check_call(conv, 1));
    if (window == nullptr || y == nullptr) { return fail(NEO_B200_ERR_INVALID, "null buffer"); }
    if (conv->cfg.kind != NEO_B200_UPOLA || conv->cfg.topology != NEO_B200_DIAGONAL || conv->cfg.frame_blocks != 0 || conv->sharded) {
        return fail(NEO_B200_ERR_INVALID, "process_window needs an unsharded overlap-add diagonal bank in the direct form");
    }
    if (conv->cfg.dtype == NEO_B200_F32) { return conv_window_impl<float>(conv, conv->f32, window, y, commit, memspace); }
    return conv_window_impl<double>(conv, conv->f64, window, y, commit, memspace);
}

int neo_b200_conv_tail(neo_b200_conv* conv, void* tail, int memspace)
{
    if (conv == nullptr || tail == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (conv->cfg.kind != NEO_B200_UPOLA) { return fail(NEO_B200_ERR_INVALID, "only overlap-add handles keep a tail"); }
    NEO_CUDA_TRY(cudaSetDevice(conv->device));
    device_buffer const& buf = conv->cfg.dtype == NEO_B200_F32 ? conv->f32.tail : conv->f64.tail;
    NEO_CUDA_TRY(cudaMemcpyAsync(tail, buf.ptr, buf.bytes, memspace == NEO_B200_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice,
                                 conv->stream.stream));
    NEO_CUDA_TRY(cudaStreamSynchronize(conv->stream.stream));
    return NEO_B200_OK;
}

int neo_b200_conv_set_stream(neo_b200_conv* conv, void* cuda_stream)
{
    if (conv == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    conv->stream.adopt(cuda_stream);
    return NEO_B200_OK;
}

int neo_b200_conv_synchronize(neo_b200_conv* conv)
{
    if (conv == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    NEO_CUDA_TRY(cudaStreamSynchronize(conv->stream.stream));
    return NEO_B200_OK;
}

int neo_b200_conv_profile_enable(neo_b200_conv* conv, int enable)
{
    if (conv == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    conv->f32.profiling = conv->f64.profiling = (enable != 0);
    return NEO_B200_OK;
}

int neo_b200_conv_profile_read(neo_b200_conv* conv, double* phase_ms, uint64_t* mac_launches)
{
    if (conv == nullptr || phase_ms == nullptr || mac_launches == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    return NEO_CONV_ENGINE(conv, read_profile(phase_ms, mac_launches, conv->stream.stream));
}

size_t neo_b200_conv_device_bytes(neo_b200_conv const* conv)
{
    if (conv == nullptr) { return 0; }
    return conv->cfg.dtype == NEO_B200_F32 ? conv->f32.device_bytes() : conv->f64.device_bytes();
}

// ---- filter preparation -------------------------------------------------------------------------------------------------------
size_t neo_b200_num_partitions(size_t taps, size_t block)
{
    // num_sftf_frames(signal, frame, overlap=0) = idiv(signal - frame, frame) + 1 (fft/stft.hpp:21-25, math/idiv.hpp:11-14)
    if (block == 0 || taps < block) { return 0; }
    return (taps - block + block - 1) / block + 1;
}

extern "C++" template<typename T>
int uniform_partition_impl(void const* ir, size_t channels, size_t taps, size_t block, void* out, int memspace)
{
    int const logb = int(log2_exact(block));
    if (logb > max_cta_logm<T>()) { return fail(NEO_B200_ERR_UNSUPPORTED, "block size %zu exceeds the single-CTA transform range", block); }
    size_t const parts = neo_b200_num_partitions(taps, block);
    stream_ref stream;
    NEO_TRY(stream.create());
    cudaStream_t const s = stream.stream;
    fft_tables<T> tables;
    NEO_TRY(tables.build(logb, true, s));
    device_buffer d_in, d_out;
    T const* src  = static_cast<T const*>(ir);
    cx<T>* dst    = static_cast<cx<T>*>(out);
    size_t const out_row = parts * (block + 1) * sizeof(cx<T>);
    size_t chunk         = channels;
    if (memspace == NEO_B200_HOST) {
        chunk = std::max<size_t>(1, std::min(channels, (size_t(256) << 20) / out_row));
        NEO_TRY(d_in.reserve(chunk * taps * sizeof(T)));
        NEO_TRY(d_out.reserve(chunk * out_row));
    }
    for (size_t c = 0; c < channels; c += chunk) {
        size_t const n = std::min(chunk, channels - c);
        T const* in_dev = src + c * taps;
        cx<T>* out_dev  = dst + c * parts * (block + 1);
        if (memspace == NEO_B200_HOST) {
            NEO_CUDA_TRY(cudaMemcpyAsync(d_in.ptr, src + c * taps, n * taps * sizeof(T), cudaMemcpyHostToDevice, s));
            in_dev  = d_in.template as<T>();
            out_dev = d_out.template as<cx<T>>();
        }
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_DISPATCH_LOGM(T, logb, {
            if constexpr (LOGM >= 1 && LOGM <= max_cta_logm<T>()) {
                partition_r2c_io<T, LOGM> io{in_dev, taps, 0, int(parts), out_dev, 0};
                status = launch_r2c<T, LOGM>(io, tables.tw(), tables.rtw(), n * parts, s);
            }
        });
        if (status != NEO_B200_OK) { return status; }
        if (memspace == NEO_B200_HOST) {
            NEO_CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(dst) + c * out_row, d_out.ptr, n * out_row, cudaMemcpyDeviceToHost, s));
        }
        NEO_CUDA_TRY(cudaStreamSynchronize(s));
    }
    return NEO_B200_OK;
}

int neo_b200_uniform_partition(void const* ir, size_t channels, size_t taps, size_t block, void* out, int dtype, int memspace)
{
    if (ir == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (!is_pow2(block) || block < 2) { return fail(NEO_B200_ERR_INVALID, "block size must be a power of two >= 2"); }
    if (taps < block) { return fail(NEO_B200_ERR_INVALID, "impulse response shorter than one block"); }
    if (channels == 0) { return NEO_B200_OK; }
    NEO_TRY(require_device());
    if (dtype == NEO_B200_F32) { return uniform_partition_impl<float>(ir, channels, taps, block, out, memspace); }
    if (dtype == NEO_B200_F64) { return uniform_partition_impl<double>(ir, channels, taps, block, out, memspace); }
    return fail(NEO_B200_ERR_INVALID, "bad dtype %d", dtype);
}

size_t neo_b200_num_stft_frames(size_t signal, size_t frame, size_t overlap)
{
    // num_sftf_frames (fft/stft.hpp:21-25): idiv(signal - frame + overlap, frame - overlap) + 1, idiv rounds up (math/idiv.hpp:11-14)
    if (frame == 0 || overlap >= frame || signal < frame) { return 0; }
    size_t const hop = frame - overlap;
    return (signal - frame + overlap + hop - 1) / hop + 1;
}

extern "C++" template<typename T>
int stft_impl(void const* x, size_t channels, size_t len, size_t frame, size_t transform, size_t overlap, void const* window, void* out,
              int memspace)
{
    size_t const order = neo_b200_next_order(transform);  // rfft_plan{from_order, next_order(transform_size)}, stft.hpp:104
    if (order < 1) { return fail(NEO_B200_ERR_INVALID, "transform size must be at least 2"); }
    int const logm = int(order) - 1;
    if (logm > max_cta_logm<T>()) { return fail(NEO_B200_ERR_UNSUPPORTED, "transform size %zu exceeds the single-CTA transform range", transform); }
    size_t const n      = size_t(1) << order;
    size_t const bins   = n / 2 + 1;
    size_t const frames = neo_b200_num_stft_frames(len, frame, overlap);
    if (frame > n) { return fail(NEO_B200_ERR_INVALID, "frame size %zu larger than the transform size %zu", frame, n); }
    stream_ref stream;
    NEO_TRY(stream.create());
    cudaStream_t const s = stream.stream;
    fft_tables<T> tables;
    NEO_TRY(tables.build(logm, true, s));
    device_buffer d_win, d_in, d_out;
    T const* win = static_cast<T const*>(window);
    if (window != nullptr && memspace == NEO_B200_HOST) {
        NEO_TRY(d_win.reserve(n * sizeof(T)));
        NEO_CUDA_TRY(cudaMemcpyAsync(d_win.ptr, window, n * sizeof(T), cudaMemcpyHostToDevice, s));
        win = d_win.template as<T>();
    }
    size_t const out_row = frames * bins * sizeof(cx<T>);
    size_t chunk         = channels;
    if (memspace == NEO_B200_HOST) {
        chunk = std::max<size_t>(1, std::min(channels, (size_t(256) << 20) / std::max<size_t>(out_row, 1)));
        NEO_TRY(d_in.reserve(chunk * len * sizeof(T)));
        NEO_TRY(d_out.reserve(chunk * out_row));
    }
    for (size_t c = 0; c < channels; c += chunk) {
        size_t const cnt = std::min(chunk, channels - c);
        T const* in_dev  = static_cast<T const*>(x) + c * len;
        cx<T>* out_dev   = static_cast<cx<T>*>(out) + c * frames * bins;
        if (memspace == NEO_B200_HOST) {
            NEO_CUDA_TRY(cudaMemcpyAsync(d_in.ptr, in_dev, cnt * len * sizeof(T), cudaMemcpyHostToDevice, s));
            in_dev  = d_in.template as<T>();
            out_dev = d_out.template as<cx<T>>();
        }
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_DISPATCH_LOGM(T, logm, {
            if constexpr (LOGM <= max_cta_logm<T>()) {
                stft_r2c_io<T, LOGM> io{in_dev, len, frame, frame - overlap, frames, win, out_dev};
                status = launch_r2c<T, LOGM>(io, tables.tw(), tables.rtw(), cnt * frames, s);
            }
        });
        if (status != NEO_B200_OK) { return status; }
        if (memspace == NEO_B200_HOST) {
            NEO_CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(out) + c * out_row, d_out.ptr, cnt * out_row, cudaMemcpyDeviceToHost, s));
        }
        NEO_CUDA_TRY(cudaStreamSynchronize(s));
    }
    return NEO_B200_OK;
}

int neo_b200_stft(void const* x, size_t channels, size_t len, size_t frame_size, size_t transform_size, size_t overlap_size,
                  void const* window, void* out, int dtype, int memspace)
{
    if (x == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (frame_size == 0 || overlap_size >= frame_size) { return fail(NEO_B200_ERR_INVALID, "need 0 <= overlap < frame size"); }
    if (len < frame_size) { return fail(NEO_B200_ERR_INVALID, "signal shorter than one frame"); }  // stft.hpp:24 underflows
    if (channels == 0) { return NEO_B200_OK; }
    NEO_TRY(require_device());
    if (dtype == NEO_B200_F32) { return stft_impl<float>(x, channels, len, frame_size, transform_size, overlap_size, window, out, memspace); }
    if (dtype == NEO_B200_F64) { return stft_impl<double>(x, channels, len, frame_size, transform_size, overlap_size, window, out, memspace); }
    return fail(NEO_B200_ERR_INVALID, "bad dtype %d", dtype);
}

extern "C++" template<typename T>
int normalize_impulse_impl(void* ir, size_t channels, size_t taps, int memspace)
{
    stream_ref stream;
    NEO_TRY(stream.create());
    cudaStream_t const s = stream.stream;
    device_buffer data, energy;
    size_t const bytes = channels * taps * sizeof(T);
    T* dev             = static_cast<T*>(ir);
    if (memspace == NEO_B200_HOST) {
        NEO_TRY(data.reserve(bytes));
        dev = data.template as<T>();
        NEO_CUDA_TRY(cudaMemcpyAsync(dev, ir, bytes, cudaMemcpyHostToDevice, s));
    }
    NEO_TRY(energy.reserve(channels * sizeof(double)));
    channel_energy_kernel<T><<<unsigned(channels), 256, 0, s>>>(dev, taps, energy.as<double>());
    NEO_TRY(check_launch("channel_energy_kernel"));
    scale_by_min_factor_kernel<T><<<1184, 256, 0, s>>>(dev, channels * taps, energy.as<double>(), unsigned(channels));
    NEO_TRY(check_launch("scale_by_min_factor_kernel"));
    if (memspace == NEO_B200_HOST) { NEO_CUDA_TRY(cudaMemcpyAsync(ir, dev, bytes, cudaMemcpyDeviceToHost, s)); }
    NEO_CUDA_TRY(cudaStreamSynchronize(s));
    return NEO_B200_OK;
}

int neo_b200_normalize_impulse(void* ir, size_t channels, size_t taps, int dtype, int memspace)
{
    if (ir == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (channels == 0 || taps == 0) { return NEO_B200_OK; }  // normalize_impulse.hpp:20-22
    if (channels > 0x7fffffffULL) { return fail(NEO_B200_ERR_INVALID, "too many channels"); }
    NEO_TRY(require_device());
    if (dtype == NEO_B200_F32) { return normalize_impulse_impl<float>(ir, channels, taps, memspace); }
    if (dtype == NEO_B200_F64) { return normalize_impulse_impl<double>(ir, channels, taps, memspace); }
    return fail(NEO_B200_ERR_INVALID, "bad dtype %d", dtype);
}

// ---- index tables -----------------------------------------------------------------------------------------------------------------
static int table_to_host(device_buffer& buf, uint32_t* out, size_t count)
{
    NEO_CUDA_TRY(cudaMemcpy(out, buf.ptr, count * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return NEO_B200_OK;
}

int neo_b200_bitrev_table(size_t order, uint32_t* out)
{
    if (out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (order > 30) { return fail(NEO_B200_ERR_UNSUPPORTED, "order %zu too large", order); }
    NEO_TRY(require_device());
    size_t const n = size_t(1) << order;
    device_buffer buf;
    NEO_TRY(buf.reserve(n * sizeof(uint32_t)));
    bitrev_table_kernel<<<unsigned((n + 255) / 256), 256>>>(unsigned(order), buf.as<unsigned>());
    NEO_TRY(check_launch("bitrev_table_kernel"));
    return table_to_host(buf, out, n);
}

int neo_b200_digitrev_perm(size_t radix, size_t size, uint32_t* out)
{
    if (out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (radix < 2 || size == 0) { return fail(NEO_B200_ERR_INVALID, "bad radix/size"); }
    size_t digits = 0, pow = 1;
    while (pow < size) {
        pow *= radix;
        ++digits;
    }
    if (pow != size) { return fail(NEO_B200_ERR_INVALID, "size %zu is not a power of radix %zu", size, radix); }
    NEO_TRY(require_device());
    device_buffer buf;
    NEO_TRY(buf.reserve(size * sizeof(uint32_t)));
    digitrev_perm_kernel<<<unsigned((size + 255) / 256), 256>>>(unsigned(radix), unsigned(digits), unsigned(size), buf.as<unsigned>());
    NEO_TRY(check_launch("digitrev_perm_kernel"));
    return table_to_host(buf, out, size);
}

}  // extern "C"

// compressed delay line: [rows][cols] int8 / int16 complex on the device
struct neo_b200_compressed_fdl
{
    int device{0};
    int dtype{NEO_B200_F32};
    int bits{16};
    size_t rows{0}, cols{0};
    device_buffer store, stage;

    size_t part_bytes() const { return bits == 8 ? 1 : 2; }
    template<typename T, typename I>
    int insert(void const* row, size_t index, int memspace)
    {
        size_t const n = 2 * cols;
        T const* src   = static_cast<T const*>(row);
        if (memspace == NEO_B200_HOST) {
            NEO_TRY(stage.reserve(n * sizeof(double)));
            NEO_CUDA_TRY(cudaMemcpy(stage.ptr, row, n * sizeof(T), cudaMemcpyHostToDevice));
            src = stage.as<T>();
        }
        compress_parts_kernel<T, I><<<unsigned((n + 255) / 256), 256>>>(src, store.as<I>() + index * n, n);
        NEO_TRY(check_launch("compress_parts_kernel"));
        NEO_CUDA_TRY(cudaDeviceSynchronize());
        return NEO_B200_OK;
    }
    template<typename T, typename I>
    int read(size_t index, void* out, int memspace)
    {
        size_t const n = 2 * cols;
        T* dst         = static_cast<T*>(out);
        if (memspace == NEO_B200_HOST) {
            NEO_TRY(stage.reserve(n * sizeof(double)));
            dst = stage.as<T>();
        }
        decompress_parts_kernel<T, I><<<unsigned((n + 255) / 256), 256>>>(store.as<I>() + index * n, dst, n);
        NEO_TRY(check_launch("decompress_parts_kernel"));
        if (memspace == NEO_B200_HOST) { NEO_CUDA_TRY(cudaMemcpy(out, stage.ptr, n * sizeof(T), cudaMemcpyDeviceToHost)); }
        else { NEO_CUDA_TRY(cudaDeviceSynchronize()); }
        return NEO_B200_OK;
    }
};

extern "C" {

int neo_b200_compressed_fdl_create(neo_b200_compressed_fdl** fdl, size_t rows, size_t cols, int dtype, int bits)
{
    if (fdl == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    *fdl = nullptr;
    if ((dtype != NEO_B200_F32 && dtype != NEO_B200_F64) || (bits != 8 && bits != 16) || rows == 0 || cols == 0) {
        return fail(NEO_B200_ERR_INVALID, "compressed_fdl: dtype F32/F64, bits 8/16, rows and cols > 0");
    }
    NEO_TRY(require_device());
    auto h = std::make_unique<neo_b200_compressed_fdl>();
    cudaGetDevice(&h->device);
    h->dtype = dtype;
    h->bits  = bits;
    h->rows  = rows;
    h->cols  = cols;
    NEO_TRY(h->store.reserve(rows * cols * 2 * h->part_bytes()));
    NEO_CUDA_TRY(cudaMemset(h->store.ptr, 0, h->store.bytes));  // the reference's mdarray is value-initialised
    *fdl = h.release();
    return NEO_B200_OK;
}

void neo_b200_compressed_fdl_destroy(neo_b200_compressed_fdl* fdl) { delete fdl; }

int neo_b200_compressed_fdl_insert(neo_b200_compressed_fdl* fdl, void const* row, size_t index, int memspace)
{
    if (fdl == nullptr || row == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (index >= fdl->rows) { return fail(NEO_B200_ERR_INVALID, "compressed_fdl: row %zu of %zu", index, fdl->rows); }
    NEO_CUDA_TRY(cudaSetDevice(fdl->device));
    if (fdl->dtype == NEO_B200_F32) {
        return fdl->bits == 8 ? fdl->insert<float, std::int8_t>(row, index, memspace) : fdl->insert<float, std::int16_t>(row, index, memspace);
    }
    return fdl->bits == 8 ? fdl->insert<double, std::int8_t>(row, index, memspace) : fdl->insert<double, std::int16_t>(row, index, memspace);
}

int neo_b200_compressed_fdl_row(neo_b200_compressed_fdl* fdl, size_t index, void* out, int memspace)
{
    if (fdl == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (index >= fdl->rows) { return fail(NEO_B200_ERR_INVALID, "compressed_fdl: row %zu of %zu", index, fdl->rows); }
    NEO_CUDA_TRY(cudaSetDevice(fdl->device));
    if (fdl->dtype == NEO_B200_F32) {
        return fdl->bits == 8 ? fdl->read<float, std::int8_t>(index, out, memspace) : fdl->read<float, std::int16_t>(index, out, memspace);
    }
    return fdl->bits == 8 ? fdl->read<double, std::int8_t>(index, out, memspace) : fdl->read<double, std::int16_t>(index, out, memspace);
}

int neo_b200_compressed_fdl_raw(neo_b200_compressed_fdl* fdl, size_t index, void* out_host)
{
    if (fdl == nullptr || out_host == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (index >= fdl->rows) { return fail(NEO_B200_ERR_INVALID, "compressed_fdl: row %zu of %zu", index, fdl->rows); }
    NEO_CUDA_TRY(cudaSetDevice(fdl->device));
    size_t const bytes = 2 * fdl->cols * fdl->part_bytes();
    NEO_CUDA_TRY(cudaMemcpy(out_host, static_cast<char const*>(fdl->store.ptr) + index * bytes, bytes, cudaMemcpyDeviceToHost));
    return NEO_B200_OK;
}

int neo_b200_fdl_index_sequence(size_t parts, size_t calls, uint32_t* write_pos, uint32_t* pairs)
{
    if (write_pos == nullptr || pairs == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (parts == 0 || calls == 0) { return NEO_B200_OK; }
    NEO_TRY(require_device());
    device_buffer wp, pr;
    NEO_TRY(wp.reserve(calls * sizeof(uint32_t)));
    NEO_TRY(pr.reserve(parts * calls * 2 * sizeof(uint32_t)));
    size_t const n = parts * calls;
    fdl_index_kernel<<<unsigned((n + 255) / 256), 256>>>(unsigned(parts), unsigned(calls), wp.as<unsigned>(), pr.as<unsigned>());
    NEO_TRY(check_launch("fdl_index_kernel"));
    NEO_TRY(table_to_host(wp, write_pos, calls));
    return table_to_host(pr, pairs, n * 2);
}

}  // extern "C"

// ---- one-block-latency convolver (neo_b200_lowlat_*): head kernel per block, frame-mode levels on side streams ----------------------
namespace neo_b200 {
namespace {

constexpr size_t k_lowlat_default_t1    = 8;
constexpr size_t k_lowlat_default_ratio = 4;  // T_1 x {4, 8} x {2, 4, 8, 16} on C5: 8, 32, 128 was fastest (DESIGN §4.7)

// validates the configuration, resolves the default schedule and yields the head range (ranges[0]) and one range per live level
int lowlat_resolve(neo_b200_lowlat_config const* c, size_t* levels, size_t fb[k_lowlat_max_levels], size_t ranges[k_lowlat_max_levels + 1][2])
{
    if (c == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (c->dtype != NEO_B200_F32 && c->dtype != NEO_B200_F64) { return fail(NEO_B200_ERR_INVALID, "bad dtype %d", c->dtype); }
    if (c->channels == 0 || c->channels > 65535) { return fail(NEO_B200_ERR_INVALID, "channels must be in [1, 65535], got %zu", c->channels); }
    size_t const max_block = size_t(1) << (c->dtype == NEO_B200_F32 ? max_cta_logm<float>() : max_cta_logm<double>());
    if (!is_pow2(c->block) || c->block < 2 || c->block > max_block) {
        return fail(NEO_B200_ERR_INVALID, "block size must be a power of two in [2, %zu], got %zu", max_block, c->block);
    }
    if (c->partitions == 0 || c->partitions > (size_t(1) << 30)) { return fail(NEO_B200_ERR_INVALID, "partitions must be in [1, 2^30]"); }
    if (c->levels > size_t(k_lowlat_max_levels)) {
        return fail(NEO_B200_ERR_INVALID, "at most %d levels, got %zu", k_lowlat_max_levels, c->levels);
    }
    size_t const P = c->partitions;
    size_t t[k_lowlat_max_levels] = {};
    size_t n                      = c->levels;
    if (n == 0) {  // library default: T_1 = 8, times 4 while the level would start inside the filter
        for (size_t v = k_lowlat_default_t1; v <= k_max_frame_blocks && n < size_t(k_lowlat_max_levels) && 2 * v < P; v *= k_lowlat_default_ratio) {
            t[n++] = v;
        }
    } else {
        for (size_t i = 0; i < n; ++i) {
            t[i] = c->frame_blocks[i];
            if (!is_pow2(t[i]) || t[i] < 2 || t[i] > k_max_frame_blocks) {
                return fail(NEO_B200_ERR_INVALID, "frame_blocks[%zu] must be a power of two in [2, %zu], got %zu", i, k_max_frame_blocks, t[i]);
            }
            if (i > 0 && t[i] <= t[i - 1]) {
                return fail(NEO_B200_ERR_INVALID, "frame_blocks must increase: frame_blocks[%zu]=%zu after %zu", i, t[i], t[i - 1]);
            }
        }
    }
    size_t live = 0;
    while (live < n && 2 * t[live] < P) { ++live; }  // levels that would start at or past the end of the filter are dropped
    size_t const t1 = n > 0 ? t[0] : k_lowlat_default_t1;
    ranges[0][0]    = 0;
    ranges[0][1]    = std::min(2 * t1, P);
    for (size_t i = 0; i < size_t(k_lowlat_max_levels); ++i) {
        fb[i]            = i < live ? t[i] : 0;
        ranges[i + 1][0] = i < live ? 2 * t[i] : 0;
        ranges[i + 1][1] = i < live ? (i + 1 < live ? 2 * t[i + 1] : P) : 0;
    }
    *levels = live;
    return NEO_B200_OK;
}

template<typename T>
struct lowlat_state
{
    conv_engine<T> head;                       // direct form over the head partitions (filter, delay line, half-window)
    conv_engine<T> level[k_lowlat_max_levels];  // frame mode, input_delayed, partitions [2 T_i, end_i)
    device_buffer in_ring;                     // [C][2 T_n][B] the last 2 T_n input blocks: every level's frame is contiguous
    device_buffer plane[k_lowlat_max_levels];  // [C][2 T_i][B] level i's partial output of block t at slot t mod 2 T_i
    device_buffer head_y, stage_in, stage_out; // unfused head output; HOST staging

    size_t device_bytes(size_t levels) const
    {
        size_t n = head.device_bytes() + in_ring.bytes + head_y.bytes + stage_in.bytes + stage_out.bytes;
        for (size_t i = 0; i < levels; ++i) { n += level[i].device_bytes() + plane[i].bytes; }
        return n;
    }
};

}  // namespace
}  // namespace neo_b200

struct neo_b200_lowlat
{
    neo_b200_lowlat_config cfg{};
    size_t levels{0};
    size_t t[k_lowlat_max_levels]{};
    size_t ranges[k_lowlat_max_levels + 1][2]{};
    size_t ring_blocks{1};  // 2 T_n
    int device{0};
    stream_ref stream;      // the head's stream (highest priority when the handle creates it)
    cudaStream_t side[k_lowlat_max_levels]{};
    cudaEvent_t ready[k_lowlat_max_levels]{};    // recorded on the head's stream when a level's frame is complete
    cudaEvent_t done[k_lowlat_max_levels][2]{};  // level i's frame f is in its plane: done[i][f % 2]
    bool sync{false};       // NEO_B200_LOWLAT_SYNC: level work on the head's stream
    bool fused{false};      // lowlat_head_kernel; else the head engine + lowlat_combine_kernel (NEO_B200_LOWLAT_UNFUSED)
    bool has_filter{false};
    size_t block_pos{0};    // blocks since the last reset
    lowlat_state<float> f32;
    lowlat_state<double> f64;

    int sync_all()
    {
        NEO_CUDA_TRY(cudaStreamSynchronize(stream.stream));
        for (size_t i = 0; i < levels; ++i) { NEO_CUDA_TRY(cudaStreamSynchronize(side[i])); }
        return NEO_B200_OK;
    }

    ~neo_b200_lowlat()
    {
        if (stream.stream != nullptr) { cudaStreamSynchronize(stream.stream); }
        for (size_t i = 0; i < size_t(k_lowlat_max_levels); ++i) {
            if (side[i] != nullptr) {
                cudaStreamSynchronize(side[i]);
                cudaStreamDestroy(side[i]);
            }
            for (cudaEvent_t ev : {ready[i], done[i][0], done[i][1]}) {
                if (ev != nullptr) { cudaEventDestroy(ev); }
            }
        }
    }
};

namespace neo_b200 {
namespace {

template<typename T>
lowlat_state<T>& lowlat_of(neo_b200_lowlat* h);
template<>
lowlat_state<float>& lowlat_of<float>(neo_b200_lowlat* h) { return h->f32; }
template<>
lowlat_state<double>& lowlat_of<double>(neo_b200_lowlat* h) { return h->f64; }

template<typename T>
int lowlat_init(neo_b200_lowlat* h)
{
    lowlat_state<T>& s   = lowlat_of<T>(h);
    cudaStream_t const st = h->stream.stream;
    size_t const C = h->cfg.channels, B = h->cfg.block;
    neo_b200_conv_config hc{NEO_B200_UPOLS, h->cfg.dtype, NEO_B200_DIAGONAL, C, C, B, h->cfg.partitions, 1, 0, h->ranges[0][1], 0, 0};
    NEO_TRY(validate(hc));
    NEO_TRY(s.head.init(hc, st));
    for (size_t i = 0; i < h->levels; ++i) {
        neo_b200_conv_config lc{NEO_B200_UPOLS, h->cfg.dtype, NEO_B200_DIAGONAL, C, C, B, h->cfg.partitions, h->t[i],
                                h->ranges[i + 1][0], h->ranges[i + 1][1], h->t[i], 1};
        NEO_TRY(validate(lc));
        NEO_TRY(s.level[i].init(lc, st));
        NEO_TRY(s.plane[i].reserve(C * 2 * h->t[i] * B * sizeof(T)));
    }
    NEO_TRY(s.in_ring.reserve(C * h->ring_blocks * B * sizeof(T)));
    if (!h->fused) { NEO_TRY(s.head_y.reserve(C * B * sizeof(T))); }
    return NEO_B200_OK;
}

// zero every piece of stream state; the caller has synchronised the side streams
template<typename T>
int lowlat_clear(neo_b200_lowlat* h)
{
    lowlat_state<T>& s   = lowlat_of<T>(h);
    cudaStream_t const st = h->stream.stream;
    NEO_TRY(s.head.clear_state(st));
    for (size_t i = 0; i < h->levels; ++i) {
        NEO_TRY(s.level[i].clear_state(st));
        NEO_CUDA_TRY(cudaMemsetAsync(s.plane[i].ptr, 0, s.plane[i].bytes, st));
    }
    NEO_CUDA_TRY(cudaMemsetAsync(s.in_ring.ptr, 0, s.in_ring.bytes, st));
    h->block_pos = 0;
    NEO_CUDA_TRY(cudaStreamSynchronize(st));
    return NEO_B200_OK;
}

template<typename T, int LOGM>
int lowlat_launch_head(lowlat_head_args<T> const& a, conv_engine<T> const& head, cudaStream_t st)
{
    using cfg   = fft_cfg<T, LOGM>;
    auto kernel = lowlat_head_kernel<T, LOGM>;
    NEO_TRY(enable_smem(kernel, cfg::SMEM));
    kernel<<<unsigned((a.channels + cfg::G - 1) / cfg::G), cfg::THREADS, cfg::SMEM, st>>>(a, head.tables.tw(), head.tables.rtw());
    return check_launch("lowlat_head_kernel");
}

// one block for every channel: `in` / `out` point at the block of channel 0
template<typename T>
int lowlat_block(neo_b200_lowlat* h, T const* in, size_t in_stride, T* out, size_t out_stride)
{
    lowlat_state<T>& s   = lowlat_of<T>(h);
    cudaStream_t const st = h->stream.stream;
    size_t const C = h->cfg.channels, B = h->cfg.block, tb = h->block_pos;

    // the partial output of level i for block tb comes from its frame tb / T_i - 2
    lowlat_levels<T> lv{};
    lv.count = int(h->levels);
    for (size_t i = 0; i < h->levels; ++i) {
        size_t const ti = h->t[i];
        if (!h->sync && tb % ti == 0 && tb >= 2 * ti) { NEO_CUDA_TRY(cudaStreamWaitEvent(st, h->done[i][(tb / ti - 2) & 1], 0)); }
        lv.plane[i]  = s.plane[i].template as<T>() + (tb % (2 * ti)) * B;
        lv.stride[i] = 2 * ti * B;
    }
    T* const ring_slot       = s.in_ring.template as<T>() + (tb % h->ring_blocks) * B;
    size_t const ring_stride = h->ring_blocks * B;

    if (h->fused) {
        conv_engine<T>& e = s.head;
        lowlat_head_args<T> a{in, in_stride, out, out_stride, e.prev[e.prev_flip].template as<T>(), e.prev[e.prev_flip ^ 1].template as<T>(),
                              ring_slot, ring_stride, e.fdl.template as<cx<T>>(), e.filter.template as<cx<T>>(), e.ring, int(e.write_pos),
                              e.parts, e.logw, C, lv};
        int status = NEO_B200_ERR_UNSUPPORTED;
        NEO_DISPATCH_LOGM(T, e.logb, {
            if constexpr (LOGM >= 6 && LOGM <= (sizeof(T) == 4 ? 12 : 11)) { status = lowlat_launch_head<T, LOGM>(a, e, st); }
        });
        if (status != NEO_B200_OK) { return status == NEO_B200_ERR_UNSUPPORTED ? fail(status, "fused head: block %zu not covered", B) : status; }
        e.advance(1);
    } else {
        conv_engine<T>& e = s.head;
        NEO_TRY(e.forward(in, in_stride, 1, st));
        NEO_TRY(e.inverse(static_cast<cx<T> const*>(e.acc_r()), 0, 1, s.head_y.template as<T>(), B, 0, C, 1, st));
        dim3 const grid(unsigned((B + 255) / 256), unsigned(C));
        lowlat_combine_kernel<T><<<grid, 256, 0, st>>>(s.head_y.template as<T>(), int(B), in, in_stride, out, out_stride, ring_slot, ring_stride, lv);
        NEO_TRY(check_launch("lowlat_combine_kernel"));
    }
    h->block_pos = tb + 1;

    // Levels whose frame this block completes. Frame f of level i (blocks f T_i .. f T_i + T_i - 1) runs on side stream i behind
    // `ready` and yields the partial output of blocks (f + 2) T_i .. (f + 3) T_i - 1 into plane slots (f % 2) T_i ..; the head waits for
    // done[i][f % 2] before block (f + 2) T_i. No slot is overwritten while it is still being read:
    //   - input ring: the head rewrites the slot of block b at block b + 2 T_n >= (f + 2) T_i, i.e. after its wait for the reader;
    //   - plane slot (f % 2): its previous readers are the head blocks f T_i .. f T_i + T_i - 1 (frame f - 2's output), all enqueued on
    //     the head's stream before `ready`;
    //   - done[i][f % 2] is re-recorded for frame f + 2 only after the head's wait for frame f has been enqueued.
    // Every kernel sums in a fixed order and none uses atomics, so the bits do not depend on how the streams interleave
    // (NEO_B200_LOWLAT_SYNC runs the same kernels on the head's stream).
    for (size_t i = 0; i < h->levels; ++i) {
        size_t const ti = h->t[i];
        if ((tb + 1) % ti != 0) { continue; }
        size_t const f      = tb / ti;
        cudaStream_t const ls = h->sync ? st : h->side[i];
        if (!h->sync) {
            NEO_CUDA_TRY(cudaEventRecord(h->ready[i], st));
            NEO_CUDA_TRY(cudaStreamWaitEvent(ls, h->ready[i], 0));
        }
        conv_engine<T>& e = s.level[i];
        NEO_TRY(e.forward(s.in_ring.template as<T>() + ((f * ti) % h->ring_blocks) * B, ring_stride, ti, ls));
        NEO_TRY(e.inverse(static_cast<cx<T> const*>(e.acc_r()), 0, 1, s.plane[i].template as<T>() + (f % 2) * ti * B, 2 * ti * B, 0, C, ti, ls));
        if (!h->sync) { NEO_CUDA_TRY(cudaEventRecord(h->done[i][f & 1], ls)); }
    }
    return NEO_B200_OK;
}

template<typename T>
int lowlat_process(neo_b200_lowlat* h, void const* in, void* out, size_t blocks, int memspace)
{
    lowlat_state<T>& s   = lowlat_of<T>(h);
    cudaStream_t const st = h->stream.stream;
    size_t const B = h->cfg.block, stride = blocks * B, bytes = h->cfg.channels * stride * sizeof(T);
    T const* din = static_cast<T const*>(in);
    T* dout      = static_cast<T*>(out);
    if (memspace == NEO_B200_HOST) {
        NEO_TRY(s.stage_in.reserve(bytes));
        NEO_TRY(s.stage_out.reserve(bytes));
        NEO_CUDA_TRY(cudaMemcpyAsync(s.stage_in.ptr, in, bytes, cudaMemcpyHostToDevice, st));
        din  = s.stage_in.template as<T>();
        dout = s.stage_out.template as<T>();
    }
    for (size_t b = 0; b < blocks; ++b) { NEO_TRY(lowlat_block<T>(h, din + b * B, stride, dout + b * B, stride)); }
    if (memspace == NEO_B200_HOST) {
        NEO_CUDA_TRY(cudaMemcpyAsync(out, dout, bytes, cudaMemcpyDeviceToHost, st));
        NEO_CUDA_TRY(cudaStreamSynchronize(st));
    }
    return NEO_B200_OK;
}

}  // namespace
}  // namespace neo_b200

extern "C" {

int neo_b200_lowlat_layout(neo_b200_lowlat_config const* config, size_t* levels, size_t frame_blocks[4], size_t ranges[5][2])
{
    if (levels == nullptr || frame_blocks == nullptr || ranges == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    return lowlat_resolve(config, levels, frame_blocks, ranges);
}

int neo_b200_lowlat_create(neo_b200_lowlat** handle, neo_b200_lowlat_config const* config)
{
    if (handle == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    *handle = nullptr;
    auto p  = std::unique_ptr<neo_b200_lowlat>(new (std::nothrow) neo_b200_lowlat{});
    if (!p) { return fail(NEO_B200_ERR_ALLOC, "out of host memory"); }
    NEO_TRY(lowlat_resolve(config, &p->levels, p->t, p->ranges));
    p->cfg         = *config;
    p->ring_blocks = p->levels > 0 ? 2 * p->t[p->levels - 1] : 1;
    p->sync        = std::getenv("NEO_B200_LOWLAT_SYNC") != nullptr;
    int const logb = int(log2_exact(config->block));
    p->fused       = logb >= 6 && logb <= (config->dtype == NEO_B200_F32 ? 12 : 11) && std::getenv("NEO_B200_LOWLAT_UNFUSED") == nullptr;
    NEO_TRY(require_device());
    NEO_CUDA_TRY(cudaGetDevice(&p->device));
    // the head is due every block, so its stream has the highest priority; smaller levels (due sooner) above larger ones
    int least = 0, greatest = 0;
    NEO_CUDA_TRY(cudaDeviceGetStreamPriorityRange(&least, &greatest));
    NEO_CUDA_TRY(cudaStreamCreateWithPriority(&p->stream.stream, cudaStreamNonBlocking, greatest));
    p->stream.owned = true;
    for (size_t i = 0; i < p->levels; ++i) {
        int const prio = std::min(least, greatest + 1 + int(i));
        NEO_CUDA_TRY(cudaStreamCreateWithPriority(&p->side[i], cudaStreamNonBlocking, prio));
        for (cudaEvent_t* ev : {&p->ready[i], &p->done[i][0], &p->done[i][1]}) { NEO_CUDA_TRY(cudaEventCreateWithFlags(ev, cudaEventDisableTiming)); }
    }
    NEO_TRY(config->dtype == NEO_B200_F32 ? lowlat_init<float>(p.get()) : lowlat_init<double>(p.get()));
    NEO_CUDA_TRY(cudaStreamSynchronize(p->stream.stream));
    *handle = p.release();
    return NEO_B200_OK;
}

void neo_b200_lowlat_destroy(neo_b200_lowlat* handle) { delete handle; }

extern "C++" template<typename T>
int lowlat_set_filter_impl(neo_b200_lowlat* h, void const* H, void const* ir, size_t taps, int memspace)
{
    lowlat_state<T>& s   = lowlat_of<T>(h);
    cudaStream_t const st = h->stream.stream;
    NEO_TRY(h->sync_all());
    h->has_filter = false;
    if (ir != nullptr) {
        NEO_TRY(s.head.set_impulse(ir, taps, memspace, st));
        for (size_t i = 0; i < h->levels; ++i) { NEO_TRY(s.level[i].set_impulse(ir, taps, memspace, st)); }
    } else {
        NEO_TRY(s.head.set_filter(H, memspace, st));
        for (size_t i = 0; i < h->levels; ++i) { NEO_TRY(s.level[i].set_filter(H, memspace, st)); }
    }
    NEO_TRY(lowlat_clear<T>(h));
    h->has_filter = true;
    return NEO_B200_OK;
}

int neo_b200_lowlat_set_filter(neo_b200_lowlat* handle, void const* H, int memspace)
{
    if (handle == nullptr || H == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    NEO_CUDA_TRY(cudaSetDevice(handle->device));
    if (handle->cfg.dtype == NEO_B200_F32) { return lowlat_set_filter_impl<float>(handle, H, nullptr, 0, memspace); }
    return lowlat_set_filter_impl<double>(handle, H, nullptr, 0, memspace);
}

int neo_b200_lowlat_set_impulse(neo_b200_lowlat* handle, void const* ir, size_t taps, int memspace)
{
    if (handle == nullptr || ir == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (taps < handle->cfg.block) { return fail(NEO_B200_ERR_INVALID, "impulse response shorter than one block"); }
    if (neo_b200_num_partitions(taps, handle->cfg.block) != handle->cfg.partitions) {
        return fail(NEO_B200_ERR_INVALID, "taps=%zu gives %zu partitions, handle was created for %zu", taps,
                    neo_b200_num_partitions(taps, handle->cfg.block), handle->cfg.partitions);
    }
    NEO_CUDA_TRY(cudaSetDevice(handle->device));
    if (handle->cfg.dtype == NEO_B200_F32) { return lowlat_set_filter_impl<float>(handle, nullptr, ir, taps, memspace); }
    return lowlat_set_filter_impl<double>(handle, nullptr, ir, taps, memspace);
}

int neo_b200_lowlat_reset(neo_b200_lowlat* handle)
{
    if (handle == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    NEO_CUDA_TRY(cudaSetDevice(handle->device));
    NEO_TRY(handle->sync_all());
    return handle->cfg.dtype == NEO_B200_F32 ? lowlat_clear<float>(handle) : lowlat_clear<double>(handle);
}

int neo_b200_lowlat_process(neo_b200_lowlat* handle, void const* in, void* out, size_t blocks, int memspace)
{
    if (handle == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (!handle->has_filter) { return fail(NEO_B200_ERR_INVALID, "no filter set"); }
    if (in == nullptr || out == nullptr) { return fail(NEO_B200_ERR_INVALID, "null buffer"); }
    if (blocks == 0) { return fail(NEO_B200_ERR_INVALID, "blocks must be >= 1"); }
    NEO_CUDA_TRY(cudaSetDevice(handle->device));
    if (handle->cfg.dtype == NEO_B200_F32) { return lowlat_process<float>(handle, in, out, blocks, memspace); }
    return lowlat_process<double>(handle, in, out, blocks, memspace);
}

int neo_b200_lowlat_set_stream(neo_b200_lowlat* handle, void* cuda_stream)
{
    if (handle == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    NEO_CUDA_TRY(cudaSetDevice(handle->device));
    NEO_CUDA_TRY(cudaStreamSynchronize(handle->stream.stream));  // work already enqueued stays ordered before the new stream's
    handle->stream.adopt(cuda_stream);
    return NEO_B200_OK;
}

int neo_b200_lowlat_synchronize(neo_b200_lowlat* handle)
{
    if (handle == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    NEO_CUDA_TRY(cudaSetDevice(handle->device));
    return handle->sync_all();
}

size_t neo_b200_lowlat_device_bytes(neo_b200_lowlat const* handle)
{
    if (handle == nullptr) { return 0; }
    return handle->cfg.dtype == NEO_B200_F32 ? handle->f32.device_bytes(handle->levels) : handle->f64.device_bytes(handle->levels);
}

}  // extern "C"
