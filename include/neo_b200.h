/* neo_b200.h -- C ABI of the B200-native FFT / partitioned-convolution backend for neo-sonar/neo-dsp.
 *
 * The reference has no FFI: its backend seam is a compile-time alias over C++ "plan" / "convolver" duck types
 * (src/neo/fft/fft.hpp:36-52, src/neo/fft/rfft.hpp:15-23, src/neo/convolution/dense_convolver.hpp:20-41).
 * This header is what one more backend behind those aliases binds to; the C++ facade that satisfies the duck types
 * on top of it is include/neo_b200.hpp, and INTEGRATION.md shows the alias branches a maintainer adds.
 *
 * Conventions
 *   - complex data is interleaved [re, im] (layout of std::complex<T> and neo::scalar_complex<T>,
 *     src/neo/complex/scalar_complex.hpp:113);
 *   - `dtype` names the REAL element type (NEO_B200_F32 / NEO_B200_F64);
 *   - transforms are UNNORMALISED in both directions, like every reference plan (c2c_dit2_plan.hpp:84-95,
 *     fallback_rfft_plan.hpp:39-55); forward is exp(-2 pi i nk/N) (fft/direction.hpp:8-12);
 *   - `memspace` says where in/out live. HOST: any host memory; the call returns when the result is in `out`. Transform plans and
 *     short convolver calls copy straight from / to the caller's pointer (pinned memory gets DMA speed, pageable memory the
 *     driver's own staging). Convolver calls of >= 4 blocks on a diagonal bank are cut into channel groups and pipelined over
 *     three streams (H2D of group g+1 and D2H of group g-1 overlap the kernels of group g); page-locked caller memory is used as it
 *     is, pageable memory is staged through two pinned chunks per direction by the calling thread and a few helper threads.
 *     DEVICE: buffers are used in place, the work is enqueued on the handle's stream and the call returns immediately (use
 *     *_synchronize or the stream);
 *   - every function returns a neo_b200_status (0 = ok); neo_b200_last_error() gives the message of the last
 *     failure on the calling thread. The C++ facade turns failures of create/set_filter into std::runtime_error,
 *     which is what the reference throws from plan construction (c2c_dit2_plan.hpp:98-104, backend/ipp.hpp:30-51);
 *   - handles are not re-entrant; distinct handles are independent (the reference's plans hold mutable scratch too);
 *   - there is NO CPU fallback: without a usable sm_100 device every compute entry point fails with
 *     NEO_B200_ERR_CUDA.
 */
#ifndef NEO_B200_H
#define NEO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
    #define NEO_B200_API __declspec(dllexport)
#else
    #define NEO_B200_API __attribute__((visibility("default")))
#endif

typedef enum neo_b200_status
{
    NEO_B200_OK              = 0,
    NEO_B200_ERR_INVALID     = 1, /* bad argument (null handle, extent mismatch, ...) */
    NEO_B200_ERR_UNSUPPORTED = 2, /* e.g. order > max_order: the reference throws std::runtime_error here */
    NEO_B200_ERR_CUDA        = 3, /* CUDA runtime failure / no device */
    NEO_B200_ERR_ALLOC       = 4
} neo_b200_status;

typedef enum neo_b200_dtype
{
    NEO_B200_F32 = 0,
    NEO_B200_F64 = 1
} neo_b200_dtype;

/* src/neo/fft/direction.hpp:8-12 */
typedef enum neo_b200_direction
{
    NEO_B200_FORWARD  = -1,
    NEO_B200_BACKWARD = 1
} neo_b200_direction;

typedef enum neo_b200_memspace
{
    NEO_B200_HOST   = 0,
    NEO_B200_DEVICE = 1
} neo_b200_memspace;

/* ---- library ------------------------------------------------------------------------------------------------- */
NEO_B200_API const char* neo_b200_last_error(void);
NEO_B200_API const char* neo_b200_version(void);
NEO_B200_API int neo_b200_device_count(void);                /* number of CUDA devices, 0 when none */
NEO_B200_API int neo_b200_set_device(int device);            /* device used by handles created afterwards on this thread */
NEO_B200_API int neo_b200_kernel_launches(uint64_t* count);  /* kernels launched by this library since load */

/* ---- c2c plan: replaces neo::fft::fft_plan<Complex> == c2c_dit2_plan (fft/reference/c2c_dit2_plan.hpp:22-104) ---- */
typedef struct neo_b200_fft_plan neo_b200_fft_plan;

/* ctor `Plan(from_order, order)` (c2c_dit2_plan.hpp:55-56). order > max_order -> NEO_B200_ERR_UNSUPPORTED. */
NEO_B200_API int neo_b200_fft_plan_create(neo_b200_fft_plan** plan, size_t order, int dtype);
NEO_B200_API void neo_b200_fft_plan_destroy(neo_b200_fft_plan* plan);
NEO_B200_API size_t neo_b200_fft_plan_order(neo_b200_fft_plan const* plan); /* c2c_dit2_plan.hpp:71-75 */
NEO_B200_API size_t neo_b200_fft_plan_size(neo_b200_fft_plan const* plan);  /* c2c_dit2_plan.hpp:77-81 */
NEO_B200_API size_t neo_b200_fft_max_order(void);                           /* c2c_dit2_plan.hpp:59-62: 27 */

/* `plan(x, dir)` (c2c_dit2_plan.hpp:84-95) on `batch` contiguous transforms [batch][size]; in == out is in place,
 * otherwise out-of-place (the optional 3-argument overload looked up by fft/fft.hpp:65,84). */
NEO_B200_API int neo_b200_fft_exec(neo_b200_fft_plan* plan, void const* in, void* out, size_t batch, int direction, int memspace);

/* the same on split-complex data (neo::split_complex, complex/split_complex.hpp:10): separate [batch][size] real and imaginary
 * planes; replaces neo::fft::split_fft_plan<Float> (fft/fallback/fallback_split_fft_plan.hpp:16-137). in == out planes allowed. */
NEO_B200_API int neo_b200_fft_exec_split(neo_b200_fft_plan* plan, void const* re_in, void const* im_in, void* re_out, void* im_out,
                                         size_t batch, int direction, int memspace);

/* one transform over a strided rank-1 view (strides in complex elements; layout_stride mdspan, fft_test.cpp:114-128);
 * HOST memory only: staged through a contiguous buffer like backend/ipp.hpp:150-158 */
NEO_B200_API int neo_b200_fft_exec_strided(
    neo_b200_fft_plan* plan, void const* in, ptrdiff_t in_stride, void* out, ptrdiff_t out_stride, int direction);

NEO_B200_API int neo_b200_fft_plan_set_stream(neo_b200_fft_plan* plan, void* cuda_stream);
NEO_B200_API int neo_b200_fft_plan_synchronize(neo_b200_fft_plan* plan);

/* ---- dft plan: replaces neo::fft::dft_plan<Complex> == fallback_dft_plan (fft/dft.hpp:28-30,
 *      fft/fallback/fallback_dft_plan.hpp:24-96): complex transform of ANY size > 0 through Bluestein's chirp-z on a
 *      power-of-two transform of next_order(2*size+1); unnormalised in both directions like the reference. -------- */
typedef struct neo_b200_dft_plan neo_b200_dft_plan;

/* `dft_plan{size}` (fallback_dft_plan.hpp:29); dtype = precision of the complex elements (F32 -> complex<float>) */
NEO_B200_API int neo_b200_dft_plan_create(neo_b200_dft_plan** plan, size_t size, int dtype);
NEO_B200_API void neo_b200_dft_plan_destroy(neo_b200_dft_plan* plan);
NEO_B200_API size_t neo_b200_dft_plan_size(neo_b200_dft_plan const* plan);
/* `plan(x, dir)` (fallback_dft_plan.hpp:48-82) for `batch` contiguous rows of `size` interleaved complex; in == out allowed */
NEO_B200_API int neo_b200_dft_exec(neo_b200_dft_plan* plan, void const* in, void* out, size_t batch, int direction, int memspace);
NEO_B200_API int neo_b200_dft_plan_set_stream(neo_b200_dft_plan* plan, void* cuda_stream);

/* ---- fft_convolver: replaces neo::convolution::fft_convolver<Float> (convolution/fft_convolver.hpp:18-93), mode::full: one-shot
 *      linear convolution of signal[signal_size] with patch[patch_size] through zero padded real transforms of
 *      bit_ceil(signal_size + patch_size - 1) points; `batch` independent (signal, patch) pairs per call. ---------------------- */
typedef struct neo_b200_fft_convolver neo_b200_fft_convolver;

NEO_B200_API int neo_b200_fft_convolver_create(neo_b200_fft_convolver** conv, size_t signal_size, size_t patch_size, int dtype);
NEO_B200_API void neo_b200_fft_convolver_destroy(neo_b200_fft_convolver* conv);
NEO_B200_API size_t neo_b200_fft_convolver_output_size(neo_b200_fft_convolver const* conv);
/* `convolver(signal, patch, output)` (fft_convolver.hpp:39-54): signal [batch][signal_size], patch [batch][patch_size] ->
 * out [batch][signal_size + patch_size - 1] reals */
NEO_B200_API int neo_b200_fft_convolver_exec(
    neo_b200_fft_convolver* conv, void const* signal, void const* patch, void* out, size_t batch, int memspace);

/* ---- dct2 plan: replaces neo::fft::fallback_dct2_plan<Float> (fft/dct.hpp:24-68): unnormalised type-2 DCT of 2^order reals
 *      (scipy.fft.dct(x, type=2), dct_test.cpp:24-39) through one complex transform of the same size. Order 0 is undefined in
 *      the reference (its order-0 c2c plan reads past the buffer) and yields 2*x[0] here. ------------------------------------- */
typedef struct neo_b200_dct2_plan neo_b200_dct2_plan;

NEO_B200_API int neo_b200_dct2_plan_create(neo_b200_dct2_plan** plan, size_t order, int dtype);
NEO_B200_API void neo_b200_dct2_plan_destroy(neo_b200_dct2_plan* plan);
NEO_B200_API size_t neo_b200_dct2_plan_order(neo_b200_dct2_plan const* plan);
NEO_B200_API size_t neo_b200_dct2_plan_size(neo_b200_dct2_plan const* plan);
/* `plan(x)` (dct.hpp:36-63) for `batch` contiguous rows of 2^order reals; in == out allowed (the reference is in place) */
NEO_B200_API int neo_b200_dct2_exec(neo_b200_dct2_plan* plan, void const* in, void* out, size_t batch, int memspace);
NEO_B200_API int neo_b200_dct2_plan_set_stream(neo_b200_dct2_plan* plan, void* cuda_stream);

/* ---- rfft plan: replaces neo::fft::rfft_plan<Float, Complex> == fallback_rfft_plan
 *      (fft/fallback/fallback_rfft_plan.hpp:15-61) ---------------------------------------------------------------- */
typedef struct neo_b200_rfft_plan neo_b200_rfft_plan;

NEO_B200_API int neo_b200_rfft_plan_create(neo_b200_rfft_plan** plan, size_t order, int dtype);
NEO_B200_API void neo_b200_rfft_plan_destroy(neo_b200_rfft_plan* plan);
NEO_B200_API size_t neo_b200_rfft_plan_order(neo_b200_rfft_plan const* plan);
NEO_B200_API size_t neo_b200_rfft_plan_size(neo_b200_rfft_plan const* plan);

/* r2c `plan(real_in, complex_out)` (fallback_rfft_plan.hpp:28-36): in [batch][N] reals -> out [batch][N/2+1] complex */
NEO_B200_API int neo_b200_rfft_exec(neo_b200_rfft_plan* plan, void const* in, void* out, size_t batch, int memspace);

/* c2r `plan(complex_in, real_out)` (fallback_rfft_plan.hpp:39-55): in [batch][in_row_len] complex of which the
 * first N/2+1 per row are used (callers may hand N-long rows, overlap_save.hpp:57,107) -> out [batch][N] reals.
 * UNNORMALISED; the imaginary parts of bins 0 and N/2 do not influence the result (the reference takes .real()). */
NEO_B200_API int neo_b200_irfft_exec(
    neo_b200_rfft_plan* plan, void const* in, size_t in_row_len, void* out, size_t batch, int memspace);

NEO_B200_API int neo_b200_rfft_plan_set_stream(neo_b200_rfft_plan* plan, void* cuda_stream);
NEO_B200_API int neo_b200_rfft_plan_synchronize(neo_b200_rfft_plan* plan);

/* ---- index tables: bit-exact with the reference ------------------------------------------------------------------ */
/* bitrevorder_plan's table (fft/reference/bitrevorder.hpp:65-75): out[i] = reverse_bits(i, order), 2^order entries */
NEO_B200_API int neo_b200_bitrev_table(size_t order, uint32_t* out);
/* permutation applied by digitrevorder_plan<radix> (fft/reference/digitrevorder.hpp:13-48) to iota(size) */
NEO_B200_API int neo_b200_digitrev_perm(size_t radix, size_t size, uint32_t* out);
/* fdl_index (convolution/fdl_index.hpp:24-36): for each of `calls` blocks the write position and the `parts`
 * (fdl row, filter row) pairs; evaluated with the indexer the MAC kernel uses. pairs: [calls][parts][2] */
NEO_B200_API int neo_b200_fdl_index_sequence(size_t parts, size_t calls, uint32_t* write_pos, uint32_t* pairs);
/* neo::convolution::compressed_fdl<FloatComplex, IntComplex> (convolution/compressed_fdl.hpp:17-52): a delay line of `rows` rows
 * of `cols` complex bins kept on the device as int8 or int16 complex (bits = 8 / 16; a quarter / half of the float32 bytes).
 * insert (:36-48) stores (int) lround(part * (float) max) for every real and imaginary part, max = 127 / 32767 -- the reference's
 * integers, bit for bit (parts are expected in [-1, 1], as there); row = `fdl[index]` through compressed_accessor
 * (container/compressed_accessor.hpp:27-45): (Float) q * (1 / max). dtype: NEO_B200_F32 / F64 of the complex rows handed in and out;
 * raw: the stored integers of a row ([cols][2] int8_t or int16_t) to HOST memory. */
typedef struct neo_b200_compressed_fdl neo_b200_compressed_fdl;
NEO_B200_API int neo_b200_compressed_fdl_create(neo_b200_compressed_fdl** fdl, size_t rows, size_t cols, int dtype, int bits);
NEO_B200_API void neo_b200_compressed_fdl_destroy(neo_b200_compressed_fdl* fdl);
NEO_B200_API int neo_b200_compressed_fdl_insert(neo_b200_compressed_fdl* fdl, void const* row, size_t index, int memspace);
NEO_B200_API int neo_b200_compressed_fdl_row(neo_b200_compressed_fdl* fdl, size_t index, void* out, int memspace);
NEO_B200_API int neo_b200_compressed_fdl_raw(neo_b200_compressed_fdl* fdl, size_t index, void* out_host);
/* number of partitions of an L-tap impulse response at block size B (fft/stft.hpp:21-25, overlap 0): ceil(L/B) */
NEO_B200_API size_t neo_b200_num_partitions(size_t taps, size_t block);
/* fft/order.hpp:33-39 */
NEO_B200_API size_t neo_b200_next_order(size_t size);

/* ---- filter preparation: replaces neo::convolution::uniform_partition (convolution/uniform_partition.hpp:13-26 ->
 *      fft/stft.hpp:58-99) ------------------------------------------------------------------------------------------ */
/* ir [channels][taps] reals -> out [channels][P][block+1] complex, P = neo_b200_num_partitions(taps, block); unscaled.
 * block must be a power of two (overlap_save.hpp:53 vs stft.hpp:104 agree only then) and taps >= block. */
NEO_B200_API int neo_b200_uniform_partition(
    void const* ir, size_t channels, size_t taps, size_t block, void* out, int dtype, int memspace);

/* neo::convolution::normalize_impulse (convolution/normalize_impulse.hpp:13-33, algorithm/normalize_energy.hpp:17-44) in place on
 * ir [channels][taps]: every sample is scaled by the smallest per-channel 1/sqrt(sum x^2) (1 for an all-zero channel). */
/* `stft_plan{options}(x)` (fft/stft.hpp:39-109): x [channels][len] reals -> out [channels][frames][n/2+1] complex, n = bit_ceil(
 * transform_size), frames = neo_b200_num_stft_frames(len, frame_size, overlap_size); frame f starts at f*(frame_size-overlap_size),
 * is clipped at the end of the signal, zero padded to n and multiplied by `window` ([n] reals in the same memory space; NULL =
 * rectangular; the reference default is hann_window, math/windowing.hpp:27-41). uniform_partition is the frame = B, transform = 2B,
 * overlap = 0, rectangular case. */
NEO_B200_API size_t neo_b200_num_stft_frames(size_t signal, size_t frame_size, size_t overlap_size);
NEO_B200_API int neo_b200_stft(void const* x, size_t channels, size_t len, size_t frame_size, size_t transform_size,
                               size_t overlap_size, void const* window, void* out, int dtype, int memspace);

NEO_B200_API int neo_b200_normalize_impulse(void* ir, size_t channels, size_t taps, int dtype, int memspace);

/* ---- partitioned convolver: replaces neo::convolution::upols_convolver / upola_convolver
 *      (convolution/uniform_partitioned_convolver.hpp:14-65, dense_convolver.hpp:20-41), one handle = a bank of
 *      channels ------------------------------------------------------------------------------------------------------ */
typedef struct neo_b200_conv neo_b200_conv;

typedef enum neo_b200_conv_kind
{
    NEO_B200_UPOLS = 0, /* overlap-save  (convolution/overlap_save.hpp:85-112) */
    NEO_B200_UPOLA = 1  /* overlap-add   (convolution/overlap_add.hpp:78-107)  */
} neo_b200_conv_kind;

typedef enum neo_b200_conv_topology
{
    NEO_B200_DIAGONAL = 0, /* channel c is convolved with its own filter c: a bank of independent reference convolvers */
    NEO_B200_MATRIX   = 1  /* out[o] = sum_i in[i] * h[o][i]: every (o,i) pair is one reference convolver, summed per o */
} neo_b200_conv_topology;

typedef struct neo_b200_conv_config
{
    int kind;           /* neo_b200_conv_kind */
    int dtype;          /* neo_b200_dtype */
    int topology;       /* neo_b200_conv_topology */
    size_t outputs;     /* output channels */
    size_t inputs;      /* input channels (== outputs for DIAGONAL) */
    size_t block;       /* B, power of two >= 2 */
    size_t partitions;  /* P of the WHOLE filter */
    size_t max_blocks;  /* largest number of blocks T handed to one process call (>= 1) */
    /* partition sharding of long impulse responses across devices: this handle holds partitions
     * [partition_begin, partition_end) of every filter and yields PARTIAL spectra. 0,0 = all partitions. */
    size_t partition_begin;
    size_t partition_end;
    /* 0: direct form. T = 2..512 (power of two): "frame mode" -- every process/forward call carries exactly T blocks and the
     * per-bin sum over partitions is itself evaluated by partitioned overlap-save along block time (frame transforms of length
     * 2T, ceil(P/T) streamed rows): HBM-bound instead of FP32-bound for long filters. Same results up to rounding; max_blocks is
     * forced to T; a sharded handle needs partition_begin % T == 0. */
    size_t frame_blocks;
    /* partition-sharded handles only. 0: the handle receives the live input and reaches back partition_begin blocks into its own
     * delay line of spectra. != 0: the CALLER delays the time-domain input of this handle by partition_begin blocks (zeros first);
     * the handle then pairs its first partition with the newest spectrum and keeps a ring of only its own partitions -- what a
     * multi-device bank does (neo_b200_bank_*), exact because the delay line is linear (fdl_index.hpp:24-36). */
    size_t input_delayed;
} neo_b200_conv_config;

NEO_B200_API int neo_b200_conv_create(neo_b200_conv** conv, neo_b200_conv_config const* config);
NEO_B200_API void neo_b200_conv_destroy(neo_b200_conv* conv);

/* `convolver.filter(partitions)` (uniform_partitioned_convolver.hpp:38-45): deep-copies H and zeroes all state
 * (window, FDL, write position). H: DIAGONAL [outputs][P][block+1], MATRIX [outputs][inputs][P][block+1] complex,
 * P = config.partitions; a sharded handle reads only its own partition range from it. */
NEO_B200_API int neo_b200_conv_set_filter(neo_b200_conv* conv, void const* H, int memspace);
/* `sparse_filter::filter(partitions, sparsity)` (sparse_filter.hpp:25-28, behind sparse_upols_convolver / sparse_upola_convolver,
 * sparse_convolver.hpp:14-22): the filters of a DIAGONAL bank as the CSR matrices neo::csr_matrix builds from the partitions and
 * the caller's sparsity predicate (container/csr_matrix.hpp:64-98): rows = partitions, columns = the block+1 bins, stored elements
 * in row-major order. Filter f owns entries [filter_base[f], filter_base[f+1]) of `values` (complex) and `cols`; row_ptr[f*(P+1)+p]
 * is relative to filter_base[f]; filter_base has outputs+1 entries. All four arrays in HOST memory (the predicate is host code).
 * The device keeps only the stored elements (a bitmap form of the same matrix: 32-bin presence words + packed values) and the MAC
 * touches only them (algorithm/multiply_add.hpp:306-324), skipping the delay-line rows of empty 32-bin segments as well.
 * Direct form only (frame_blocks = 0), unsharded partitions. Zeroes all state like neo_b200_conv_set_filter. */
NEO_B200_API int neo_b200_conv_set_filter_csr(neo_b200_conv* conv, void const* values, uint64_t const* cols, uint64_t const* row_ptr,
                                              uint64_t const* filter_base);
/* same, starting from time-domain impulse responses [filters][taps] (uniform_partition fused in, on the device) */
NEO_B200_API int neo_b200_conv_set_impulse(neo_b200_conv* conv, void const* ir, size_t taps, int memspace);
/* zero window / FDL / write position, keep the filter */
NEO_B200_API int neo_b200_conv_reset(neo_b200_conv* conv);

/* `convolver(block)` (uniform_partitioned_convolver.hpp:48-65) for every channel of the bank, `blocks` consecutive
 * blocks per call: in [inputs][blocks*B] -> out [outputs][blocks*B] reals; in == out allowed for DIAGONAL (the
 * reference is in place). blocks == 1 is the reference's streaming call; blocks > 1 gives identical results to
 * `blocks` successive calls but reuses each filter partition across the blocks. */
NEO_B200_API int neo_b200_conv_process(neo_b200_conv* conv, void const* in, void* out, size_t blocks, int memspace);

/* split form for partition-sharded handles: forward = window + r2c + FDL insert + spectral MAC -> partial spectra
 * [outputs][blocks][B] complex in an internal packed layout (device pointer below; sum across shards elementwise);
 * inverse = c2r + overlap handling of (already summed) spectra for outputs [first, first+count). */
NEO_B200_API int neo_b200_conv_forward(neo_b200_conv* conv, void const* in, size_t blocks, int memspace);
/* the same for the channel range [first, first+count) only (diagonal topology, DEVICE memory, `in` is still the whole
 * [inputs][blocks*B] array): lets a caller overlap the reduction of one channel group with the MAC of the next.
 * The ranges of one call tile the bank in ascending order (the first starts at channel 0, each next one where the previous ended),
 * all with the same `blocks`; pass final != 0 with the range that ends at the last channel (the ring position then advances).
 * Anything else is rejected, and neo_b200_conv_process / _forward are rejected while such a call is in progress. */
NEO_B200_API int neo_b200_conv_forward_range(
    neo_b200_conv* conv, void const* in, size_t blocks, size_t first, size_t count, int final);
/* device pointer of the partial spectra of the most recent forward / forward_range call (the call in progress, if its final
 * range is still to come). A partition-sharded handle alternates between two buffers: the pointer stays valid (not overwritten)
 * until the second-next call, so the reduction of call i may overlap call i+1; ask again AFTER the (first) forward of every call. */
NEO_B200_API int neo_b200_conv_spectra(neo_b200_conv* conv, void** device_ptr, size_t* bytes_per_output_block);
NEO_B200_API int neo_b200_conv_inverse(
    neo_b200_conv* conv, void const* spectra_device, void* out, size_t first, size_t count, size_t blocks, int memspace);

/* the chunk step of neo::convolution::overlap_add_convolver == upola_convolver_v2 (convolution/overlap_add_convolver.hpp:85-132), which
 * accepts calls of any length >= one block and therefore calls that END INSIDE a block: `window` [channels][2B] reals is transformed AS
 * IT STANDS (:92; after a partial chunk it holds the previous inverse transform's output with new samples written over part of it), its
 * spectrum replaces the newest delay-line row (:94), all partitions are accumulated (:96-111), and the inverse transform scaled by 1/2B
 * comes back in `y` [channels][2B] (:114-115). commit != 0: the chunk completed a block and the delay line advances (:122-131). The
 * caller keeps window, overlap and input position, as the reference object does (include/neo_b200.hpp: overlap_add_convolver).
 * Unsharded overlap-add diagonal banks in the direct form. */
NEO_B200_API int neo_b200_conv_process_window(neo_b200_conv* conv, void const* window, void* y, int commit, int memspace);
/* the overlap-add tail [outputs][B] a handle carries between neo_b200_conv_process calls (overlap_add.hpp:106): lets a caller move
 * from whole-block calls to the chunk step above without losing state */
NEO_B200_API int neo_b200_conv_tail(neo_b200_conv* conv, void* tail, int memspace);

NEO_B200_API int neo_b200_conv_set_stream(neo_b200_conv* conv, void* cuda_stream);
NEO_B200_API int neo_b200_conv_synchronize(neo_b200_conv* conv);
/* per-phase device time, measured with CUDA events on the handle's stream while enabled: phase_ms[5] = window+r2c+FDL
 * insert, spectral MAC, c2r+overlap, frame transform forward, frame transform inverse (the last two are 0 outside frame
 * mode; summed since the last read; the read synchronises the stream);
 * mac_launches = MAC kernel launches in that span. Measurement aid for benchmarks, no effect on results. */
NEO_B200_API int neo_b200_conv_profile_enable(neo_b200_conv* conv, int enable);
NEO_B200_API int neo_b200_conv_profile_read(neo_b200_conv* conv, double* phase_ms, uint64_t* mac_launches);
/* bytes of device memory held by the handle (filter + FDL + scratch) */
NEO_B200_API size_t neo_b200_conv_device_bytes(neo_b200_conv const* conv);

/* ---- one-block-latency convolver: what upols_convolver computes (overlap-save, diagonal bank), at one block of latency for long
 *      impulse responses, through non-uniform partitioning (Gardner 1995; Garcia 2002). With levels T_1 < ... < T_n (powers of two
 *      in [2, 512], n <= 4) and P partitions:
 *        head     partitions [0, min(2 T_1, P)): direct form, one fused kernel per block for the whole bank;
 *        level i  partitions [2 T_i, 2 T_{i+1}) (the last one ends at P): frame mode with frame_blocks = T_i on its own stream, started
 *                 when a frame of T_i input blocks is complete and due 2 T_i blocks after the frame began -- one frame period of slack.
 *      Levels that would start at or past P are dropped. Results are the reference's up to rounding (a regrouping of the same sum over
 *      partitions), independent of timing: fixed summation order, no atomics; n-block calls give the bits of n one-block calls.
 *      Environment, read at creation: NEO_B200_LOWLAT_SYNC runs the level work on the handle's stream (same bits);
 *      NEO_B200_LOWLAT_UNFUSED runs the head through the direct-form kernels plus a combine kernel (what block sizes outside
 *      2^6 .. 2^12 (float) / 2^11 (double) always use). ----------------------------------------------------------------------- */
typedef struct neo_b200_lowlat neo_b200_lowlat;

typedef struct neo_b200_lowlat_config
{
    int dtype;               /* neo_b200_dtype */
    size_t channels;         /* C, each with its own filter */
    size_t block;            /* B, power of two >= 2 (the single-CTA transform range: 8192 float, 4096 double) */
    size_t partitions;       /* P of the whole filter */
    size_t levels;           /* 0 = library default: T_1 = 8, then x4 while 2 T_i < P */
    size_t frame_blocks[4];  /* T_1 < ... < T_levels */
} neo_b200_lowlat_config;

/* validates `config` and resolves the schedule without touching a device: the live levels, their T, and [begin, end) partition ranges
 * (ranges[0] = head, ranges[1 + i] = level i; unused entries 0) */
NEO_B200_API int neo_b200_lowlat_layout(neo_b200_lowlat_config const* config, size_t* levels, size_t frame_blocks[4], size_t ranges[5][2]);
NEO_B200_API int neo_b200_lowlat_create(neo_b200_lowlat** handle, neo_b200_lowlat_config const* config);
NEO_B200_API void neo_b200_lowlat_destroy(neo_b200_lowlat* handle);
/* H [channels][P][block+1] complex (uniform_partition layout) / ir [channels][taps] reals; both zero all state */
NEO_B200_API int neo_b200_lowlat_set_filter(neo_b200_lowlat* handle, void const* H, int memspace);
NEO_B200_API int neo_b200_lowlat_set_impulse(neo_b200_lowlat* handle, void const* ir, size_t taps, int memspace);
NEO_B200_API int neo_b200_lowlat_reset(neo_b200_lowlat* handle);
/* `convolver(block)` for every channel, `blocks` >= 1 consecutive blocks: in [channels][blocks*B] -> out, in == out allowed. HOST:
 * returns with the result in `out`; DEVICE: enqueued on the handle's stream, level work continues on the handle's side streams. */
NEO_B200_API int neo_b200_lowlat_process(neo_b200_lowlat* handle, void const* in, void* out, size_t blocks, int memspace);
NEO_B200_API int neo_b200_lowlat_set_stream(neo_b200_lowlat* handle, void* cuda_stream);
/* waits for the handle's stream and its side streams */
NEO_B200_API int neo_b200_lowlat_synchronize(neo_b200_lowlat* handle);
NEO_B200_API size_t neo_b200_lowlat_device_bytes(neo_b200_lowlat const* handle);

/* ---- multi-GPU bank: one convolver bank spread over the GPUs of one box -----------------------------------------------------------
 * What a caller of the reference does with N host threads -- one private convolver per channel
 * (convolution/uniform_partitioned_convolver.hpp:28-34; extra/cli/src/convolver.cpp:37-40 builds one per channel) -- and, for one very
 * long impulse response, what the linearity of the delay line allows (convolution/fdl_index.hpp:24-36: partition p pairs with the
 * spectrum of p blocks ago): N = channel_groups x partition_shards ranks, rank = group * partition_shards + shard.
 *   - rank (g, s) holds partitions [lo_s, hi_s) of the filters of channel group g (matrix topology: OUTPUT channel group g) and yields
 *     partial spectra; the partition_shards partial spectra of a group are summed over NVLink and every rank finishes (c2r + overlap)
 *     1/N of the bank's output rows;
 *   - every rank moves only 1/N of the input rows and 1/N of the output rows across ITS host link; ranks that need the same input
 *     rows exchange them over NVLink;
 *   - results are those of the single-device handle up to float rounding of the split sum (same tolerance as the reference parity).
 * Two ways to build it:
 *   neo_b200_bank_create       every rank lives in the calling process (a C++ host with N GPUs); the devices exchange data through
 *                              peer-mapped memory and the reduction is fused into the c2r kernel. The same device may be named
 *                              more than once.
 *   neo_b200_bank_create_rank  one rank per process (torchrun / MPI); data exchange through NCCL (ncclAllGather of input rows,
 *                              ncclReduceScatter of partial spectra), loaded at run time from libnccl.so.2 (or $NEO_B200_NCCL_LIB).
 *                              Rank 0 calls neo_b200_bank_unique_id and hands the 128 bytes to every rank out of band.
 * Row pointers: `in_rows[l]` / `out_rows[l]` belong to LOCAL rank l (0 .. neo_b200_bank_local_ranks-1) and point at the rows that rank
 * moves: [in_count][blocks*B] / [out_count][blocks*B] reals, rows in_first.. / out_first.. of the bank (neo_b200_bank_local_rank).
 * With every rank local and one [channels][blocks*B] array, in_rows[l] = array + in_first_l * blocks * B. HOST memory should be pinned
 * for the copies to overlap; DEVICE pointers must live on the rank's own device, and their contents must be complete when submit is
 * called (the bank works on its own streams and does not wait for the caller's).
 * How the partial spectra of a group reach the rank that finishes a channel (environment NEO_B200_BANK_EXCHANGE, read at creation):
 *   dma        (default) every shard's kernels write their partial spectra locally and the copy engines move each owner's rows into
 *              its inbox over NVLink (peer-mapped memory; CUDA IPC mappings between processes, with a one-word ncclAllGather per
 *              step as the cross-process gate); the c2r kernel sums its own rows and its inbox slots -- no SM and no store queue of a
 *              compute kernel is spent on the exchange;
 *   kernel     the fused frame kernel stores the result rows straight into the owners' inboxes (peer stores from inside the kernel);
 *   collective ncclReduceScatter of the partial spectra (rank-per-process banks) / peer loads inside the c2r kernel (devices[] banks).
 * dma, kernel and the peer-load form sum in shard order and give identical bits; ncclReduceScatter sums in NCCL's own order. */
typedef struct neo_b200_bank neo_b200_bank;

typedef struct neo_b200_bank_layout
{
    size_t channel_groups;    /* Gc */
    size_t partition_shards;  /* Gp, at most 8; in frame mode shards start on frame boundaries of the partition axis */
} neo_b200_bank_layout;

typedef struct neo_b200_bank_rank_info
{
    int rank;                 /* global rank = channel_group * partition_shards + partition_shard */
    int device;               /* CUDA device (-1 from neo_b200_bank_layout_info) */
    size_t channel_group, partition_shard;
    size_t group_first, group_count;          /* channels (matrix: outputs) whose filters the rank holds */
    size_t in_first, in_count;                /* input rows the rank brings in */
    size_t out_first, out_count;              /* output rows the rank finishes and returns */
    size_t partition_begin, partition_end;    /* partitions of every filter of the group held by the rank */
    size_t delay_blocks;                      /* frame mode: the rank transforms its input this many blocks late instead of keeping a
                                                 deeper ring of spectra (neo_b200_conv_config::input_delayed) */
} neo_b200_bank_rank_info;

#define NEO_B200_BANK_ID_BYTES 128
NEO_B200_API int neo_b200_bank_unique_id(void* id /* NEO_B200_BANK_ID_BYTES */);
/* config: the WHOLE bank (outputs, inputs, partitions of the whole filter; partition_begin/end = 0). outputs and inputs must be
 * multiples of the number of ranks. */
NEO_B200_API int neo_b200_bank_create(neo_b200_bank** bank, neo_b200_conv_config const* config, neo_b200_bank_layout const* layout,
                                      int const* devices, size_t n_devices);
NEO_B200_API int neo_b200_bank_create_rank(neo_b200_bank** bank, neo_b200_conv_config const* config, neo_b200_bank_layout const* layout,
                                           int device, int rank, int world, void const* unique_id);
NEO_B200_API void neo_b200_bank_destroy(neo_b200_bank* bank);
NEO_B200_API int neo_b200_bank_local_ranks(neo_b200_bank const* bank, size_t* count);
NEO_B200_API int neo_b200_bank_local_rank(neo_b200_bank const* bank, size_t local_index, neo_b200_bank_rank_info* info);
/* the same facts for any rank of a layout, without building anything (lets a launcher prepare each rank's rows and filters) */
NEO_B200_API int neo_b200_bank_layout_info(neo_b200_conv_config const* config, neo_b200_bank_layout const* layout, size_t rank,
                                           neo_b200_bank_rank_info* info);

/* `convolver.filter(...)` for every convolver of the bank (uniform_partitioned_convolver.hpp:38-45). per local rank: the impulse
 * responses / partitions of ITS channel group, all P partitions of them (the rank picks its own range): DIAGONAL [group_count][taps]
 * or [group_count][P][B+1], MATRIX [group_count][inputs][taps] or [group_count][inputs][P][B+1]; HOST, or DEVICE on the rank's device. */
NEO_B200_API int neo_b200_bank_set_impulse(neo_b200_bank* bank, void const* const* ir_per_rank, size_t taps, int memspace);
NEO_B200_API int neo_b200_bank_set_filter(neo_b200_bank* bank, void const* const* h_per_rank, int memspace);
NEO_B200_API int neo_b200_bank_reset(neo_b200_bank* bank);

/* `convolver(block)` for every channel of the bank, `blocks` blocks per call (uniform_partitioned_convolver.hpp:48-65).
 * submit only enqueues; wait returns when the OLDEST outstanding submit has delivered its output rows. Up to three submits may be
 * outstanding (a fourth waits inside submit), so the input copy of step i+2 and the output copy of step i-1 overlap the kernels of
 * step i and both directions of the host link stay busy. In rank-per-process banks every rank must make the same sequence of calls. process = submit + wait until idle. */
NEO_B200_API int neo_b200_bank_submit(neo_b200_bank* bank, void const* const* in_rows, void* const* out_rows, size_t blocks, int memspace);
NEO_B200_API int neo_b200_bank_wait(neo_b200_bank* bank);
NEO_B200_API int neo_b200_bank_process(neo_b200_bank* bank, void const* const* in_rows, void* const* out_rows, size_t blocks, int memspace);

/* device time of a run of steps, CUDA events on the bank's own streams: start waits for outstanding work and records at the head of
 * every local rank's input stream; stop records behind the last submitted step on every output stream, waits, and yields the
 * longest span over the local ranks in milliseconds. */
NEO_B200_API int neo_b200_bank_timer_start(neo_b200_bank* bank);
NEO_B200_API int neo_b200_bank_timer_stop(neo_b200_bank* bank, double* ms);
/* per-phase device time of one local rank (see neo_b200_conv_profile_read) and its device memory */
NEO_B200_API int neo_b200_bank_profile_enable(neo_b200_bank* bank, int enable);
NEO_B200_API int neo_b200_bank_profile_read(neo_b200_bank* bank, size_t local_index, double* phase_ms, uint64_t* mac_launches);
NEO_B200_API size_t neo_b200_bank_device_bytes(neo_b200_bank const* bank, size_t local_index);

#ifdef __cplusplus
}
#endif

#endif /* NEO_B200_H */
