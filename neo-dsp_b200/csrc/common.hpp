// common.hpp -- host-side plumbing shared by the C-ABI translation units: error reporting, launch accounting,
// device / pinned buffers. No compute here.
#pragma once

#include "../../include/neo_b200.h"

#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <utility>

namespace neo_b200 {

// last error text of the calling thread (neo_b200_last_error)
inline std::string& last_error_slot()
{
    thread_local std::string slot;
    return slot;
}

inline int fail(int status, char const* fmt, ...)
{
    char buf[512];
    va_list args;
    va_start(args, fmt);
    std::vsnprintf(buf, sizeof(buf), fmt, args);
    va_end(args);
    last_error_slot() = buf;
    return status;
}

// every kernel this library launches is counted (bench.py reports it as gpu_launches)
std::atomic<std::uint64_t>& launch_counter();
inline void count_launch(std::uint64_t n = 1) { launch_counter().fetch_add(n, std::memory_order_relaxed); }

#define NEO_CUDA_TRY(expr)                                                                                             \
    do {                                                                                                               \
        cudaError_t const neo_err_ = (expr);                                                                           \
        if (neo_err_ != cudaSuccess) {                                                                                 \
            return ::neo_b200::fail(NEO_B200_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(neo_err_),   \
                                    __FILE__, __LINE__);                                                               \
        }                                                                                                              \
    } while (0)

#define NEO_TRY(...)                                                                                                   \
    do {                                                                                                               \
        int const neo_st_ = (__VA_ARGS__);                                                                                    \
        if (neo_st_ != NEO_B200_OK) { return neo_st_; }                                                                \
    } while (0)

inline int check_launch(char const* what)
{
    cudaError_t const err = cudaGetLastError();
    if (err != cudaSuccess) { return fail(NEO_B200_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(err)); }
    count_launch();
    return NEO_B200_OK;
}

// grow-only device allocation
struct device_buffer
{
    void* ptr{nullptr};
    size_t bytes{0};

    device_buffer() = default;
    device_buffer(device_buffer const&)            = delete;
    device_buffer& operator=(device_buffer const&) = delete;
    ~device_buffer() { release(); }

    void release()
    {
        if (ptr != nullptr) { cudaFree(ptr); }
        ptr   = nullptr;
        bytes = 0;
    }

    int reserve(size_t want)
    {
        if (want <= bytes) { return NEO_B200_OK; }
        release();
        cudaError_t const err = cudaMalloc(&ptr, want);
        if (err != cudaSuccess) {
            ptr = nullptr;
            return fail(NEO_B200_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(err));
        }
        bytes = want;
        return NEO_B200_OK;
    }

    template<typename U>
    U* as() const
    {
        return static_cast<U*>(ptr);
    }

    void swap(device_buffer& o) noexcept
    {
        std::swap(ptr, o.ptr);
        std::swap(bytes, o.bytes);
    }
};

// grow-only pinned host allocation (staging for HOST memspace calls)
struct pinned_buffer
{
    void* ptr{nullptr};
    size_t bytes{0};

    pinned_buffer() = default;
    pinned_buffer(pinned_buffer const&)            = delete;
    pinned_buffer& operator=(pinned_buffer const&) = delete;
    ~pinned_buffer() { release(); }

    void release()
    {
        if (ptr != nullptr) { cudaFreeHost(ptr); }
        ptr   = nullptr;
        bytes = 0;
    }

    int reserve(size_t want)
    {
        if (want <= bytes) { return NEO_B200_OK; }
        release();
        cudaError_t const err = cudaMallocHost(&ptr, want);
        if (err != cudaSuccess) {
            ptr = nullptr;
            return fail(NEO_B200_ERR_ALLOC, "cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(err));
        }
        bytes = want;
        return NEO_B200_OK;
    }
};

// the stream a handle enqueues on: its own non-blocking stream unless the caller supplies one
struct stream_ref
{
    cudaStream_t stream{nullptr};
    bool owned{false};

    int create()
    {
        NEO_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        owned = true;
        return NEO_B200_OK;
    }

    void adopt(void* external)
    {
        if (owned && stream != nullptr) { cudaStreamDestroy(stream); }
        stream = static_cast<cudaStream_t>(external);
        owned  = false;
    }

    ~stream_ref()
    {
        if (owned && stream != nullptr) { cudaStreamDestroy(stream); }
    }
};

inline size_t elem_size(int dtype) { return dtype == NEO_B200_F64 ? sizeof(double) : sizeof(float); }

inline bool is_pow2(size_t x) { return x != 0 && (x & (x - 1)) == 0; }

inline size_t log2_exact(size_t x)
{
    size_t l = 0;
    while ((size_t(1) << l) < x) { ++l; }
    return l;
}

// verifies a usable device exists (no CPU fallback: callers fail loudly otherwise)
int require_device();

}  // namespace neo_b200
