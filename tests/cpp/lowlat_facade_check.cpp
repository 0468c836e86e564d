// lowlat_facade_check.cpp -- the reference CLI's per-channel loop (extra/cli/src/convolver.cpp:25-59: one convolver per channel,
// filter(partitions of that channel), one call per block through a pageable block buffer) run with neo::b200::low_latency_convolver and
// with neo::b200::upols_convolver; the two outputs must agree to 1e-5 relative L2. Prints "lowlat facade ok" on success.
#include "../../include/neo_b200.hpp"

#include <cuda/std/mdspan>

#include <algorithm>
#include <cmath>
#include <complex>
#include <cstdio>
#include <random>
#include <vector>

namespace stdex = cuda::std;
template<typename T>
using vec = stdex::mdspan<T, stdex::dextents<std::size_t, 1>>;
template<typename T>
using mat = stdex::mdspan<T, stdex::dextents<std::size_t, 2>>;
template<typename T>
using cube = stdex::mdspan<T, stdex::dextents<std::size_t, 3>>;

static auto noise(std::size_t n, unsigned seed) -> std::vector<float>
{
    auto rng  = std::mt19937{seed};
    auto dist = std::uniform_real_distribution<float>{-1.0F, 1.0F};
    auto v    = std::vector<float>(n);
    for (auto& x : v) { x = dist(rng); }
    return v;
}

template<typename Convolver>
static auto convolve(mat<float const> signal, cube<std::complex<float> const> partitions, mat<float> output, std::size_t block_size) -> void
{
    auto block_buffer = std::vector<float>(block_size);
    for (std::size_t channel = 0; channel < signal.extent(0); ++channel) {
        auto convolver = Convolver{};
        convolver.filter(mat<std::complex<float> const>{&partitions(channel, 0, 0), partitions.extent(1), partitions.extent(2)});
        for (std::size_t i = 0; i < output.extent(1); i += block_size) {
            std::fill(block_buffer.begin(), block_buffer.end(), 0.0F);
            auto const num_samples = std::min(output.extent(1) - i, block_size);
            std::copy_n(&signal(channel, i), num_samples, block_buffer.begin());
            convolver(vec<float>{block_buffer.data(), block_size});
            std::copy_n(block_buffer.begin(), num_samples, &output(channel, i));
        }
    }
}

auto main() -> int
{
    std::size_t const channels = 2, blocks = 64, block = 256, taps = 40 * 256 - 100;
    try {
        auto impulse = noise(channels * taps, 11);
        neo::b200::detail::check(neo_b200_normalize_impulse(impulse.data(), channels, taps, NEO_B200_F32, NEO_B200_HOST));
        auto const parts = neo_b200_num_partitions(taps, block);
        auto partitions  = std::vector<std::complex<float>>(channels * parts * (block + 1));
        neo::b200::uniform_partition(impulse.data(), channels, taps, block, partitions.data());
        auto const signal = noise(channels * blocks * block, 13);
        auto low = std::vector<float>(signal.size()), direct = std::vector<float>(signal.size());
        auto const sig = mat<float const>{signal.data(), channels, blocks * block};
        auto const H   = cube<std::complex<float> const>{partitions.data(), channels, parts, block + 1};
        convolve<neo::b200::low_latency_convolver<std::complex<float>>>(sig, H, mat<float>{low.data(), channels, blocks * block}, block);
        convolve<neo::b200::upols_convolver<std::complex<float>>>(sig, H, mat<float>{direct.data(), channels, blocks * block}, block);
        double num = 0, den = 0;
        for (std::size_t i = 0; i < low.size(); ++i) {
            num += (double(low[i]) - double(direct[i])) * (double(low[i]) - double(direct[i]));
            den += double(direct[i]) * double(direct[i]);
        }
        double const rel = std::sqrt(num / den);
        std::printf("relative L2 low_latency_convolver vs upols_convolver: %.3e\n", rel);
        if (!(rel <= 1e-5)) { return 1; }
        std::printf("lowlat facade ok\n");
    } catch (std::exception const& e) {
        std::fprintf(stderr, "lowlat_facade_check: %s\n", e.what());
        return 1;
    }
    return 0;
}
