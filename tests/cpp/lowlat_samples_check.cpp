// lowlat_samples_check.cpp -- a plugin host's loop through neo::b200::low_latency_convolver::process: one convolver per channel, each
// called with a buffer size that changes from call to call (seeded, 1 .. 3 blocks, different per channel), in place, every output
// returned by the call that delivers its input. The result must match a float64 direct convolution to 1e-5 relative L2 per channel.
// One call per channel also goes through a strided view. Prints "lowlat samples ok" on success.
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
using strided = stdex::mdspan<T, stdex::dextents<std::size_t, 1>, stdex::layout_stride>;
template<typename T>
using mat = stdex::mdspan<T, stdex::dextents<std::size_t, 2>>;

static auto noise(std::size_t n, unsigned seed) -> std::vector<float>
{
    auto rng  = std::mt19937{seed};
    auto dist = std::uniform_real_distribution<float>{-1.0F, 1.0F};
    auto v    = std::vector<float>(n);
    for (auto& x : v) { x = dist(rng); }
    return v;
}

auto main() -> int
{
    std::size_t const channels = 2, block = 128, taps = 20 * 128 - 37, samples = 48 * 128;
    try {
        auto impulse = noise(channels * taps, 21);
        neo::b200::detail::check(neo_b200_normalize_impulse(impulse.data(), channels, taps, NEO_B200_F32, NEO_B200_HOST));
        auto const parts = neo_b200_num_partitions(taps, block);
        auto partitions  = std::vector<std::complex<float>>(channels * parts * (block + 1));
        neo::b200::uniform_partition(impulse.data(), channels, taps, block, partitions.data());
        auto const signal = noise(channels * samples, 23);
        for (std::size_t c = 0; c < channels; ++c) {
            auto convolver = neo::b200::low_latency_convolver<std::complex<float>>{std::vector<std::size_t>{2, 4}};
            convolver.filter(mat<std::complex<float> const>{&partitions[c * parts * (block + 1)], parts, block + 1});
            auto rng  = std::mt19937{unsigned(31 + c)};
            auto size = std::uniform_int_distribution<std::size_t>{1, 3 * block};
            auto out  = std::vector<float>(signal.begin() + std::ptrdiff_t(c * samples), signal.begin() + std::ptrdiff_t((c + 1) * samples));
            std::size_t calls = 0;
            for (std::size_t i = 0; i < samples; ++calls) {
                auto const n = std::min(samples - i, calls == 0 ? std::size_t(1) : size(rng));
                if (calls == 3) {  // every other sample of a scratch buffer: the facade stages the strided view
                    auto scratch = std::vector<float>(2 * n);
                    for (std::size_t k = 0; k < n; ++k) { scratch[2 * k] = out[i + k]; }
                    auto const map = stdex::layout_stride::mapping<stdex::dextents<std::size_t, 1>>{stdex::dextents<std::size_t, 1>{n},
                                                                                                  stdex::array<std::size_t, 1>{2}};
                    convolver.process(strided<float>{scratch.data(), map});
                    for (std::size_t k = 0; k < n; ++k) { out[i + k] = scratch[2 * k]; }
                } else {
                    convolver.process(vec<float>{out.data() + i, n});
                }
                i += n;
            }
            double num = 0, den = 0;
            for (std::size_t t = 0; t < samples; ++t) {
                double want = 0;
                for (std::size_t k = 0; k < taps && k <= t; ++k) { want += double(impulse[c * taps + k]) * double(signal[c * samples + t - k]); }
                num += (double(out[t]) - want) * (double(out[t]) - want);
                den += want * want;
            }
            double const rel = std::sqrt(num / den);
            std::printf("channel %zu: %zu calls, relative L2 against float64 direct convolution %.3e\n", c, calls, rel);
            if (!(rel <= 1e-5)) { return 1; }
        }
        std::printf("lowlat samples ok\n");
    } catch (std::exception const& e) {
        std::fprintf(stderr, "lowlat_samples_check: %s\n", e.what());
        return 1;
    }
    return 0;
}
