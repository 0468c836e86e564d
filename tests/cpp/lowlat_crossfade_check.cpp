// lowlat_crossfade_check.cpp -- a plugin swapping its impulse response while audio runs, through
// neo::b200::low_latency_convolver::crossfade_to: one convolver per channel, called with a buffer size that changes from call to call
// (seeded, 1 .. 3 blocks), in place; after a few calls the host switches to a second response with a linear crossfade. The result must
// match, to 1e-5 relative L2 per channel, a float64 reference computed here: the direct convolution with the first response before the
// returned start, the second response's from start + fade on, and the linear blend between. Prints "lowlat crossfade ok" on success.
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

static auto noise(std::size_t n, unsigned seed) -> std::vector<float>
{
    auto rng  = std::mt19937{seed};
    auto dist = std::uniform_real_distribution<float>{-1.0F, 1.0F};
    auto v    = std::vector<float>(n);
    for (auto& x : v) { x = dist(rng); }
    return v;
}

static auto direct(std::vector<float> const& ir, std::size_t taps, float const* x, std::size_t t) -> double
{
    double y = 0;
    for (std::size_t k = 0; k < taps && k <= t; ++k) { y += double(ir[k]) * double(x[t - k]); }
    return y;
}

auto main() -> int
{
    std::size_t const channels = 2, block = 128, taps = 20 * 128 - 37, samples = 48 * 128, switch_call = 5, fade = 3 * 128 + 11;
    try {
        auto const parts = neo_b200_num_partitions(taps, block);
        auto const signal = noise(channels * samples, 23);
        for (std::size_t c = 0; c < channels; ++c) {
            std::vector<float> ir[2];
            std::vector<std::complex<float>> H[2];
            for (int r = 0; r < 2; ++r) {
                ir[r] = noise(taps, unsigned(41 + 2 * c + r));
                neo::b200::detail::check(neo_b200_normalize_impulse(ir[r].data(), 1, taps, NEO_B200_F32, NEO_B200_HOST));
                H[r].resize(parts * (block + 1));
                neo::b200::uniform_partition(ir[r].data(), 1, taps, block, H[r].data());
            }
            auto convolver = neo::b200::low_latency_convolver<std::complex<float>>{std::vector<std::size_t>{2, 4}};
            convolver.filter(mat<std::complex<float> const>{H[0].data(), parts, block + 1});
            auto rng  = std::mt19937{unsigned(31 + c)};
            auto size = std::uniform_int_distribution<std::size_t>{1, 3 * block};
            auto out  = std::vector<float>(signal.begin() + std::ptrdiff_t(c * samples), signal.begin() + std::ptrdiff_t((c + 1) * samples));
            float const* x    = signal.data() + c * samples;
            std::size_t calls = 0, start = 0, at = 0;
            for (std::size_t i = 0; i < samples; ++calls) {
                if (calls == switch_call) {
                    start = convolver.crossfade_to(mat<std::complex<float> const>{H[1].data(), parts, block + 1}, fade);
                    at    = i;
                }
                auto const n = std::min(samples - i, size(rng));
                convolver.process(vec<float>{out.data() + i, n});
                i += n;
            }
            if (start < at || start + fade > samples) {
                std::printf("channel %zu: start %zu out of range (switch requested at %zu)\n", c, start, at);
                return 1;
            }
            double num = 0, den = 0;
            for (std::size_t t = 0; t < samples; ++t) {
                double const ya = t < start + fade ? direct(ir[0], taps, x, t) : 0.0;
                double const yb = t >= start ? direct(ir[1], taps, x, t) : 0.0;
                double const g  = t < start ? 0.0 : t >= start + fade ? 1.0 : double(t - start) / double(fade);
                double const want = g == 0.0 ? ya : g == 1.0 ? yb : ya + g * (yb - ya);
                num += (double(out[t]) - want) * (double(out[t]) - want);
                den += want * want;
            }
            double const rel = std::sqrt(num / den);
            std::printf("channel %zu: %zu calls, switch requested at %zu, fade [%zu, %zu), relative L2 against float64 %.3e\n", c, calls, at, start,
                        start + fade, rel);
            if (!(rel <= 1e-5)) { return 1; }
        }
        std::printf("lowlat crossfade ok\n");
    } catch (std::exception const& e) {
        std::fprintf(stderr, "lowlat_crossfade_check: %s\n", e.what());
        return 1;
    }
    return 0;
}
