// conv_crossfade_check.cpp -- a command-line renderer swapping its impulse response mid-file, through
// neo::b200::upols_convolver::crossfade_to: one convolver per channel, called block by block in place as a CLI host's loop does; after a
// few blocks the host switches each channel to a second response with a linear crossfade, then later to a third one. The result must
// match, to 1e-5 relative L2 per channel, a float64 reference computed here: the direct convolution with the current response before the
// returned start, the next response's from start + fade on, and the linear blend between. Prints "conv crossfade ok" on success.
#include "../../include/neo_b200.hpp"

#include <cuda/std/mdspan>

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
    std::size_t const channels = 2, block = 128, taps = 12 * 128 - 37, blocks = 40;
    std::size_t const switch_at[2] = {5, 21}, fades[2] = {3 * 128 + 11, 1};  // calls before which a crossfade is requested
    std::size_t const samples = blocks * block;
    try {
        auto const parts  = neo_b200_num_partitions(taps, block);
        auto const signal = noise(channels * samples, 29);
        for (std::size_t c = 0; c < channels; ++c) {
            std::vector<float> ir[3];
            std::vector<std::complex<float>> H[3];
            for (int r = 0; r < 3; ++r) {
                ir[r] = noise(taps, unsigned(53 + 3 * c + r));
                neo::b200::detail::check(neo_b200_normalize_impulse(ir[r].data(), 1, taps, NEO_B200_F32, NEO_B200_HOST));
                H[r].resize(parts * (block + 1));
                neo::b200::uniform_partition(ir[r].data(), 1, taps, block, H[r].data());
            }
            auto convolver = neo::b200::upols_convolver<std::complex<float>>{};
            convolver.filter(mat<std::complex<float> const>{H[0].data(), parts, block + 1});
            auto out       = std::vector<float>(signal.begin() + std::ptrdiff_t(c * samples), signal.begin() + std::ptrdiff_t((c + 1) * samples));
            float const* x = signal.data() + c * samples;
            std::size_t start[2] = {0, 0};
            for (std::size_t b = 0, k = 0; b < blocks; ++b) {
                if (k < 2 && b == switch_at[k]) {
                    start[k] = convolver.crossfade_to(mat<std::complex<float> const>{H[k + 1].data(), parts, block + 1}, fades[k]);
                    if (start[k] != b * block) {
                        std::printf("channel %zu: crossfade %zu starts at %zu, expected the next sample %zu\n", c, k, start[k], b * block);
                        return 1;
                    }
                    ++k;
                }
                convolver(vec<float>{out.data() + b * block, block});
            }
            double num = 0, den = 0;
            for (std::size_t t = 0; t < samples; ++t) {
                // response r is current before the fade into r + 1 ends
                auto const at = [&](int r) { return direct(ir[r], taps, x, t); };
                double want   = at(0);
                for (int k = 0; k < 2; ++k) {
                    if (t < start[k]) { break; }
                    double const g = t >= start[k] + fades[k] ? 1.0 : double(t - start[k]) / double(fades[k]);
                    double const y = at(k + 1);
                    want           = g == 1.0 ? y : want + g * (y - want);
                }
                num += (double(out[t]) - want) * (double(out[t]) - want);
                den += want * want;
            }
            double const rel = std::sqrt(num / den);
            std::printf("channel %zu: fades [%zu, %zu) and [%zu, %zu), relative L2 against float64 %.3e\n", c, start[0], start[0] + fades[0],
                        start[1], start[1] + fades[1], rel);
            if (!(rel <= 1e-5)) { return 1; }
        }
        std::printf("conv crossfade ok\n");
    } catch (std::exception const& e) {
        std::fprintf(stderr, "conv_crossfade_check: %s\n", e.what());
        return 1;
    }
    return 0;
}
