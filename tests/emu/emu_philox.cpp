// TEST INFRASTRUCTURE ONLY - CPU emulator of the Philox sensor read-out (B200CAM_SENSOR_NOISE_PHILOX).
//
// Same scheme as tests/emu/emu.cpp (kernels.cuh compiled with g++, each barrier phase a loop over the block's thread ids): the
// Philox4x32-10 block function, the materialiser body and the normalise body with the Philox epilogue next to its tensor-epilogue
// instantiation, so tests/test_host_philox.py compares them in the same binary.  The host Box-Muller uses the host libm (and a
// sincospi computed in double), so its values are not the device's; the integers are.  Never linked into libb200cam.so.
#include <vector>

#include "../../privacy-preserving-vision_b200/csrc/kernels.cuh"

using namespace b200cam;

namespace {

template <class F>
void grid1(int gx, int threads, F&& f) {
    for (int x = 0; x < gx; ++x) {
        HostExec ex{x, 0, threads};
        f(ex);
    }
}

constexpr int EW_GRID = 7;   // any grid works for the grid-stride bodies; a small odd one on purpose

}  // namespace

extern "C" {

// Philox4x32-10 of n counters ctr[n][4] under keys key[n][2] -> out[n][4]
int emup_philox(const unsigned* ctr, const unsigned* key, unsigned* out, long long n) {
    for (long long i = 0; i < n; ++i) {
        uint32_t c[4] = {ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3]};
        philox4x32_10(c, key[2 * i], key[2 * i + 1]);
        for (int k = 0; k < 4; ++k) out[4 * i + k] = c[k];
    }
    return 0;
}

// b200cam_sensor_noise's body: out[e] = n(e), e < count (count % 4 == 0), seed block {key, first4}
int emup_noise(const unsigned long long* seed_block, float* out, long long count) {
    if (count % 4 != 0) return -1;
    const auto* seed = reinterpret_cast<const b200cam_noise_seed*>(seed_block);
    grid1(EW_GRID, EW_THREADS, [&](HostExec& ex) { philox_noise_body(ex, seed, out, count / 4, EW_GRID); });
    return 0;
}

// the normalise body on y [B][3][N][N] (in place, fp32 out) with the Philox epilogue (seed_block != NULL) or the tensor one
// (noise, nullable); levels <= 0: no quantisation
int emup_normalise(int N, int B, float* y, const float* img_max, int* tie_count, int* tie_pos, const unsigned long long* seed_block,
                   const float* noise, float noise_scale, float levels) {
    const long long n4 = static_cast<long long>(B) * 3 * N * N / 4;
    const auto* seed = reinterpret_cast<const b200cam_noise_seed*>(seed_block);
    const SensorEpilogue epi{noise, noise_scale, levels, seed};
    const NormaliseParams p{y, img_max, tie_count, tie_pos, n4, 3 * N * N / 4, epi};
    grid1(EW_GRID, EW_THREADS, [&](HostExec& ex) {
        if (seed != nullptr)
            normalise_body<float, true>(ex, p, EW_GRID);
        else
            normalise_body(ex, p, EW_GRID);
    });
    return 0;
}

}  // extern "C"
