// TEST INFRASTRUCTURE ONLY - CPU emulator of the uint8-image variants of the sensor kernel bodies.
//
// Same scheme as tests/emu/emu.cpp (kernels.cuh compiled with g++, each barrier phase a loop over the block's thread ids): the
// forward row passes on uint8 images (K1 and the TMA-staged K1s) and the arg-max gather of the backward (K8 tie_term) on a
// uint8 batch, next to their fp32 instantiations in the same library, so tests/test_emulator_u8.py compares the two bodies in
// the same binary.  It is never linked into libb200cam.so and never used by the product.
#include <cstring>
#include <type_traits>
#include <vector>

#include "../../privacy-preserving-vision_b200/csrc/kernels.cuh"

using namespace b200cam;

namespace {

std::vector<float2> make_twiddle(int N) {
    std::vector<float2> tw(N);
    for (int j = 0; j < N; ++j) {
        const double a = -2.0 * M_PI * j / N;
        tw[j] = make_float2(static_cast<float>(cos(a)), static_cast<float>(sin(a)));
    }
    return tw;
}

template <class F>
void grid2(int gx, int gy, int threads, F&& f) {
    for (int y = 0; y < gy; ++y)
        for (int x = 0; x < gx; ++x) {
            HostExec ex{x, y, threads};
            f(ex);
        }
}

template <class F>
int dispatch_n(int N, F&& f) {
    switch (N) {
        case 64: return f(std::integral_constant<int, 64>{});
        case 128: return f(std::integral_constant<int, 128>{});
        case 256: return f(std::integral_constant<int, 256>{});
        case 512: return f(std::integral_constant<int, 512>{});
        case 1024: return f(std::integral_constant<int, 1024>{});
        default: return -1;
    }
}

}  // namespace

extern "C" {

// the value the kernels read for a uint8 byte (compat.cuh to_float(u8)), for all 256 bytes
int emu8_convert(float* out) {
    for (int v = 0; v < 256; ++v) out[v] = to_float(u8{static_cast<unsigned char>(v)});
    return 0;
}

// the forward row pass over `planes` N x N planes: K1 (stream = 0) or the persistent TMA-staged K1s (stream = 1, odd grid),
// on fp32 (u8_in = 0) or uint8 (u8_in = 1) images; init_max / init_count (nullable, [planes/3]) as the sensor forward passes
// them; st [planes][N/2+1][N] complex
int emu8_rows_r2c(int N, int planes, int stream, int u8_in, const void* x, float* st, float* init_max, int* init_count) {
    return dispatch_n(N, [&](auto tag) -> int {
        constexpr int NN_ = decltype(tag)::value;
        using T = Tile<NN_>;
        auto tw = make_twiddle(NN_);
        float2* out = reinterpret_cast<float2*>(st);
        auto go = [&](auto in_tag) {
            using In = decltype(in_tag);
            const RowsR2CParamsT<In> p{static_cast<const In*>(x), out, tw.data(), init_max, init_count};
            if (stream) {
                const int total = (NN_ / T::ROWS) * planes, nctas = 5;
                std::vector<float2> ssmem(RowsStreamSmem<NN_, In>::FLOAT2S);
                grid2(nctas, 1, RowsStreamSmem<NN_, In>::THREADS, [&](HostExec& ex) {
                    rows_r2c_stream_body<NN_>(ex, p, ssmem.data(), total, nctas);
                });
            } else {
                std::vector<float2> smem(RowsR2CSmem<NN_>::FLOAT2S);
                grid2(NN_ / T::ROWS, planes, RowsR2CSmem<NN_>::THREADS, [&](HostExec& ex) { rows_r2c_body<NN_>(ex, p, smem.data()); });
            }
        };
        if (u8_in) go(u8{}); else go(float{});
        return 0;
    });
}

// the arg-max term of the amax backward (K8 tie_term_body) on an fp32 (u8_in = 0) or uint8 (u8_in = 1) batch x [B][3][N][N]:
// gpsf [3][N][N] is updated in place from the ties (tie_count [B], tie_pos [B][MAX_TIES]) weighted by coef [B]
int emu8_tie_term(int N, int B, int u8_in, const void* x, float* gpsf, const int* tie_count, const int* tie_pos, const float* coef) {
    if ((N != 64 && N != 128 && N != 256 && N != 512 && N != 1024) || B < 1) return -1;
    std::vector<float> s_coef(TIE_PASS * MAX_TIES);
    std::vector<int> s_meta(3 * TIE_PASS * MAX_TIES), s_cnt(TIE_PASS + 1);
    const int per_ch = 3;                      // any grid works for the grid-stride body; a small odd one on purpose
    auto go = [&](auto in_tag) {
        using Img = decltype(in_tag);
        const TieTermParamsT<Img> p{gpsf, static_cast<const Img*>(x), tie_count, tie_pos, coef, B, N};
        grid2(per_ch, 3, EW_THREADS, [&](HostExec& ex) { tie_term_body(ex, p, per_ch, s_coef.data(), s_meta.data(), s_cnt.data()); });
    };
    if (u8_in) go(u8{}); else go(float{});
    return 0;
}

}  // extern "C"
