// TEST INFRASTRUCTURE ONLY - CPU emulator of the bf16 variants of the sensor kernel bodies.
//
// Same scheme as tests/emu/emu.cpp (kernels.cuh compiled with g++, each barrier phase a loop over the block's thread ids):
// the bf16 normalise body, the forward row passes on bf16 input (K1 and the TMA-staged K1s), the host rounding rule of
// compat.cuh, and the generic sensor forward / backward with a bf16 sensor image / bf16 upstream gradient next to their fp32
// instantiations - built into one library, so tests/test_emulator_bf16.py compares the two in the same binary.
// It is never linked into libb200cam.so and never used by the product.
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

constexpr int EW_GRID = 7;   // any grid works for the grid-stride bodies; a small odd one on purpose

int accum_chunks(int N, int B) {          // the library sizes this from the device's occupancy; any value works
    const int colgroups = (3 * (N / 2 + 1) + 7) / 8;
    int n = 444 / colgroups;
    if (n > 16) n = 16;
    if (n > B) n = B;
    if (n < 1) n = 1;
    return n;
}

template <int N>
void otf_impl(const float* psf, float2* otf, const float2* tw) {
    using T = Tile<N>;
    std::vector<float2> smem(RowsR2CSmem<N>::FLOAT2S > ColsSmem<N>::FLOAT2S ? RowsR2CSmem<N>::FLOAT2S : ColsSmem<N>::FLOAT2S);
    grid2(N / T::ROWS, 3, RowsR2CSmem<N>::THREADS, [&](HostExec& ex) {
        rows_r2c_body<N>(ex, RowsR2CParams{psf, otf, tw, nullptr, nullptr}, smem.data());
    });
    const int total = 3 * T::NC;
    grid2((total + T::COLS - 1) / T::COLS, 1, ColsSmem<N>::THREADS, [&](HostExec& ex) {
        cols_fwd_body<N>(ex, ColsFwdParams{otf, tw, total, 1, 1.0f / (static_cast<float>(N) * N), nullptr, 0}, smem.data());
    });
}

int conv_chunks(int N, int B) {
    const int colgroups = (3 * (N / 2 + 1) + 7) / 8;
    int n = 592 / colgroups;
    if (n > 16) n = 16;
    if (n > B) n = B;
    if (n < 1) n = 1;
    return n;
}

// out16 != nullptr: bf16 sensor image (sensor is then the fp32 conv scratch), as b200cam_sensor_fwd_bf16
template <int N>
int sensor_fwd_impl(int B, const float* img, const float* psf, float* sensor, float* img_max, int* tie_count,
                    int* tie_pos, float2* otf, float2* spectrum, bf16* out16 = nullptr) {
    using T = Tile<N>;
    auto tw = make_twiddle(N);
    otf_impl<N>(psf, otf, tw.data());
    const int planes = 3 * B;
    std::vector<float2> stx(static_cast<size_t>(planes) * T::NC * N), st2(static_cast<size_t>(planes) * T::NC * N);
    float2* srow = spectrum != nullptr ? spectrum : stx.data();
    std::vector<float2> smem(RowsR2CSmem<N>::FLOAT2S > ColsSmem<N>::FLOAT2S ? RowsR2CSmem<N>::FLOAT2S : ColsSmem<N>::FLOAT2S);
    {   // the library runs the image rows as a persistent, TMA-staged grid: same here with a small odd grid
        const int total = (N / T::ROWS) * planes, nctas = 5;
        std::vector<float2> ssmem(RowsStreamSmem<N>::FLOAT2S);
        grid2(nctas, 1, RowsStreamSmem<N>::THREADS, [&](HostExec& ex) {
            rows_r2c_stream_body<N>(ex, RowsR2CParams{img, srow, tw.data(), img_max, tie_count}, ssmem.data(), total, nctas);
        });
    }
    const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS;
    const int nchunks = conv_chunks(N, B);
    std::vector<ConvState<N>> cst(ColsSmem<N>::THREADS);
    grid2(colgroups, nchunks, ColsSmem<N>::THREADS, [&](HostExec& ex) {
        cols_conv_body<N>(ex, ColsConvParams{srow, st2.data(), otf, tw.data(), nullptr, B, nchunks, 0, 1.0f}, smem.data(), cst.data());
    });
    {
        const int total = (N / T::ROWS) * planes, nctas = 7;
        std::vector<float2> ssmem(RowsC2RStreamSmem<N>::FLOAT2S);
        grid2(nctas, 1, RowsC2RStreamSmem<N>::THREADS, [&](HostExec& ex) {
            rows_c2r_stream_body<N>(ex, RowsC2RParams{st2.data(), sensor, tw.data(), img_max, 1.0f, nullptr, nullptr, 0},
                                    ssmem.data(), total, nctas);
        });
    }
    const long long n4 = static_cast<long long>(planes) * N * N / 4;
    grid2(EW_GRID, 1, EW_THREADS, [&](HostExec& ex) {
        if (out16 != nullptr)
            normalise_body<bf16>(ex, NormaliseParams{sensor, img_max, tie_count, tie_pos, n4, 3 * N * N / 4}, EW_GRID, out16);
        else
            normalise_body(ex, NormaliseParams{sensor, img_max, tie_count, tie_pos, n4, 3 * N * N / 4}, EW_GRID);
    });
    return 0;
}

// In = bf16: the upstream gradient in bf16, as b200cam_sensor_bwd_bf16
template <int N, class In = float>
int sensor_bwd_impl(int B, const In* g, const float* img, const float* sensor, const float* img_max,
                    const int* tie_count, const int* tie_pos, const float* psf, const float2* otf,
                    const float2* spectrum, float* grad_psf, float* grad_img) {
    using T = Tile<N>;
    auto tw = make_twiddle(N);
    const int planes = 3 * B, tiles = N / T::ROWS;
    const size_t plane_sz = static_cast<size_t>(T::NC) * N;
    std::vector<float2> stx(planes * plane_sz), stg(planes * plane_sz), stp(3 * plane_sz);
    const int nchunks = accum_chunks(N, B);
    const int used_chunks = nchunks;
    std::vector<float2> partial(static_cast<size_t>(nchunks) * 3 * plane_sz);
    std::vector<float> dot_lanes(static_cast<size_t>(B) * 3 * T::NC * 32), coef(B);
    (void)sensor;
    std::vector<float2> smem(RowsR2CSmem<N>::FLOAT2S > ColsSmem<N>::FLOAT2S ? RowsR2CSmem<N>::FLOAT2S : ColsSmem<N>::FLOAT2S);
    const float2* srow = spectrum;
    if (srow == nullptr) {
        grid2(tiles, planes, RowsR2CSmem<N>::THREADS, [&](HostExec& ex) {
            rows_r2c_body<N>(ex, RowsR2CParams{img, stx.data(), tw.data(), nullptr, nullptr}, smem.data());
        });
        srow = stx.data();
    }
    grid2(tiles, planes, RowsR2CSmem<N>::THREADS, [&](HostExec& ex) {
        rows_r2c_body<N>(ex, RowsR2CParamsT<In>{g, stg.data(), tw.data(), nullptr, nullptr}, smem.data());
    });
    const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS;
    std::vector<AccumState<N>> states(ColsSmem<N>::THREADS);
    // the arg-max term of the amax backward is folded into cols_reduce_inv (spectral form, the library's default): the warp
    // partials of the Parseval dot product replace the per-thread ones, the spatial tie_term kernel is not run
    const int dot_count = colgroups * ColsSmem<N>::WARPS;
    std::vector<float> dot_warps(static_cast<size_t>(B) * dot_count);
    grid2(colgroups, used_chunks, ColsSmem<N>::THREADS, [&](HostExec& ex) {
        cols_accum_body<N>(ex, ColsAccumParams{srow, stg.data(), partial.data(), tw.data(), img_max, otf,
                                               dot_lanes.data(), B, nchunks, 0, dot_warps.data()}, smem.data(), states.data());
    });
    std::vector<float2> rsmem(ReduceInvSmem<N>::FLOAT2S);
    const bool side_job = grad_img != nullptr;
    grid2(3 * T::NC + (side_job ? B : 0), 1, ReduceInvSmem<N>::THREADS, [&](HostExec& ex) {
        cols_reduce_inv_body<N>(ex, ColsReduceInvParams{partial.data(), stp.data(), tw.data(), used_chunks,
                                                        1.0f / (static_cast<float>(N) * N), side_job ? dot_lanes.data() : nullptr, img_max,
                                                        tie_count, coef.data(), B, nullptr, tie_pos, srow, dot_warps.data(), dot_count},
                                rsmem.data());
    });
    grid2(tiles, 3, RowsR2CSmem<N>::THREADS, [&](HostExec& ex) {
        rows_c2r_body<N>(ex, RowsC2RParams{stp.data(), grad_psf, tw.data(), nullptr, 1.0f}, smem.data());
    });
    (void)img;
    if (grad_img != nullptr) {
        const int cchunks = conv_chunks(N, B);
        std::vector<ConvState<N>> cst(ColsSmem<N>::THREADS);
        grid2(colgroups, cchunks, ColsSmem<N>::THREADS, [&](HostExec& ex) {
            cols_conv_body<N>(ex, ColsConvParams{stg.data(), stg.data(), otf, tw.data(), img_max, B, cchunks, 1, 1.0f}, smem.data(),
                              cst.data());
        });
        grid2(tiles, planes, RowsR2CSmem<N>::THREADS, [&](HostExec& ex) {
            rows_c2r_body<N>(ex, RowsC2RParams{stg.data(), grad_img, tw.data(), nullptr, 1.0f}, smem.data());
        });
        grid2(EW_GRID, 1, EW_THREADS, [&](HostExec& ex) {
            tie_term_img_body(ex, TieTermImgParams{grad_img, psf, tie_count, tie_pos, coef.data(), B, N}, EW_GRID);
        });
    }
    return 0;
}

}  // namespace

#define DISPATCH_N(N_, CALL)                                   \
    switch (N_) {                                              \
        case 64: { constexpr int NN_ = 64; return CALL; }      \
        case 128: { constexpr int NN_ = 128; return CALL; }    \
        case 256: { constexpr int NN_ = 256; return CALL; }    \
        case 512: { constexpr int NN_ = 512; return CALL; }    \
        case 1024: { constexpr int NN_ = 1024; return CALL; }  \
        default: return -1;                                    \
    }


extern "C" {

// the host rounding rule of compat.cuh (bf16_bits_rn), element by element
int emu16_round(const float* x, unsigned short* out, long long n) {
    for (long long i = 0; i < n; ++i) out[i] = bf16_bits_rn(x[i]);
    return 0;
}

// the normalise body alone on a given conv [B][3][N][N]: out16 == NULL -> fp32, in place in y; else bf16 into out16 (y read only).
// levels > 0: quantisation; noise != NULL: additive noise (the read-out epilogue)
int emu16_normalise(int N, int B, float* y, const float* img_max, int* tie_count, int* tie_pos, unsigned short* out16,
                  const float* noise, float noise_scale, float levels) {
    const long long n4 = static_cast<long long>(B) * 3 * N * N / 4;
    const SensorEpilogue epi{noise, noise_scale, levels};
    grid2(EW_GRID, 1, EW_THREADS, [&](HostExec& ex) {
        const NormaliseParams p{y, img_max, tie_count, tie_pos, n4, 3 * N * N / 4, epi};
        if (out16 != nullptr)
            normalise_body<bf16>(ex, p, EW_GRID, reinterpret_cast<bf16*>(out16));
        else
            normalise_body(ex, p, EW_GRID);
    });
    return 0;
}

// the forward row pass over `planes` N x N planes: K1 (stream = 0) or the persistent TMA-staged K1s (stream = 1, odd grid),
// on fp32 (bf16_in = 0) or bf16 (bf16_in = 1) input; st [planes][N/2+1][N] complex
int emu16_rows_r2c(int N, int planes, int stream, int bf16_in, const void* x, float* st) {
    auto run = [&](auto tag) -> int {
        constexpr int NN_ = decltype(tag)::value;
        using T = Tile<NN_>;
        auto tw = make_twiddle(NN_);
        float2* out = reinterpret_cast<float2*>(st);
        auto go = [&](auto in_tag) {
            using In = decltype(in_tag);
            const RowsR2CParamsT<In> p{static_cast<const In*>(x), out, tw.data(), nullptr, nullptr};
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
        if (bf16_in) go(bf16{}); else go(float{});
        return 0;
    };
    switch (N) {
        case 64: return run(std::integral_constant<int, 64>{});
        case 128: return run(std::integral_constant<int, 128>{});
        case 256: return run(std::integral_constant<int, 256>{});
        case 512: return run(std::integral_constant<int, 512>{});
        case 1024: return run(std::integral_constant<int, 1024>{});
        default: return -1;
    }
}

// the generic sensor forward: bf16_out = 0 -> fp32 sensor image in `sensor` (as emu.cpp's emu_sensor_fwd); 1 -> `sensor` is the
// fp32 conv scratch and the image goes to `sensor16` in bf16 (as b200cam_sensor_fwd_bf16)
int emu16_sensor_fwd(int bf16_out, int N, int B, const float* img, const float* psf, float* sensor, unsigned short* sensor16,
                     float* img_max, int* tie_count, int* tie_pos, float* otf, float* spectrum) {
    bf16* out = bf16_out ? reinterpret_cast<bf16*>(sensor16) : nullptr;
    DISPATCH_N(N, (sensor_fwd_impl<NN_>(B, img, psf, sensor, img_max, tie_count, tie_pos, reinterpret_cast<float2*>(otf),
                                        reinterpret_cast<float2*>(spectrum), out)));
}

// the generic sensor backward on an fp32 (bf16_in = 0) or bf16 (bf16_in = 1, as b200cam_sensor_bwd_bf16) upstream gradient
int emu16_sensor_bwd(int bf16_in, int N, int B, const void* g, const float* img, const float* img_max, const int* tie_count,
                     const int* tie_pos, const float* psf, const float* otf, const float* spectrum, float* grad_psf, float* grad_img) {
    const float2* o = reinterpret_cast<const float2*>(otf);
    const float2* sp = reinterpret_cast<const float2*>(spectrum);
    if (bf16_in) {
        DISPATCH_N(N, (sensor_bwd_impl<NN_, bf16>(B, static_cast<const bf16*>(g), img, nullptr, img_max, tie_count, tie_pos, psf, o, sp,
                                                  grad_psf, grad_img)));
    }
    DISPATCH_N(N, (sensor_bwd_impl<NN_, float>(B, static_cast<const float*>(g), img, nullptr, img_max, tie_count, tie_pos, psf, o, sp,
                                               grad_psf, grad_img)));
}

}  // extern "C"
