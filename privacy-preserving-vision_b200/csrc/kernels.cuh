// b200cam: phase-structured kernel bodies of the generic (any power-of-two N) pipeline.
//
// Data layouts in HBM
//   image planes        x[plane][y][x]                 fp32, plane = b*3 + c (NCHW contiguous)
//   half spectrum  "ST" s[plane][u][y or v]            complex64, u < NC = N/2+1, TRANSPOSED:
//                       each spectral column u is a contiguous run of N complex values, so the
//                       column pass streams 8N-byte runs and the row passes write/read 128-byte
//                       segments (16 rows x 8 B) per u.
//   full spectrum  (PSF chain, complex fields)  f[lambda][u][y], u < N, same transposed form.
//
// Reference lines each body replaces are cited at the body.
#pragma once

#include "../../include/b200cam.h"
#include "compat.cuh"
#include "exec.cuh"
#include "fft_plan.cuh"

namespace b200cam {

template <int N>
struct Tile {
    static constexpr int ROWS = (N <= 512) ? 16 : 8;   // image rows per CTA in the row passes (16 rows = 128-byte spectrum segments)
    static constexpr int NP = ROWS / 2;                // real rows are transformed in pairs
    static constexpr int NC = N / 2 + 1;
    static constexpr int FP_PAIR = N + 16 / NP;        // natural-order smem row pitch (float2)
    static constexpr int FP_ROW = N + 16 / ROWS;
    static constexpr int COLS = 8;                     // spectral columns per CTA in column passes
    static constexpr int CROWS = (N >= 256) ? 2 : 4;   // rows per CTA in the complex (PSF chain) row passes: these kernels are
                                                       // latency chains - more, smaller CTAs shorten the chain per thread
    static constexpr int FP_CROW = N + 16 / CROWS;
    static constexpr int RCOLS = 2;                    // columns per CTA in the small batch-independent column passes
};

// ---------------------------------------------------------------------------------------------
// K1  rows_r2c : real rows -> transposed half spectrum (first half of rfftn, Utils.py:8-9)
//      grid (N/ROWS, planes), block NP*LANES.
//      init_max/init_count (tile 0 of channel 0) reset the per-image max / tie counters for the
//      kernels that follow in the stream.
// ---------------------------------------------------------------------------------------------
// `In`: element type of x - fp32, bf16 (an upstream gradient handed over in bf16; widened exactly in registers) or u8 (a uint8
// image, converted in registers as byte * fp32(1/255))
template <class In>
struct RowsR2CParamsT {
    const In* x;             // [planes][N][N]
    float2* st;              // [planes][NC][N]
    const float2* tw;
    float* init_max;         // nullable, [planes/3]
    int* init_count;         // nullable, [planes/3]
};
using RowsR2CParams = RowsR2CParamsT<float>;

// Shared memory of the row passes: one block of PA float2 per row pair, used first as the exchange array E of the
// two-pass FFT and then, IN PLACE, as the natural-order line F of the same pair (only the 16/32 lanes of the pair touch
// the block in between, so a warp-level sync separates the two uses).  Half the footprint of separate E and F arrays
// = twice the resident CTAs: these kernels are latency bound and live on occupancy.
// PA == FP_PAIR (mod 16 float2) keeps the transposing accesses of the unpack phase on distinct banks.
template <int N>
struct RowsR2CSmem {
    using P = Plan<N>;
    using T = Tile<N>;
    static constexpr int PA = P::E_SIZE + (((T::FP_PAIR - P::E_SIZE) % 16) + 16) % 16;
    static_assert(PA >= P::E_SIZE && PA >= T::FP_PAIR, "pair block too small");
    static constexpr int RED_OFF = T::NP * PA;                                 // float2 units
    static constexpr int FLOAT2S = RED_OFF + (T::NP * P::LANES + 2) / 2 + 1;   // reduction scratch (floats) of rows_c2r
    static constexpr int BYTES = FLOAT2S * 8;
    static constexpr int THREADS = T::NP * P::LANES;
};

template <int N>
struct RowState {
    float2 v[Plan<N>::R2];
};

template <int N, class Exec, class In>
B200_HD void rows_r2c_body(Exec& ex, const RowsR2CParamsT<In>& p, float2* smem) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = RowsR2CSmem<N>;
    const int tile = ex.bx(), plane = ex.by();
    const int y0 = tile * T::ROWS;
    RowState<N> st[Exec::IS_HOST ? S::THREADS : 1];

    ex.warp_phase([&](int tid) {
        const int j = tid / P::LANES, a = tid % P::LANES;
        if (a < P::R2) {
            const In* r0 = p.x + (static_cast<size_t>(plane) * N + y0 + 2 * j) * N;
            const In* r1 = r0 + N;
            float2 v[P::R1];
#pragma unroll
            for (int i = 0; i < P::R1; ++i) v[i] = make_float2(load_elem(r0 + P::R2 * i + a), load_elem(r1 + P::R2 * i + a));
            P::stepA(v, a, smem + j * S::PA, p.tw);
        }
        if (tid == 0 && tile == 0 && plane % 3 == 0) {
            if (p.init_max != nullptr) p.init_max[plane / 3] = neg_inf();
            if (p.init_count != nullptr) p.init_count[plane / 3] = 0;
        }
    });
    ex.warp_phase([&](int tid) {
        const int j = tid / P::LANES, b = tid % P::LANES;
        if (b < P::R1) P::stepB(st[ex.slot(tid)].v, b, smem + j * S::PA);
    });
    ex.phase([&](int tid) {                       // every lane of the pair has read E: overwrite it with the line
        const int j = tid / P::LANES, b = tid % P::LANES;
        if (b < P::R1) {
            const RowState<N>& s = st[ex.slot(tid)];
#pragma unroll
            for (int i = 0; i < P::R2; ++i) smem[j * S::PA + b + P::R1 * i] = s.v[i];
        }
    });
    ex.phase([&](int tid) {
        // unpack the pair spectrum Z = FFT(row_even + i*row_odd) into the two Hermitian halves
        for (int w = tid; w < T::NP * T::NC; w += S::THREADS) {
            const int u = w / T::NP, j = w % T::NP;
            const float2 z1 = smem[j * S::PA + u];
            const float2 z2 = smem[j * S::PA + ((N - u) & (N - 1))];
            const float4 o = make_float4(0.5f * (z1.x + z2.x), 0.5f * (z1.y - z2.y),    // X_even[u]
                                         0.5f * (z1.y + z2.y), -0.5f * (z1.x - z2.x));  // X_odd[u]
            *reinterpret_cast<float4*>(p.st + (static_cast<size_t>(plane) * T::NC + u) * N + y0 + 2 * j) = o;
        }
    });
}

// ---------------------------------------------------------------------------------------------
// K1s rows_r2c_stream : the same row pass as a PERSISTENT grid with TMA-staged image tiles.
//      CTA k walks tiles k, k + nctas, ...; a tile (ROWS image rows) is one contiguous ROWS*N*4-byte block in global
//      memory, fetched by a single 1-D bulk copy (cp.async.bulk + mbarrier) into one of two staging buffers while
//      the previous tile is being transformed.  Compared with K1: no 4-byte strided global loads (each 128-byte line
//      was fetched by two different instructions), the loads are asynchronous, and - the kernel being persistent - the
//      lane's twiddles stay in registers.  grid = any (the launch picks the resident CTAs per SM), block NP*LANES.
// ---------------------------------------------------------------------------------------------
template <int N, class In = float>
struct RowsStreamSmem {
    using R = RowsR2CSmem<N>;
    using T = Tile<N>;
    // Each image row is copied by its own bulk copy into a staging row of pitch N + 8 floats: the two row pairs that
    // share a warp then read from banks 16 apart (with contiguous rows, 2N floats = 0 mod 32 banks put them on the SAME
    // banks: ncu showed a quarter of this kernel's shared-memory wavefronts to be such conflicts).
    // bf16 rows (In = bf16): pitch N + 8 elements as well, i.e. 16 padding bytes.  Two lanes read the two halves of one
    // 4-byte word (a broadcast, not a conflict), so a row pair's R2 lanes touch R2/2 consecutive banks, and the rows of the
    // pairs that share a warp are 2 * (N + 8) / 2 = N + 8 words = 8 banks apart: the 2 (N = 128, 256) or 4 (N = 64) pairs of a
    // warp read disjoint banks.  The pitch stays a multiple of 16 bytes, as the bulk copies need.
    // uint8 rows (In = u8): pitch N + 16 bytes (N + 8 would not be a multiple of 16).  Four lanes read the four bytes of one word
    // (a broadcast), so a row pair's R2 lanes touch R2/4 consecutive banks, and the rows of the pairs that share a warp are
    // 2 * (N + 16) / 4 = N/2 + 8 words = 8 banks apart (N/2 = 0 mod 32 for N >= 64): the 2 pairs (N = 128, 256, R2/4 = 4 banks
    // each) or 4 pairs (N = 64, 2 banks each) of a warp again read disjoint banks.
    static constexpr int ROW_PITCH = N + (sizeof(In) == 1 ? 16 : 8);          // elements; ROW_PITCH * sizeof(In) is a multiple of 16 bytes
    static constexpr int TILE_ELEMS = T::ROWS * ROW_PITCH;
    static constexpr int TILE_BYTES = T::ROWS * N * static_cast<int>(sizeof(In));   // bytes that arrive per tile
    static constexpr int STAGE_OFF = (R::RED_OFF + 15) / 16 * 16;            // float2 units, 128-byte aligned
    static constexpr int BAR_OFF = STAGE_OFF + (2 * TILE_ELEMS * static_cast<int>(sizeof(In)) + 7) / 8;   // two tiles, in float2 units
    static constexpr int FLOAT2S = BAR_OFF + 2;                               // two 8-byte mbarriers
    static constexpr int BYTES = FLOAT2S * 8;
    static constexpr int THREADS = R::THREADS;
    static_assert(T::ROWS <= R::THREADS, "one issuing thread per row");
};

template <int N, class Exec, class In>
B200_HD void rows_r2c_stream_body(Exec& ex, const RowsR2CParamsT<In>& p, float2* smem, int total_tiles, int nctas) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = RowsR2CSmem<N>;
    using Q = RowsStreamSmem<N, In>;
    constexpr int TILES = N / T::ROWS;
    constexpr bool RT = P::REG_TW;
    In* stage = reinterpret_cast<In*>(smem + Q::STAGE_OFF);
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + Q::BAR_OFF);
    RowState<N> st[Exec::IS_HOST ? S::THREADS : 1];
    float2 wreg[RT ? P::R1 : 1];
    const int first = ex.bx();
    // thread r < ROWS copies row r of tile t (tiles are contiguous in x) into staging buffer `buf`; thread 0 arms the barrier
    auto issue = [&](int tid, int t, int buf) {
        if (tid == 0) ex.bulk_expect(bars + buf, Q::TILE_BYTES);
        if (tid < T::ROWS)
            ex.bulk_load(stage + buf * Q::TILE_ELEMS + tid * Q::ROW_PITCH, p.x + (static_cast<size_t>(t) * T::ROWS + tid) * N,
                         N * static_cast<unsigned>(sizeof(In)), bars + buf);
    };

    ex.phase([&](int tid) {
        if (tid == 0) {
            ex.bulk_init(bars + 0);
            ex.bulk_init(bars + 1);
            ex.bulk_fence_init();
        }
        if constexpr (RT && !Exec::IS_HOST) P::load_tw(wreg, p.tw, tid % P::LANES);
    });
    ex.phase([&](int tid) {
        if (first < total_tiles) issue(tid, first, 0);
    });
    int it = 0;
    for (int t = first; t < total_tiles; t += nctas, ++it) {
        const int buf = it & 1;
        const int plane = t / TILES, tile = t % TILES;
        const int y0 = tile * T::ROWS;
        ex.warp_phase([&](int tid) {
            // the other buffer was last read two block barriers ago: refill it with this CTA's next tile
            if (t + nctas < total_tiles) issue(tid, t + nctas, buf ^ 1);
            ex.bulk_wait(bars + buf, (it >> 1) & 1);
            const int j = tid / P::LANES, a = tid % P::LANES;
            if (a < P::R2) {
                const In* r0 = stage + buf * Q::TILE_ELEMS + (2 * j) * Q::ROW_PITCH;
                const In* r1 = r0 + Q::ROW_PITCH;
                float2 v[P::R1];
#pragma unroll
                for (int i = 0; i < P::R1; ++i) v[i] = make_float2(to_float(r0[P::R2 * i + a]), to_float(r1[P::R2 * i + a]));
                if constexpr (RT) {
                    if constexpr (Exec::IS_HOST) P::load_tw(wreg, p.tw, a);
                    P::stepA(v, a, smem + j * S::PA, wreg);
                } else {
                    P::stepA(v, a, smem + j * S::PA, p.tw);
                }
            }
            if (tid == 0 && tile == 0 && plane % 3 == 0) {
                if (p.init_max != nullptr) p.init_max[plane / 3] = neg_inf();
                if (p.init_count != nullptr) p.init_count[plane / 3] = 0;
            }
        });
        ex.warp_phase([&](int tid) {
            const int j = tid / P::LANES, b = tid % P::LANES;
            if (b < P::R1) P::stepB(st[ex.slot(tid)].v, b, smem + j * S::PA);
        });
        ex.phase([&](int tid) {
            const int j = tid / P::LANES, b = tid % P::LANES;
            if (b < P::R1) {
                const RowState<N>& s = st[ex.slot(tid)];
#pragma unroll
                for (int i = 0; i < P::R2; ++i) smem[j * S::PA + b + P::R1 * i] = s.v[i];
            }
        });
        ex.phase([&](int tid) {
            for (int w = tid; w < T::NP * T::NC; w += S::THREADS) {
                const int u = w / T::NP, j = w % T::NP;
                const float2 z1 = smem[j * S::PA + u];
                const float2 z2 = smem[j * S::PA + ((N - u) & (N - 1))];
                const float4 o = make_float4(0.5f * (z1.x + z2.x), 0.5f * (z1.y - z2.y),    // X_even[u]
                                             0.5f * (z1.y + z2.y), -0.5f * (z1.x - z2.x));  // X_odd[u]
                *reinterpret_cast<float4*>(p.st + (static_cast<size_t>(plane) * T::NC + u) * N + y0 + 2 * j) = o;
            }
        });
    }
}

// ---------------------------------------------------------------------------------------------
// K2  cols_conv : per spectral column  FFT_v -> x OTF -> IFFT_v, in place on ST
//      (second half of rfftn, the multiply Utils.py:10 and first half of irfftn Utils.py:11)
//      grid ceil(planes*NC / COLS), block COLS*LANES.  OTF layout [3][NC][N] (column = channel,u),
//      pre-scaled by 1/N^2.  conj_otf: multiply by conj(OTF) (adjoint, for dL/dimg).
//      col_scale (nullable, [planes/3]): extra per-image factor (1/max for the backward).
// ---------------------------------------------------------------------------------------------
struct ColsConvParams {
    const float2* in;        // [B*3][NC][N]
    float2* out;             // same layout (may alias in)
    const float2* otf;       // [3][NC][N]
    const float2* tw;
    const float* img_scale;  // nullable: per image multiplier is 1/img_scale[b]
    int B;
    int nchunks;             // = gridDim.y: CTA (., y) owns images [B*y/nchunks, B*(y+1)/nchunks) (balanced split)
    int conj_otf;
    float otf_scale;         // extra factor on the OTF
    int* zero_ints;          // nullable: n_zero ints zeroed by CTA (0,0) for the kernel that follows (arrival counters)
    int n_zero;
};

template <int N>
struct ColsSmem {
    using P = Plan<N>;
    static constexpr int COLS = Tile<N>::COLS;
    static constexpr int THREADS = COLS * P::LANES;
    static constexpr int WARPS = THREADS / 32;
    static constexpr int WCOLS = 32 / P::LANES;                   // columns owned by one warp
    // TMA staging: a warp's WCOLS columns of one image are one contiguous run of WCOLS*N float2 in the spectrum
    // layout; lane 0 fetches it with a single bulk copy (cp.async.bulk + the warp's own mbarrier) into the warp's slice
    // of the staging area, and re-issues the copy for the NEXT image as soon as the warp has consumed the slice - the
    // copy then flies while the current image is transformed.  No LSU instruction, no register, warp-level syncs only.
    // Used by the accumulate kernel (two operands per image: 25.6 -> 23.6 us at N = 256, B = 64).  The convolution
    // kernel keeps direct loads: staging costs it the registers that let 4 CTAs share an SM (measured 21.9 -> 24.7 us).
    static constexpr bool STAGED_ACCUM = N <= 512;                // N = 1024: the slices do not fit beside the exchange buffers
    static constexpr int STAGE_OFF = 2 * COLS * P::E_SIZE;        // float2 units (E_SIZE is a multiple of 8: 64-B aligned)
    static constexpr int STAGE1 = COLS * N;                       // one operand
    static constexpr int BAR_OFF_ACCUM = STAGE_OFF + (STAGED_ACCUM ? 2 * STAGE1 : 0);
    static constexpr int FLOAT2S_CONV = STAGE_OFF;
    static constexpr int FLOAT2S_ACCUM = BAR_OFF_ACCUM + WARPS;   // one 8-byte mbarrier per warp
    static constexpr int FLOAT2S = FLOAT2S_ACCUM;
    static constexpr int BYTES_CONV = FLOAT2S_CONV * 8;
    static constexpr int BYTES = FLOAT2S * 8;
    static_assert((2 * COLS * P::E_SIZE) % 2 == 0, "staging area must be 16-byte aligned");
};

template <int N>
struct ConvState {
    float2 k[Plan<N>::R2];   // this lane's OTF values, loaded once per CTA
};

// grid (ceil(3*NC/COLS), nchunks), block COLS*LANES.  A CTA owns COLS columns of one channel
// (flat index cu over [3][NC]) and walks its chunk of images, so the OTF - and, for R1 == R2, the lane's FFT
// twiddles - are read once per CTA and stay in registers.  (These passes are bound by the shared/L1 data pipe:
// every look-up that does not go through it counts.)
template <int N, class Exec>
B200_HD void cols_conv_body(Exec& ex, const ColsConvParams& p, float2* smem, ConvState<N>* st) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = ColsSmem<N>;
    float2* E1 = smem;
    float2* E2 = smem + S::COLS * P::E_SIZE;
    constexpr int TOTAL = 3 * T::NC;
    constexpr bool RT = P::REG_TW;
    const int cu0 = ex.bx() * S::COLS;
    const int b0 = static_cast<int>(static_cast<long long>(p.B) * ex.by() / p.nchunks);
    const int b1 = static_cast<int>(static_cast<long long>(p.B) * (ex.by() + 1) / p.nchunks);
    float2 wreg[RT ? P::R1 : 1];                 // device: loaded once; host emulator: reloaded inside every phase

    ex.warp_phase([&](int tid) {
        const int jc = tid / P::LANES, b = tid % P::LANES;
        const int cu = cu0 + jc;
        if (p.zero_ints != nullptr && ex.bx() == 0 && ex.by() == 0)
            for (int i = tid; i < p.n_zero; i += S::THREADS) p.zero_ints[i] = 0;
        if (cu < TOTAL && b < P::R1) {
            ConvState<N>& s = st[ex.slot(tid)];
            const float2* k = p.otf + static_cast<size_t>(cu) * N;
#pragma unroll
            for (int i = 0; i < P::R2; ++i) {
                const float2 kk = cscale(ld_ro(k + b + P::R1 * i), p.otf_scale);
                s.k[i] = p.conj_otf ? cconj(kk) : kk;
            }
        }
        if constexpr (RT && !Exec::IS_HOST) P::load_tw(wreg, p.tw, b);
    });
    for (int img = b0; img < b1; ++img) {
        ex.warp_phase([&](int tid) {
            const int jc = tid / P::LANES, a = tid % P::LANES;
            const int cu = cu0 + jc;
            if (cu < TOTAL && a < P::R2) {
                const int c = cu / T::NC, u = cu % T::NC;
                const float2* src = p.in + (static_cast<size_t>(img * 3 + c) * T::NC + u) * N;   // may alias out: plain loads
                float2 v[P::R1];
#pragma unroll
                for (int i = 0; i < P::R1; ++i) v[i] = src[P::R2 * i + a];
                if constexpr (RT) {
                    if constexpr (Exec::IS_HOST) P::load_tw(wreg, p.tw, a);
                    P::stepA(v, a, E1 + jc * P::E_SIZE, wreg);
                } else {
                    P::stepA(v, a, E1 + jc * P::E_SIZE, p.tw);
                }
            }
        });
        ex.warp_phase([&](int tid) {
            const int jc = tid / P::LANES, b = tid % P::LANES;
            const int cu = cu0 + jc;
            if (cu < TOTAL && b < P::R1) {
                const ConvState<N>& s = st[ex.slot(tid)];
                const float sc = p.img_scale != nullptr ? 1.0f / ld_ro(p.img_scale + img) : 1.0f;
                float2 v[P::R2];
                P::stepB(v, b, E1 + jc * P::E_SIZE);
#pragma unroll
                for (int i = 0; i < P::R2; ++i) {
                    v[i] = cmul(v[i], s.k[i]);
                    if (p.img_scale != nullptr) v[i] = cscale(v[i], sc);
                }
                if constexpr (RT) {
                    if constexpr (Exec::IS_HOST) P::load_tw(wreg, p.tw, b);
                    P::stepC(v, b, E2 + jc * P::E_SIZE, wreg);
                } else {
                    P::stepC(v, b, E2 + jc * P::E_SIZE, p.tw);
                }
            }
        });
        ex.warp_phase([&](int tid) {
            const int jc = tid / P::LANES, a = tid % P::LANES;
            const int cu = cu0 + jc;
            if (cu < TOTAL && a < P::R2) {
                const int c = cu / T::NC, u = cu % T::NC;
                float2 v[P::R1];
                P::stepD(v, a, E2 + jc * P::E_SIZE);
                float2* dst = p.out + (static_cast<size_t>(img * 3 + c) * T::NC + u) * N;
#pragma unroll
                for (int i = 0; i < P::R1; ++i) dst[P::R2 * i + a] = v[i];
            }
        });
    }
}

// ---------------------------------------------------------------------------------------------
// K2b cols_fwd : per spectral column FFT_v only, then a point-wise sign/scale, in place
//      (used for the OTF: K = rfft2(roll(psf,-N/2)) = (-1)^(u+v) rfft2(psf), Optics.py:126 + Utils.py:9)
// ---------------------------------------------------------------------------------------------
struct ColsFwdParams {
    float2* st;          // [planes][NC][N] in place; output is written in Q order = natural v index
    const float2* tw;
    int total_cols;
    int checker_sign;    // multiply by (-1)^(u+v)
    float scale;
    // optional: divide by S = sum(partials) as well - the OTF of psf = |U|^2 / S taken straight from |U|^2, so that it
    // does not have to wait for psf_finalise.  Every CTA adds the same values in the same order.
    const float* sum_partials;
    int npartials;
    const float2* in = nullptr;   // nullable: read the columns from here instead of `st` (out of place)
};

template <int N, class Exec>
B200_HD void cols_fwd_body(Exec& ex, const ColsFwdParams& p, float2* smem) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = ColsSmem<N>;
    float2* E1 = smem;
    float* red = reinterpret_cast<float*>(smem + S::COLS * P::E_SIZE);      // second exchange buffer: unused here
    const int col0 = ex.bx() * S::COLS;
    if (p.sum_partials != nullptr) {
        ex.phase([&](int tid) {
            float acc = 0.f;
            for (int i = tid; i < p.npartials; i += S::THREADS) acc += p.sum_partials[i];
            red[tid] = acc;
        });
        ex.phase([&](int tid) {
            if (tid == 0) {
                float tot = 0.f;
                for (int t = 0; t < S::THREADS; ++t) tot += red[t];
                red[S::THREADS] = tot;
            }
        });
    }
    const float scale = p.sum_partials != nullptr ? p.scale / red[S::THREADS] : p.scale;
    ex.warp_phase([&](int tid) {
        const int jc = tid / P::LANES, a = tid % P::LANES;
        const int col = col0 + jc;
        if (col < p.total_cols && a < P::R2) {
            const float2* src = (p.in != nullptr ? p.in : p.st) + static_cast<size_t>(col) * N;
            float2 v[P::R1];
#pragma unroll
            for (int i = 0; i < P::R1; ++i) v[i] = src[P::R2 * i + a];
            P::stepA(v, a, E1 + jc * P::E_SIZE, p.tw);
        }
    });
    ex.warp_phase([&](int tid) {
        const int jc = tid / P::LANES, b = tid % P::LANES;
        const int col = col0 + jc;
        if (col < p.total_cols && b < P::R1) {
            const int u = col % T::NC;
            float2 v[P::R2];
            P::stepB(v, b, E1 + jc * P::E_SIZE);
            float2* dst = p.st + static_cast<size_t>(col) * N;
#pragma unroll
            for (int i = 0; i < P::R2; ++i) {
                const int k = b + P::R1 * i;
                const float s = (p.checker_sign && ((u + k) & 1)) ? -scale : scale;
                dst[k] = cscale(v[i], s);
            }
        }
    });
}

// ---------------------------------------------------------------------------------------------
// K3  rows_c2r : transposed half spectrum (already inverse-transformed along v) -> real rows
//      (second half of irfftn, Utils.py:11) + per-image max (Optics.py:128, amax part)
//      grid (N/ROWS, planes), block NP*LANES
// ---------------------------------------------------------------------------------------------
constexpr int C2R_MAX_TIES = 8;     // = MAX_TIES (declared with the normalise kernel below)

// Opt-in sensor read-out epilogue of both cameras (north_star step 5; SURVEY trap T6: the reference has NO live sensor
// noise and no quantisation - its gaussian_noise call is commented out, Image_Caption/Camera/Lens.py:295-301,
// Utils.py:300-302 - so both are OFF unless asked for):
//     y <- conv / max ;  y += noise_scale * noise[idx] ;  y <- round(clamp(y,0,1) * L) / L
// Face-DeId `Camera`: applied where the sensor kernels write y (one-pass inverse rows, normalise kernel; b200cam.cu);
// Image_Caption `OpticsZernike`: in the normalise kernel of lens_conv.cu, after the batch-global maximum.
// `noise` is a caller-supplied N(0,1) tensor shaped like the image batch (drawn with torch's generator, so a run is
// reproducible against the oracle); L = 2^bits - 1.  Or `seed` (B200CAM_SENSOR_NOISE_PHILOX): the element-wise kernels draw
// the normals with philox_normal4 below instead of reading a tensor - their own instantiations, which add them through
// add_noise / quantise exactly as apply_epilogue adds a tensor's values.  The backward is straight through (dL/dconv as if
// the epilogue were the identity), the usual treatment of a quantiser.
struct SensorEpilogue {
    const float* noise;      // nullable
    float noise_scale;
    float levels;            // <= 0: no quantisation
    const b200cam_noise_seed* seed;   // nullable; set: the Philox read-out (noise == nullptr then)
};
B200_HD float add_noise(const SensorEpilogue& e, float y, float n) { return y + e.noise_scale * n; }
B200_HD float quantise(const SensorEpilogue& e, float y) {
    if (e.levels > 0.f) {
        y = fminf(fmaxf(y, 0.f), 1.f);
        y = rintf(y * e.levels) / e.levels;
    }
    return y;
}
B200_HD float apply_epilogue(const SensorEpilogue& e, float y, size_t idx) {
    if (e.noise != nullptr) y = add_noise(e, y, ld_ro(e.noise + idx));
    return quantise(e, y);
}

// ---- the sensor noise of B200CAM_SENSOR_NOISE_PHILOX (include/b200cam.h): Philox4x32-10 + Box-Muller ------------------------
// One counter j gives the standard normals of the four elements 4j'..4j'+3 of the call's batch, j = first4 + j'.  Every kernel
// that draws them (the normalise kernels of both cameras, the materialiser) calls philox_normal4, so the fused read-out and the
// materialised tensor agree bit for bit.
struct Normal4 { float n[4]; };
B200_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return static_cast<uint32_t>((static_cast<uint64_t>(a) * b) >> 32);
#endif
}
// Philox4x32-10 of Random123 (the cuRAND constants): 10 rounds, the key bumped between rounds
B200_HD void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r > 0) {
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        const uint32_t hi0 = mulhi32(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = mulhi32(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t c1 = c[1], c3 = c[3];
        c[0] = hi1 ^ c1 ^ k0;
        c[1] = lo1;
        c[2] = hi0 ^ c3 ^ k1;
        c[3] = lo0;
    }
}
// sin(pi x), cos(pi x).  Host (emulator): computed in double and rounded - host and device values are not compared.
B200_HD void sincospi_f(float x, float* s, float* c) {
#if defined(__CUDA_ARCH__)
    sincospif(x, s, c);
#else
    const double a = M_PI * static_cast<double>(x);
    *s = static_cast<float>(sin(a));
    *c = static_cast<float>(cos(a));
#endif
}
// (2 (x >> 9) + 1) 2^-24: a 24-bit odd integer times a power of two, exact; never 0 or 1
B200_HD float philox_uniform(uint32_t x) { return static_cast<float>(2u * (x >> 9) + 1u) * 5.9604644775390625e-8f; }
B200_HD void box_muller(float u0, float u1, float* n0, float* n1) {
    const float r = sqrtf(-2.0f * logf(u0));
    float s, c;
    sincospi_f(2.0f * u1, &s, &c);
#if defined(__CUDA_ARCH__)
    *n0 = __fmul_rn(r, c);          // (no contraction into the caller's noise_scale * n + y)
    *n1 = __fmul_rn(r, s);
#else
    *n0 = r * c;
    *n1 = r * s;
#endif
}
B200_HD Normal4 philox_normal4(unsigned long long key, unsigned long long j) {
    uint32_t c[4] = {static_cast<uint32_t>(j), static_cast<uint32_t>(j >> 32), 0u, 0u};
    philox4x32_10(c, static_cast<uint32_t>(key), static_cast<uint32_t>(key >> 32));
    Normal4 o;
    box_muller(philox_uniform(c[0]), philox_uniform(c[1]), &o.n[0], &o.n[1]);
    box_muller(philox_uniform(c[2]), philox_uniform(c[3]), &o.n[2], &o.n[3]);
    return o;
}
// the seed block as the kernels read it (device memory, so that a graph replay sees the key drawn in that replay)
struct NoiseSeed { unsigned long long key, first4; };
B200_HD NoiseSeed load_seed(const b200cam_noise_seed* s) {
    const unsigned long long* w = reinterpret_cast<const unsigned long long*>(s);
    return NoiseSeed{ld_ro(w), ld_ro(w + 1)};
}

// Validates the (flags, noise, noise_scale, quant_bits) arguments of the _ex entry points of both cameras (include/b200cam.h)
// and builds the epilogue they select; host side, before anything is enqueued.
inline int make_epilogue(int flags, const float* noise, float noise_scale, int quant_bits, SensorEpilogue* epi) {
    *epi = SensorEpilogue{nullptr, 0.f, 0.f, nullptr};
    if (flags & ~(B200CAM_SENSOR_NOISE | B200CAM_SENSOR_QUANT | B200CAM_SENSOR_NOISE_PHILOX)) return B200CAM_E_BAD_SIZE;
    if ((flags & B200CAM_SENSOR_NOISE) && (flags & B200CAM_SENSOR_NOISE_PHILOX)) return B200CAM_E_BAD_SIZE;
    if (flags & B200CAM_SENSOR_NOISE) {
        if (noise == nullptr) return B200CAM_E_NULL;
        epi->noise = noise;
        epi->noise_scale = noise_scale;
    }
    if (flags & B200CAM_SENSOR_NOISE_PHILOX) {
        if (!(noise_scale > 0.f)) return B200CAM_E_BAD_SIZE;      // a zero-amplitude draw: ask for no noise instead
        if (noise == nullptr) return B200CAM_E_NULL;
        if (reinterpret_cast<uintptr_t>(noise) % 8 != 0) return B200CAM_E_ALIGN;
        epi->seed = reinterpret_cast<const b200cam_noise_seed*>(noise);
        epi->noise_scale = noise_scale;
    }
    if (flags & B200CAM_SENSOR_QUANT) {
        if (quant_bits < 1 || quant_bits > 16) return B200CAM_E_BAD_SIZE;
        epi->levels = static_cast<float>((1 << quant_bits) - 1);
    }
    return 0;
}

struct RowsC2RParams {
    const float2* st;    // [planes][NC][N]
    float* out;          // [planes][N][N]; nullptr: nothing is stored (max-only pass)
    const float2* tw;
    float* img_max;      // nullable, [planes/3]: atomically maximised (norm = 0) or read (norm = 1)
    float scale;
    // norm = 1: second pass over the same spectrum - the rows are recomputed (bit-identical), divided by the
    // image maximum found by the first pass (Optics.py:128) and the positions that attain it are recorded
    // (torch's amax backward splits the gradient evenly between exact ties).  Saves writing and re-reading conv.
    int* tie_count;      // [planes/3], zero on entry
    int* tie_pos;        // [planes/3][MAX_TIES] flat index into (3,N,N)
    int norm;
    int discard_input;   // stream kernel: `st` is dead after this pass - drop its lines from L2 instead of writing them back
    // stream kernel, arrivals > 0: ONE pass - y = conv / max is written directly.  A tile's outputs wait in the thread's
    // registers while its CTA max is published ({atomic max, arrival count} per image); the CTA finishes the
    // tile one iteration later, when the `arrivals` tiles of that image - all processed in the same wave of the
    // persistent grid - have long arrived.  No un-normalised image, no normalise pass (Optics.py:128).
    int* arrive;         // [planes/3], zero on entry
    int arrivals;        // tiles per image = 3 * N / ROWS
    SensorEpilogue epi;  // applied by the one-pass mode where it writes y
};

template <int N, class Exec>
B200_HD void rows_c2r_body(Exec& ex, const RowsC2RParams& p, float2* smem) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = RowsR2CSmem<N>;
    const int tile = ex.bx(), plane = ex.by();
    const int y0 = tile * T::ROWS;
    float* red = reinterpret_cast<float*>(smem + S::RED_OFF);
    RowState<N> st[Exec::IS_HOST ? S::THREADS : 1];

    ex.phase([&](int tid) {
        // all of the thread's 16-byte loads are issued before the first one is consumed (latency, not bandwidth, bounds
        // this gather of 128-byte segments)
        constexpr int ITEMS = (T::NP * T::NC + S::THREADS - 1) / S::THREADS;
        float4 q[ITEMS];
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const int w = tid + k * S::THREADS;
            if (w < T::NP * T::NC) {
                const int u = w / T::NP, j = w % T::NP;
                q[k] = ld_ro(reinterpret_cast<const float4*>(p.st + (static_cast<size_t>(plane) * T::NC + u) * N + y0 + 2 * j));
            }
        }
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const int w = tid + k * S::THREADS;
            if (w < T::NP * T::NC) {
                const int u = w / T::NP, j = w % T::NP;
                // Z = X_even + i X_odd ; Z[N-u] = conj(X_even[u]) + i conj(X_odd[u])
                float2* F = smem + j * S::PA;
                if (u == 0 || u == N / 2) {
                    F[u] = make_float2(q[k].x, q[k].z);   // irfft ignores Im at DC/Nyquist
                } else {
                    F[u] = make_float2(q[k].x - q[k].w, q[k].y + q[k].z);
                    F[N - u] = make_float2(q[k].x + q[k].w, q[k].z - q[k].y);
                }
            }
        }
    });
    ex.warp_phase([&](int tid) {
        const int j = tid / P::LANES, b = tid % P::LANES;
        if (b < P::R1) {
            RowState<N>& s = st[ex.slot(tid)];
#pragma unroll
            for (int i = 0; i < P::R2; ++i) s.v[i] = smem[j * S::PA + b + P::R1 * i];
        }
    });
    ex.warp_phase([&](int tid) {                  // every lane of the pair holds its part of the line: reuse it as E
        const int j = tid / P::LANES, b = tid % P::LANES;
        if (b < P::R1) P::stepC(st[ex.slot(tid)].v, b, smem + j * S::PA, p.tw);
    });
    ex.phase([&](int tid) {
        const int j = tid / P::LANES, a = tid % P::LANES;
        float mx = neg_inf();
        if (a < P::R2) {
            float2 v[P::R1];
            P::stepD(v, a, smem + j * S::PA);
            const size_t row = (static_cast<size_t>(plane) * N + y0 + 2 * j) * N;
            if (p.norm) {
                const int img = plane / 3;
                const float m = *(p.img_max + img);
                const int base = (plane % 3) * N * N + (y0 + 2 * j) * N;
#pragma unroll
                for (int i = 0; i < P::R1; ++i) {
                    const float e = v[i].x * p.scale, o = v[i].y * p.scale;
                    const int x = P::R2 * i + a;
                    if (e == m) {
                        const int slot = atomic_add_int(p.tie_count + img, 1);
                        if (slot < C2R_MAX_TIES) p.tie_pos[img * C2R_MAX_TIES + slot] = base + x;
                    }
                    if (o == m) {
                        const int slot = atomic_add_int(p.tie_count + img, 1);
                        if (slot < C2R_MAX_TIES) p.tie_pos[img * C2R_MAX_TIES + slot] = base + N + x;
                    }
                    p.out[row + x] = e / m;
                    p.out[row + N + x] = o / m;
                }
            } else {
#pragma unroll
                for (int i = 0; i < P::R1; ++i) {
                    const float e = v[i].x * p.scale, o = v[i].y * p.scale;
                    if (p.out != nullptr) {
                        p.out[row + P::R2 * i + a] = e;
                        p.out[row + N + P::R2 * i + a] = o;
                    }
                    mx = fmaxf(mx, fmaxf(e, o));
                }
            }
        }
        red[tid] = mx;
    });
    if (p.img_max != nullptr && !p.norm) {
        ex.phase([&](int tid) {
            if (tid == 0) {
                float mx = red[0];
                for (int t = 1; t < S::THREADS; ++t) mx = fmaxf(mx, red[t]);
                atomic_max_float(p.img_max + plane / 3, mx);
            }
        });
    }
}

// ---------------------------------------------------------------------------------------------
// K3s rows_c2r_stream : K3 (norm = 0) as a persistent grid with TMA-staged spectrum tiles.  A tile is NC segments of
//      ROWS*8 bytes (one per spectral column u, 8N bytes apart): thread u issues the bulk copy of segment u, all on
//      one mbarrier; two staging buffers, so the next tile lands while this one is transformed.
// ---------------------------------------------------------------------------------------------
template <int N>
struct RowsC2RStreamSmem {
    using R = RowsR2CSmem<N>;
    using T = Tile<N>;
    static constexpr int SEG = T::ROWS;                                       // float2 per segment
    static constexpr int TILE_FLOAT2S = T::NC * SEG;
    static constexpr int STAGE_OFF = (R::FLOAT2S + 15) / 16 * 16;             // float2 units, 128-byte aligned
    static constexpr int BAR_OFF = STAGE_OFF + 2 * ((TILE_FLOAT2S + 15) / 16 * 16);
    static constexpr int FLOAT2S = BAR_OFF + 2;
    static constexpr int BYTES = FLOAT2S * 8;
    static constexpr int THREADS = R::THREADS;
};

// ONE_PASS = false compiles the stash of the one-pass mode away (it costs the two-pass kernel its registers: 128 with spills
// instead of 96, 35 us instead of 22 us at B = 64)
template <int N, class Exec, bool ONE_PASS = true>
B200_HD void rows_c2r_stream_body(Exec& ex, const RowsC2RParams& p, float2* smem, int total_tiles, int nctas) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = RowsR2CSmem<N>;
    using Q = RowsC2RStreamSmem<N>;
    constexpr int TILES = N / T::ROWS;
    constexpr bool RT = P::REG_TW;
    constexpr int STAGE_STRIDE = (Q::TILE_FLOAT2S + 15) / 16 * 16;
    float2* stage = smem + Q::STAGE_OFF;
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + Q::BAR_OFF);
    float* red = reinterpret_cast<float*>(smem + S::RED_OFF);
    RowState<N> st[Exec::IS_HOST ? S::THREADS : 1];
    float2 wreg[RT ? P::R1 : 1];
    const int first = ex.bx();
    // thread tid copies segments tid, tid + THREADS, ... of tile t into staging buffer `buf`
    auto issue = [&](int tid, int t, int buf) {
        const int plane = t / TILES, y0 = (t % TILES) * T::ROWS;
        for (int u = tid; u < T::NC; u += S::THREADS)
            ex.bulk_load(stage + buf * STAGE_STRIDE + u * Q::SEG, p.st + (static_cast<size_t>(plane) * T::NC + u) * N + y0,
                         Q::SEG * 8, bars + buf);
    };

    // one-pass normalise (see RowsC2RParams::arrive): every lane holds a full transform output (LANES == R2) of <= 16 values
    constexpr bool FUSABLE = ONE_PASS && (P::R1 <= 16) && (P::LANES == P::R2);
    const bool fused = FUSABLE && p.arrivals > 0 && p.arrive != nullptr && p.img_max != nullptr && p.out != nullptr;
    // the previous tile's outputs wait here (registers, or thread-private local memory where the compiler spills them: tensor
    // memory would be the natural stash, but a kernel that contains tcgen05.alloc is limited to ONE CTA per SM by the
    // launch machinery - measured: grid 592 -> 148)
    struct OutState { float2 v[P::R1]; };
    OutState keep[(Exec::IS_HOST && FUSABLE) ? S::THREADS : 1], cur[(Exec::IS_HOST && FUSABLE) ? S::THREADS : 1];
    // write the stashed tile `tt` as conv / max of its image; the positions that attain the max are recorded for the backward
    // one-pass mode: the tiles of an image publish their maxima as never-zero keys in the image's slot row (zeroed by the
    // column kernel before); a warp reads the row (k0: slots 0..31, k1: slots 32..), polls until every word is non-zero
    // and takes the maximum - no atomic, no fence, no counter
    constexpr int SLOTS = 64;                       // words per image row in p.arrive
    static_assert(!FUSABLE || 3 * TILES <= SLOTS, "slot row too short");
    constexpr int NS0 = 3 * TILES < 32 ? 3 * TILES : 32, NS1 = 3 * TILES > 32 ? 3 * TILES - 32 : 0;   // live slots per half row
    // lanes without a slot carry the smallest key (1): "present", never the maximum
    auto finish = [&](int tid, int tt, unsigned k0, unsigned k1) {
        const int fplane = tt / TILES, fy0 = (tt % TILES) * T::ROWS, img = fplane / 3;
        float m = 0.f;
        {
            const unsigned* row = reinterpret_cast<const unsigned*>(p.arrive) + static_cast<size_t>(img) * SLOTS;
            if (!ex.key_wait(row, tid & 31, k0, k1, &m)) ex.report(1u);
            if (tt % (3 * TILES) == 0 && tid == 0) p.img_max[img] = m;      // kept for the backward
        }
        const float inv = 1.0f / m;
        const int j = tid / P::LANES, a = tid % P::LANES;
        const float2 (&v)[P::R1] = keep[ex.slot(tid)].v;
        const size_t row = (static_cast<size_t>(fplane) * N + fy0 + 2 * j) * N;
        unsigned eq = 0u;
#pragma unroll
        for (int i = 0; i < P::R1; ++i) {
            eq |= (v[i].x == m ? 1u : 0u) << (2 * i);
            eq |= (v[i].y == m ? 1u : 0u) << (2 * i + 1);
            const size_t i0 = row + P::R2 * i + a, i1 = i0 + N;
            p.out[i0] = apply_epilogue(p.epi, v[i].x == m ? 1.0f : v[i].x * inv, i0);    // the arg-max itself: exactly 1 (torch: x / x)
            p.out[i1] = apply_epilogue(p.epi, v[i].y == m ? 1.0f : v[i].y * inv, i1);
        }
        while (eq != 0u) {                                                         // rare
            int bit = 0;
            while (((eq >> bit) & 1u) == 0u) ++bit;
            eq &= eq - 1u;
            const int slot = atomic_add_int(p.tie_count + img, 1);
            if (slot < C2R_MAX_TIES)
                p.tie_pos[img * C2R_MAX_TIES + slot] = (fplane % 3) * N * N + (fy0 + 2 * j + (bit & 1)) * N + P::R2 * (bit >> 1) + a;
        }
    };

    ex.phase([&](int tid) {
        if (tid == 0) {
            ex.bulk_init(bars + 0);
            ex.bulk_init(bars + 1);
            ex.bulk_fence_init();
        }
        if constexpr (RT && !Exec::IS_HOST) P::load_tw(wreg, p.tw, tid % P::LANES);
    });
    ex.phase([&](int tid) {
        if (first < total_tiles) {
            if (tid == 0) ex.bulk_expect(bars + 0, T::NC * Q::SEG * 8);
            issue(tid, first, 0);
        }
    });
    int it = 0;
    // one-pass mode: the arrival count and the maximum of the PREVIOUS tile's image are fetched at the top of the iteration
    // (two dependent L2 round trips that fly while this tile is transformed) instead of inside finish()
    unsigned pre_k0 = 0u, pre_k1 = 0u;
    for (int t = first; t < total_tiles; t += nctas, ++it) {
        const int buf = it & 1;
        const int plane = t / TILES, y0 = (t % TILES) * T::ROWS;
        ex.phase([&](int tid) {
            if (t + nctas < total_tiles) {        // the other buffer was consumed before the last block barrier
                if (tid == 0) ex.bulk_expect(bars + (buf ^ 1), T::NC * Q::SEG * 8);
                issue(tid, t + nctas, buf ^ 1);
            }
            ex.bulk_wait(bars + buf, (it >> 1) & 1);
            if (p.discard_input && Q::SEG * 8 == 128)
                for (int u = tid; u < T::NC; u += S::THREADS)
                    discard_line(p.st + (static_cast<size_t>(plane) * T::NC + u) * N + y0);
            const float2* sg = stage + buf * STAGE_STRIDE;
            for (int w = tid; w < T::NP * T::NC; w += S::THREADS) {
                const int u = w / T::NP, j = w % T::NP;
                const float4 q = *reinterpret_cast<const float4*>(sg + u * Q::SEG + 2 * j);
                // Z = X_even + i X_odd ; Z[N-u] = conj(X_even[u]) + i conj(X_odd[u])
                float2* F = smem + j * S::PA;
                if (u == 0 || u == N / 2) {
                    F[u] = make_float2(q.x, q.z);   // irfft ignores Im at DC/Nyquist
                } else {
                    F[u] = make_float2(q.x - q.w, q.y + q.z);
                    F[N - u] = make_float2(q.x + q.w, q.z - q.y);
                }
            }
        });
        ex.warp_phase([&](int tid) {
            const int j = tid / P::LANES, b = tid % P::LANES;
            if constexpr (FUSABLE && !Exec::IS_HOST) {
                if (fused && it > 0) {               // the previous tile's image: its keys fly in while this tile is transformed
                    const unsigned* row = reinterpret_cast<const unsigned*>(p.arrive) + static_cast<size_t>(((t - nctas) / TILES) / 3) * SLOTS;
                    pre_k0 = (tid & 31) < NS0 ? ex.key_load(row + (tid & 31)) : 1u;
                    pre_k1 = (tid & 31) < NS1 ? ex.key_load(row + 32 + (tid & 31)) : 1u;
                }
            }
            if (b < P::R1) {
                RowState<N>& s = st[ex.slot(tid)];
#pragma unroll
                for (int i = 0; i < P::R2; ++i) s.v[i] = smem[j * S::PA + b + P::R1 * i];
            }
        });
        ex.warp_phase([&](int tid) {
            const int j = tid / P::LANES, b = tid % P::LANES;
            if (b < P::R1) {
                if constexpr (RT) {
                    if constexpr (Exec::IS_HOST) P::load_tw(wreg, p.tw, b);
                    P::stepC(st[ex.slot(tid)].v, b, smem + j * S::PA, wreg);
                } else {
                    P::stepC(st[ex.slot(tid)].v, b, smem + j * S::PA, p.tw);
                }
            }
        });
        ex.phase([&](int tid) {
            const int j = tid / P::LANES, a = tid % P::LANES;
            float mx = neg_inf();
            if (a < P::R2) {
                float2 v[P::R1];
                P::stepD(v, a, smem + j * S::PA);
                const size_t row = (static_cast<size_t>(plane) * N + y0 + 2 * j) * N;
#pragma unroll
                for (int i = 0; i < P::R1; ++i) {
                    const float e = v[i].x * p.scale, o = v[i].y * p.scale;
                    if (p.out != nullptr && !fused) {
                        p.out[row + P::R2 * i + a] = e;
                        p.out[row + N + P::R2 * i + a] = o;
                    }
                    if constexpr (FUSABLE) cur[ex.slot(tid)].v[i] = make_float2(e, o);
                    mx = fmaxf(mx, fmaxf(e, o));
                }
            }
            ex.stage_max(mx, red, tid);
        });
        if (p.img_max != nullptr) {
            ex.phase([&](int tid) {
                if (tid == 0) {
                    float mx = red[0];
                    for (int k = 1; k < ex.staged(S::THREADS); ++k) mx = fmaxf(mx, red[k]);
                    if constexpr (FUSABLE && !Exec::IS_HOST) {
                        if (fused)
                            ex.key_store(reinterpret_cast<unsigned*>(p.arrive) + static_cast<size_t>(plane / 3) * SLOTS + t % (3 * TILES), mx);
                        else
                            atomic_max_float(p.img_max + plane / 3, mx);
                    } else {
                        atomic_max_float(p.img_max + plane / 3, mx);
                    }
                }
                if constexpr (FUSABLE) {
                    if (fused) {
                        if (it > 0) finish(tid, t - nctas, pre_k0, pre_k1);            // the previous tile's image is complete by now
#pragma unroll
                        for (int i = 0; i < P::R1; ++i) keep[ex.slot(tid)].v[i] = cur[ex.slot(tid)].v[i];
                    }
                }
            });
        }
    }
    if constexpr (FUSABLE) {
        if (fused && it > 0) ex.phase([&](int tid) { finish(tid, first + (it - 1) * nctas, (tid & 31) < NS0 ? 0u : 1u, (tid & 31) < NS1 ? 0u : 1u); });
    }
}

// ---------------------------------------------------------------------------------------------
// K4  normalise : y = conv / max_b  (Optics.py:128) + record positions that attain the max
//      (torch's amax backward splits the gradient evenly between exact ties)
//      1-D grid-stride over float4 elements; tie_pos[b][MAX_TIES], tie_count[b]
// ---------------------------------------------------------------------------------------------
constexpr int MAX_TIES = 8;
static_assert(MAX_TIES == C2R_MAX_TIES, "tie buffers");

struct NormaliseParams {
    float* y;               // [B][3][N][N] in place: conv -> sensor
    const float* img_max;   // [B]
    int* tie_count;         // [B]
    int* tie_pos;           // [B][MAX_TIES] flat index into (3,N,N)
    long long n4;           // number of float4 elements
    int per_image4;         // 3*N*N/4
    SensorEpilogue epi;
};

// Four independent float4 per thread and iteration (the kernel is a pure stream: keep loads in flight).
// y = conv * (1/max) instead of a division per element; the arg-max element itself is written as exactly 1.
// A CTA works on a slice of ONE image at a time (unit = image x slice): the maximum is loaded once per unit and no
// per-element index division is left (the flat-index version spent ~120 instructions per float4, 11.6 M warp instructions).
// Out = float: in place, p.y holds conv on entry and the sensor image on exit.  Out = bf16: p.y (the fp32 conv) is only
// read and the sensor image goes to `out`, each value the fp32 result rounded to nearest-even as the very last step (after
// the tie recording and the epilogue), i.e. exactly the fp32 image cast with torch.
// PHILOX: the Philox read-out (p.epi.seed): one philox_normal4 per float4, counter first4 + the float4's index in the batch.
template <class Out = float, bool PHILOX = false, class Exec>
B200_HD void normalise_body(Exec& ex, const NormaliseParams& p, int grid_x, Out* out = nullptr) {
    ex.phase([&](int tid) {
        constexpr int U = 4;
        NoiseSeed seed{0ull, 0ull};
        if constexpr (PHILOX) seed = load_seed(p.epi.seed);
        const int B = static_cast<int>(p.n4 / p.per_image4);
        const int spi = grid_x / B > 1 ? grid_x / B : 1;               // slices per image
        const int nthr = ex.nthreads();
        const int stride = spi * nthr;
        float4* y4 = reinterpret_cast<float4*>(p.y);
        for (int unit = ex.bx(); unit < B * spi; unit += grid_x) {
            const int b = unit / spi, sl = unit - b * spi;
            const float m = ld_ro(p.img_max + b);
            const float inv = 1.0f / m;
            float4* img4 = y4 + static_cast<size_t>(b) * p.per_image4;
            for (int i0 = sl * nthr + tid; i0 < p.per_image4; i0 += U * stride) {
                float4 v[U];
#pragma unroll
                for (int k = 0; k < U; ++k)
                    if (i0 + k * stride < p.per_image4) v[k] = img4[i0 + k * stride];
#pragma unroll
                for (int k = 0; k < U; ++k) {
                    const int i = i0 + k * stride;
                    if (i >= p.per_image4) continue;
                    float e[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
                    Normal4 nz{};
                    if constexpr (PHILOX) nz = philox_normal4(seed.key, seed.first4 + static_cast<unsigned long long>(b) * p.per_image4 + i);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        if (e[q] == m) {
                            const int slot = atomic_add_int(p.tie_count + b, 1);
                            if (slot < MAX_TIES) p.tie_pos[b * MAX_TIES + slot] = i * 4 + q;
                            e[q] = 1.0f;
                        } else {
                            e[q] *= inv;
                        }
                        if constexpr (PHILOX)
                            e[q] = quantise(p.epi, add_noise(p.epi, e[q], nz.n[q]));
                        else
                            e[q] = apply_epilogue(p.epi, e[q], (static_cast<size_t>(b) * p.per_image4 + i) * 4 + q);
                    }
                    if constexpr (sizeof(Out) == sizeof(float))
                        img4[i] = make_float4(e[0], e[1], e[2], e[3]);
                    else
                        store4(out, static_cast<long long>(b) * p.per_image4 + i, e[0], e[1], e[2], e[3]);
                }
            }
        }
    });
}

// The noise of the Philox read-out materialised (b200cam_sensor_noise): out[e] = n(e), n4 float4s, 1-D grid-stride
template <class Exec>
B200_HD void philox_noise_body(Exec& ex, const b200cam_noise_seed* seed_block, float* out, long long n4, int grid_x) {
    ex.phase([&](int tid) {
        const NoiseSeed seed = load_seed(seed_block);
        const long long stride = static_cast<long long>(grid_x) * ex.nthreads();
        for (long long i = static_cast<long long>(ex.bx()) * ex.nthreads() + tid; i < n4; i += stride) {
            const Normal4 nz = philox_normal4(seed.key, seed.first4 + static_cast<unsigned long long>(i));
            store4(out, i, nz.n[0], nz.n[1], nz.n[2], nz.n[3]);
        }
    });
}

// ---------------------------------------------------------------------------------------------
// K6  cols_accum : batch reduction of the backward pass in the frequency domain
//        acc[c][u][v] = sum_{b in chunk} conj(X_b[c][v,u]) * G_b[c][v,u] / max_b
//      (closed form of autograd through Utils.py:7-12 w.r.t. the kernel; SURVEY 8a row a14)
//      grid (ceil(3*NC/COLS), nchunks), block COLS*LANES.  Output partial[chunk][3][NC][N].
//      Deterministic: fixed b order inside a chunk, chunks summed in order by K7.
//
//      With `otf` the same registers also give the amax backward's  sum(g_b * conv_b)  (Optics.py:128) by
//      Parseval:  sum_{y,x} g conv = sum_{u<=N/2,v} wt_u Re( G conj(X K) ),  K = OTF (already / N^2), wt = 1 at
//      u = 0, N/2 and 2 elsewhere.  Every thread stores its own partial (dot_lanes[b][column][lane], summed in a
//      fixed order by K7) - the upstream gradient's row pass then needs no second operand (sensor image) at all.
// ---------------------------------------------------------------------------------------------
struct ColsAccumParams {
    const float2* stx;      // [B*3][NC][N] row-transformed image
    const float2* stg;      // [B*3][NC][N] row-transformed upstream gradient
    float2* partial;        // [nchunks][3][NC][N]
    const float2* tw;
    const float* img_max;   // [B]; nullptr: no per-image scale (plain convolution adjoint)
    const float2* otf;      // nullable [3][NC][N]: also emit the per-thread partials of sum(g * conv)
    float* dot_lanes;       // [B][3*NC][R1]
    int B;
    int nchunks;            // = gridDim.y: chunk y owns images [B*y/nchunks, B*(y+1)/nchunks) (balanced split)
    int discard_stg;        // stg is dead after this pass: drop its lines from L2 instead of writing them back
    // nullable [B][gridDim.x][WARPS]: the Parseval partials summed over each warp (one store per warp and image instead of one
    // per thread) - what the spectral arg-max term of K7 reads; dot_lanes is not written then
    float* dot_warps = nullptr;
};

template <int N>
struct AccumState {
    float2 acc[Plan<N>::R2];
};

template <int N, class Exec>
B200_HD void cols_accum_body(Exec& ex, const ColsAccumParams& p, float2* smem, AccumState<N>* st) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = ColsSmem<N>;
    float2* Ex = smem;
    float2* Eg = smem + S::COLS * P::E_SIZE;
    float2* stage_x = smem + S::STAGE_OFF;
    float2* stage_g = stage_x + S::STAGE1;
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + S::BAR_OFF_ACCUM);
    const int cu0 = ex.bx() * S::COLS;
    const int b0 = static_cast<int>(static_cast<long long>(p.B) * ex.by() / p.nchunks);
    const int b1 = static_cast<int>(static_cast<long long>(p.B) * (ex.by() + 1) / p.nchunks);
    constexpr int TOTAL = 3 * T::NC;
    constexpr bool RT = P::REG_TW;
    float2 wreg[RT ? P::R1 : 1];                 // the lane's twiddles, in registers for the whole chunk (see cols_conv)
    // lane 0 of warp w: bulk copies of the warp's columns of image b (both operands, one mbarrier) - see ColsSmem
    auto fetch = [&](int tid, int b) {
        const int w = tid / 32, cu = cu0 + w * S::WCOLS;
        if (tid % 32 == 0 && cu < TOTAL) {
            const int ncols = TOTAL - cu < S::WCOLS ? TOTAL - cu : S::WCOLS;
            const size_t off = (static_cast<size_t>(b) * TOTAL + cu) * N;
            ex.bulk_expect(bars + w, 2 * ncols * N * 8);
            ex.bulk_load(stage_x + w * S::WCOLS * N, p.stx + off, ncols * N * 8, bars + w);
            ex.bulk_load(stage_g + w * S::WCOLS * N, p.stg + off, ncols * N * 8, bars + w);
        }
    };

    ex.warp_phase([&](int tid) {
        AccumState<N>& s = st[ex.slot(tid)];
#pragma unroll
        for (int i = 0; i < P::R2; ++i) s.acc[i] = make_float2(0.f, 0.f);
        if constexpr (S::STAGED_ACCUM) {
            if (tid % 32 == 0) {
                ex.bulk_init(bars + tid / 32);
                ex.bulk_fence_init();
            }
            if (b0 < b1) fetch(tid, b0);
        }
        if constexpr (RT && !Exec::IS_HOST) P::load_tw(wreg, p.tw, tid % P::LANES);
    });
    for (int b = b0; b < b1; ++b) {
        ex.warp_phase([&](int tid) {
            const int jc = tid / P::LANES, a = tid % P::LANES;
            const int cu = cu0 + jc;
            if constexpr (S::STAGED_ACCUM) {
                if (cu0 + (tid / 32) * S::WCOLS < TOTAL) {
                    ex.bulk_wait(bars + tid / 32, (b - b0) & 1);
                    if (p.discard_stg) {             // the warp's WCOLS columns = WCOLS*N*8 bytes, one 128-byte line per lane and pass
                        const int wcu = cu0 + (tid / 32) * S::WCOLS;
                        const int ncols = TOTAL - wcu < S::WCOLS ? TOTAL - wcu : S::WCOLS;
                        const char* base = reinterpret_cast<const char*>(p.stg + (static_cast<size_t>(b) * TOTAL + wcu) * N);
                        for (int ln = tid % 32; ln < ncols * N * 8 / 128; ln += 32) discard_line(base + ln * 128);
                    }
                }
            }
            if (cu < TOTAL && a < P::R2) {
                const size_t off = (static_cast<size_t>(b) * TOTAL + cu) * N;
                float2 vx[P::R1], vg[P::R1];
#pragma unroll
                for (int i = 0; i < P::R1; ++i)
                    vx[i] = S::STAGED_ACCUM ? stage_x[jc * N + P::R2 * i + a] : ld_ro(p.stx + off + P::R2 * i + a);
#pragma unroll
                for (int i = 0; i < P::R1; ++i)
                    vg[i] = S::STAGED_ACCUM ? stage_g[jc * N + P::R2 * i + a] : ld_ro(p.stg + off + P::R2 * i + a);
                if constexpr (RT) {
                    if constexpr (Exec::IS_HOST) P::load_tw(wreg, p.tw, a);
                    P::stepA(vx, a, Ex + jc * P::E_SIZE, wreg);
                    P::stepA(vg, a, Eg + jc * P::E_SIZE, wreg);
                } else {
                    P::stepA(vx, a, Ex + jc * P::E_SIZE, p.tw);
                    P::stepA(vg, a, Eg + jc * P::E_SIZE, p.tw);
                }
            }
        });
        ex.warp_phase([&](int tid) {
            const int jc = tid / P::LANES, bb = tid % P::LANES;
            const int cu = cu0 + jc;
            if constexpr (S::STAGED_ACCUM) {
                if (b + 1 < b1) fetch(tid, b + 1);   // both slices are consumed (warp sync above): refill them
            }
            float dpart = 0.f;
            if (cu < TOTAL && bb < P::R1) {
                AccumState<N>& s = st[ex.slot(tid)];
                const float inv_m = p.img_max != nullptr ? 1.0f / ld_ro(p.img_max + b) : 1.0f;
                float2 vx[P::R2], vg[P::R2];
                P::stepB(vx, bb, Ex + jc * P::E_SIZE);
                P::stepB(vg, bb, Eg + jc * P::E_SIZE);
                float2 d2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < P::R2; ++i) {
                    const float2 t = cmulc(vg[i], vx[i]);   // G * conj(X)
                    if (p.otf != nullptr) {
                        // Re(G conj(X K)) = Re(t conj(K)) = t.x K.x + t.y K.y  (kept as two lanes: one packed FMA)
                        const float2 k = ld_ro(p.otf + static_cast<size_t>(cu) * N + bb + P::R1 * i);
                        d2.x += t.x * k.x;
                        d2.y += t.y * k.y;
                    }
                    s.acc[i].x += t.x * inv_m;
                    s.acc[i].y += t.y * inv_m;
                }
                if (p.otf != nullptr) {
                    const int u = cu % T::NC;
                    const float wt = (u == 0 || u == N / 2) ? 1.0f : 2.0f;
                    dpart = wt * (d2.x + d2.y);
                    if (p.dot_warps == nullptr) p.dot_lanes[(static_cast<size_t>(b) * TOTAL + cu) * P::R1 + bb] = dpart;
                }
            }
            if (p.otf != nullptr && p.dot_warps != nullptr)      // every lane of the warp: a CTA's tail columns contribute 0
                ex.warp_sum_store(dpart, p.dot_warps + (static_cast<size_t>(b) * ((TOTAL + S::COLS - 1) / S::COLS) + ex.bx()) * S::WARPS + tid / 32, tid);
        });
    }
    ex.warp_phase([&](int tid) {
        const int jc = tid / P::LANES, bb = tid % P::LANES;
        const int cu = cu0 + jc;
        if (cu < TOTAL && bb < P::R1) {
            const AccumState<N>& s = st[ex.slot(tid)];
            float2* dst = p.partial + (static_cast<size_t>(ex.by()) * TOTAL + cu) * N;
#pragma unroll
            for (int i = 0; i < P::R2; ++i) dst[bb + P::R1 * i] = s.acc[i];
        }
    });
}

// ---------------------------------------------------------------------------------------------
// K7  cols_reduce_inv : sum the chunk partials in order, apply (-1)^(u+v) (the adjoint of the
//      roll at Optics.py:126) and 1/N^2, inverse FFT along v -> ST layout for rows_c2r
// ---------------------------------------------------------------------------------------------
struct ColsReduceInvParams {
    const float2* partial;   // [nchunks][3][NC][N]
    float2* st;              // [3][NC][N]
    const float2* tw;
    int nchunks;
    float scale;
    // side job (dot_lanes != nullptr, grid = 3*NC + B): CTA 3*NC + b reduces image b's partials of sum(g*conv) written by K6 into
    //   coef[b] = sum(g_b*y_b) / (n_b m_b) = sum(g_b*conv_b) / (n_b m_b^2)     (weight of the arg-max term, Optics.py:128)
    const float* dot_lanes;  // nullable [B][3*NC*R1]
    const float* img_max;    // [B]
    const int* tie_count;    // [B]
    float* coef;             // [B]
    int B;
    // the side-job CTA of image b also pulls the planes that the arg-max term (K8) is about to gather from - x_b[c*] for every
    // recorded arg-max - into L2: K8 runs two small kernels later and would otherwise pay a DRAM miss per gather (the images
    // were last read a whole step ago)
    const void* x = nullptr;         // nullable [B][3][N][N] of x_elem-byte elements (fp32, or uint8: N^2 bytes per plane)
    const int* tie_pos = nullptr;    // [B][MAX_TIES]
    // Arg-max term of the amax backward folded into this pass (srow != nullptr; replaces K8 tie_term and its launch):
    //   gpsf[c][p] -= sum_t coef_t x_b[c][(p*_t - p + N/2) mod N]
    // is, after the row transform in x and BEFORE the one in y, a flipped copy of the image's own row-spectrum column:
    //   st[c][u][y'] -= scale N coef_t (-1)^u e^{-2 pi i u px_t / N} conj( X~_b[c][u][(py_t + N/2 - y') mod N] )
    // (X~ = srow, the row spectra kept from the forward) - no transform, 8 contiguous bytes per tie and output element.
    // coef_t comes from the warp partials of K6 (dot_warps), summed in a fixed order by the thread that stages the tie.
    const float2* srow = nullptr;    // nullable [B*3][NC][N]
    const float* dot_warps = nullptr;   // [B][dot_count]
    int dot_count = 0;
    int x_elem = 4;                  // bytes per element of x (4: fp32 images, 1: uint8 images)
};
constexpr int RINV_PASS = 64;        // images staged per pass of the tie list (<= RINV_PASS * MAX_TIES entries)

// grid 3*NC (one spectral column per CTA), block N (thread = v): the chunk sum is spread over N threads with
// coalesced 8N-byte reads; the first LANES threads then run the inverse transform of the column.
// shared: line[N] + E[E_SIZE] float2
template <int N>
struct ReduceInvSmem {
    static constexpr int THREADS = N;
    static constexpr int TIE_OFF = N + Plan<N>::E_SIZE;                       // float2 units
    // tie list of one pass: per entry {coef * phase (float2), image, source row} + per image {count, coef}
    static constexpr int TIE_FLOAT2S = RINV_PASS * 8 * 2 + RINV_PASS + 2;      // ... + per image {count, sum(g conv)} as 2 x 4 bytes
    static constexpr int FLOAT2S = TIE_OFF + TIE_FLOAT2S;
    static constexpr int BYTES = FLOAT2S * 8;
};

template <int N, class Exec>
B200_HD void cols_reduce_inv_body(Exec& ex, const ColsReduceInvParams& p, float2* smem) {
    using P = Plan<N>;
    using T = Tile<N>;
    float2* line = smem;
    float2* E = smem + N;
    const int cu = ex.bx();
    constexpr int TOTAL = 3 * T::NC;
    const int u = cu % T::NC;
    if (cu >= TOTAL) {
        // extra CTAs (grid = 3*NC + B when dot_lanes is given): CTA TOTAL + b reduces image b's Parseval partials, beside -
        // not in front of - the column work of the other CTAs
        const int PER_IMAGE = p.dot_warps != nullptr ? p.dot_count : TOTAL * P::R1;
        float* red = reinterpret_cast<float*>(E);
        const int b = cu - TOTAL;
        if (p.x != nullptr && p.tie_pos != nullptr) {
            ex.phase([&](int t) {
                const int n = p.tie_count[b] < C2R_MAX_TIES ? p.tie_count[b] : C2R_MAX_TIES;
                for (int k = 0; k < n; ++k) {
                    const int c = p.tie_pos[b * C2R_MAX_TIES + k] / (N * N);
                    const char* plane = static_cast<const char*>(p.x) + (static_cast<size_t>(b) * 3 + c) * N * N * p.x_elem;
                    for (int line = t; line < N * N * p.x_elem / 128; line += N) prefetch_l2(plane + static_cast<size_t>(line) * 128);
                }
            });
        }
        ex.phase([&](int t) {
            const float* src = (p.dot_warps != nullptr ? p.dot_warps : p.dot_lanes) + static_cast<size_t>(b) * PER_IMAGE;
            float s = 0.f;
            int i = t;
            for (; i + 7 * N < PER_IMAGE; i += 8 * N) {              // eight loads in flight; fixed order: deterministic
                float v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) v[k] = src[i + k * N];
#pragma unroll
                for (int k = 0; k < 8; ++k) s += v[k];
            }
            for (; i < PER_IMAGE; i += N) s += src[i];
            red[t] = s;
        });
        ex.phase([&](int t) {
            if (t < 16) {
                float s = 0.f;
                for (int i = t; i < N; i += 16) s += red[i];
                red[N + t] = s;
            }
        });
        ex.phase([&](int t) {
            if (t == 0) {
                float s = 0.f;
                for (int i = 0; i < 16; ++i) s += red[N + i];
                const int n = p.tie_count[b] > 0 ? p.tie_count[b] : 1;
                const float m = p.img_max[b];
                p.coef[b] = s / (static_cast<float>(n) * m * m);
            }
        });
        return;
    }
    // ---- arg-max term (see ColsReduceInvParams::srow): its staging runs INSIDE the phases of the column work ----
    using RS = ReduceInvSmem<N>;
    const bool spectral = p.srow != nullptr && p.dot_warps != nullptr && p.tie_pos != nullptr;
    const int c = cu / T::NC;
    float2* t_w = smem + RS::TIE_OFF;                                            // [PASS*8] coef * phase
    int* t_meta = reinterpret_cast<int*>(smem + RS::TIE_OFF + RINV_PASS * 8);    // [PASS*8][2] image, source row
    int* t_cnt = reinterpret_cast<int*>(smem + RS::TIE_OFF + RINV_PASS * 8 * 2); // [PASS + 1] ties of this channel per image
    float* t_sdot = reinterpret_cast<float*>(t_cnt + RINV_PASS + 1);             // [PASS] sum(g_b conv_b)
    float2 acc = make_float2(0.f, 0.f);                                          // thread y' (device: lives across the passes)
    float2 acc_host[Exec::IS_HOST ? N : 1];
    if constexpr (Exec::IS_HOST)
        for (int i = 0; i < N; ++i) acc_host[i] = make_float2(0.f, 0.f);
    // (1) ties of this channel per image of the pass
    auto tie_count = [&](int t, int b0, int nb) {
        for (int i = t; i < nb; i += N) {
            const int b = b0 + i;
            const int n = p.tie_count[b] < C2R_MAX_TIES ? p.tie_count[b] : C2R_MAX_TIES;
            int cnt = 0;
            for (int k = 0; k < n; ++k) cnt += (p.tie_pos[b * C2R_MAX_TIES + k] / (N * N) == c) ? 1 : 0;
            t_cnt[i] = cnt;
        }
    };
    // (2) sum(g_b * conv_b) of the images that have an arg-max here: one warp per image, the lanes stride over the warp
    //     partials of K6, fixed shuffle tree (a single thread adding them one after the other pays a load latency each)
    auto tie_sdot = [&](int t, int b0, int nb) {
        constexpr int NW = N / 32 > 0 ? N / 32 : 1;
        for (int i = t / 32; i < nb; i += NW) {
            if (t_cnt[i] == 0) continue;                                        // uniform over the warp
            const float* d = p.dot_warps + static_cast<size_t>(b0 + i) * p.dot_count;
            float part = 0.f;
            for (int q0 = t % 32; q0 < p.dot_count; q0 += 8 * 32) {             // eight loads in flight per lane, fixed order
                float vals[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) vals[k] = q0 + 32 * k < p.dot_count ? ld_ro(d + q0 + 32 * k) : 0.f;
#pragma unroll
                for (int k = 0; k < 8; ++k) part += vals[k];
            }
            ex.warp_sum_store(part, t_sdot + i, t);
        }
    };
    // (3) the list {coef * phase, image, source row}; ordered by image: the sum order is fixed
    auto tie_list = [&](int t, int b0, int nb) {
        for (int i = t; i < nb; i += N) {
            if (t_cnt[i] == 0) continue;
            int k0 = 0;
            for (int q = 0; q < i; ++q) k0 += t_cnt[q];
            const int b = b0 + i;
            const int nt = p.tie_count[b] > 0 ? p.tie_count[b] : 1;
            const float m = ld_ro(p.img_max + b);
            const float coef = t_sdot[i] / (static_cast<float>(nt) * m * m) * p.scale * static_cast<float>(N);
            const int n = p.tie_count[b] < C2R_MAX_TIES ? p.tie_count[b] : C2R_MAX_TIES;
            for (int k = 0; k < n; ++k) {
                const int pos = p.tie_pos[b * C2R_MAX_TIES + k];
                if (pos / (N * N) != c) continue;
                const int py = (pos % (N * N)) / N, px = pos % N;
                const float2 ph = ld_ro(p.tw + ((u * px) & (N - 1)));              // e^{-2 pi i u px / N}
                const float sg = (u & 1) ? -coef : coef;
                t_w[k0] = make_float2(sg * ph.x, sg * ph.y);
                t_meta[2 * k0] = b;
                t_meta[2 * k0 + 1] = (py + N / 2) & (N - 1);
                ++k0;
            }
        }
        if (t == 0) {
            int tot = 0;
            for (int q = 0; q < nb; ++q) tot += t_cnt[q];
            t_cnt[RINV_PASS] = tot;
        }
    };
    // (4) thread y': the listed row-spectrum columns, flipped; eight gathers in flight, fixed order
    auto tie_gather = [&](int y) {
        const int tot = t_cnt[RINV_PASS];
        float2 a2 = Exec::IS_HOST ? acc_host[Exec::IS_HOST ? y : 0] : acc;
        constexpr int G = 12;                      // gathers in flight per thread
        for (int e0 = 0; e0 < tot; e0 += G) {
            // Unconditional loads (clamped index) and unconditional FMAs (zero weight past the end): a conditional use lets
            // the compiler sink each load next to its use - measured: 4 of 8 loads exposed their full latency one by one
            float2 xs[G], ws[G];
#pragma unroll
            for (int k = 0; k < G; ++k) {
                const int e = e0 + k < tot ? e0 + k : tot - 1;
                xs[k] = ld_ro(p.srow + (static_cast<size_t>(t_meta[2 * e] * 3 + c) * T::NC + u) * N + ((t_meta[2 * e + 1] - y) & (N - 1)));
                const float2 w = t_w[e];
                ws[k] = e0 + k < tot ? w : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int k = 0; k < G; ++k) {                                       // w * conj(xs)
                a2.x += ws[k].x * xs[k].x + ws[k].y * xs[k].y;
                a2.y += ws[k].y * xs[k].x - ws[k].x * xs[k].y;
            }
        }
        if constexpr (Exec::IS_HOST) acc_host[Exec::IS_HOST ? y : 0] = a2;
        else acc = a2;
    };
    const int nb0 = p.B < RINV_PASS ? p.B : RINV_PASS;

    ex.phase([&](int v) {
        const float2* src = p.partial + static_cast<size_t>(cu) * N + v;
        const size_t step = static_cast<size_t>(TOTAL) * N;
        float2 s = make_float2(0.f, 0.f);
        for (int ch0 = 0; ch0 < p.nchunks; ch0 += 8) {   // eight chunk loads in flight; fixed order: deterministic
            float2 tv[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) tv[k] = ch0 + k < p.nchunks ? ld_ro(src + (ch0 + k) * step) : make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 0; k < 8; ++k) s = cadd(s, tv[k]);
        }
        line[v] = cscale(s, ((u + v) & 1) ? -p.scale : p.scale);
        if (spectral) tie_count(v, 0, nb0);
    });
    ex.phase([&](int b) {
        if (b < P::R1) {
            float2 q[P::R2];
#pragma unroll
            for (int i = 0; i < P::R2; ++i) q[i] = line[b + P::R1 * i];
            P::stepC(q, b, E, p.tw);
        }
        if (spectral) tie_sdot(b, 0, nb0);
    });
    ex.phase([&](int a) {
        if (a < P::R2) {
            float2 q[P::R1];
            P::stepD(q, a, E);
            float2* dst = spectral ? line : p.st + static_cast<size_t>(cu) * N;     // spectral: the tie term is subtracted first
#pragma unroll
            for (int i = 0; i < P::R1; ++i) dst[P::R2 * i + a] = q[i];
        }
        if (spectral) tie_list(a, 0, nb0);
    });
    if (!spectral) return;
    ex.phase([&](int y) { tie_gather(y); });
    for (int b0 = RINV_PASS; b0 < p.B; b0 += RINV_PASS) {       // further passes (batches above RINV_PASS images)
        const int nb = p.B - b0 < RINV_PASS ? p.B - b0 : RINV_PASS;
        ex.phase([&](int t) { tie_count(t, b0, nb); });
        ex.phase([&](int t) { tie_sdot(t, b0, nb); });
        ex.phase([&](int t) { tie_list(t, b0, nb); });
        ex.phase([&](int y) { tie_gather(y); });
    }
    ex.phase([&](int y) {
        const float2 a2 = Exec::IS_HOST ? acc_host[Exec::IS_HOST ? y : 0] : acc;
        const float2 v = line[y];
        p.st[static_cast<size_t>(cu) * N + y] = make_float2(v.x - a2.x, v.y - a2.y);
    });
}

// ---------------------------------------------------------------------------------------------
// K8  tie_term : the arg-max part of the amax backward, in the spatial domain
//      gpsf[c][p] -= sum_b sum_{ties t of image b in channel c} (s_b/(n_b m_b)) * x_b[c][(p*_t - p + N/2) mod N]
//      with s_b = sum(g_b * y_b) from the Parseval partials of K6, reduced by K7 (coef).
//      grid-stride over 3*N*N outputs.
//      `Img` = u8: the gather reads the uint8 image and converts each value in registers (to_float), so every gathered
//      value - and with it the sum, in the same order - is that of the fp32 kernel on the converted image.
// ---------------------------------------------------------------------------------------------
template <class Img>
struct TieTermParamsT {
    float* gpsf;              // [3][N][N] in place
    const Img* x;             // [B][3][N][N]
    const int* tie_count;     // [B]
    const int* tie_pos;       // [B][MAX_TIES]
    const float* coef;        // [B]: s_b / (n_b m_b), written by K7
    int B, N;
};
using TieTermParams = TieTermParamsT<float>;

constexpr int TIE_PASS = 256;   // images staged per pass (= block size of the kernel)

// grid (blocks_per_channel, 3), block TIE_PASS.  A block only applies the ties of its own channel.
// Staging is parallel (thread t <-> image b0+t) and the compaction offsets come from an ordered
// scan, so the list - and therefore the floating-point subtraction order - is deterministic.
// shared: s_coef[TIE_PASS*MAX_TIES], s_meta[3*TIE_PASS*MAX_TIES], s_cnt[TIE_PASS+1]
template <class Exec, class Img>
B200_HD void tie_term_body(Exec& ex, const TieTermParamsT<Img>& p, int grid_x, float* s_coef, int* s_meta, int* s_cnt) {
    const int N = p.N, NN = N * N, c = ex.by();
    for (int b0 = 0; b0 < p.B; b0 += TIE_PASS) {
        const int nb = (p.B - b0 < TIE_PASS) ? p.B - b0 : TIE_PASS;
        ex.phase([&](int tid) {
            int cnt = 0;
            if (tid < nb) {
                const int b = b0 + tid;
                const int n = p.tie_count[b] < MAX_TIES ? p.tie_count[b] : MAX_TIES;
                for (int t = 0; t < n; ++t) cnt += (p.tie_pos[b * MAX_TIES + t] / NN == c) ? 1 : 0;
            }
            if (tid < TIE_PASS) s_cnt[tid] = cnt;
        });
        ex.phase([&](int tid) {
            if (tid < nb) {
                // exclusive prefix of the counts: every thread sums the (broadcast) counts below it - no serial scan
                int k = 0;
                for (int t = 0; t < tid; ++t) k += s_cnt[t];
                if (tid == nb - 1) s_cnt[TIE_PASS] = k + s_cnt[tid];
                const int b = b0 + tid;
                const int n = p.tie_count[b] < MAX_TIES ? p.tie_count[b] : MAX_TIES;
                for (int t = 0; t < n; ++t) {
                    const int pos = p.tie_pos[b * MAX_TIES + t];
                    if (pos / NN != c) continue;
                    s_coef[k] = p.coef[b];
                    s_meta[3 * k + 0] = b;
                    s_meta[3 * k + 1] = (pos % NN) / N;
                    s_meta[3 * k + 2] = pos % N;
                    ++k;
                }
            }
        });
        ex.phase([&](int tid) {
            const int k = s_cnt[TIE_PASS];
            if (k > 0) {
                // a thread owns two adjacent pixels; 16 ties x 2 pixels = 32 gathers in flight (they miss L2: the images
                // were last read a whole step ago).  Tail entries are clamped to the last valid one and skipped in the
                // sum: same additions, fixed order.
                const int stride = grid_x * ex.nthreads();
                for (int idx = ex.bx() * ex.nthreads() + tid; idx < NN / 2; idx += stride) {
                    const int py = idx / (N / 2), px = 2 * (idx % (N / 2));
                    float acc0 = 0.f, acc1 = 0.f;
                    for (int e = 0; e < k; e += 16) {
                        float v0[16], v1[16];
#pragma unroll
                        for (int q = 0; q < 16; ++q) {
                            const int ee = e + q < k ? e + q : k - 1;
                            const int sy = (s_meta[3 * ee + 1] - py + N / 2 + N) & (N - 1);
                            const int sx = (s_meta[3 * ee + 2] - px + N / 2 + N) & (N - 1);
                            const Img* row = p.x + (static_cast<size_t>(s_meta[3 * ee]) * 3 + c) * NN + sy * N;
                            v0[q] = load_elem(row + sx);
                            v1[q] = load_elem(row + ((sx - 1) & (N - 1)));
                        }
#pragma unroll
                        for (int q = 0; q < 16; ++q) {
                            // unconditional FMAs (zero weight past the end): with a conditional use the compiler sinks each
                            // load next to its use and the gathers expose their latency one by one (seen in SASS, round 2)
                            const float cf = e + q < k ? s_coef[e + q] : 0.f;
                            acc0 += cf * v0[q];
                            acc1 += cf * v1[q];
                        }
                    }
                    float2* dst = reinterpret_cast<float2*>(p.gpsf + c * NN + py * N + px);
                    const float2 old = *dst;
                    *dst = make_float2(old.x - acc0, old.y - acc1);
                }
            }
        });
    }
}

// K9  tie_term_img : the same arg-max term for dL/dimg (optional output)
//      gimg[b][c][q] -= coef_b * sum_{ties t of b in channel c} psf[c][(p*_t - q + N/2) mod N]
struct TieTermImgParams {
    float* gimg;              // [B][3][N][N] in place
    const float* psf;         // [3][N][N] centred
    const int* tie_count;
    const int* tie_pos;
    const float* coef;        // [B]
    int B, N;
};

template <class Exec>
B200_HD void tie_term_img_body(Exec& ex, const TieTermImgParams& p, int grid_x) {
    ex.phase([&](int tid) {
        const int N = p.N, NN = N * N;
        const long long total = static_cast<long long>(p.B) * 3 * NN;
        const long long stride = static_cast<long long>(grid_x) * ex.nthreads();
        for (long long idx = static_cast<long long>(ex.bx()) * ex.nthreads() + tid; idx < total; idx += stride) {
            const int b = static_cast<int>(idx / (3 * NN));
            const int r = static_cast<int>(idx % (3 * NN));
            const int c = r / NN, qy = (r % NN) / N, qx = r % N;
            const int n = p.tie_count[b] < MAX_TIES ? p.tie_count[b] : MAX_TIES;
            float acc = 0.f;
            for (int t = 0; t < n; ++t) {
                const int pos = p.tie_pos[b * MAX_TIES + t];
                if (pos / NN != c) continue;
                const int ty = (pos % NN) / N, tx = pos % N;
                const int sy = (ty - qy + N / 2 + N) & (N - 1), sx = (tx - qx + N / 2 + N) & (N - 1);
                acc += ld_ro(p.psf + c * NN + sy * N + sx);
            }
            if (acc != 0.f) p.gimg[idx] -= p.coef[b] * acc;
        }
    });
}

// =============================================================================================
//                      PSF chain (complex fields, 3 wavelengths)
// =============================================================================================

// loaders / epilogues of the complex row passes
// Loaders are split in two stages - fetch() only issues the global loads, make() does the arithmetic - so that a
// row's 16/32 elements are all in flight before the first one is used (the PSF chain is a latency chain).
struct PupilLoad {     // V = A * exp(i*kappa_l*h)   (Optics.py:89-100)
    const float2* A;   // [3][N][N] constant pupil table (aperture, lens, defocus and pre-phase)
    const float* h;    // [N][N]
    float kappa[3];
    int N;
    struct Raw { float2 a; float h; };
    // selects instead of kappa[l]: a dynamically indexed kernel-parameter array is copied to local memory
    B200_HD float kap(int l) const { return l == 0 ? kappa[0] : (l == 1 ? kappa[1] : kappa[2]); }
    B200_HD void bind(float*) {}
    template <class Exec>
    B200_HD void prologue(Exec&, float*) const {}
    B200_HD Raw fetch(int l, int y, int x) const {
        const size_t i = static_cast<size_t>(y) * N + x;
        return Raw{ld_ro(A + static_cast<size_t>(l) * N * N + i), ld_ro(h + i)};
    }
    B200_HD float2 make(int l, const Raw& r) const {
        float s, c;
#if defined(__CUDA_ARCH__)
        // exp(i phi) through sincospi: exact range reduction, straight-line code (sincosf carries a Payne-Hanek slow
        // path with a stack frame, which keeps the 16 evaluations of a row from overlapping).  phi/pi costs one
        // rounding of the argument: |error| <= 6e-8 |phi| rad.
        sincospif((kap(l) * r.h) * 0.31830988618379067154f, &s, &c);
#else
        const float phi = kap(l) * r.h;
        s = sinf(phi); c = cosf(phi);
#endif
        return cmul(r.a, make_float2(c, s));
    }
    B200_HD float2 operator()(int l, int y, int x) const { return make(l, fetch(l, y, x)); }
};

struct GradFieldLoad {  // GU = 2 * (gtot - dot)/S * U      (adjoint of |U|^2 / sum, Optics.py:109-110)
    const float2* U;       // [3][N][N]
    const float* gtot;     // [3][N][N]
    const float* scal;     // device scalars: [0]=S
    const float* partial;  // [npartial] partial sums of gtot*psf written by psf_grad_prepare
    float* dot_smem;       // two floats of shared memory: dot = sum(partial) (reduced by every CTA in the same order), 2/S
    int npartial;
    int N;
    struct Raw { float2 u; float g; };
    B200_HD void bind(float* scratch) { dot_smem = scratch; }
    template <class Exec>
    B200_HD void prologue(Exec& ex, float* red) const {
        const int nt = ex.nthreads();
        ex.phase([&](int tid) {
            float acc = 0.f;
            for (int i = tid; i < npartial; i += nt) acc += partial[i];
            red[tid] = acc;
        });
        ex.phase([&](int tid) {
            if (tid == 0) {
                float s = 0.f;
                for (int t = 0; t < nt; ++t) s += red[t];
                dot_smem[0] = s;
                dot_smem[1] = 2.0f / ld_ro(scal + 0);
            }
        });
    }
    B200_HD Raw fetch(int l, int y, int x) const {
        const size_t i = (static_cast<size_t>(l) * N + y) * N + x;
        return Raw{ld_ro(U + i), ld_ro(gtot + i)};
    }
    B200_HD float2 make(int, const Raw& r) const { return cscale(r.u, (r.g - dot_smem[0]) * dot_smem[1]); }
};

// P1  crows_fwd : complex rows -> transposed full spectrum.  grid (N/CROWS, 3), block CROWS*LANES
template <int N>
struct CRowsSmem {
    using P = Plan<N>;
    using T = Tile<N>;
    static constexpr int THREADS = T::CROWS * P::LANES;
    static constexpr int E_OFF = 0;
    static constexpr int F_OFF = T::CROWS * P::E_SIZE;
    static constexpr int RED_OFF = F_OFF + T::CROWS * T::FP_CROW;
    static constexpr int FLOAT2S = RED_OFF + THREADS + 2;   // 2 floats per thread of scratch + 2 scalars
    static constexpr int BYTES = FLOAT2S * 8;
};

struct CRowsFwdParams {
    float2* st;         // [3][N][N] transposed: st[l][u][y]
    const float2* tw;
};

template <int N, class Load, class Exec>
B200_HD void crows_fwd_body(Exec& ex, const CRowsFwdParams& p, Load load, float2* smem) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = CRowsSmem<N>;
    const int tile = ex.bx(), l = ex.by();
    const int y0 = tile * T::CROWS;
    float2* E = smem + S::E_OFF;
    float2* F = smem + S::F_OFF;
    load.bind(reinterpret_cast<float*>(smem + S::RED_OFF) + S::THREADS);
    load.prologue(ex, reinterpret_cast<float*>(smem + S::RED_OFF));
    ex.phase([&](int tid) {
        const int j = tid / P::LANES, a = tid % P::LANES;
        if (a < P::R2) {
            typename Load::Raw raw[P::R1];
#pragma unroll
            for (int i = 0; i < P::R1; ++i) raw[i] = load.fetch(l, y0 + j, P::R2 * i + a);
            float2 v[P::R1];
#pragma unroll
            for (int i = 0; i < P::R1; ++i) v[i] = load.make(l, raw[i]);
            P::stepA(v, a, E + j * P::E_SIZE, p.tw);
        }
    });
    ex.phase([&](int tid) {
        const int j = tid / P::LANES, b = tid % P::LANES;
        if (b < P::R1) {
            float2 v[P::R2];
            P::stepB(v, b, E + j * P::E_SIZE);
#pragma unroll
            for (int i = 0; i < P::R2; ++i) F[j * T::FP_CROW + b + P::R1 * i] = v[i];
        }
    });
    ex.phase([&](int tid) {
        for (int w = tid; w < T::CROWS * N; w += S::THREADS) {
            const int u = w / T::CROWS, j = w % T::CROWS;
            p.st[(static_cast<size_t>(l) * N + u) * N + y0 + j] = F[j * T::FP_CROW + u];
        }
    });
}

// P2  ccols_mix : per spectral column u, for the three wavelengths together:
//      FFT_v, 3-point DFT across wavelength, x H_m (or conj), inverse 3-point DFT, IFFT_v, in place.
//      This is `fftn` / `ifftn` WITHOUT a dim argument at Optics.py:101,105 (they also transform
//      the wavelength axis; H is indexed by the DFT bin m - SURVEY trap T1).
//      grid ceil(N/CC), block CC*3*LANES.  H layout [m][u][v] (the reference's table transposed);
//      scale = 1/(3 N^2) makes the pair an exact (normalised) inverse.
struct CColsMixParams {
    float2* st;         // [3][N][N] transposed, in place
    const float2* H;    // [3][N][N] TRANSPOSED (m, u, v) so that a column's run is contiguous
    const float2* tw;
    int conj_h;
    float scale;
};

template <int N>
struct CColsSmem {
    using P = Plan<N>;
    // columns per CTA: 128 CTAs at N=256.  N = 1024: two columns need 149 KB of shared memory = one CTA per SM and 512 CTAs in
    // 3.5 rounds; one column per CTA (75 KB, three CTAs per SM, 1024 CTAs in 2.3 shorter rounds) is faster
    static constexpr int CC = N >= 1024 ? 1 : 2;
    static constexpr int THREADS = CC * 3 * P::LANES;
    static constexpr int E_OFF = 0;
    static constexpr int G_OFF = CC * 3 * P::E_SIZE;  // natural-order exchange for the 3-pt DFT
    static constexpr int GP = N + 1;
    static constexpr int FLOAT2S = G_OFF + 2 * CC * 3 * GP;
    static constexpr int BYTES = FLOAT2S * 8;
};

template <int N, class Exec>
B200_HD void ccols_mix_body(Exec& ex, const CColsMixParams& p, float2* smem) {
    using P = Plan<N>;
    using S = CColsSmem<N>;
    float2* E = smem + S::E_OFF;
    float2* G1 = smem + S::G_OFF;
    float2* G2 = G1 + S::CC * 3 * S::GP;
    const int u0 = ex.bx() * S::CC;
    // w3 = exp(-2*pi*i/3)
    const float2 w3 = make_float2(-0.5f, -0.86602540378443864676f);

    ex.phase([&](int tid) {
        const int f = tid / P::LANES, a = tid % P::LANES;   // f = jc*3 + l
        const int jc = f / 3, l = f % 3, u = u0 + jc;
        if (u < N && a < P::R2) {
            const float2* src = p.st + (static_cast<size_t>(l) * N + u) * N;
            float2 v[P::R1];
#pragma unroll
            for (int i = 0; i < P::R1; ++i) v[i] = src[P::R2 * i + a];
            P::stepA(v, a, E + f * P::E_SIZE, p.tw);
        }
    });
    ex.phase([&](int tid) {
        const int f = tid / P::LANES, b = tid % P::LANES;
        const int u = u0 + f / 3;
        if (u < N && b < P::R1) {
            float2 v[P::R2];
            P::stepB(v, b, E + f * P::E_SIZE);
#pragma unroll
            for (int i = 0; i < P::R2; ++i) G1[f * S::GP + b + P::R1 * i] = v[i];
        }
    });
    ex.phase([&](int tid) {
        // thread (jc, m, b): W_m[k] = H_m[k,u] * sum_l w3^(m*l) Vhat_l[k]
        const int f = tid / P::LANES, b = tid % P::LANES;
        const int jc = f / 3, m = f % 3, u = u0 + jc;
        if (u < N && b < P::R1) {
            const float2 wa = (m == 0) ? make_float2(1.f, 0.f) : (m == 1 ? w3 : cconj(w3));   // w3^m
            const float2 wb = (m == 0) ? make_float2(1.f, 0.f) : (m == 1 ? cconj(w3) : w3);   // w3^(2m)
            float2 h[P::R2];                        // the transfer function is not in L2 any more: all loads first
#pragma unroll
            for (int i = 0; i < P::R2; ++i) h[i] = ld_ro(p.H + (static_cast<size_t>(m) * N + u) * N + b + P::R1 * i);
#pragma unroll
            for (int i = 0; i < P::R2; ++i) {
                const int k = b + P::R1 * i;
                const float2 a0 = G1[(jc * 3 + 0) * S::GP + k];
                const float2 a1 = G1[(jc * 3 + 1) * S::GP + k];
                const float2 a2 = G1[(jc * 3 + 2) * S::GP + k];
                const float2 s = cadd(a0, cadd(cmul(a1, wa), cmul(a2, wb)));
                G2[f * S::GP + k] = p.conj_h ? cmulc(s, h[i]) : cmul(s, h[i]);
            }
        }
    });
    ex.phase([&](int tid) {
        // thread (jc, l', b): out_l'[k] = scale * sum_m conj(w3)^(m*l') W_m[k]; then IFFT along v
        const int f = tid / P::LANES, b = tid % P::LANES;
        const int jc = f / 3, l = f % 3, u = u0 + jc;
        if (u < N && b < P::R1) {
            const float2 wa = (l == 0) ? make_float2(1.f, 0.f) : (l == 1 ? cconj(w3) : w3);
            const float2 wb = (l == 0) ? make_float2(1.f, 0.f) : (l == 1 ? w3 : cconj(w3));
            float2 v[P::R2];
#pragma unroll
            for (int i = 0; i < P::R2; ++i) {
                const int k = b + P::R1 * i;
                const float2 a0 = G2[(jc * 3 + 0) * S::GP + k];
                const float2 a1 = G2[(jc * 3 + 1) * S::GP + k];
                const float2 a2 = G2[(jc * 3 + 2) * S::GP + k];
                v[i] = cscale(cadd(a0, cadd(cmul(a1, wa), cmul(a2, wb))), p.scale);
            }
            P::stepC(v, b, E + f * P::E_SIZE, p.tw);
        }
    });
    ex.phase([&](int tid) {
        const int f = tid / P::LANES, a = tid % P::LANES;
        const int jc = f / 3, l = f % 3, u = u0 + jc;
        if (u < N && a < P::R2) {
            float2 v[P::R1];
            P::stepD(v, a, E + f * P::E_SIZE);
            float2* dst = p.st + (static_cast<size_t>(l) * N + u) * N;
#pragma unroll
            for (int i = 0; i < P::R1; ++i) dst[P::R2 * i + a] = v[i];
        }
    });
}

// P3  crows_inv : transposed spectrum (already inverse-transformed along v) -> complex rows,
//      with an epilogue functor.  grid (N/ROWS, 3), block ROWS*LANES.
struct CRowsInvParams {
    const float2* st;   // [3][N][N] transposed
    const float2* tw;
};

// forward epilogue: save the field, emit intensity and a per-CTA partial sum (Optics.py:109-110)
struct IntensityEpilogue {
    float2* U;          // [3][N][N]
    float* I;           // [3][N][N]
    float* partial;     // [3][N/CROWS]
    int* arrive;        // counter of psf_finalise, zeroed here (it runs next in the stream)
    int N;
    // nullable [3][NC][N]: the CTA also row-transforms its rows of |U|^2 (pairs of real rows as one complex transform) into the
    // transposed half spectrum the OTF's column pass starts from - the first half of rfft2(psf) (Utils.py:9) without a kernel
    // of its own in the latency chain of the step's head
    float2* otf_rows = nullptr;
    B200_HD float operator()(int l, int y, int x, float2 v) const {
        const size_t i = (static_cast<size_t>(l) * N + y) * N + x;
        U[i] = v;
        const float in = v.x * v.x + v.y * v.y;
        I[i] = in;
        return in;
    }
    B200_HD void finish(int l, int tile, int tiles, float s) const {
        partial[l * tiles + tile] = s;
        if (l == 0 && tile == 0) *arrive = 0;
    }
};

template <int N, class Epi, class Exec>
B200_HD void crows_inv_body(Exec& ex, const CRowsInvParams& p, const Epi& epi, float2* smem) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = CRowsSmem<N>;
    const int tile = ex.bx(), l = ex.by();
    const int y0 = tile * T::CROWS;
    float2* E = smem + S::E_OFF;
    float2* F = smem + S::F_OFF;
    float* Irow = reinterpret_cast<float*>(F);                     // [CROWS][N] intensities (OTF row transform)
    float* red = reinterpret_cast<float*>(smem + S::RED_OFF);
    ex.phase([&](int tid) {
        constexpr int ITEMS = T::CROWS * N / S::THREADS;         // loads first, stores after (latency chain)
        float2 q[ITEMS];
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const int w = tid + k * S::THREADS;
            q[k] = ld_ro(p.st + (static_cast<size_t>(l) * N + w / T::CROWS) * N + y0 + w % T::CROWS);
        }
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const int w = tid + k * S::THREADS;
            F[(w % T::CROWS) * T::FP_CROW + w / T::CROWS] = q[k];
        }
    });
    ex.phase([&](int tid) {
        const int j = tid / P::LANES, b = tid % P::LANES;
        if (b < P::R1) {
            float2 v[P::R2];
#pragma unroll
            for (int i = 0; i < P::R2; ++i) v[i] = F[j * T::FP_CROW + b + P::R1 * i];
            P::stepC(v, b, E + j * P::E_SIZE, p.tw);
        }
    });
    ex.phase([&](int tid) {
        const int j = tid / P::LANES, a = tid % P::LANES;
        float s = 0.f;
        if (a < P::R2) {
            float2 v[P::R1];
            P::stepD(v, a, E + j * P::E_SIZE);
#pragma unroll
            for (int i = 0; i < P::R1; ++i) {
                const float in = epi(l, y0 + j, P::R2 * i + a, v[i]);
                s += in;
                if (epi.otf_rows != nullptr) Irow[j * N + P::R2 * i + a] = in;     // F is free: phase 2 consumed it
            }
        }
        red[tid] = s;
    });
    if (epi.otf_rows != nullptr) {
        // rows (2jp, 2jp+1) of |U|^2 as ONE complex transform, un-mixed by Hermitian symmetry - as K1 (rows_r2c) does
        constexpr int PAIRS = T::CROWS / 2;
        static_assert(T::CROWS % 2 == 0, "row pairs");
        ex.phase([&](int tid) {
            const int jp = tid / P::LANES, a = tid % P::LANES;
            if (jp < PAIRS && a < P::R2) {
                float2 v[P::R1];
#pragma unroll
                for (int i = 0; i < P::R1; ++i)
                    v[i] = make_float2(Irow[(2 * jp) * N + P::R2 * i + a], Irow[(2 * jp + 1) * N + P::R2 * i + a]);
                P::stepA(v, a, E + jp * P::E_SIZE, p.tw);
            }
        });
        ex.phase([&](int tid) {
            const int jp = tid / P::LANES, b = tid % P::LANES;
            if (jp < PAIRS && b < P::R1) {
                float2 q[P::R2];
                P::stepB(q, b, E + jp * P::E_SIZE);
#pragma unroll
                for (int i = 0; i < P::R2; ++i) F[jp * N + b + P::R1 * i] = q[i];     // the intensities are consumed: reuse F
            }
        });
        ex.phase([&](int tid) {
            for (int w = tid; w < PAIRS * T::NC; w += S::THREADS) {
                const int u = w / PAIRS, jp = w % PAIRS;
                const float2 z1 = F[jp * N + u];
                const float2 z2 = F[jp * N + ((N - u) & (N - 1))];
                const float4 o = make_float4(0.5f * (z1.x + z2.x), 0.5f * (z1.y - z2.y),    // row 2jp
                                             0.5f * (z1.y + z2.y), -0.5f * (z1.x - z2.x));  // row 2jp + 1
                *reinterpret_cast<float4*>(epi.otf_rows + (static_cast<size_t>(l) * T::NC + u) * N + y0 + 2 * jp) = o;
            }
        });
    }
    ex.phase([&](int tid) {
        if (tid == 0) {
            float s = 0.f;
            for (int t = 0; t < S::THREADS; ++t) s += red[t];
            epi.finish(l, tile, N / T::CROWS, s);
        }
    });
}

// P3b crows_inv_hgrad : the backward's last stage.  grid (N/CROWS), block 3*CROWS*LANES.  The three
//      wavelengths of a row tile are three thread groups of one CTA; kappa_l * Im(GV_l conj V_l) is summed
//      over l through shared memory in fixed order, so dL/dh is written once (sum over wavelengths of
//      Optics.py:89-90's adjoint) - no per-wavelength planes, no extra pass.
template <int N>
struct HGradSmem {
    using C = CRowsSmem<N>;
    static constexpr int THREADS = 3 * C::THREADS;
    static constexpr int PART = C::FLOAT2S;                                 // float2 per wavelength group
    static constexpr int SUM_OFF = 3 * PART;                                // [2][CROWS][N] floats
    static constexpr int FLOAT2S = SUM_OFF + Tile<N>::CROWS * N;            // 2 * CROWS*N floats
    static constexpr int BYTES = FLOAT2S * 8;
};

template <int N, class Exec>
B200_HD void crows_inv_hgrad_body(Exec& ex, const CRowsInvParams& p, const PupilLoad& pupil, float* gh, float2* smem) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = CRowsSmem<N>;
    using H = HGradSmem<N>;
    const int tile = ex.bx();
    const int y0 = tile * T::CROWS;
    float* sum = reinterpret_cast<float*>(smem + H::SUM_OFF);      // partial sums of wavelengths 1 and 2
    ex.phase([&](int tid) {
        const int l = tid / S::THREADS, t = tid % S::THREADS;
        float2* F = smem + l * H::PART + S::F_OFF;
        constexpr int ITEMS = T::CROWS * N / S::THREADS;         // loads first, stores after (latency chain)
        float2 q[ITEMS];
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const int w = t + k * S::THREADS;
            q[k] = ld_ro(p.st + (static_cast<size_t>(l) * N + w / T::CROWS) * N + y0 + w % T::CROWS);
        }
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const int w = t + k * S::THREADS;
            F[(w % T::CROWS) * T::FP_CROW + w / T::CROWS] = q[k];
        }
    });
    ex.phase([&](int tid) {
        const int l = tid / S::THREADS, t = tid % S::THREADS;
        const int j = t / P::LANES, b = t % P::LANES;
        float2* F = smem + l * H::PART + S::F_OFF;
        float2* E = smem + l * H::PART + S::E_OFF;
        if (b < P::R1) {
            float2 v[P::R2];
#pragma unroll
            for (int i = 0; i < P::R2; ++i) v[i] = F[j * T::FP_CROW + b + P::R1 * i];
            P::stepC(v, b, E + j * P::E_SIZE, p.tw);
        }
    });
    ex.phase([&](int tid) {
        const int l = tid / S::THREADS, t = tid % S::THREADS;
        const int j = t / P::LANES, a = t % P::LANES;
        const float2* E = smem + l * H::PART + S::E_OFF;
        if (a < P::R2) {
            PupilLoad::Raw raw[P::R1];               // issue the pupil loads before the transform needs its registers
#pragma unroll
            for (int i = 0; i < P::R1; ++i) raw[i] = pupil.fetch(l, y0 + j, P::R2 * i + a);
            float2 v[P::R1];
            P::stepD(v, a, E + j * P::E_SIZE);
#pragma unroll
            for (int i = 0; i < P::R1; ++i) {
                const int x = P::R2 * i + a;
                const float2 pv = pupil.make(l, raw[i]);
                const float g = pupil.kap(l) * cmulc(v[i], pv).y;
                if (l > 0) sum[((l - 1) * T::CROWS + j) * N + x] = g;
                else v[i].x = g;
            }
            if (l == 0) {
                // keep wavelength 0 in registers across the barrier through the group's own E buffer
                float* keep = reinterpret_cast<float*>(smem + S::F_OFF);      // F of group 0 is free now
#pragma unroll
                for (int i = 0; i < P::R1; ++i) keep[j * N + P::R2 * i + a] = v[i].x;
            }
        }
    });
    ex.phase([&](int tid) {
        const float* keep = reinterpret_cast<const float*>(smem + S::F_OFF);
        for (int w = tid; w < T::CROWS * N; w += H::THREADS) {
            const int j = w / N, x = w % N;
            gh[static_cast<size_t>(y0 + j) * N + x] = (keep[w] + sum[w]) + sum[T::CROWS * N + w];
        }
    });
}

// ---------------------------------------------------------------------------------------------
// small element-wise / reduction bodies of the PSF chain.  Device scalars `scal`:
//   [0] S = sum |U|^2   [1] loss_rad   [2] centering_loss   [3] dot = sum(gtot * psf)
// ---------------------------------------------------------------------------------------------
constexpr int EW_THREADS = 256;

// P4  psf_finalise: psf = I/S (Optics.py:110); partial sums for loss_rad (:113) and the centering loss (:124-125)
struct PsfFinaliseParams {
    const float* I;        // [3][N][N]
    const float* rho;      // [N][N]
    float* scal;           // out: [0]=S, [1]=loss_rad, [2]=centering_loss
    float* psf;            // [3][N][N]
    float* partial;        // [3 sets][grid]
    const float* row_partial;  // [nrow] partial sums of |U|^2 from the inverse row pass
    int* arrive;           // one counter, zero on entry, reset to zero by the last CTA
    int nrow;
    int N;
};

template <class Exec>
B200_HD void psf_finalise_body(Exec& ex, const PsfFinaliseParams& p, int grid_x, float* red) {
    const int N = p.N, NN = N * N, total = 3 * NN;
    // S = sum |U|^2: every CTA adds the same partials in the same order (deterministic, no extra launch)
    ex.phase([&](int tid) {
        float acc = 0.f;
        for (int i = tid; i < p.nrow; i += EW_THREADS) acc += p.row_partial[i];
        red[tid] = acc;
    });
    for (int half = EW_THREADS / 2; half > 0; half /= 2) {
        ex.phase([&](int tid) {
            if (tid < half) red[tid] += red[tid + half];
        });
    }
    ex.phase([&](int tid) {
        if (tid == 0) {
            red[3 * EW_THREADS] = red[0];
            if (ex.bx() == 0) p.scal[0] = red[0];
        }
    });
    ex.phase([&](int tid) {
        const float S = red[3 * EW_THREADS];
        float r2 = 0.f, cy = 0.f, cx = 0.f;
        const int stride = grid_x * EW_THREADS;
        for (int idx = ex.bx() * EW_THREADS + tid; idx < total; idx += stride) {
            const int l = idx / NN, y = (idx % NN) / N, x = idx % N;
            const float v = p.I[idx] / S;
            const float vy = p.I[l * NN + ((y + N / 2) & (N - 1)) * N + x] / S;
            const float vx = p.I[l * NN + y * N + ((x + N / 2) & (N - 1))] / S;
            p.psf[idx] = v;
            const float r = p.rho[y * N + x] * v;
            r2 += r * r;
            cy += (v - vy) * (v - vy);
            cx += (v - vx) * (v - vx);
        }
        red[tid] = r2; red[EW_THREADS + tid] = cy; red[2 * EW_THREADS + tid] = cx;
    });
    for (int half = EW_THREADS / 2; half > 0; half /= 2) {
        ex.phase([&](int tid) {
            if (tid < half)
                for (int s = 0; s < 3; ++s) red[s * EW_THREADS + tid] += red[s * EW_THREADS + tid + half];
        });
    }
    ex.phase([&](int tid) {
        if (tid < 3) p.partial[tid * grid_x + ex.bx()] = red[tid * EW_THREADS];
    });
    // the last CTA to arrive turns the partials into the two regulariser values (Optics.py:113, :124-125)
    ex.phase([&](int tid) {
        if (tid == 0) {
            ex.threadfence();
            const int old = atomic_add_int(p.arrive, 1);
            red[3 * EW_THREADS + 1] = (old == grid_x - 1) ? 1.f : 0.f;
        }
    });
    if (red[3 * EW_THREADS + 1] != 0.f) {
        ex.phase([&](int tid) {
            ex.threadfence();
            for (int s = 0; s < 3; ++s) {
                float acc = 0.f;
                for (int i = tid; i < grid_x; i += EW_THREADS) acc += ex.load_cg(p.partial + s * grid_x + i);
                red[s * EW_THREADS + tid] = acc;
            }
        });
        for (int half = EW_THREADS / 2; half > 0; half /= 2) {
            ex.phase([&](int tid) {
                if (tid < half)
                    for (int s = 0; s < 3; ++s) red[s * EW_THREADS + tid] += red[s * EW_THREADS + tid + half];
            });
        }
        ex.phase([&](int tid) {
            if (tid == 0) {
                p.scal[1] = sqrtf(red[0]);
                p.scal[2] = red[EW_THREADS] / (3.0f * N * N) + red[2 * EW_THREADS] / (3.0f * N * N);
                *p.arrive = 0;
            }
        });
    }
}

// Q1  psf_grad_prepare: gtot = gpsf + g_rad * d loss_rad/dpsf + g_cen * d centering/dpsf ; partial sum(gtot*psf)
struct PsfGradPrepParams {
    const float* gpsf;     // nullable [3][N][N]
    const float* g_rad;    // nullable device scalar: upstream gradient of loss_rad
    const float* g_cen;    // nullable device scalar: upstream gradient of centering_loss
    const float* psf;      // [3][N][N]
    const float* rho;
    const float* scal;
    float* gtot;           // [3][N][N]
    float* partial;        // [grid]
    int N;
};

template <class Exec>
B200_HD void psf_grad_prepare_body(Exec& ex, const PsfGradPrepParams& p, int grid_x, float* red) {
    const int N = p.N, NN = N * N, total = 3 * NN;
    ex.phase([&](int tid) {
        const float g_rad = p.g_rad != nullptr ? *p.g_rad : 0.f;
        const float g_cen = p.g_cen != nullptr ? *p.g_cen : 0.f;
        const float loss_rad = p.scal[1];
        const float kc = g_cen * 4.0f / static_cast<float>(total);
        float dot = 0.f;
        const int stride = grid_x * EW_THREADS;
        for (int idx = ex.bx() * EW_THREADS + tid; idx < total; idx += stride) {
            const int l = idx / NN, y = (idx % NN) / N, x = idx % N;
            const float v = p.psf[idx];
            float g = p.gpsf != nullptr ? p.gpsf[idx] : 0.f;
            if (g_rad != 0.f) g += g_rad * p.rho[y * N + x] * v / loss_rad;
            if (g_cen != 0.f) {
                const float vy = p.psf[l * NN + ((y + N / 2) & (N - 1)) * N + x];
                const float vx = p.psf[l * NN + y * N + ((x + N / 2) & (N - 1))];
                g += kc * ((v - vy) + (v - vx));
            }
            p.gtot[idx] = g;
            dot += g * v;
        }
        red[tid] = dot;
    });
    for (int half = EW_THREADS / 2; half > 0; half /= 2) {
        ex.phase([&](int tid) {
            if (tid < half) red[tid] += red[tid + half];
        });
    }
    ex.phase([&](int tid) {
        if (tid == 0) p.partial[ex.bx()] = red[0];
    });
}


// =============================================================================================
//        Zernike projection  h = sum_j coef_j * Z_j   and its adjoint   (SURVEY 8 f1)
//        (Face-DeId/Camera/Optics.py:79-83 `get_Heith_Map`, Image_Caption/Camera/Lens.py:158-177)
// =============================================================================================
// A GEMV over the T x (N*N) basis volume (78.6 MB at T=300, N=256): one pass over Z each way, nothing materialised
// (torch's  sum(coef * volume, 0)  writes and re-reads the product).
//
// Z1  zernike_fwd : grid (ceil(NN4/EW_THREADS), KS), block EW_THREADS.  CTA (x, k) adds terms [T*k/KS, T*(k+1)/KS) for
//      its EW_THREADS pixel quads into partial[k]; the last of the KS CTAs of a pixel block to finish adds the partials
//      in order k = 0..KS-1 (deterministic) and writes h.  arrive[x] must be zero on entry and is left zero.
struct ZernikeFwdParams {
    const float* coef;     // [T]
    const float4* Z;       // [T][NN4]
    float4* partial;       // [KS][NN4]
    float4* h;             // [NN4]
    int* arrive;           // [gridDim.x]
    int T, NN4, KS;
    // nullable: the float4 positions that are non-zero in at least one basis plane (the Zernike basis is zero outside the unit
    // disc: 21 % of the square) - the grid then covers `nactive` positions instead of NN4; h must be zero elsewhere (the entry
    // point clears it)
    const int* active = nullptr;
    int nactive = 0;
};

template <class Exec>
B200_HD void zernike_fwd_body(Exec& ex, const ZernikeFwdParams& p, int* flag) {
    const int k = ex.by();
    const int j0 = static_cast<int>(static_cast<long long>(p.T) * k / p.KS);
    const int j1 = static_cast<int>(static_cast<long long>(p.T) * (k + 1) / p.KS);
    const int nq = p.active != nullptr ? p.nactive : p.NN4;
    ex.phase([&](int tid) {
        const int qi = ex.bx() * EW_THREADS + tid;
        if (qi < nq) {
            const int q = p.active != nullptr ? ld_ro(p.active + qi) : qi;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            int j = j0;
            for (; j + 8 <= j1; j += 8) {                 // eight independent 16-byte loads in flight per thread
                float4 z[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) z[i] = ld_ro(p.Z + static_cast<size_t>(j + i) * p.NN4 + q);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float c = ld_ro(p.coef + j + i);
                    acc.x += c * z[i].x; acc.y += c * z[i].y; acc.z += c * z[i].z; acc.w += c * z[i].w;
                }
            }
            for (; j < j1; ++j) {
                const float4 z = ld_ro(p.Z + static_cast<size_t>(j) * p.NN4 + q);
                const float c = ld_ro(p.coef + j);
                acc.x += c * z.x; acc.y += c * z.y; acc.z += c * z.z; acc.w += c * z.w;
            }
            p.partial[static_cast<size_t>(k) * p.NN4 + q] = acc;
        }
    });
    ex.phase([&](int tid) {
        if (tid == 0) {
            ex.threadfence();
            *flag = (atomic_add_int(p.arrive + ex.bx(), 1) == p.KS - 1) ? 1 : 0;
        }
    });
    if (*flag) {
        ex.phase([&](int tid) {
            ex.threadfence();
            const int qi = ex.bx() * EW_THREADS + tid;
            if (qi < nq) {
                const int q = p.active != nullptr ? ld_ro(p.active + qi) : qi;
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int kk = 0; kk < p.KS; ++kk) {
                    const float4 v = ex.load_cg4(p.partial + static_cast<size_t>(kk) * p.NN4 + q);
                    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
                }
                p.h[q] = acc;
            }
            if (tid == 0) p.arrive[ex.bx()] = 0;
        });
    }
}

// Z2  zernike_bwd : gcoef_j = sum_p Z_j[p] * gh[p].  grid (T, splits), block EW_THREADS; fixed-order tree.
//     splits > 1 (few terms, e.g. the single trainable defocus term of the Image_Caption camera): CTA (j, s) reduces the
//     s-th slice of the plane into partial[j * splits + s]; k_zernike_bwd_fin adds the slices in order.
struct ZernikeBwdParams {
    const float4* gh;      // [NN4]
    const float4* Z;       // [T][NN4]
    float* gcoef;          // [T]  (splits == 1) or the partials [T][splits]
    int NN4;
    int splits = 1;
    const int* active = nullptr;   // as ZernikeFwdParams::active: only these float4 positions are visited
    int nactive = 0;
};

template <class Exec>
B200_HD void zernike_bwd_body(Exec& ex, const ZernikeBwdParams& p, float* red) {
    const int j = ex.bx();
    const int nq = p.active != nullptr ? p.nactive : p.NN4;
    const int slice = (nq + p.splits - 1) / p.splits;
    const int q0 = ex.by() * slice;
    const int q1 = q0 + slice < nq ? q0 + slice : nq;
    ex.phase([&](int tid) {
        const float4* z = p.Z + static_cast<size_t>(j) * p.NN4;
        float acc = 0.f;
        int q = q0 + tid;
        for (; q + 7 * EW_THREADS < q1; q += 8 * EW_THREADS) {
            float4 a[8], g[8];
            int at[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) at[i] = p.active != nullptr ? ld_ro(p.active + q + i * EW_THREADS) : q + i * EW_THREADS;
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = ld_ro(z + at[i]);
#pragma unroll
            for (int i = 0; i < 8; ++i) g[i] = ld_ro(p.gh + at[i]);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc += (a[i].x * g[i].x + a[i].y * g[i].y) + (a[i].z * g[i].z + a[i].w * g[i].w);
        }
        for (; q < q1; q += EW_THREADS) {
            const int at = p.active != nullptr ? ld_ro(p.active + q) : q;
            const float4 a = ld_ro(z + at), g = ld_ro(p.gh + at);
            acc += (a.x * g.x + a.y * g.y) + (a.z * g.z + a.w * g.w);
        }
        red[tid] = acc;
    });
    for (int half = EW_THREADS / 2; half > 0; half /= 2) {
        ex.phase([&](int tid) {
            if (tid < half) red[tid] += red[tid + half];
        });
    }
    ex.phase([&](int tid) {
        if (tid == 0) p.gcoef[j * p.splits + ex.by()] = red[0];
    });
}

// =============================================================================================
//   Image_Caption sensor epilogue:  |.|, crop and nearest 255 -> 256 resize in one pass
//   (img_psf_conv, Image_Caption/Camera/Utils.py:289-295:  abs -> [129:-128] crop -> nearest resize
//    out[i] = crop[max(i-1, 0)])  and its adjoint.  Replaces five element-wise / gather torch kernels over the
//    (B,3,2P,2P) convolution output (and seven in the backward) by one read of the P x P window.
// =============================================================================================
struct CropAbsResizeParams {
    const float* conv;     // [planes][n][n]
    float* out;            // [planes][P][P]
    int planes, n, P, off; // window origin (off, off); source row of output row i is off + max(i - 1, 0)
};

template <class Exec>
B200_HD void crop_abs_resize_fwd_body(Exec& ex, const CropAbsResizeParams& p, int grid_x) {
    ex.phase([&](int tid) {
        const long long total = static_cast<long long>(p.planes) * p.P * p.P;
        const long long stride = static_cast<long long>(grid_x) * ex.nthreads();
        for (long long idx = static_cast<long long>(ex.bx()) * ex.nthreads() + tid; idx < total; idx += stride) {
            const int j = static_cast<int>(idx % p.P), i = static_cast<int>((idx / p.P) % p.P);
            const long long pl = idx / (static_cast<long long>(p.P) * p.P);
            const int r = p.off + (i > 0 ? i - 1 : 0), c = p.off + (j > 0 ? j - 1 : 0);
            p.out[idx] = fabsf(ld_ro(p.conv + (pl * p.n + r) * p.n + c));
        }
    });
}

struct CropAbsResizeBwdParams {
    const float* g_out;    // [planes][P][P]
    const float* conv;     // [planes][n][n]  (sign of the forward's argument)
    float* g_conv;         // [planes][n][n]  every element is written (zero outside the window)
    int planes, n, P, off;
};

template <class Exec>
B200_HD void crop_abs_resize_bwd_body(Exec& ex, const CropAbsResizeBwdParams& p, int grid_x) {
    ex.phase([&](int tid) {
        const long long total = static_cast<long long>(p.planes) * p.n * p.n;
        const long long stride = static_cast<long long>(grid_x) * ex.nthreads();
        for (long long idx = static_cast<long long>(ex.bx()) * ex.nthreads() + tid; idx < total; idx += stride) {
            const int c = static_cast<int>(idx % p.n), r = static_cast<int>((idx / p.n) % p.n);
            const long long pl = idx / (static_cast<long long>(p.n) * p.n);
            const int rr = r - p.off, cc = c - p.off;          // position in the (P-1)^2 crop
            float g = 0.f;
            if (rr >= 0 && rr < p.P - 1 && cc >= 0 && cc < p.P - 1) {
                // crop row rr feeds output row rr+1, and output row 0 as well when rr == 0 (same for columns)
                const float* go = p.g_out + pl * p.P * p.P;
                const int i1 = rr + 1, j1 = cc + 1;
                g = ld_ro(go + i1 * p.P + j1);
                if (rr == 0) g += ld_ro(go + j1);
                if (cc == 0) g += ld_ro(go + i1 * p.P);
                if (rr == 0 && cc == 0) g += ld_ro(go);
                const float v = ld_ro(p.conv + idx);
                g = v > 0.f ? g : (v < 0.f ? -g : 0.f);      // d|v|/dv, 0 at v == 0 as torch.abs
            }
            p.g_conv[idx] = g;
        }
    });
}

}  // namespace b200cam
