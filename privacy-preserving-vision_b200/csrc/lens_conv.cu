// b200cam: the sensor image of the Image_Caption camera - img_psf_conv (Image_Caption/Camera/Utils.py:251-297) and the
// batch-global normalisation (Lens.py:312) - with the zero padding, the crop / nearest resize and |.| folded into the
// transform kernels.
//
//   reference:  pad img P -> n = 2P (P/2 zeros each side) ; FFT2 ; x OTF ; IFFT2 ; abs ; crop [pt+1 : n-pb] ; nearest resize
//               (P-1 -> P: out[i] = crop[max(i-1,0)]) ; / max over the whole batch
//   here:       the padded image is never written: the row pass transforms the P live rows only (zero columns filled in
//               shared memory), the column pass reads / writes the P live rows of every spectral column, the inverse row pass
//               transforms the P rows the crop keeps and writes  raw[i][j] = conv[pt + max(i,1)][pt + max(j,1)]  (signed) plus
//               the batch maximum of |raw| (integer atomics); one element-wise pass then gives |raw| / max, optionally followed by
//               the read-out epilogue of kernels.cuh (sensor noise, quantisation).
// The row pass reads fp32 images or uint8 images (converted in registers exactly as torch's u8.float() / 255.0 on the GPU).
//   Spectrum traffic is half that of the padded transform, the 4x padded image and the 4x conv output never exist.
// The backward reads (g, raw) in the loader of the gradient's row pass: dL/dconv = sign(raw) (g / m - tie s / (m n)).
//
// Same two-pass FFT building blocks (fft_plan.cuh) and spectrum layout st[plane][u][y] as the Face-DeId pipeline
// (kernels.cuh); n in {128, 256, 512, 1024}.
#include <cuda_runtime.h>

#include <type_traits>

#include "../../include/b200cam.h"
#include "kernels.cuh"

namespace b200cam {
void note_launches(int n);
const float2* lens_twiddle(int N);                                                             // b200cam.cu
int lens_otf(int N, const float* kern, float2* otf, cudaStream_t s);                           // b200cam.cu: rows + cols of the padded PSF
int lens_grad_kernel_tail(int N, const float2* partial, float2* stp, float* grad_kern, int nchunks, cudaStream_t s);   // reduce + inverse
namespace lconv {

extern __shared__ __align__(16) unsigned char lsmem_raw[];
#define LSMEM2 reinterpret_cast<float2*>(lsmem_raw)

// ---- loaders of the live P x P region of a padded plane ----------------------------------------------------------------
struct ImgLoad {        // the image itself (Utils.py:266-277)
    const float* x;     // [planes][P][P]
    __device__ __forceinline__ void init() {}
    __device__ __forceinline__ float operator()(int plane, int r, int c, int P) const {
        return __ldg(x + (static_cast<size_t>(plane) * P + r) * P + c);
    }
};
struct ImgLoadU8 {      // a uint8 image: a quarter of the bytes; = torch's u8.float() / 255.0 on the GPU, which multiplies by the
    const unsigned char* x;   // [planes][P][P]                                   fp32 reciprocal of a CPU scalar divisor
    __device__ __forceinline__ void init() {}
    __device__ __forceinline__ float operator()(int plane, int r, int c, int P) const {
        return __fmul_rn(static_cast<float>(__ldg(x + (static_cast<size_t>(plane) * P + r) * P + c)), 1.0f / 255.0f);
    }
};
template <class G>      // G: element type of dL/dy - fp32, or bf16 (widened exactly in registers)
struct GradLoadT {      // dL/dconv from dL/dy: adjoint of / max, |.|, crop and nearest resize (Utils.py:289-295, Lens.py:312)
    const G* g;         // [planes][P][P] dL/dy
    const float* raw;   // [planes][P][P] signed un-normalised sensor image of the forward
    const float* gmax;  // device scalar: batch maximum m (all ranks)
    const float* coef;  // device scalar: s / (m n), s = sum(g y), n = number of positions that attain m
    float inv_m, cf, m;
    __device__ __forceinline__ void init() {
        m = __ldg(gmax);
        inv_m = 1.0f / m;
        cf = __ldg(coef);
    }
    __device__ __forceinline__ float draw(size_t o) const {
        const float rv = __ldg(raw + o), gv = load_elem(g + o);
        const float d = gv * inv_m - (fabsf(rv) == m ? cf : 0.f);
        return rv > 0.f ? d : (rv < 0.f ? -d : 0.f);
    }
    __device__ __forceinline__ float operator()(int plane, int r, int c, int P) const {
        if (r == 0 || c == 0) return 0.f;                  // conv row / column pt is cropped away
        const size_t base = static_cast<size_t>(plane) * P * P;
        float v = draw(base + static_cast<size_t>(r) * P + c);
        // the nearest resize duplicates crop row 0 / column 0 into output row / column 0: only r == 1 / c == 1 collect two terms.
        // Both tests are rare and warp-uniform enough to be branches, not selects around extra loads.
        if (c == 1 || r == 1) {
            if (c == 1) v += draw(base + static_cast<size_t>(r) * P);
            if (r == 1) {
                v += draw(base + c);
                if (c == 1) v += draw(base);
            }
        }
        return v;
    }
};
using GradLoad = GradLoadT<float>;

// ---- KA: zero-padded real rows -> transposed half spectrum, live rows only.  grid (P / ROWS, planes), block NP * LANES ------
// MIN_CTAS > 0: held to that many resident CTAs per SM (__launch_bounds__ minimum; 0 emits no bound).  Used for the bf16
// gradient loader at n = 512, which otherwise costs ptxas 4 registers more than the fp32 one (84 vs 80: 2 instead of 3 CTAs of
// 256 threads per SM; measured 77 against 64 us per launch at B = 64, one B200).
template <int N, class Load, int MIN_CTAS = 0>
__global__ void __launch_bounds__(RowsR2CSmem<N>::THREADS, MIN_CTAS) k_lrows_r2c(Load load, float2* __restrict__ st, const float2* __restrict__ tw) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = RowsR2CSmem<N>;
    constexpr int PP = N / 2, PT = N / 4;
    float2* smem = LSMEM2;
    const int tile = blockIdx.x, plane = blockIdx.y;
    const int r0 = tile * T::ROWS;                 // first live row of the tile
    const int tid = threadIdx.x;
    const int j = tid / P::LANES, a = tid % P::LANES;
    load.init();
    if (a < P::R2) {
        float2 v[P::R1];
#pragma unroll
        for (int i = 0; i < P::R1; ++i) {
            const int c = P::R2 * i + a - PT;
            v[i] = (c >= 0 && c < PP) ? make_float2(load(plane, r0 + 2 * j, c, PP), load(plane, r0 + 2 * j + 1, c, PP)) : make_float2(0.f, 0.f);
        }
        P::stepA(v, a, smem + j * S::PA, tw);
    }
    __syncthreads();
    float2 q[P::R2];
    if (a < P::R1) P::stepB(q, a, smem + j * S::PA);
    __syncthreads();
    if (a < P::R1) {
#pragma unroll
        for (int i = 0; i < P::R2; ++i) smem[j * S::PA + a + P::R1 * i] = q[i];
    }
    __syncthreads();
    for (int w = tid; w < T::NP * T::NC; w += S::THREADS) {
        const int u = w / T::NP, jj = w % T::NP;
        const float2 z1 = smem[jj * S::PA + u];
        const float2 z2 = smem[jj * S::PA + ((N - u) & (N - 1))];
        const float4 o = make_float4(0.5f * (z1.x + z2.x), 0.5f * (z1.y - z2.y), 0.5f * (z1.y + z2.y), -0.5f * (z1.x - z2.x));
        *reinterpret_cast<float4*>(st + (static_cast<size_t>(plane) * T::NC + u) * N + PT + r0 + 2 * jj) = o;
    }
}

// ---- KB: per spectral column FFT_v -> x OTF (or conj) -> IFFT_v over the live rows [PT, PT + P).  grid (colgroups, nchunks) ----
template <int N>
__global__ void __launch_bounds__(ColsSmem<N>::THREADS, N <= 512 ? 2 : 1) k_lcols_conv(const float2* in, float2* out, const float2* __restrict__ otf,
                                                                      const float2* __restrict__ tw, int B, int nchunks, int conj_otf) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = ColsSmem<N>;
    constexpr int PT = N / 4;
    static_assert(PT % P::R2 == 0, "live range must be a whole number of register rows");
    constexpr int I0 = PT / P::R2, I1 = 3 * PT / P::R2;          // live i range of y = R2 * i + a
    float2* E1 = LSMEM2;
    float2* E2 = E1 + S::COLS * P::E_SIZE;
    constexpr int TOTAL = 3 * T::NC;
    const int tid = threadIdx.x;
    const int jc = tid / P::LANES, a = tid % P::LANES;
    const int cu = blockIdx.x * S::COLS + jc;
    const int b0 = static_cast<int>(static_cast<long long>(B) * blockIdx.y / nchunks);
    const int b1 = static_cast<int>(static_cast<long long>(B) * (blockIdx.y + 1) / nchunks);
    const bool live = cu < TOTAL;
    float2 k[P::R2];
    if (live && a < P::R1) {
#pragma unroll
        for (int i = 0; i < P::R2; ++i) {
            const float2 kk = __ldg(otf + static_cast<size_t>(cu) * N + a + P::R1 * i);
            k[i] = conj_otf ? cconj(kk) : kk;
        }
    }
    const int c = live ? cu / T::NC : 0, u = live ? cu % T::NC : 0;
    for (int img = b0; img < b1; ++img) {
        const size_t col = (static_cast<size_t>(img * 3 + c) * T::NC + u) * N;
        if (live && a < P::R2) {
            float2 v[P::R1];
#pragma unroll
            for (int i = 0; i < P::R1; ++i) v[i] = (i >= I0 && i < I1) ? in[col + P::R2 * i + a] : make_float2(0.f, 0.f);
            P::stepA(v, a, E1 + jc * P::E_SIZE, tw);
        }
        __syncwarp();        // a column lives in one warp (LANES <= 32): no block barrier
        if (live && a < P::R1) {
            float2 v[P::R2];
            P::stepB(v, a, E1 + jc * P::E_SIZE);
#pragma unroll
            for (int i = 0; i < P::R2; ++i) v[i] = cmul(v[i], k[i]);
            P::stepC(v, a, E2 + jc * P::E_SIZE, tw);
        }
        __syncwarp();        // a column lives in one warp (LANES <= 32): no block barrier
        if (live && a < P::R2) {
            float2 v[P::R1];
            P::stepD(v, a, E2 + jc * P::E_SIZE);
#pragma unroll
            for (int i = I0; i < I1; ++i) out[col + P::R2 * i + a] = v[i];
        }
    }
}

// ---- KC: inverse rows of the live rows, fused crop.  grid (P / ROWS, planes) ----------------------------------------------
//   MODE 0: raw[i][j] = conv[PT + max(i,1)][PT + max(j,1)] (abs / crop / nearest resize, Utils.py:289-295; the sign is kept for the
//           backward) and the batch maximum of |raw|
//   MODE 1: out[i][j] = conv[PT + i][PT + j]   (adjoint of the zero padding: dL/dimg)
template <int N, int MODE>
__global__ void __launch_bounds__(RowsR2CSmem<N>::THREADS) k_lrows_c2r(const float2* __restrict__ st, float* __restrict__ out, const float2* __restrict__ tw,
                                                                        float* gmax) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = RowsR2CSmem<N>;
    constexpr int PP = N / 2, PT = N / 4;
    float2* smem = LSMEM2;
    float* red = reinterpret_cast<float*>(smem + S::RED_OFF);
    const int tile = blockIdx.x, plane = blockIdx.y;
    const int r0 = tile * T::ROWS;
    const int tid = threadIdx.x;
    {
        constexpr int ITEMS = (T::NP * T::NC + S::THREADS - 1) / S::THREADS;
        float4 q[ITEMS];
#pragma unroll
        for (int kk = 0; kk < ITEMS; ++kk) {
            const int w = tid + kk * S::THREADS;
            if (w < T::NP * T::NC) {
                const int u = w / T::NP, j = w % T::NP;
                q[kk] = __ldg(reinterpret_cast<const float4*>(st + (static_cast<size_t>(plane) * T::NC + u) * N + PT + r0 + 2 * j));
            }
        }
#pragma unroll
        for (int kk = 0; kk < ITEMS; ++kk) {
            const int w = tid + kk * S::THREADS;
            if (w < T::NP * T::NC) {
                const int u = w / T::NP, j = w % T::NP;
                float2* F = smem + j * S::PA;
                if (u == 0 || u == N / 2) {
                    F[u] = make_float2(q[kk].x, q[kk].z);
                } else {
                    F[u] = make_float2(q[kk].x - q[kk].w, q[kk].y + q[kk].z);
                    F[N - u] = make_float2(q[kk].x + q[kk].w, q[kk].z - q[kk].y);
                }
            }
        }
    }
    __syncthreads();
    const int j = tid / P::LANES, a = tid % P::LANES;
    float2 q[P::R2];
    if (a < P::R1) {
#pragma unroll
        for (int i = 0; i < P::R2; ++i) q[i] = smem[j * S::PA + a + P::R1 * i];
    }
    __syncthreads();
    if (a < P::R1) P::stepC(q, a, smem + j * S::PA, tw);
    __syncthreads();
    float mx = 0.f;
    if (a < P::R2) {
        float2 v[P::R1];
        P::stepD(v, a, smem + j * S::PA);
        float* po = out + static_cast<size_t>(plane) * PP * PP;
#pragma unroll
        for (int i = 0; i < P::R1; ++i) {
            const int c = P::R2 * i + a - PT;
            if (c < 0 || c >= PP) continue;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int r = r0 + 2 * j + h;
                const float val = h ? v[i].y : v[i].x;
                if (MODE == 1) {
                    po[static_cast<size_t>(r) * PP + c] = val;
                } else if (r >= 1 && c >= 1) {
                    mx = fmaxf(mx, fabsf(val));
                    po[static_cast<size_t>(r) * PP + c] = val;
                    if (c == 1) po[static_cast<size_t>(r) * PP] = val;
                    if (r == 1) {
                        po[c] = val;
                        if (c == 1) po[0] = val;
                    }
                }
            }
        }
    }
    if (MODE == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if ((tid & 31) == 0) red[tid >> 5] = mx;
        __syncthreads();
        if (tid == 0) {
            float t = red[0];
            for (int w = 1; w < S::THREADS / 32; ++w) t = fmaxf(t, red[w]);
            atomicMax(reinterpret_cast<int*>(gmax), __float_as_int(t));          // t >= 0: integer order = float order
        }
    }
}

// ---- KD: sum over the chunk's images of G * conj(X) per spectral column (live rows only).  grid (colgroups, nchunks) --------
template <int N>
__global__ void __launch_bounds__(ColsSmem<N>::THREADS, N <= 512 ? 2 : 1) k_lcols_accum(const float2* __restrict__ stx, const float2* __restrict__ stg,
                                                                       float2* __restrict__ partial, const float2* __restrict__ tw, int B,
                                                                       int nchunks) {
    using P = Plan<N>;
    using T = Tile<N>;
    using S = ColsSmem<N>;
    constexpr int PT = N / 4;
    constexpr int I0 = PT / P::R2, I1 = 3 * PT / P::R2;
    float2* Ex = LSMEM2;
    float2* Eg = Ex + S::COLS * P::E_SIZE;
    constexpr int TOTAL = 3 * T::NC;
    const int tid = threadIdx.x;
    const int jc = tid / P::LANES, a = tid % P::LANES;
    const int cu = blockIdx.x * S::COLS + jc;
    const int b0 = static_cast<int>(static_cast<long long>(B) * blockIdx.y / nchunks);
    const int b1 = static_cast<int>(static_cast<long long>(B) * (blockIdx.y + 1) / nchunks);
    const bool live = cu < TOTAL;
    float2 acc[P::R2];
#pragma unroll
    for (int i = 0; i < P::R2; ++i) acc[i] = make_float2(0.f, 0.f);
    for (int b = b0; b < b1; ++b) {
        if (live && a < P::R2) {
            const size_t off = (static_cast<size_t>(b) * TOTAL + cu) * N;
            // the two operands one after the other: the load phase then holds R1 values, not 2 R1 (two CTAs per SM)
            {
                float2 v[P::R1];
#pragma unroll
                for (int i = 0; i < P::R1; ++i) v[i] = (i >= I0 && i < I1) ? __ldg(stx + off + P::R2 * i + a) : make_float2(0.f, 0.f);
                P::stepA(v, a, Ex + jc * P::E_SIZE, tw);
            }
            {
                float2 v[P::R1];
#pragma unroll
                for (int i = 0; i < P::R1; ++i) v[i] = (i >= I0 && i < I1) ? __ldg(stg + off + P::R2 * i + a) : make_float2(0.f, 0.f);
                P::stepA(v, a, Eg + jc * P::E_SIZE, tw);
            }
        }
        __syncwarp();
        if (live && a < P::R1) {
            float2 vx[P::R2], vg[P::R2];
            P::stepB(vx, a, Ex + jc * P::E_SIZE);
            P::stepB(vg, a, Eg + jc * P::E_SIZE);
#pragma unroll
            for (int i = 0; i < P::R2; ++i) {
                const float2 t = cmulc(vg[i], vx[i]);
                acc[i].x += t.x;
                acc[i].y += t.y;
            }
        }
        __syncwarp();
    }
    if (live && a < P::R1) {
        float2* dst = partial + (static_cast<size_t>(blockIdx.y) * TOTAL + cu) * N;
#pragma unroll
        for (int i = 0; i < P::R2; ++i) dst[a + P::R1 * i] = acc[i];
    }
}

// ---- element-wise: y = |raw| / m [-> read-out epilogue] ; partial sums of g * y and the number of positions that attain m -----
// Out = bf16: the fp32 value rounded to nearest-even as the last step (= the fp32 sensor image cast with torch)
constexpr int EWT = 256;
// PHILOX (with EPI): the Philox read-out (epi.seed), one philox_normal4 per float4 at counter first4 + i
template <bool EPI, class Out = float, bool PHILOX = false>
__global__ void __launch_bounds__(EWT) k_lnormalise(const float4* __restrict__ raw, const float* __restrict__ gmax, Out* __restrict__ y, long long n4,
                                                    SensorEpilogue epi) {
    const float m = __ldg(gmax);
    NoiseSeed seed{0ull, 0ull};
    if constexpr (PHILOX) seed = load_seed(epi.seed);
    for (long long i = blockIdx.x * static_cast<long long>(EWT) + threadIdx.x; i < n4; i += static_cast<long long>(gridDim.x) * EWT) {
        const float4 v = __ldg(raw + i);
        float4 o = make_float4(fabsf(v.x) / m, fabsf(v.y) / m, fabsf(v.z) / m, fabsf(v.w) / m);
        if constexpr (PHILOX) {
            const Normal4 nz = philox_normal4(seed.key, seed.first4 + static_cast<unsigned long long>(i));
            o = make_float4(quantise(epi, add_noise(epi, o.x, nz.n[0])), quantise(epi, add_noise(epi, o.y, nz.n[1])),
                            quantise(epi, add_noise(epi, o.z, nz.n[2])), quantise(epi, add_noise(epi, o.w, nz.n[3])));
        } else if (EPI) {
            const size_t e = static_cast<size_t>(i) * 4;
            o = make_float4(apply_epilogue(epi, o.x, e), apply_epilogue(epi, o.y, e + 1), apply_epilogue(epi, o.z, e + 2),
                            apply_epilogue(epi, o.w, e + 3));
        }
        if constexpr (sizeof(Out) == sizeof(float))
            reinterpret_cast<float4*>(y)[i] = o;
        else
            store4(y, i, o.x, o.y, o.z, o.w);
    }
}
// part[block] = {sum g y, ties} in double / as a count; fixed order inside a block, blocks summed in order by k_ldot_final
template <class G = float>     // G: element type of dL/dy (fp32 / bf16)
__global__ void __launch_bounds__(EWT) k_ldot(const G* __restrict__ g, const float4* __restrict__ raw, const float* __restrict__ gmax, long long n4,
                                              double* __restrict__ part) {
    __shared__ double rs[EWT / 32];
    __shared__ double rt[EWT / 32];
    const float m = __ldg(gmax);
    const float inv = 1.0f / m;
    double s = 0.0, t = 0.0;
    for (long long i = blockIdx.x * static_cast<long long>(EWT) + threadIdx.x; i < n4; i += static_cast<long long>(gridDim.x) * EWT) {
        const float4 v = __ldg(raw + i), gg = load4(g, i);
        const float ax = fabsf(v.x), ay = fabsf(v.y), az = fabsf(v.z), aw = fabsf(v.w);
        s += static_cast<double>(gg.x * (ax * inv)) + static_cast<double>(gg.y * (ay * inv)) + static_cast<double>(gg.z * (az * inv)) +
             static_cast<double>(gg.w * (aw * inv));
        t += (ax == m) + (ay == m) + (az == m) + (aw == m);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_down_sync(0xffffffffu, s, o);
        t += __shfl_down_sync(0xffffffffu, t, o);
    }
    if ((threadIdx.x & 31) == 0) {
        rs[threadIdx.x >> 5] = s;
        rt[threadIdx.x >> 5] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < EWT / 32; ++w) {
            a += rs[w];
            b += rt[w];
        }
        part[2 * blockIdx.x] = a;
        part[2 * blockIdx.x + 1] = b;
    }
}
__global__ void __launch_bounds__(EWT) k_ldot_final(const double* __restrict__ part, int nblocks, float* __restrict__ out) {   // one CTA, fixed order
    __shared__ double ra[EWT];
    __shared__ double rb[EWT];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += EWT) {
        a += part[2 * i];
        b += part[2 * i + 1];
    }
    ra[threadIdx.x] = a;
    rb[threadIdx.x] = b;
    __syncthreads();
    for (int o = EWT / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            ra[threadIdx.x] += ra[threadIdx.x + o];
            rb[threadIdx.x] += rb[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = static_cast<float>(ra[0]);
        out[1] = static_cast<float>(rb[0]);
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------------
#define LCK(expr)                                               \
    do {                                                        \
        cudaError_t e_ = (expr);                                \
        if (e_ != cudaSuccess) return static_cast<int>(e_);     \
    } while (0)
#define LLAUNCH()                 \
    do {                          \
        LCK(cudaGetLastError());  \
        note_launches(1);         \
    } while (0)

constexpr int MAX_LCHUNKS = 16;
static int lchunks(int N, int B) {
    const int colgroups = (3 * (N / 2 + 1) + 7) / 8;
    const int per_sm = N <= 512 ? 2 : 1;                       // resident CTAs per SM (launch bounds of the column kernels)
    int n = (per_sm * 148) / colgroups;                        // one wave: a second, partly filled wave costs as much as a full one
    if (n > MAX_LCHUNKS) n = MAX_LCHUNKS;
    if (n > B) n = B;
    return n < 1 ? 1 : n;
}
static int ew_grid(long long n4) {
    const long long b = (n4 + EWT - 1) / EWT;
    return static_cast<int>(b < 148 * 8 ? (b < 1 ? 1 : b) : 148 * 8);
}

struct Ws {
    float2* st2; float2* stg; float2* partial; float2* stp; double* dpart;
    size_t bytes;
    Ws(void* base, int N, int B) {
        size_t off = 0;
        auto take = [&](size_t b) {
            void* p = base ? static_cast<char*>(base) + off : nullptr;
            off += (b + 255) / 256 * 256;
            return p;
        };
        const size_t plane = static_cast<size_t>(N / 2 + 1) * N * sizeof(float2);
        st2 = static_cast<float2*>(take(plane * 3 * B));               // forward: product spectrum; backward: gradient spectrum
        stg = st2;
        partial = static_cast<float2*>(take(plane * 3 * (B < MAX_LCHUNKS ? B : MAX_LCHUNKS)));
        stp = static_cast<float2*>(take(plane * 3));
        dpart = static_cast<double*>(take(sizeof(double) * 2 * 148 * 8));
        bytes = off;
    }
};

template <class K>
static cudaError_t optin(K kernel, size_t bytes) {
    return bytes > 48 * 1024 ? cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)) : cudaSuccess;
}

template <int N, class Load>
static int fwd_impl(Load load, const float* kern, float* raw, float* gmax, float2* otf, float2* spectrum, void* wsp, int B, cudaStream_t s) {
    using T = Tile<N>;
    const float2* tw = lens_twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    Ws ws(wsp, N, B);
    int rc = lens_otf(N, kern, otf, s);
    if (rc) return rc;
    const int planes = 3 * B, tiles = (N / 2) / T::ROWS;
    const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS, nch = lchunks(N, B);
    LCK(optin(k_lrows_r2c<N, Load>, RowsR2CSmem<N>::BYTES));
    LCK(optin(k_lcols_conv<N>, ColsSmem<N>::BYTES_CONV));
    LCK(optin(k_lrows_c2r<N, 0>, RowsR2CSmem<N>::BYTES));
    k_lrows_r2c<N, Load><<<dim3(tiles, planes), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s>>>(load, spectrum, tw);
    LLAUNCH();
    k_lcols_conv<N><<<dim3(colgroups, nch), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV, s>>>(spectrum, ws.st2, otf, tw, B, nch, 0);
    LLAUNCH();
    k_lrows_c2r<N, 0><<<dim3(tiles, planes), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s>>>(ws.st2, raw, tw, gmax);
    LLAUNCH();
    return 0;
}

template <int N, class G = float>
static int bwd_impl(const G* g, const float* raw, const float* gmax, const float* coef, const float2* otf, const float2* spectrum,
                    float* grad_kern, float* grad_img, void* wsp, int B, cudaStream_t s) {
    using T = Tile<N>;
    const float2* tw = lens_twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    Ws ws(wsp, N, B);
    const int planes = 3 * B, tiles = (N / 2) / T::ROWS;
    const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS, nch = lchunks(N, B);
    constexpr int MIN_CTAS = (N == 512 && !std::is_same<G, float>::value) ? 3 : 0;
    auto rows = k_lrows_r2c<N, GradLoadT<G>, MIN_CTAS>;
    LCK(optin(rows, RowsR2CSmem<N>::BYTES));
    LCK(optin(k_lcols_accum<N>, ColsSmem<N>::BYTES_CONV));
    rows<<<dim3(tiles, planes), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s>>>(GradLoadT<G>{g, raw, gmax, coef, 0.f, 0.f, 0.f}, ws.stg, tw);
    LLAUNCH();
    k_lcols_accum<N><<<dim3(colgroups, nch), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV, s>>>(spectrum, ws.stg, ws.partial, tw, B, nch);
    LLAUNCH();
    int rc = lens_grad_kernel_tail(N, ws.partial, ws.stp, grad_kern, nch, s);
    if (rc) return rc;
    if (grad_img != nullptr) {
        LCK(optin(k_lcols_conv<N>, ColsSmem<N>::BYTES_CONV));
        LCK(optin(k_lrows_c2r<N, 1>, RowsR2CSmem<N>::BYTES));
        k_lcols_conv<N><<<dim3(colgroups, nch), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV, s>>>(ws.stg, ws.stg, otf, tw, B, nch, 1);
        LLAUNCH();
        k_lrows_c2r<N, 1><<<dim3(tiles, planes), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s>>>(ws.stg, grad_img, tw, nullptr);
        LLAUNCH();
    }
    return 0;
}

}  // namespace lconv
}  // namespace b200cam

using namespace b200cam;
using namespace b200cam::lconv;

static bool lens_n_ok(int P) { return P == 64 || P == 128 || P == 256 || P == 512; }
static bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// the checks and the dispatch of both forward entry points; `Load` reads the image (ImgLoad: fp32, ImgLoadU8: uint8)
template <class Load>
static int lens_fwd(Load load, const void* img, const float* kernel, float* raw, float* gmax, float* otf, float* spectrum, void* workspace,
                    size_t workspace_bytes, int B, int P, void* stream) {
    if (!lens_n_ok(P) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!img || !kernel || !raw || !gmax || !otf || !spectrum || !workspace) return B200CAM_E_NULL;
    if (!al16(img) || !al16(raw) || !al16(spectrum) || !al16(workspace)) return B200CAM_E_ALIGN;
    const int N = 2 * P;
    if (workspace_bytes < Ws(nullptr, N, B).bytes) return B200CAM_E_WORKSPACE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float2* o = reinterpret_cast<float2*>(otf);
    float2* sp = reinterpret_cast<float2*>(spectrum);
    switch (N) {
        case 128: return fwd_impl<128>(load, kernel, raw, gmax, o, sp, workspace, B, s);
        case 256: return fwd_impl<256>(load, kernel, raw, gmax, o, sp, workspace, B, s);
        case 512: return fwd_impl<512>(load, kernel, raw, gmax, o, sp, workspace, B, s);
        default: return fwd_impl<1024>(load, kernel, raw, gmax, o, sp, workspace, B, s);
    }
}

// checks and launches of the element-wise / backward entry points; Out / G: fp32, or bf16 (the _bf16 entry points)
template <class Out>
static int lens_normalise(const float* raw, const float* gmax, Out* y, long long count, void* stream, int flags, const float* noise,
                          float noise_scale, int quant_bits) {
    SensorEpilogue epi;
    if (const int rc = make_epilogue(flags, noise, noise_scale, quant_bits, &epi)) return rc;
    if (!raw || !gmax || !y) return B200CAM_E_NULL;
    if (count < 0 || count % 4 != 0) return B200CAM_E_BAD_SIZE;
    if (!al16(raw) || !al16(y)) return B200CAM_E_ALIGN;
    if (count == 0) return 0;
    const auto r4 = reinterpret_cast<const float4*>(raw);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (epi.seed != nullptr)
        k_lnormalise<true, Out, true><<<ew_grid(count / 4), EWT, 0, s>>>(r4, gmax, y, count / 4, epi);
    else if (flags)
        k_lnormalise<true><<<ew_grid(count / 4), EWT, 0, s>>>(r4, gmax, y, count / 4, epi);
    else
        k_lnormalise<false><<<ew_grid(count / 4), EWT, 0, s>>>(r4, gmax, y, count / 4, epi);
    LLAUNCH();
    return 0;
}

template <class G>
static int lens_dot(const G* grad_y, const float* raw, const float* gmax, float* dot_ties, void* workspace, size_t workspace_bytes, int B,
                    int P, void* stream) {
    if (!lens_n_ok(P) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!grad_y || !raw || !gmax || !dot_ties || !workspace) return B200CAM_E_NULL;
    if (!al16(grad_y) || !al16(raw)) return B200CAM_E_ALIGN;
    Ws ws(workspace, 2 * P, B);
    if (workspace_bytes < ws.bytes) return B200CAM_E_WORKSPACE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const long long n4 = static_cast<long long>(B) * 3 * P * P / 4;
    const int grid = ew_grid(n4);
    k_ldot<<<grid, EWT, 0, s>>>(grad_y, reinterpret_cast<const float4*>(raw), gmax, n4, ws.dpart);
    LLAUNCH();
    k_ldot_final<<<1, EWT, 0, s>>>(ws.dpart, grid, dot_ties);
    LLAUNCH();
    return 0;
}

template <class G>
static int lens_bwd(const G* grad_y, const float* raw, const float* gmax, const float* coef, const float* otf, const float* spectrum,
                    float* grad_kernel, float* grad_img, void* workspace, size_t workspace_bytes, int B, int P, void* stream) {
    if (!lens_n_ok(P) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!grad_y || !raw || !gmax || !coef || !otf || !spectrum || !grad_kernel || !workspace) return B200CAM_E_NULL;
    if (!al16(grad_y) || !al16(raw) || !al16(spectrum) || !al16(workspace)) return B200CAM_E_ALIGN;
    const int N = 2 * P;
    if (workspace_bytes < Ws(nullptr, N, B).bytes) return B200CAM_E_WORKSPACE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const float2* o = reinterpret_cast<const float2*>(otf);
    const float2* sp = reinterpret_cast<const float2*>(spectrum);
    switch (N) {
        case 128: return bwd_impl<128>(grad_y, raw, gmax, coef, o, sp, grad_kernel, grad_img, workspace, B, s);
        case 256: return bwd_impl<256>(grad_y, raw, gmax, coef, o, sp, grad_kernel, grad_img, workspace, B, s);
        case 512: return bwd_impl<512>(grad_y, raw, gmax, coef, o, sp, grad_kernel, grad_img, workspace, B, s);
        default: return bwd_impl<1024>(grad_y, raw, gmax, coef, o, sp, grad_kernel, grad_img, workspace, B, s);
    }
}

extern "C" {

size_t b200cam_lens_sensor_workspace_bytes(int P, int B) {
    if (!lens_n_ok(P) || B < 1) return 0;
    return Ws(nullptr, 2 * P, B).bytes;
}

int b200cam_lens_sensor_fwd(const float* img, const float* kernel, float* raw, float* gmax, float* otf, float* spectrum, void* workspace,
                            size_t workspace_bytes, int B, int P, void* stream) {
    return lens_fwd(ImgLoad{img}, img, kernel, raw, gmax, otf, spectrum, workspace, workspace_bytes, B, P, stream);
}

int b200cam_lens_sensor_fwd_u8(const unsigned char* img, const float* kernel, float* raw, float* gmax, float* otf, float* spectrum,
                               void* workspace, size_t workspace_bytes, int B, int P, void* stream) {
    return lens_fwd(ImgLoadU8{img}, img, kernel, raw, gmax, otf, spectrum, workspace, workspace_bytes, B, P, stream);
}

int b200cam_lens_normalise(const float* raw, const float* gmax, float* y, long long count, void* stream) {
    return b200cam_lens_normalise_ex(raw, gmax, y, count, stream, 0, nullptr, 0.f, 0);
}

int b200cam_lens_normalise_ex(const float* raw, const float* gmax, float* y, long long count, void* stream, int flags, const float* noise,
                              float noise_scale, int quant_bits) {
    return lens_normalise(raw, gmax, y, count, stream, flags, noise, noise_scale, quant_bits);
}

int b200cam_lens_normalise_bf16(const float* raw, const float* gmax, unsigned short* y, long long count, void* stream, int flags,
                                const float* noise, float noise_scale, int quant_bits) {
    return lens_normalise(raw, gmax, reinterpret_cast<bf16*>(y), count, stream, flags, noise, noise_scale, quant_bits);
}

int b200cam_lens_sensor_dot(const float* grad_y, const float* raw, const float* gmax, float* dot_ties, void* workspace, size_t workspace_bytes,
                            int B, int P, void* stream) {
    return lens_dot(grad_y, raw, gmax, dot_ties, workspace, workspace_bytes, B, P, stream);
}

int b200cam_lens_sensor_dot_bf16(const unsigned short* grad_y, const float* raw, const float* gmax, float* dot_ties, void* workspace,
                                 size_t workspace_bytes, int B, int P, void* stream) {
    return lens_dot(reinterpret_cast<const bf16*>(grad_y), raw, gmax, dot_ties, workspace, workspace_bytes, B, P, stream);
}

int b200cam_lens_sensor_bwd(const float* grad_y, const float* raw, const float* gmax, const float* coef, const float* otf, const float* spectrum,
                            float* grad_kernel, float* grad_img, void* workspace, size_t workspace_bytes, int B, int P, void* stream) {
    return lens_bwd(grad_y, raw, gmax, coef, otf, spectrum, grad_kernel, grad_img, workspace, workspace_bytes, B, P, stream);
}

int b200cam_lens_sensor_bwd_bf16(const unsigned short* grad_y, const float* raw, const float* gmax, const float* coef, const float* otf,
                                 const float* spectrum, float* grad_kernel, float* grad_img, void* workspace, size_t workspace_bytes, int B,
                                 int P, void* stream) {
    return lens_bwd(reinterpret_cast<const bf16*>(grad_y), raw, gmax, coef, otf, spectrum, grad_kernel, grad_img, workspace,
                    workspace_bytes, B, P, stream);
}

}  // extern "C"
