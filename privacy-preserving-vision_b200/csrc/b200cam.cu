// b200cam: __global__ wrappers, launch sequencing and the C ABI (include/b200cam.h).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <type_traits>
#include <utility>

#include "../../include/b200cam.h"
#include "kernels.cuh"
#include "plane.cuh"

namespace b200cam {

// ------------------------------------------------------------------------------------------
// __global__ wrappers: one CUDA thread per Exec "tid", dynamic shared memory as float2[]
// ------------------------------------------------------------------------------------------
extern __shared__ __align__(16) unsigned char smem_raw[];
// programmatic dependent launch: let the next kernel of the stream be scheduled now, then wait until the previous one has
// completed and its writes are visible (no-ops for a kernel launched without the attribute)
__constant__ int c_pdl_trigger = 0;      // 1: signal the dependents at kernel entry (B200CAM_PDL_TRIGGER=1); 0: at completion
__device__ __forceinline__ void pdl_gate() {
#if defined(B200CAM_PDL_BUILD)
    if (c_pdl_trigger) asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    asm volatile("griddepcontrol.wait;\n" ::: "memory");
#endif
}
#define SMEM2 reinterpret_cast<float2*>(smem_raw)

template <int N, class In = float>
__global__ void __launch_bounds__(RowsR2CSmem<N>::THREADS) k_rows_r2c(RowsR2CParamsT<In> p) {
    pdl_gate();
    DeviceExec ex;
    rows_r2c_body<N>(ex, p, SMEM2);
}
// the same row pass as a persistent grid of `gridDim.x` CTAs walking the tiles: the number of resident CTAs per SM is
// then the launch's choice, not the occupancy limit - used for the image rows that run BESIDE the PSF chain, whose
// small high-priority kernels need free registers / shared memory on every SM the moment they are launched
template <int N, class In = float>
__global__ void __launch_bounds__(RowsStreamSmem<N, In>::THREADS) k_rows_r2c_persist(RowsR2CParamsT<In> p, int tiles_total) {
    pdl_gate();
    DeviceExec ex;
    rows_r2c_stream_body<N>(ex, p, SMEM2, tiles_total, static_cast<int>(gridDim.x));
}
template <int N, bool ONE_PASS>
__global__ void __launch_bounds__(RowsC2RStreamSmem<N>::THREADS, N <= 256 ? 4 : (N == 512 ? 2 : 1)) k_rows_c2r_persist(RowsC2RParams p, int tiles_total, unsigned* err) {
    pdl_gate();
    DeviceExec ex;
    ex.err = err;
    rows_c2r_stream_body<N, DeviceExec, ONE_PASS>(ex, p, SMEM2, tiles_total, static_cast<int>(gridDim.x));
}
template <int N>
__global__ void __launch_bounds__(ColsSmem<N>::THREADS, N <= 256 ? 4 : (N == 512 ? 2 : 1)) k_cols_conv(ColsConvParams p) {
    pdl_gate();
    DeviceExec ex;
    ConvState<N> st;
    cols_conv_body<N>(ex, p, SMEM2, &st);
}
template <int N>
__global__ void __launch_bounds__(ColsSmem<N>::THREADS) k_cols_fwd(ColsFwdParams p) {
    pdl_gate();
    DeviceExec ex;
    cols_fwd_body<N>(ex, p, SMEM2);
}
template <int N>
__global__ void __launch_bounds__(RowsR2CSmem<N>::THREADS) k_rows_c2r(RowsC2RParams p) {
    pdl_gate();
    DeviceExec ex;
    rows_c2r_body<N>(ex, p, SMEM2);
}
__global__ void __launch_bounds__(EW_THREADS) k_normalise(NormaliseParams p) {
    pdl_gate();
    DeviceExec ex;
    normalise_body(ex, p, gridDim.x);
}
// bf16 sensor image: reads the fp32 conv (p.y), writes the rounded image to `out`
__global__ void __launch_bounds__(EW_THREADS) k_normalise_bf16(NormaliseParams p, bf16* out) {
    pdl_gate();
    DeviceExec ex;
    normalise_body<bf16>(ex, p, gridDim.x, out);
}
// the same two with the Philox read-out (p.epi.seed): the noise is drawn in the kernel, no tensor is read
__global__ void __launch_bounds__(EW_THREADS) k_normalise_philox(NormaliseParams p) {
    pdl_gate();
    DeviceExec ex;
    normalise_body<float, true>(ex, p, gridDim.x);
}
__global__ void __launch_bounds__(EW_THREADS) k_normalise_bf16_philox(NormaliseParams p, bf16* out) {
    pdl_gate();
    DeviceExec ex;
    normalise_body<bf16, true>(ex, p, gridDim.x, out);
}
__global__ void __launch_bounds__(EW_THREADS) k_philox_noise(const b200cam_noise_seed* seed, float* out, long long n4) {
    DeviceExec ex;
    philox_noise_body(ex, seed, out, n4, gridDim.x);
}
template <int N>
__global__ void __launch_bounds__(ColsSmem<N>::THREADS, N <= 256 ? 3 : 1) k_cols_accum(ColsAccumParams p) {
    pdl_gate();
    DeviceExec ex;
    AccumState<N> st;
    cols_accum_body<N>(ex, p, SMEM2, &st);
}
template <int N>
__global__ void __launch_bounds__(ReduceInvSmem<N>::THREADS) k_cols_reduce_inv(ColsReduceInvParams p) {
    pdl_gate();
    DeviceExec ex;
    cols_reduce_inv_body<N>(ex, p, SMEM2);
}
template <class Img = float>
__global__ void __launch_bounds__(EW_THREADS) k_tie_term(TieTermParamsT<Img> p) {
    pdl_gate();
    __shared__ float s_coef[TIE_PASS * MAX_TIES];
    __shared__ int s_meta[3 * TIE_PASS * MAX_TIES];
    __shared__ int s_cnt[TIE_PASS + 1];
    DeviceExec ex;
    tie_term_body(ex, p, gridDim.x, s_coef, s_meta, s_cnt);
}
__global__ void __launch_bounds__(EW_THREADS) k_tie_term_img(TieTermImgParams p) {
    pdl_gate();
    DeviceExec ex;
    tie_term_img_body(ex, p, gridDim.x);
}
template <int N, class Load>
__global__ void __launch_bounds__(CRowsSmem<N>::THREADS) k_crows_fwd(CRowsFwdParams p, Load load) {
    pdl_gate();
    DeviceExec ex;
    crows_fwd_body<N>(ex, p, load, SMEM2);
}
template <int N>
__global__ void __launch_bounds__(CColsSmem<N>::THREADS) k_ccols_mix(CColsMixParams p) {
    pdl_gate();
    DeviceExec ex;
    ccols_mix_body<N>(ex, p, SMEM2);
}
template <int N, class Epi>
__global__ void __launch_bounds__(CRowsSmem<N>::THREADS) k_crows_inv(CRowsInvParams p, Epi epi) {
    pdl_gate();
    DeviceExec ex;
    crows_inv_body<N>(ex, p, epi, SMEM2);
}
template <int N>
__global__ void __launch_bounds__(HGradSmem<N>::THREADS) k_crows_inv_hgrad(CRowsInvParams p, PupilLoad pupil, float* gh) {
    pdl_gate();
    DeviceExec ex;
    crows_inv_hgrad_body<N>(ex, p, pupil, gh, SMEM2);
}
// ------------------------------------------------------------------------------------------
// dL/dh tile + all-reduce over NVLink peer memory in ONE kernel (data parallel: SURVEY 8e).
// Every rank owns a symmetric buffer  [epochs 8 KB][2 parities][world][N*N] of 8-byte words  (value, epoch).
// CTA t computes its CROWS rows of the local dL/dh (same body as k_crows_inv_hgrad) and PUSHES them into slot[rank] of
// every peer's buffer as (value, epoch) words - data and flag travel in ONE 8-byte store (delivered atomically over
// NVLink), so there is no fence, no remote atomic and no separate flag: the receiver polls each word until its epoch
// half shows the current step (the low-latency protocol of collective libraries; half the link bandwidth, which a
// 256 KB gradient does not need).  Each thread then sums the `world` slots of its elements in rank order - every rank
// holds the bit-identical sum.  No grid-wide barrier: an element only ever waits for the same element of the peers.
// Epochs are monotone per-tile counters kept in the buffer itself (CUDA-graph replays reuse the frozen kernel
// arguments); slots are double buffered by epoch parity (a peer can be at most one step ahead), so a word carrying
// epoch e-2 is recognisably stale.
// ------------------------------------------------------------------------------------------
constexpr int COMM_MAX_WORLD = 16;
constexpr size_t COMM_HEADER_BYTES = 8192;
struct CommDev {
    unsigned char* buf[COMM_MAX_WORLD];     // every rank's buffer, as mapped in this process
    int rank, world;
    float scale;
    long long timeout_clk;                  // give-up deadline of the receive loop in SM clocks (B200CAM_COMM_TIMEOUT_S, default 30 s)
};

template <int N>
__global__ void __launch_bounds__(HGradSmem<N>::THREADS) k_crows_inv_hgrad_allreduce(CRowsInvParams p, PupilLoad pupil,
                                                                                     float* gh, CommDev c, unsigned* err) {
    pdl_gate();
    DeviceExec ex;
    crows_inv_hgrad_body<N>(ex, p, pupil, gh, SMEM2);            // local dL/dh rows of this tile -> gh (ends with a barrier)
    __shared__ unsigned s_epoch;
    constexpr int COUNT = Tile<N>::CROWS * N;
    const int tile = blockIdx.x, tid = threadIdx.x;
    const size_t NN = static_cast<size_t>(N) * N, base = static_cast<size_t>(tile) * COUNT;
    if (tid == 0) {
        unsigned* ep = reinterpret_cast<unsigned*>(c.buf[c.rank]) + tile;
        s_epoch = *ep + 1;
        *ep = s_epoch;
    }
    __syncthreads();
    const unsigned epoch = s_epoch;
    const size_t parity_off = static_cast<size_t>(epoch & 1) * c.world * NN;
    for (int i = tid; i < COUNT; i += blockDim.x) {
        const uint2 word = make_uint2(__float_as_uint(gh[base + i]), epoch);
        for (int r = 0; r < c.world; ++r) {
            uint2* slot = reinterpret_cast<uint2*>(c.buf[r] + COMM_HEADER_BYTES) + parity_off + c.rank * NN + base;
            slot[i] = word;                                      // one 8-byte store: value and flag together
        }
    }
    // receive: a thread's elements x four ranks are polled as ONE batch of loads (each volatile load is an L2 round trip;
    // polled one after the other they cost more than the exchange itself), summed in rank order once all have arrived
    const uint2* slots = reinterpret_cast<const uint2*>(c.buf[c.rank] + COMM_HEADER_BYTES) + parity_off + base;
    constexpr int THREADS = HGradSmem<N>::THREADS;
    constexpr int K = (COUNT + THREADS - 1) / THREADS;
    float acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.f;
    // A peer that never arrives (died, or the ranks called the collective a different number of times) must not hang the
    // device for ever, and must not yield a result either: after `c.timeout_clk` cycles the tile gives up, raises the
    // device error word (b200cam_device_error -> RuntimeError in the wrapper) and fills its rows of dL/dh with NaN.
    const long long t0 = clock64();
    bool gave_up = false;
    for (int r0 = 0; r0 < c.world; r0 += 4) {
        uint2 w[K][4];
        bool ok;
        do {
            ok = true;
#pragma unroll
            for (int k = 0; k < K; ++k) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int i = tid + k * THREADS;
                    w[k][q] = make_uint2(0u, epoch);
                    if (i < COUNT && r0 + q < c.world) {
                        const uint2* src = slots + static_cast<size_t>(r0 + q) * NN + i;
                        asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];\n" : "=r"(w[k][q].x), "=r"(w[k][q].y) : "l"(src) : "memory");
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int q = 0; q < 4; ++q) ok = ok && (w[k][q].y == epoch);
            if (!ok && clock64() - t0 > c.timeout_clk) {
                gave_up = true;
                break;
            }
        } while (!ok);
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[k] += __uint_as_float(w[k][q].x);      // rank order; absent ranks add +0
    }
    if (gave_up && err != nullptr) atomicExch(err, B200CAM_DEVERR_ALLREDUCE_WAIT);
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int i = tid + k * THREADS;
        if (i < COUNT) gh[base + i] = gave_up ? __int_as_float(0x7fc00000) : acc[k] * c.scale;
    }
}

__global__ void __launch_bounds__(EW_THREADS) k_psf_finalise(PsfFinaliseParams p) {
    pdl_gate();
    __shared__ float red[3 * EW_THREADS + 2];
    DeviceExec ex;
    psf_finalise_body(ex, p, gridDim.x, red);
}
__global__ void __launch_bounds__(EW_THREADS) k_psf_grad_prepare(PsfGradPrepParams p) {
    pdl_gate();
    __shared__ float red[EW_THREADS];
    DeviceExec ex;
    psf_grad_prepare_body(ex, p, gridDim.x, red);
}
// ------------------------------------------------------------------------------------------
// Plane-resident N = 256 sensor kernels (plane.cuh): device execution policy and __global__ wrappers
// ------------------------------------------------------------------------------------------
struct PlaneCtx {
    int rank, tid;
    plane::Thread& t;
    float2* smem;
    unsigned* err;          // device error word (mapped host memory): set when a wait gives up
    __device__ __forceinline__ float2 shfl_v(int idx, int src, bool half) {
        const unsigned mask = half ? (0xffffu << (threadIdx.x & 16)) : 0xffffffffu;
        const int s = (threadIdx.x & 16) | src;
        return make_float2(__shfl_sync(mask, t.v[idx].x, s), __shfl_sync(mask, t.v[idx].y, s));
    }
    __device__ __forceinline__ float2 shfl_u(int idx, int src, bool half) {
        const unsigned mask = half ? (0xffffu << (threadIdx.x & 16)) : 0xffffffffu;
        const int s = (threadIdx.x & 16) | src;
        return make_float2(__shfl_sync(mask, t.u[idx].x, s), __shfl_sync(mask, t.u[idx].y, s));
    }
    __device__ __forceinline__ unsigned lane0_key() { return __shfl_sync(0xffffffffu, t.key, 0); }
    __device__ __forceinline__ unsigned warp_max_key() { return __reduce_max_sync(0xffffffffu, t.key); }
    __device__ __forceinline__ float warp_sum_dot() {
        float s = t.dot;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);     // fixed tree: deterministic
        return s;
    }
    __device__ __forceinline__ void bulk_init(unsigned long long* bar) { BulkOps::init(bar); }
    __device__ __forceinline__ void bulk_fence_init() { BulkOps::fence_init(); }
    __device__ __forceinline__ void bulk_expect(unsigned long long* bar, unsigned bytes) { BulkOps::expect(bar, bytes); }
    __device__ __forceinline__ void bulk_load(void* dst, const void* src, unsigned bytes, unsigned long long* bar) { BulkOps::copy(dst, src, bytes, bar); }
    __device__ __forceinline__ void bulk_wait(unsigned long long* bar, unsigned parity) { BulkOps::wait(bar, parity); }
    // The per-image maximum is taken across the 3 x 8 CTAs that hold the image's planes: max first, then the arrival.
    // No acquire fences anywhere on this path: an acquire at gpu / cluster scope makes ptxas emit CCTL.IVALL (the whole
    // L1 of the SM is invalidated - measured: 30 % of this kernel's stall samples sat on it).  Release on the writer
    // (membar + atomic) and L2-coherent accesses on the reader (relaxed.gpu load, then an atomic read of the max) order
    // the two words without touching L1.
    __device__ __forceinline__ void publish_max(unsigned* s, unsigned key) {
        asm volatile("red.relaxed.gpu.global.max.u32 [%0], %1;\n" ::"l"(s), "r"(key) : "memory");
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;\n" ::"l"(s + 1) : "memory");
    }
    // All 24 CTAs are resident (the grid is one wave of co-scheduled clusters, sized from the occupancy API) and published
    // a whole pipeline step ago.  A wait that outlives ~2 s means a broken launch: it is reported through the device
    // error word (b200cam_device_error), never turned into a silent result.
    __device__ __forceinline__ unsigned wait_max(unsigned* s, unsigned target) {
        unsigned n;
        long long t0 = 0;
        for (int spin = 0;; ++spin) {
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];\n" : "=r"(n) : "l"(s + 1) : "memory");
            if (n >= target) break;
            if (spin == 64) t0 = clock64();
            if (spin > 64 && clock64() - t0 > 4000000000LL) {
                if (err != nullptr) atomicExch(err, B200CAM_DEVERR_IMAGE_MAX_WAIT);
                break;
            }
        }
        unsigned key;
        asm volatile("atom.relaxed.gpu.global.max.u32 %0, [%1], 0;\n" : "=r"(key) : "l"(s) : "memory");
        return key;
    }
};
// The barrier of a cluster is NOT barrier.cluster: its wait carries acquire semantics, for which ptxas emits CCTL.IVALL
// (invalidate the SM's whole L1) - with bulk copies in flight that instruction alone held 30 % of k_pconv's stall samples.
// The crossing data is read with L1-bypassing loads, so no invalidation is needed; what is needed is a release on the
// writers and an arrival count the readers can poll:  bar.sync ; thread 0: red.release.gpu (membar + add) on the cluster's
// word in global memory ... thread 0: poll with relaxed loads ; bar.sync.  The word is never reset: every CTA reads it
// before an initial (hardware) cluster barrier, i.e. before any arrival of this launch, and counts from there - so the
// workspace needs no initialisation and CUDA-graph replays just keep counting.
struct PlaneExec {
    PlaneCtx ctx;
    unsigned* ctr = nullptr;
    unsigned base = 0, waits = 0;
    template <class F>
    __device__ __forceinline__ void each(F&& f) { f(ctx); }
    __device__ __forceinline__ void sync_warp() { __syncwarp(); }
    __device__ __forceinline__ void sync_cta() { __syncthreads(); }
    __device__ __forceinline__ void cluster_begin(unsigned* word) {
        ctr = word;
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];\n" : "=r"(base) : "l"(ctr) : "memory");
        asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
        asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
    }
    __device__ __forceinline__ void cluster_arrive() {
        __syncthreads();
        if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;\n" ::"l"(ctr) : "memory");
    }
    __device__ __forceinline__ void cluster_wait() {
        ++waits;
        if (threadIdx.x == 0) {
            unsigned n;
            long long t0 = 0;
            for (int spin = 0;; ++spin) {
                asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];\n" : "=r"(n) : "l"(ctr) : "memory");
                if (n - base >= waits * plane::C) break;
                if (spin == 64) t0 = clock64();
                if (spin > 64 && clock64() - t0 > 4000000000LL) {
                    if (ctx.err != nullptr) atomicExch(ctx.err, B200CAM_DEVERR_GRID_BARRIER);
                    break;
                }
            }
        }
        __syncthreads();
    }
};

__global__ void __launch_bounds__(plane::THREADS, 4) k_prow(plane::RowParams p) {
    pdl_gate();
    plane::Thread t;
    PlaneExec x{{0, static_cast<int>(threadIdx.x), t, SMEM2, nullptr}};
    plane::prow_body(x, p, static_cast<int>(blockIdx.x), static_cast<int>(gridDim.x));
}
__global__ void __cluster_dims__(plane::C, 1, 1) __launch_bounds__(plane::THREADS, 2) k_pconv(plane::ConvParams p, unsigned* ctr, unsigned* err) {
    pdl_gate();
    plane::Thread t;
    const int cluster = blockIdx.x / plane::C;
    PlaneExec x{{static_cast<int>(blockIdx.x % plane::C), static_cast<int>(threadIdx.x), t, SMEM2, err}};
    const int T = plane::planes_of_cluster(cluster, p.B, p.G3);
    if (T == 0) return;
    x.cluster_begin(ctr + 32 * cluster);
    plane::pconv_init(x, p, cluster);
    for (int it = 0; it <= T + 1; ++it) plane::pconv_step(x, p, cluster, it);
}
__global__ void __cluster_dims__(plane::C, 1, 1) __launch_bounds__(plane::THREADS, 2) k_pacc(plane::AccParams p, unsigned* ctr, unsigned* err) {
    pdl_gate();
    plane::Thread t;
    const int cluster = blockIdx.x / plane::C;
    PlaneExec x{{static_cast<int>(blockIdx.x % plane::C), static_cast<int>(threadIdx.x), t, SMEM2, err}};
    x.cluster_begin(ctr + 32 * cluster);
    plane::pacc_body(x, p, cluster);
}
// coef[b] = sum(g_b * y_b) / (n_b m_b) = sum(g_b * conv_b) / (n_b m_b^2) from the 24 per-CTA Parseval partials of k_pacc
// (which carry a factor 4) - the weight of the arg-max term of the amax backward (Optics.py:128)
__global__ void __launch_bounds__(64) k_pcoef(const float* dotp, const float* img_max, const int* tie_count, float* coef, int B) {
    pdl_gate();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float s = 0.f;
    for (int i = 0; i < 3 * plane::DOT_PER_PLANE; ++i) s += dotp[b * 3 * plane::DOT_PER_PLANE + i];     // fixed order: deterministic
    const int n = tie_count[b] > 0 ? tie_count[b] : 1;
    const float m = img_max[b];
    coef[b] = 0.25f * s / (static_cast<float>(n) * m * m);
}

// ------------------------------------------------------------------------------------------
// PSF chain as ONE cooperative launch per direction: the same bodies, run as virtual blocks, with
// grid-wide barriers where the multi-kernel version had kernel boundaries.
// ------------------------------------------------------------------------------------------
// Grid-wide barrier for the cooperative PSF kernels (all CTAs are co-resident: cudaLaunchCooperativeKernel).
// One monotonically increasing arrival counter; barrier number k (1-based) waits for k * gridDim.x arrivals.
// ~1.2 us on 192 CTAs (one L2 atomic + one polled line), against ~5 us for cooperative_groups' grid.sync().
struct GridBarrier {
    unsigned* ctr;      // [2]: arrivals, departures; both zero between launches
    unsigned* err = nullptr;
    unsigned k = 0;
    __device__ __forceinline__ void sync() {
        __syncthreads();
        if (threadIdx.x == 0) {
            ++k;
            __threadfence();
            atomicAdd(ctr, 1u);
            const unsigned target = k * gridDim.x;
            const long long t0 = clock64();          // never hang the device: give up after ~2 s and say so (device error word)
            while (*reinterpret_cast<volatile unsigned*>(ctr) < target) {
                if (clock64() - t0 > 4000000000LL) {
                    if (err != nullptr) atomicExch(err, B200CAM_DEVERR_GRID_BARRIER);
                    break;
                }
            }
            __threadfence();
        }
        __syncthreads();
    }
    // after the last barrier: the last CTA to leave zeroes the counters for the next launch
    __device__ __forceinline__ void finish() {
        if (threadIdx.x == 0) {
            __threadfence();
            if (atomicAdd(ctr + 1, 1u) == gridDim.x - 1) {
                ctr[0] = 0;
                ctr[1] = 0;
                __threadfence();
            }
        }
    }
};

constexpr int COOP_THREADS = 384;   // >= the widest body (3 wavelength groups of the N=1024 row pass)

struct PsfFwdArgs {
    CRowsFwdParams rows_fwd; PupilLoad pupil;
    CColsMixParams mix;
    CRowsInvParams rows_inv; IntensityEpilogue inten;
    PsfFinaliseParams fin;
    unsigned* barrier;
    unsigned* err;
};

template <int N>
__global__ void __launch_bounds__(COOP_THREADS) k_psf_fwd_coop(PsfFwdArgs a) {
    pdl_gate();
    GridBarrier grid{a.barrier, a.err};
    __shared__ float red[3 * EW_THREADS + 2];
    using T = Tile<N>;
    const int G = gridDim.x;
    for (int vb = blockIdx.x; vb < 3 * (N / T::CROWS); vb += G) {
        VirtualExec ex{vb % (N / T::CROWS), vb / (N / T::CROWS), CRowsSmem<N>::THREADS};
        crows_fwd_body<N>(ex, a.rows_fwd, a.pupil, SMEM2);
    }
    grid.sync();
    for (int vb = blockIdx.x; vb < (N + CColsSmem<N>::CC - 1) / CColsSmem<N>::CC; vb += G) {
        VirtualExec ex{vb, 0, CColsSmem<N>::THREADS};
        ccols_mix_body<N>(ex, a.mix, SMEM2);
    }
    grid.sync();
    for (int vb = blockIdx.x; vb < 3 * (N / T::CROWS); vb += G) {
        VirtualExec ex{vb % (N / T::CROWS), vb / (N / T::CROWS), CRowsSmem<N>::THREADS};
        crows_inv_body<N>(ex, a.rows_inv, a.inten, SMEM2);
    }
    grid.sync();
    {
        VirtualExec ex{static_cast<int>(blockIdx.x), 0, EW_THREADS};
        psf_finalise_body(ex, a.fin, G, red);
    }
    grid.finish();
}

struct PsfBwdArgs {
    PsfGradPrepParams prep;
    CRowsFwdParams rows_fwd; GradFieldLoad gload;
    CColsMixParams mix;
    CRowsInvParams rows_inv; PupilLoad pupil; float* gh;
    unsigned* barrier;
    unsigned* err;
};

template <int N>
__global__ void __launch_bounds__(COOP_THREADS) k_psf_bwd_coop(PsfBwdArgs a) {
    pdl_gate();
    GridBarrier grid{a.barrier, a.err};
    __shared__ float red[3 * EW_THREADS + 2];
    using T = Tile<N>;
    const int G = gridDim.x;
    {
        VirtualExec ex{static_cast<int>(blockIdx.x), 0, EW_THREADS};
        psf_grad_prepare_body(ex, a.prep, G, red);
    }
    grid.sync();
    for (int vb = blockIdx.x; vb < 3 * (N / T::CROWS); vb += G) {
        VirtualExec ex{vb % (N / T::CROWS), vb / (N / T::CROWS), CRowsSmem<N>::THREADS};
        crows_fwd_body<N>(ex, a.rows_fwd, a.gload, SMEM2);
    }
    grid.sync();
    for (int vb = blockIdx.x; vb < (N + CColsSmem<N>::CC - 1) / CColsSmem<N>::CC; vb += G) {
        VirtualExec ex{vb, 0, CColsSmem<N>::THREADS};
        ccols_mix_body<N>(ex, a.mix, SMEM2);
    }
    grid.sync();
    for (int vb = blockIdx.x; vb < N / T::CROWS; vb += G) {
        VirtualExec ex{vb, 0, HGradSmem<N>::THREADS};
        crows_inv_hgrad_body<N>(ex, a.rows_inv, a.pupil, a.gh, SMEM2);
    }
    grid.finish();
}

template <int N>
constexpr int coop_smem_bytes() {
    return HGradSmem<N>::BYTES > CColsSmem<N>::BYTES ? HGradSmem<N>::BYTES : CColsSmem<N>::BYTES;
}
static_assert(HGradSmem<1024>::BYTES <= 227 * 1024 && HGradSmem<512>::BYTES <= 227 * 1024 && CColsSmem<1024>::BYTES <= 227 * 1024,
              "shared memory budget");
static_assert(HGradSmem<1024>::THREADS <= COOP_THREADS && HGradSmem<512>::THREADS <= COOP_THREADS && CColsSmem<1024>::THREADS <= COOP_THREADS && EW_THREADS <= COOP_THREADS,
              "cooperative block too small for a body");

__global__ void __launch_bounds__(EW_THREADS) k_zernike_fwd(ZernikeFwdParams p) {
    pdl_gate();
    __shared__ int flag;
    DeviceExec ex;
    zernike_fwd_body(ex, p, &flag);
}
__global__ void __launch_bounds__(EW_THREADS) k_zernike_bwd(ZernikeBwdParams p) {
    pdl_gate();
    __shared__ float red[EW_THREADS];
    DeviceExec ex;
    zernike_bwd_body(ex, p, red);
}
__global__ void __launch_bounds__(EW_THREADS) k_zernike_bwd_fin(const float* partial, float* gcoef, int T, int splits) {
    pdl_gate();
    const int j = blockIdx.x * EW_THREADS + threadIdx.x;
    if (j < T) {
        float acc = 0.f;
        for (int s = 0; s < splits; ++s) acc += partial[j * splits + s];
        gcoef[j] = acc;
    }
}

__global__ void __launch_bounds__(EW_THREADS) k_crop_abs_resize_fwd(CropAbsResizeParams p) {
    pdl_gate();
    DeviceExec ex;
    crop_abs_resize_fwd_body(ex, p, gridDim.x);
}
__global__ void __launch_bounds__(EW_THREADS) k_crop_abs_resize_bwd(CropAbsResizeBwdParams p) {
    pdl_gate();
    DeviceExec ex;
    crop_abs_resize_bwd_body(ex, p, gridDim.x);
}

__global__ void k_fill_twiddle(float2* tw, int N) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < N) {
        double s, c;
        sincospi(-2.0 * j / N, &s, &c);
        tw[j] = make_float2(static_cast<float>(c), static_cast<float>(s));
    }
}

// ------------------------------------------------------------------------------------------
// per-device state: twiddle tables (the only thing the library owns)
// ------------------------------------------------------------------------------------------
constexpr int MAX_DEV = 64;
// grid of the element-wise PSF kernels: one pass of 256-thread CTAs over the 3*N*N elements, at most 1024 CTAs (the size
// of their partial-sum slices in the workspace).  These kernels are latency chains: one element per thread where possible.
static int ew_grid(int N) {
    const long long want = (3LL * N * N + EW_THREADS - 1) / EW_THREADS;
    return static_cast<int>(want < 1024 ? want : 1024);
}

inline int log2i(int n) { int l = 0; while ((1 << l) < n) ++l; return l; }
struct DeviceState {
    float2* tw[11] = {nullptr}; int sms = 0; int coop_grid[11] = {0}; unsigned* bar = nullptr;
    int conv_slots[11] = {0}, accum_slots[11] = {0};     // resident CTAs of the persistent column kernels
    cudaEvent_t chain_ev = nullptr;                      // orders a caller stream behind the first PSF-chain kernel
    int r2c_fit[11] = {0}, c2r_fit[11] = {0};            // resident CTAs per SM of the persistent row kernels
    int r2c16_fit[11] = {0};                             // ... and of the bf16-input forward row kernel (upstream gradient)
    int r2c8_fit[11] = {0};                              // ... and of the uint8-input forward row kernel (uint8 images)
    float* scratch = nullptr;                            // SCRATCH_FLOATS floats: slice partials of the Zernike adjoint
    int prow_fit = 0, pconv_g3 = 0, pacc_g3 = 0;         // plane kernels (N = 256): resident CTAs per SM / co-resident cluster triples
    unsigned* err_host = nullptr; unsigned* err_dev = nullptr;   // device error word (mapped pinned host memory)
};
constexpr int SCRATCH_FLOATS = 16384;
static DeviceState g_state[MAX_DEV];
static std::mutex g_mutex;

static cudaEvent_t chain_event() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return nullptr;
    return g_state[dev].chain_ev;
}
static int sm_count() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return 0;
    return g_state[dev].sms;
}
// The PSF chain is a dozen tiny dependent steps.  Launched eagerly it runs as ONE cooperative kernel per direction
// with grid-wide barriers (GridBarrier above) where the multi-kernel version has kernel boundaries: that saves the
// CPU launch cost of 6 kernels.  Replayed from a CUDA graph the two cost the same device time (30 us per direction,
// the steps themselves are latency bound) and the multi-kernel version releases its SMs between steps, which matters
// when the image row pass runs beside it (261 vs 267 us per step) - so: cooperative unless the stream is being
// captured.  B200CAM_COOP=0/1 forces one or the other.
static int coop_grid(int N, cudaStream_t s) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return 0;
    static const int mode = [] { const char* e = getenv("B200CAM_COOP"); return e ? (e[0] == '0' ? 0 : 1) : -1; }();
    if (mode == 0 || g_state[dev].bar == nullptr) return 0;
    if (mode < 0) {
        cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(s, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) return 0;
    }
    return g_state[dev].coop_grid[log2i(N)];
}
static const float2* twiddle(int N) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return nullptr;
    return g_state[dev].tw[log2i(N)];
}

template <class K>
static cudaError_t optin(K kernel, int bytes) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

template <int N>
static cudaError_t init_kernels() {
    cudaError_t e;
    if ((e = optin(k_rows_r2c<N>, RowsR2CSmem<N>::BYTES))) return e;
    if ((e = optin(k_rows_c2r<N>, RowsR2CSmem<N>::BYTES))) return e;
    if ((e = optin(k_rows_r2c_persist<N>, RowsStreamSmem<N>::BYTES))) return e;
    if ((e = optin(k_rows_r2c<N, bf16>, RowsR2CSmem<N>::BYTES))) return e;
    if ((e = optin(k_rows_r2c_persist<N, bf16>, RowsStreamSmem<N, bf16>::BYTES))) return e;
    if ((e = optin(k_rows_r2c<N, u8>, RowsR2CSmem<N>::BYTES))) return e;
    if ((e = optin(k_rows_r2c_persist<N, u8>, RowsStreamSmem<N, u8>::BYTES))) return e;
    if ((e = optin(k_rows_c2r_persist<N, false>, RowsC2RStreamSmem<N>::BYTES))) return e;
    if ((e = optin(k_rows_c2r_persist<N, true>, RowsC2RStreamSmem<N>::BYTES))) return e;
    if ((e = optin(k_cols_conv<N>, ColsSmem<N>::BYTES_CONV))) return e;
    if ((e = optin(k_cols_fwd<N>, ColsSmem<N>::BYTES))) return e;
    if ((e = optin(k_cols_accum<N>, ColsSmem<N>::BYTES))) return e;
    if ((e = optin(k_cols_reduce_inv<N>, ReduceInvSmem<N>::BYTES))) return e;
    if ((e = optin(k_crows_fwd<N, PupilLoad>, CRowsSmem<N>::BYTES))) return e;
    if ((e = optin(k_crows_fwd<N, GradFieldLoad>, CRowsSmem<N>::BYTES))) return e;
    if ((e = optin(k_crows_inv<N, IntensityEpilogue>, CRowsSmem<N>::BYTES))) return e;
    if ((e = optin(k_crows_inv_hgrad<N>, HGradSmem<N>::BYTES))) return e;
    if ((e = optin(k_crows_inv_hgrad_allreduce<N>, HGradSmem<N>::BYTES))) return e;
    if ((e = optin(k_ccols_mix<N>, CColsSmem<N>::BYTES))) return e;
    if ((e = optin(k_psf_fwd_coop<N>, coop_smem_bytes<N>()))) return e;
    if ((e = optin(k_psf_bwd_coop<N>, coop_smem_bytes<N>()))) return e;
    return cudaSuccess;
}

// largest co-resident grid of the cooperative PSF kernels, capped at the useful number of virtual blocks
template <int N>
static cudaError_t coop_grid_size(int dev, int sms, int* out) {
    int coop = 0, nb_f = 0, nb_b = 0;
    cudaError_t e;
    if ((e = cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev))) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb_f, k_psf_fwd_coop<N>, COOP_THREADS, coop_smem_bytes<N>()))) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb_b, k_psf_bwd_coop<N>, COOP_THREADS, coop_smem_bytes<N>()))) return e;
    const int nb = nb_f < nb_b ? nb_f : nb_b;
    int g = coop ? sms * nb : 0;
    const int useful = 3 * (N / Tile<N>::CROWS);
    if (g > useful) g = useful;
    *out = g;
    return cudaSuccess;
}

// resident CTAs (one wave) of the persistent column kernels on this device
template <int N>
static cudaError_t row_fits(int* r2c, int* r2c16, int* r2c8, int* c2r) {
    cudaError_t e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(r2c, k_rows_r2c_persist<N>, RowsStreamSmem<N>::THREADS, RowsStreamSmem<N>::BYTES))) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(r2c16, k_rows_r2c_persist<N, bf16>, RowsStreamSmem<N, bf16>::THREADS,
                                                           RowsStreamSmem<N, bf16>::BYTES))) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(r2c8, k_rows_r2c_persist<N, u8>, RowsStreamSmem<N, u8>::THREADS,
                                                           RowsStreamSmem<N, u8>::BYTES))) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(c2r, k_rows_c2r_persist<N, false>, RowsC2RStreamSmem<N>::THREADS, RowsC2RStreamSmem<N>::BYTES);
}
template <int N>
static cudaError_t column_slots(int sms, int* conv, int* accum) {
    int nc = 0, na = 0;
    cudaError_t e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nc, k_cols_conv<N>, ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV))) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&na, k_cols_accum<N>, ColsSmem<N>::THREADS, ColsSmem<N>::BYTES))) return e;
    *conv = sms * nc;
    *accum = sms * na;
    return cudaSuccess;
}

// The plane kernels (N = 256) run as ONE wave of co-scheduled 8-CTA clusters: the three clusters that hold the planes of
// an image exchange the image maximum through global memory while they are resident, so the grid must never exceed what
// the device keeps resident at once (cudaOccupancyMaxActiveClusters), rounded down to whole triples.
constexpr int PLANE_MAX_G3 = 24;        // sizes the crossing scratch and the partial planes of the backward
// Measured (round 2, B = 64, one B200, CUDA-graph replay; profiles/r02_plane_kernels.md): k_prow 30 us, k_pconv 116 us,
// k_pacc 70 us against 20 + (22 + 23 + 16) + (18 + 23) us for the generic kernels doing the same work - the cluster
// kernels execute fewer bytes but every plane costs them ~6 dependent synchronisations (stage barrier, cluster arrive /
// wait, image-max exchange) and the CTAs of a cluster and the clusters of an image all run at the pace of the slowest of
// their 24 CTAs.  They stay in the tree as an opt-in (B200CAM_PLANE=1), tested, not as the default path.
static bool plane_selected() {
    static const bool on = [] { const char* e = getenv("B200CAM_PLANE"); return e && e[0] == '1'; }();
    return on;
}
template <class K>
static cudaError_t max_cluster_triples(K kernel, int smem_bytes, int* g3) {
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(plane::THREADS);
    cfg.gridDim = dim3(plane::C);
    cfg.dynamicSmemBytes = smem_bytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = plane::C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int n = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
    if (e != cudaSuccess) return e;
    static const int cap = [] { const char* v = getenv("B200CAM_PLANE_G3"); return v ? atoi(v) : PLANE_MAX_G3; }();
    int t = n / 3;
    if (t > PLANE_MAX_G3) t = PLANE_MAX_G3;
    if (cap > 0 && t > cap) t = cap;
    *g3 = t;
    return cudaSuccess;
}
static cudaError_t plane_init(int dev) {
    cudaError_t e;
    if ((e = optin(k_prow, plane::SMEM_BYTES))) return e;
    if ((e = optin(k_pconv, plane::CONV_SMEM_BYTES))) return e;
    if ((e = optin(k_pacc, plane::ACC_SMEM_BYTES))) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&g_state[dev].prow_fit, k_prow, plane::THREADS, plane::SMEM_BYTES))) return e;
    if ((e = max_cluster_triples(k_pconv, plane::CONV_SMEM_BYTES, &g_state[dev].pconv_g3))) return e;
    if ((e = max_cluster_triples(k_pacc, plane::ACC_SMEM_BYTES, &g_state[dev].pacc_g3))) return e;
    return cudaSuccess;
}
static DeviceState* cur_state() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return nullptr;
    return &g_state[dev];
}

// grid of a persistent row kernel: `want` CTAs per SM, never more than fit at once (a persistent grid larger than one
// wave runs its surplus CTAs after the first ones have finished ALL their tiles), never more than there are tiles.
// `fit` = resident CTAs per SM of that kernel, measured at init.
static int persistent_grid(int fit, int want_per_sm, int total_tiles) {
    if (fit < 1) fit = 1;
    const int sms = sm_count() > 0 ? sm_count() : 148;
    const int per_sm = want_per_sm < fit ? want_per_sm : fit;
    const long long cap = static_cast<long long>(sms) * per_sm;
    return static_cast<int>(total_tiles < cap ? total_tiles : cap);
}
// in_bytes: element size of the forward row kernel's input (4 fp32, 2 bf16, 1 uint8)
static int rows_fit(int N, bool inverse, int in_bytes = 4) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return 1;
    if (!inverse && in_bytes == 2) return g_state[dev].r2c16_fit[log2i(N)];
    if (!inverse && in_bytes == 1) return g_state[dev].r2c8_fit[log2i(N)];
    return inverse ? g_state[dev].c2r_fit[log2i(N)] : g_state[dev].r2c_fit[log2i(N)];
}

// ------------------------------------------------------------------------------------------
// workspace carving (256-byte aligned slices of the caller's buffer)
// ------------------------------------------------------------------------------------------
struct Carver {
    unsigned char* base;
    size_t off = 0;
    explicit Carver(void* p) : base(static_cast<unsigned char*>(p)) {}
    template <class T>
    T* take(size_t count) {
        T* r = reinterpret_cast<T*>(base + off);
        off += (count * sizeof(T) + 255) / 256 * 256;
        return r;
    }
};

// The column kernels are persistent over images: CTA (colgroup, chunk) walks its chunk of the batch.  The number of
// chunks is normally chosen so that the whole grid is ONE wave of resident CTAs (slots = SMs x occupancy, measured at
// init): a second, partly filled wave costs as much as a full one.  Where one wave leaves SMs idle (N = 512 accumulate:
// 97 column groups on 148 one-CTA SMs) or cannot hold the grid at all (N = 1024: 193 column groups), a simple wave model
// - CTAs start in rounds of `slots`, a CTA costs its images plus a fixed prologue - picks a finer split when that is
// predicted at least 10 % faster (N = 512: 1 -> 3 chunks = two full rounds of 11 images instead of one of 32 on 2/3 of
// the SMs; N = 1024: 1 -> 2 chunks = three rounds of 4 images instead of two of 8).
constexpr int MAX_CHUNKS = 16;          // sizes the partial-sum workspace of the backward
static int col_chunks(int N, int B, int slots) {
    const int colgroups = (3 * (N / 2 + 1) + Tile<64>::COLS - 1) / Tile<64>::COLS;
    const int cap = B < MAX_CHUNKS ? (B < 1 ? 1 : B) : MAX_CHUNKS;
    int n = slots / colgroups;
    if (n > cap) n = cap;
    if (n < 1) n = 1;
    static const bool one_wave_only = [] { const char* e = getenv("B200CAM_ONE_WAVE"); return e && e[0] == '1'; }();
    if (one_wave_only) return n;
    auto cost = [&](int k) {
        const int rounds = (colgroups * k + slots - 1) / slots;
        return static_cast<float>(rounds) * (static_cast<float>((B + k - 1) / k) + 0.5f);
    };
    float best = cost(n);
    for (int k = 1; k <= cap; ++k)
        if (cost(k) < 0.9f * best) {
            best = cost(k);
            n = k;
        }
    return n;
}
static int conv_chunks(int N, int B) {
    int dev = 0;
    const int slots = (cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < MAX_DEV) ? g_state[dev].conv_slots[log2i(N)] : 0;
    static const int forced = [] { const char* e = getenv("B200CAM_CONV_CHUNKS"); return e ? atoi(e) : 0; }();   // experiments
    if (forced > 0) return forced > B ? B : (forced > MAX_CHUNKS ? MAX_CHUNKS : forced);
    return col_chunks(N, B, slots > 0 ? slots : 592);
}
static int accum_chunks(int N, int B) {
    static const int forced = [] { const char* e = getenv("B200CAM_ACCUM_CHUNKS"); return e ? atoi(e) : 0; }();
    if (forced > 0) return forced > B ? B : (forced > MAX_CHUNKS ? MAX_CHUNKS : forced);
    int dev = 0;
    const int slots = (cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < MAX_DEV) ? g_state[dev].accum_slots[log2i(N)] : 0;
    return col_chunks(N, B, slots > 0 ? slots : 592);
}

struct PsfWs {
    float2* st; float* I; float* gtot; float* part_rows; float* part_ew; int* arrive; unsigned* bar; float2* otf_rows;
    size_t bytes;
    PsfWs(void* p, int N) {
        Carver c(p);
        const size_t NN = static_cast<size_t>(N) * N;
        st = c.take<float2>(3 * NN);
        otf_rows = c.take<float2>(3 * static_cast<size_t>(N / 2 + 1) * N);   // row spectra of |U|^2, written by the inverse-row kernel
        I = c.take<float>(3 * NN);
        gtot = c.take<float>(3 * NN);
        part_rows = c.take<float>(3 * N);
        part_ew = c.take<float>(3 * 1024);          // element-wise partials: grid <= 1024 CTAs
        arrive = c.take<int>(1);
        bar = c.take<unsigned>(4);                   // grid-barrier words of the cooperative kernels: forward [0,1], backward [2,3]
        bytes = c.off;
    }
};

struct SensorWs {
    float2* stx; float2* stg; float2* partial; float2* stp; float* dot_lanes; float* coef;
    float4* pscratch; unsigned* pctr; float2* st2; int* arrive;
    size_t bytes;
    SensorWs(void* p, int N, int B, bool backward) {
        Carver c(p);
        // N = 256 plane kernels: crossing scratch of the resident clusters, [3 * G3][2][128 x 128] float4 (L2 resident)
        pscratch = (N == 256) ? c.take<float4>(static_cast<size_t>(3) * (B < PLANE_MAX_G3 ? B : PLANE_MAX_G3) * plane::NBUF * plane::PLANE_F4) : nullptr;
        pctr = (N == 256) ? c.take<unsigned>(static_cast<size_t>(3) * PLANE_MAX_G3 * 32) : nullptr;   // one arrival word per cluster, 128 B apart
        const size_t plane = static_cast<size_t>(N / 2 + 1) * N;
        stx = c.take<float2>(static_cast<size_t>(B) * 3 * plane);
        st2 = c.take<float2>(static_cast<size_t>(B) * 3 * plane);
        arrive = c.take<int>(static_cast<size_t>(B) * 64);     // one-pass normalise: a row of 64 key slots per image
        if (backward) {
            stg = c.take<float2>(static_cast<size_t>(B) * 3 * plane);
            const int max_chunks = (N == 256 && PLANE_MAX_G3 > MAX_CHUNKS) ? PLANE_MAX_G3 : MAX_CHUNKS;
            partial = c.take<float2>(static_cast<size_t>(B < max_chunks ? B : max_chunks) * 3 * plane);
            stp = c.take<float2>(3 * plane);
            dot_lanes = c.take<float>(static_cast<size_t>(B) * 3 * (N / 2 + 1) * 32);   // [B][3*NC][R1 <= 32]
            coef = c.take<float>(B);
        } else {
            stg = nullptr; partial = nullptr; stp = nullptr; dot_lanes = nullptr; coef = nullptr;
        }
        bytes = c.off;
    }
};

#define CK(expr)                                   \
    do {                                           \
        cudaError_t e_ = (expr);                   \
        if (e_ != cudaSuccess) return static_cast<int>(e_); \
    } while (0)
static std::atomic<unsigned long long> g_launches{0};
void note_launches(int n) { g_launches.fetch_add(static_cast<unsigned long long>(n), std::memory_order_relaxed); }   // other translation units (lens_psf.cu)
#define LAUNCH_CHECK()           \
    do {                         \
        CK(cudaGetLastError());  \
        g_launches.fetch_add(1, std::memory_order_relaxed); \
    } while (0)

// ------------------------------------------------------------------------------------------
// Every kernel of the library is launched through launch_k.  Programmatic dependent launch (VERDICT r1 item 2) is wired in
// - every kernel starts with pdl_gate(), the small kernels of the PSF chain / backward tail are launched with the
// attribute - but it is OFF by default (B200CAM_PDL=1 enables; B200CAM_PDL_TRIGGER=1 also signals dependents at kernel
// entry).  Measured, B = 64, graph replay (profiles/r02_pdl.md): 173 us per step without, 179 us with completion-time
// trigger, 183-197 us with entry-time trigger: the early-resident CTAs of the next kernels take registers / shared
// memory / issue slots from the kernel that is still running (the chain's head gets 6 us shorter, the image row pass
// beside it 9 us longer, tie_term and the last kernel 6-7 us longer each).
// ------------------------------------------------------------------------------------------
static bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("B200CAM_PDL"); return e && e[0] == '1'; }();
    return on;
}
// `Pdl`: the launch may overlap the tail of its predecessor.  Only the small kernels of the PSF chain and of the backward tail
// ask for it: a big batch kernel whose CTAs start early just sits on registers / shared memory that the concurrently
// running PSF chain (side stream) needs - measured 197 us per step with every launch programmatic, 174 us with none.
struct Pdl {};
template <class... KArgs, class... Args>
static void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args);
template <class... KArgs, class... Args>
static void launch_k(Pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    (void)cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);      // errors: cudaGetLastError in LAUNCH_CHECK
}
template <class... KArgs, class... Args>
static void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    (void)cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
}

// ------------------------------------------------------------------------------------------
// launch sequences
// ------------------------------------------------------------------------------------------
// first part of the PSF synthesis: pupil -> propagated field U, |U|^2 (workspace) and S = sum |U|^2 (stats[0])
// B200CAM_OTF_ROWS=0: the OTF's row transform as a kernel of its own (k_rows_r2c on the 3 planes) instead of inside k_crows_inv
static bool fuse_otf_rows() {
    static const bool on = [] { const char* e = getenv("B200CAM_OTF_ROWS"); return !(e && e[0] == '0'); }();
    return on;
}
template <int N>
static int psf_field_impl(const float* h, const float2* A, const float2* Ht, const float* kappa, float2* field,
                          void* ws_ptr, cudaStream_t s, cudaStream_t dependent = nullptr, bool has_dependent = false) {
    using T = Tile<N>;
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    PsfWs ws(ws_ptr, N);
    PupilLoad load{A, h, {kappa[0], kappa[1], kappa[2]}, N};
    const dim3 rgrid(N / T::CROWS, 3);
    launch_k(k_crows_fwd<N, PupilLoad>, rgrid, CRowsSmem<N>::THREADS, CRowsSmem<N>::BYTES, s, CRowsFwdParams{ws.st, tw}, load);
    LAUNCH_CHECK();
    if (has_dependent) {
        // The caller's big batch kernel (image row pass) is held back until this first small kernel is done: both it and
        // our next kernel then become ready together and the higher-priority one (ours) takes its SMs first.  Launched
        // earlier, the batch kernel fills every SM and each kernel of this chain waits a wave (~7 us) for room.
        cudaEvent_t ev = chain_event();
        if (ev == nullptr) return B200CAM_E_NOT_INIT;
        CK(cudaEventRecord(ev, s));
        CK(cudaStreamWaitEvent(dependent, ev, 0));
    }
    launch_k(Pdl{}, k_ccols_mix<N>, (N + CColsSmem<N>::CC - 1) / CColsSmem<N>::CC, CColsSmem<N>::THREADS, CColsSmem<N>::BYTES, s, 
        CColsMixParams{ws.st, Ht, tw, 0, 1.0f / (3.0f * N * N)});
    LAUNCH_CHECK();
    launch_k(Pdl{}, k_crows_inv<N, IntensityEpilogue>, rgrid, CRowsSmem<N>::THREADS, CRowsSmem<N>::BYTES, s, 
        CRowsInvParams{ws.st, tw}, IntensityEpilogue{field, ws.I, ws.part_rows, ws.arrive, N, fuse_otf_rows() ? ws.otf_rows : nullptr});
    LAUNCH_CHECK();
    return 0;
}

// second part: psf = |U|^2 / S and the two regularisers
template <int N>
static int psf_finish_impl(const float* rho, float* psf, float* stats, void* ws_ptr, cudaStream_t s) {
    PsfWs ws(ws_ptr, N);
    launch_k(Pdl{}, k_psf_finalise, ew_grid(N), EW_THREADS, 0, s, PsfFinaliseParams{ws.I, rho, stats, psf, ws.part_ew, ws.part_rows, ws.arrive, 3 * (N / Tile<N>::CROWS), N});
    LAUNCH_CHECK();
    return 0;
}

template <int N>
static int psf_fwd_impl(const float* h, const float2* A, const float2* Ht, const float* rho, const float* kappa,
                        float* psf, float2* field, float* stats, void* ws_ptr, cudaStream_t s) {
    using T = Tile<N>;
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    if (const int G = coop_grid(N, s)) {
        PsfWs ws(ws_ptr, N);
        PupilLoad load{A, h, {kappa[0], kappa[1], kappa[2]}, N};
        PsfFwdArgs args{CRowsFwdParams{ws.st, tw}, load, CColsMixParams{ws.st, Ht, tw, 0, 1.0f / (3.0f * N * N)},
                        CRowsInvParams{ws.st, tw}, IntensityEpilogue{field, ws.I, ws.part_rows, ws.arrive, N},
                        PsfFinaliseParams{ws.I, rho, stats, psf, ws.part_ew, ws.part_rows, ws.arrive, 3 * (N / Tile<N>::CROWS), N}, ws.bar, cur_state() != nullptr ? cur_state()->err_dev : nullptr};
        void* kargs[] = {&args};
        CK(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(k_psf_fwd_coop<N>), dim3(G), dim3(COOP_THREADS), kargs,
                                       coop_smem_bytes<N>(), s));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return 0;
    }
    int rc = psf_field_impl<N>(h, A, Ht, kappa, field, ws_ptr, s);
    if (rc) return rc;
    return psf_finish_impl<N>(rho, psf, stats, ws_ptr, s);
}

template <int N>
static int psf_bwd_impl(const float* gpsf, const float* g_rad, const float* g_cen, const float* h, const float2* A, const float2* Ht,
                        const float* rho, const float* kappa, const float* psf, const float2* field, float* stats,
                        float* grad_h, void* ws_ptr, cudaStream_t s, const CommDev* comm = nullptr) {
    using T = Tile<N>;
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    PsfWs ws(ws_ptr, N);
    PupilLoad pupil{A, h, {kappa[0], kappa[1], kappa[2]}, N};
    CRowsFwdParams rf{ws.st, tw};
    CColsMixParams mix{ws.st, Ht, tw, 1, 1.0f / (3.0f * N * N)};
    CRowsInvParams ri{ws.st, tw};
    if (const int G = (comm != nullptr ? 0 : coop_grid(N, s))) {
        PsfBwdArgs args{PsfGradPrepParams{gpsf, g_rad, g_cen, psf, rho, stats, ws.gtot, ws.part_ew, N}, rf,
                        GradFieldLoad{field, ws.gtot, stats, ws.part_ew, nullptr, G, N}, mix, ri, pupil, grad_h,
                        ws.bar + 2, cur_state() != nullptr ? cur_state()->err_dev : nullptr};
        void* kargs[] = {&args};
        CK(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(k_psf_bwd_coop<N>), dim3(G), dim3(COOP_THREADS), kargs,
                                       coop_smem_bytes<N>(), s));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return 0;
    }
    launch_k(Pdl{}, k_psf_grad_prepare, ew_grid(N), EW_THREADS, 0, s, PsfGradPrepParams{gpsf, g_rad, g_cen, psf, rho, stats, ws.gtot, ws.part_ew, N});
    LAUNCH_CHECK();
    launch_k(Pdl{}, k_crows_fwd<N, GradFieldLoad>, dim3(N / T::CROWS, 3), CRowsSmem<N>::THREADS, CRowsSmem<N>::BYTES, s, 
        rf, GradFieldLoad{field, ws.gtot, stats, ws.part_ew, nullptr, ew_grid(N), N});
    LAUNCH_CHECK();
    launch_k(Pdl{}, k_ccols_mix<N>, (N + CColsSmem<N>::CC - 1) / CColsSmem<N>::CC, CColsSmem<N>::THREADS, CColsSmem<N>::BYTES, s, mix);
    LAUNCH_CHECK();
    if (comm != nullptr)
        launch_k(Pdl{}, k_crows_inv_hgrad_allreduce<N>, N / T::CROWS, HGradSmem<N>::THREADS, HGradSmem<N>::BYTES, s, ri, pupil, grad_h, *comm,
                 cur_state() != nullptr ? cur_state()->err_dev : nullptr);
    else
        launch_k(Pdl{}, k_crows_inv_hgrad<N>, N / T::CROWS, HGradSmem<N>::THREADS, HGradSmem<N>::BYTES, s, ri, pupil, grad_h);
    LAUNCH_CHECK();
    return 0;
}

template <int N>
static int otf_impl(const float* src, float2* otf, const float2* tw, float scale, cudaStream_t s,
                    const float* sum_partials = nullptr, int npartials = 0) {
    using T = Tile<N>;
    launch_k(Pdl{}, k_rows_r2c<N>, dim3(N / T::ROWS, 3), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
        RowsR2CParams{src, otf, tw, nullptr, nullptr});
    LAUNCH_CHECK();
    const int total = 3 * T::NC;
    launch_k(Pdl{}, k_cols_fwd<N>, (total + T::COLS - 1) / T::COLS, ColsSmem<N>::THREADS, ColsSmem<N>::BYTES, s, 
        ColsFwdParams{otf, tw, total, 1, scale, sum_partials, npartials});
    LAUNCH_CHECK();
    return 0;
}

// column half of the OTF alone: the row spectra were written by k_crows_inv (IntensityEpilogue::otf_rows)
template <int N>
static int otf_cols_impl(const float2* rows, float2* otf, const float2* tw, float scale, cudaStream_t s, const float* sum_partials,
                         int npartials) {
    using T = Tile<N>;
    const int total = 3 * T::NC;
    launch_k(Pdl{}, k_cols_fwd<N>, (total + T::COLS - 1) / T::COLS, ColsSmem<N>::THREADS, ColsSmem<N>::BYTES, s,
        ColsFwdParams{otf, tw, total, 1, scale, sum_partials, npartials, rows});
    LAUNCH_CHECK();
    return 0;
}

// first half of the generic forward: row transforms of the images (independent of the PSF, so a caller may run it on a
// second stream while b200cam_psf_fwd is still busy); also resets the per-image max / tie counters
// allow_plane = false: always the standard spectrum layout (the bf16 sensor path runs the default two-pass pipeline only)
// Img = u8: uint8 images, converted in the row kernel; always the standard layout (the plane kernels read fp32 only)
template <int N, class Img = float>
static int sensor_rows_impl(const Img* img, float2* srow, float* img_max, int* tie_count, int B, cudaStream_t s,
                            bool allow_plane = true) {
    using T = Tile<N>;
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    // B200CAM_ROWS_PER_SM resident CTAs per SM (default 3 of the 4 that fit): see k_rows_r2c_persist
    static const int per_sm = [] { const char* e = getenv("B200CAM_ROWS_PER_SM"); const int v = e ? atoi(e) : 3; return v > 0 ? v : 3; }();
    if constexpr (N == 256 && std::is_same<Img, float>::value) {
        if (allow_plane && plane_selected()) {
            // plane layout "A"; the words behind it (the buffer is sized for 129 columns, A uses 128) hold the per-image
            // {max key, arrivals} pairs of k_pconv: reset here, early, beside the PSF chain
            const DeviceState* st = cur_state();
            if (st == nullptr) return B200CAM_E_NOT_INIT;
            const int planes = 3 * B;
            float4* A = reinterpret_cast<float4*>(srow);
            if (img_max != nullptr) CK(cudaMemsetAsync(A + static_cast<size_t>(planes) * plane::PLANE_F4, 0, sizeof(unsigned) * 2 * B, s));
            if (tie_count != nullptr) CK(cudaMemsetAsync(tie_count, 0, sizeof(int) * B, s));
            const int grid = persistent_grid(st->prow_fit, per_sm, planes * 8);
            launch_k(k_prow, grid, plane::THREADS, plane::SMEM_BYTES, s, plane::RowParams{img, A, tw, planes});
            LAUNCH_CHECK();
            return 0;
        }
    }
    const int total = (N / T::ROWS) * 3 * B;
    const int grid = persistent_grid(rows_fit(N, false, static_cast<int>(sizeof(Img))), per_sm, total);
    launch_k(k_rows_r2c_persist<N, Img>, grid, RowsStreamSmem<N, Img>::THREADS, RowsStreamSmem<N, Img>::BYTES, s,
        RowsR2CParamsT<Img>{img, srow, tw, img_max, tie_count}, total);
    LAUNCH_CHECK();
    return 0;
}

// second half: OTF of the PSF, column convolution, inverse rows + per-image max, normalise
// out16 != nullptr: bf16 sensor image.  `sensor` is then the fp32 conv scratch, and the default two-pass pipeline runs
// whatever B200CAM_PLANE / B200CAM_ONE_PASS say (those opt-in kernels write fp32 only).
// allow_plane = false: `srow` is in the standard layout whatever B200CAM_PLANE says (the uint8 row pass writes no other), so
// the plane kernels are not used for this call; the one-pass kernel still is (it reads the standard layout).
template <int N>
static int sensor_finish_impl(const float* psf, float* sensor, float* img_max, int* tie_count, int* tie_pos, float2* otf,
                              const float2* srow, const SensorWs& ws, int B, int otf_ready, cudaStream_t s,
                              SensorEpilogue epi = SensorEpilogue{nullptr, 0.f, 0.f}, bf16* out16 = nullptr,
                              bool allow_plane = true) {
    using T = Tile<N>;
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    if (!otf_ready) {
        int rc = otf_impl<N>(psf, otf, tw, 1.0f / (static_cast<float>(N) * N), s);
        if (rc) return rc;
    }
    const int planes = 3 * B;
    if constexpr (N == 256) {
        if (allow_plane && out16 == nullptr && plane_selected() && epi.noise == nullptr && epi.seed == nullptr &&
            epi.levels <= 0.f) {   // (the opt-in plane kernels have no read-out epilogue)
            const DeviceState* st = cur_state();
            if (st == nullptr || st->pconv_g3 < 1) return B200CAM_E_NOT_INIT;
            const int G3 = B < st->pconv_g3 ? B : st->pconv_g3;
            float4* A = reinterpret_cast<float4*>(const_cast<float2*>(srow));
            unsigned* sync = reinterpret_cast<unsigned*>(A + static_cast<size_t>(planes) * plane::PLANE_F4);
            k_pconv<<<3 * G3 * plane::C, plane::THREADS, plane::CONV_SMEM_BYTES, s>>>(
                plane::ConvParams{A, otf, ws.pscratch, sensor, tw, sync, img_max, tie_count, tie_pos, B, G3, 1, 1}, ws.pctr, st->err_dev);
            LAUNCH_CHECK();
            return 0;
        }
    }
    const dim3 rgrid(N / T::ROWS, planes);
    const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS;
    const int nchunks = conv_chunks(N, B);
    static const int per_sm = [] { const char* e = getenv("B200CAM_C2R_PER_SM"); const int v = e ? atoi(e) : 4; return v; }();
    // one-pass normalise (RowsC2RParams::arrive, B200CAM_ONE_PASS=1): the persistent inverse-row kernel writes conv / max
    // directly.  OFF by default: measured on one box against the two-pass path (B = 64, N = 256, graph replay) the kernel takes
    // 50-56 us against 21.6 + 16-19 us - and 52.9 us even with the maximum exchange skipped, i.e. it is the stash of the
    // previous tile's outputs (128 registers / thread at 4 CTAs per SM) that costs the time, not the waiting.
    static const int one_pass = [] { const char* e = getenv("B200CAM_ONE_PASS"); return e ? atoi(e) : 0; }();
    constexpr bool FUSABLE = (Plan<N>::R1 <= 16) && (Plan<N>::LANES == Plan<N>::R2);
    // (the one-pass kernel reads a noise tensor only: the Philox read-out runs in the normalise kernel)
    const bool fused = FUSABLE && one_pass && per_sm > 0 && out16 == nullptr && epi.seed == nullptr;
    launch_k(k_cols_conv<N>, dim3(colgroups, nchunks), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV, s, 
        ColsConvParams{srow, ws.st2, otf, tw, nullptr, B, nchunks, 0, 1.0f, fused ? ws.arrive : nullptr, fused ? 64 * B : 0});
    LAUNCH_CHECK();
    {
        if (per_sm > 0) {
            const int total = (N / T::ROWS) * planes;
            const int grid = persistent_grid(rows_fit(N, true), per_sm, total);
            static const int discard = [] { const char* e = getenv("B200CAM_DISCARD"); return e ? atoi(e) : 1; }();
            const DeviceState* st = cur_state();
            const RowsC2RParams cp{ws.st2, sensor, tw, img_max, 1.0f, tie_count, tie_pos, 0, discard, fused ? ws.arrive : nullptr,
                                   fused ? 3 * (N / T::ROWS) : 0, epi};
            if (fused) {
                launch_k(k_rows_c2r_persist<N, true>, grid, RowsC2RStreamSmem<N>::THREADS, RowsC2RStreamSmem<N>::BYTES, s, cp, total,
                         st != nullptr ? st->err_dev : nullptr);
                LAUNCH_CHECK();
                return 0;
            }
            launch_k(k_rows_c2r_persist<N, false>, grid, RowsC2RStreamSmem<N>::THREADS, RowsC2RStreamSmem<N>::BYTES, s, cp, total,
                     st != nullptr ? st->err_dev : nullptr);
        } else {
            launch_k(k_rows_c2r<N>, rgrid, RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
                RowsC2RParams{ws.st2, sensor, tw, img_max, 1.0f, nullptr, nullptr, 0});
        }
    }
    LAUNCH_CHECK();
    const long long n4 = static_cast<long long>(planes) * N * N / 4;
    const int grid = static_cast<int>(n4 / EW_THREADS < 148 * 8 ? (n4 + EW_THREADS - 1) / EW_THREADS : 148 * 8);
    const NormaliseParams np{sensor, img_max, tie_count, tie_pos, n4, 3 * N * N / 4, epi};
    if (out16 != nullptr)
        launch_k(epi.seed != nullptr ? k_normalise_bf16_philox : k_normalise_bf16, grid, EW_THREADS, 0, s, np, out16);
    else
        launch_k(epi.seed != nullptr ? k_normalise_philox : k_normalise, grid, EW_THREADS, 0, s, np);
    LAUNCH_CHECK();
    return 0;
}

// Plain circular convolution with a centred kernel (no per-image normalisation): the building block of the
// Image_Caption camera's padded linear convolution (img_psf_conv, Image_Caption/Camera/Utils.py:251-297).
//   out_b = irfft2( rfft2(img_b) * rfft2(roll(kernel, -N/2)) )
template <int N>
static int conv_fwd_impl(const float* img, const float* kern, float* out, float2* otf, float2* spectrum, void* ws_ptr,
                         int B, cudaStream_t s) {
    using T = Tile<N>;
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    SensorWs ws(ws_ptr, N, B, false);
    float2* srow = spectrum != nullptr ? spectrum : ws.stx;
    int rc = sensor_rows_impl<N>(img, srow, nullptr, nullptr, B, s);
    if (rc) return rc;
    rc = otf_impl<N>(kern, otf, tw, 1.0f / (static_cast<float>(N) * N), s);
    if (rc) return rc;
    const int planes = 3 * B;
    if constexpr (N == 256) {
        if (plane_selected()) {
            const DeviceState* st = cur_state();
            if (st == nullptr || st->pconv_g3 < 1) return B200CAM_E_NOT_INIT;
            const int G3 = B < st->pconv_g3 ? B : st->pconv_g3;
            k_pconv<<<3 * G3 * plane::C, plane::THREADS, plane::CONV_SMEM_BYTES, s>>>(
                plane::ConvParams{reinterpret_cast<float4*>(srow), otf, ws.pscratch, out, tw, nullptr, nullptr, nullptr, nullptr, B, G3,
                                  1, 0}, ws.pctr, st->err_dev);
            LAUNCH_CHECK();
            return 0;
        }
    }
    const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS;
    const int nchunks = conv_chunks(N, B);
    launch_k(k_cols_conv<N>, dim3(colgroups, nchunks), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV, s, 
        ColsConvParams{srow, ws.st2, otf, tw, nullptr, B, nchunks, 0, 1.0f});
    LAUNCH_CHECK();
    launch_k(k_rows_c2r<N>, dim3(N / T::ROWS, planes), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
        RowsC2RParams{ws.st2, out, tw, nullptr, 1.0f, nullptr, nullptr, 0});
    LAUNCH_CHECK();
    return 0;
}

// adjoints of conv_fwd: grad_kern = sum_b corr(img_b, g_b) (centred frame), grad_img_b = corr(g_b, kernel) (optional)
template <int N>
static int conv_bwd_impl(const float* g, const float* img, const float2* otf, const float2* spectrum, float* grad_kern,
                         float* grad_img, void* ws_ptr, int B, cudaStream_t s) {
    using T = Tile<N>;
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    SensorWs ws(ws_ptr, N, B, true);
    const int planes = 3 * B, tiles = N / T::ROWS;
    const dim3 rgrid(tiles, planes);
    if constexpr (N == 256) {
        if (plane_selected()) {
            const DeviceState* st = cur_state();
            if (st == nullptr || st->pacc_g3 < 1 || st->pconv_g3 < 1) return B200CAM_E_NOT_INIT;
            const float4* Xh = reinterpret_cast<const float4*>(spectrum);
            if (Xh == nullptr) {
                int rc = sensor_rows_impl<N>(img, ws.stx, nullptr, nullptr, B, s);
                if (rc) return rc;
                const int G3c = B < st->pconv_g3 ? B : st->pconv_g3;
                k_pconv<<<3 * G3c * plane::C, plane::THREADS, plane::CONV_SMEM_BYTES, s>>>(
                    plane::ConvParams{reinterpret_cast<float4*>(ws.stx), otf, ws.pscratch, nullptr, tw, nullptr, nullptr, nullptr,
                                      nullptr, B, G3c, 1, 0}, ws.pctr, st->err_dev);
                LAUNCH_CHECK();
                Xh = reinterpret_cast<const float4*>(ws.stx);
            }
            const int G3 = B < st->pacc_g3 ? B : st->pacc_g3;
            k_pacc<<<3 * G3 * plane::C, plane::THREADS, plane::ACC_SMEM_BYTES, s>>>(
                plane::AccParams{g, Xh, otf, ws.pscratch, tw, nullptr, ws.partial, ws.dot_lanes, B, G3}, ws.pctr, st->err_dev);
            LAUNCH_CHECK();
            launch_k(Pdl{}, k_cols_reduce_inv<N>, 3 * T::NC, ReduceInvSmem<N>::THREADS, ReduceInvSmem<N>::BYTES, s, 
                ColsReduceInvParams{ws.partial, ws.stp, tw, G3, 0.25f / (static_cast<float>(N) * N), nullptr, nullptr, nullptr, nullptr, 0});
            LAUNCH_CHECK();
            launch_k(Pdl{}, k_rows_c2r<N>, dim3(tiles, 3), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
                RowsC2RParams{ws.stp, grad_kern, tw, nullptr, 1.0f, nullptr, nullptr, 0});
            LAUNCH_CHECK();
            if (grad_img != nullptr) {
                launch_k(k_rows_r2c<N>, rgrid, RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, RowsR2CParams{g, ws.stg, tw, nullptr, nullptr});
                LAUNCH_CHECK();
                const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS;
                const int cchunks = conv_chunks(N, B);
                launch_k(k_cols_conv<N>, dim3(colgroups, cchunks), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV, s, 
                    ColsConvParams{ws.stg, ws.stg, otf, tw, nullptr, B, cchunks, 1, 1.0f});
                LAUNCH_CHECK();
                launch_k(k_rows_c2r<N>, rgrid, RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
                    RowsC2RParams{ws.stg, grad_img, tw, nullptr, 1.0f, nullptr, nullptr, 0});
                LAUNCH_CHECK();
            }
            return 0;
        }
    }
    const float2* srow = spectrum;
    if (srow == nullptr) {
        int rc = sensor_rows_impl<N>(img, ws.stx, nullptr, nullptr, B, s);
        if (rc) return rc;
        srow = ws.stx;
    }
    int rc = sensor_rows_impl<N>(g, ws.stg, nullptr, nullptr, B, s);
    if (rc) return rc;
    const int nchunks = accum_chunks(N, B);
    const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS;
    launch_k(k_cols_accum<N>, dim3(colgroups, nchunks), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES, s, 
        ColsAccumParams{srow, ws.stg, ws.partial, tw, nullptr, nullptr, nullptr, B, nchunks});
    LAUNCH_CHECK();
    launch_k(Pdl{}, k_cols_reduce_inv<N>, 3 * T::NC, ReduceInvSmem<N>::THREADS, ReduceInvSmem<N>::BYTES, s, 
        ColsReduceInvParams{ws.partial, ws.stp, tw, nchunks, 1.0f / (static_cast<float>(N) * N),
                            nullptr, nullptr, nullptr, nullptr, 0});
    LAUNCH_CHECK();
    launch_k(Pdl{}, k_rows_c2r<N>, dim3(tiles, 3), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
        RowsC2RParams{ws.stp, grad_kern, tw, nullptr, 1.0f, nullptr, nullptr, 0});
    LAUNCH_CHECK();
    if (grad_img != nullptr) {
        const int cchunks = conv_chunks(N, B);
        launch_k(k_cols_conv<N>, dim3(colgroups, cchunks), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV, s, 
            ColsConvParams{ws.stg, ws.stg, otf, tw, nullptr, B, cchunks, 1, 1.0f});
        LAUNCH_CHECK();
        launch_k(k_rows_c2r<N>, rgrid, RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
            RowsC2RParams{ws.stg, grad_img, tw, nullptr, 1.0f, nullptr, nullptr, 0});
        LAUNCH_CHECK();
    }
    return 0;
}

template <int N, class Img = float>
static int sensor_fwd_impl(const Img* img, const float* psf, float* sensor, float* img_max, int* tie_count,
                           int* tie_pos, float2* otf, float2* spectrum, void* ws_ptr, int B, cudaStream_t s,
                           SensorEpilogue epi = SensorEpilogue{nullptr, 0.f, 0.f}, bf16* out16 = nullptr) {
    SensorWs ws(ws_ptr, N, B, false);
    float2* srow = spectrum != nullptr ? spectrum : ws.stx;      // row spectra: kept for the backward when asked
    constexpr bool FP32_IMG = std::is_same<Img, float>::value;  // (uint8 images: standard layout, no plane kernels)
    // (bf16 and the Philox read-out run the default pipeline: the rows in the standard layout)
    int rc = sensor_rows_impl<N, Img>(img, srow, img_max, tie_count, B, s, out16 == nullptr && epi.seed == nullptr);
    if (rc) return rc;
    return sensor_finish_impl<N>(psf, sensor, img_max, tie_count, tie_pos, otf, srow, ws, B, 0, s, epi, out16, FP32_IMG);
}

// In = bf16: the upstream gradient arrives in bf16 and is widened in the row kernels; everything after them is the fp32
// pipeline (the plane kernels are fp32 only: the bf16 path always runs the generic one)
// Img = u8: the images are uint8 (converted in registers wherever they are read: the row pass that rebuilds the spectra when
// the forward kept none, and the arg-max gather); likewise the generic pipeline only
template <int N, class In = float, class Img = float>
static int sensor_bwd_impl(const In* g, const Img* img, const float* sensor, const float* img_max,
                           const int* tie_count, const int* tie_pos, const float* psf, const float2* otf,
                           const float2* spectrum, float* grad_psf, float* grad_img, void* ws_ptr, int B,
                           cudaStream_t s) {
    using T = Tile<N>;
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    SensorWs ws(ws_ptr, N, B, true);
    const int planes = 3 * B, tiles = N / T::ROWS;
    const dim3 rgrid(tiles, planes);
    if constexpr (N == 256 && std::is_same<In, float>::value && std::is_same<Img, float>::value) {
        if (plane_selected()) {
            const DeviceState* st = cur_state();
            if (st == nullptr || st->pacc_g3 < 1 || st->pconv_g3 < 1) return B200CAM_E_NOT_INIT;
            const float4* Xh = reinterpret_cast<const float4*>(spectrum);
            if (Xh == nullptr) {                 // the forward did not keep X^: rebuild it (rows, then the column half of k_pconv)
                int rc = sensor_rows_impl<N>(img, ws.stx, nullptr, nullptr, B, s);
                if (rc) return rc;
                const int G3c = B < st->pconv_g3 ? B : st->pconv_g3;
                k_pconv<<<3 * G3c * plane::C, plane::THREADS, plane::CONV_SMEM_BYTES, s>>>(
                    plane::ConvParams{reinterpret_cast<float4*>(ws.stx), otf, ws.pscratch, nullptr, tw, nullptr, nullptr, nullptr,
                                      nullptr, B, G3c, 1, 0}, ws.pctr, st->err_dev);
                LAUNCH_CHECK();
                Xh = reinterpret_cast<const float4*>(ws.stx);
            }
            const int G3 = B < st->pacc_g3 ? B : st->pacc_g3;
            k_pacc<<<3 * G3 * plane::C, plane::THREADS, plane::ACC_SMEM_BYTES, s>>>(
                plane::AccParams{g, Xh, otf, ws.pscratch, tw, img_max, ws.partial, ws.dot_lanes, B, G3}, ws.pctr, st->err_dev);
            LAUNCH_CHECK();
            launch_k(Pdl{}, k_pcoef, (B + 63) / 64, 64, 0, s, ws.dot_lanes, img_max, tie_count, ws.coef, B);
            LAUNCH_CHECK();
            launch_k(Pdl{}, k_cols_reduce_inv<N>, 3 * T::NC, ReduceInvSmem<N>::THREADS, ReduceInvSmem<N>::BYTES, s, 
                ColsReduceInvParams{ws.partial, ws.stp, tw, G3, 0.25f / (static_cast<float>(N) * N), nullptr, nullptr, nullptr, nullptr, 0});
            LAUNCH_CHECK();
            launch_k(Pdl{}, k_rows_c2r<N>, dim3(tiles, 3), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
                RowsC2RParams{ws.stp, grad_psf, tw, nullptr, 1.0f});
            LAUNCH_CHECK();
            const int per_ch = N * N / 2 / EW_THREADS < 592 ? N * N / 2 / EW_THREADS : 592;
            launch_k(Pdl{}, k_tie_term<>, dim3(per_ch, 3), EW_THREADS, 0, s, TieTermParams{grad_psf, img, tie_count, tie_pos, ws.coef, B, N});
            LAUNCH_CHECK();
            if (grad_img != nullptr) {           // optional output (no reference caller asks for it): generic kernels on g
                launch_k(k_rows_r2c<N>, rgrid, RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, RowsR2CParams{g, ws.stg, tw, nullptr, nullptr});
                LAUNCH_CHECK();
                const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS;
                const int cchunks = conv_chunks(N, B);
                launch_k(k_cols_conv<N>, dim3(colgroups, cchunks), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV, s, 
                    ColsConvParams{ws.stg, ws.stg, otf, tw, img_max, B, cchunks, 1, 1.0f});
                LAUNCH_CHECK();
                launch_k(k_rows_c2r<N>, rgrid, RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
                    RowsC2RParams{ws.stg, grad_img, tw, nullptr, 1.0f});
                LAUNCH_CHECK();
                const long long tot = static_cast<long long>(planes) * N * N;
                const int grid = static_cast<int>(tot / EW_THREADS < 148 * 8 ? (tot + EW_THREADS - 1) / EW_THREADS : 148 * 8);
                launch_k(k_tie_term_img, grid, EW_THREADS, 0, s, TieTermImgParams{grad_img, psf, tie_count, tie_pos, ws.coef, B, N});
                LAUNCH_CHECK();
            }
            return 0;
        }
    }
    const float2* srow = spectrum;
    if (srow == nullptr) {                       // forward did not keep the row spectra: recompute them
        launch_k(k_rows_r2c<N, Img>, rgrid, RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s,
            RowsR2CParamsT<Img>{img, ws.stx, tw, nullptr, nullptr});
        LAUNCH_CHECK();
        srow = ws.stx;
    }
    // upstream gradient rows; sum(g*conv) of the amax term comes out of the accumulate kernel (Parseval), so the
    // sensor image is not read again
    (void)sensor;
    {
        static const int per_sm = [] { const char* e = getenv("B200CAM_GROWS_PER_SM"); return e ? atoi(e) : 3; }();
        if (per_sm > 0) {
            const int total = tiles * planes;
            const int grid = persistent_grid(rows_fit(N, false, static_cast<int>(sizeof(In))), per_sm, total);
            launch_k(k_rows_r2c_persist<N, In>, grid, RowsStreamSmem<N, In>::THREADS, RowsStreamSmem<N, In>::BYTES, s,
                RowsR2CParamsT<In>{g, ws.stg, tw, nullptr, nullptr}, total);
        } else {
            launch_k(k_rows_r2c<N, In>, rgrid, RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, RowsR2CParamsT<In>{g, ws.stg, tw, nullptr, nullptr});
        }
    }
    LAUNCH_CHECK();
    const int nchunks = accum_chunks(N, B);
    const int colgroups = (3 * T::NC + T::COLS - 1) / T::COLS;
    // arg-max term of the amax backward: the spatial gather kernel k_tie_term after the inverse rows (default), or folded into
    // k_cols_reduce_inv in the (u, y) domain (B200CAM_TIE_SPECTRAL=1: one launch less, no 17 MB gather - but the staging of the
    // tie list inside that kernel is a chain of dependent loads: measured 17.7 us against 5.7 + 10.6 us, step 168.6-174 us
    // against 165.8-171.5 us, so it stays opt-in; the CPU emulator runs this form)
    static const int tie_spectral = [] { const char* e = getenv("B200CAM_TIE_SPECTRAL"); return e ? atoi(e) : 0; }();
    const int dot_count = colgroups * ColsSmem<N>::WARPS;
    const bool spectral = tie_spectral != 0 && static_cast<size_t>(dot_count) <= static_cast<size_t>(3) * T::NC * 32;
    float* dot_warps = spectral ? ws.dot_lanes : nullptr;          // the same workspace slice, [B][colgroups][WARPS]
    launch_k(k_cols_accum<N>, dim3(colgroups, nchunks), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES, s, 
        ColsAccumParams{srow, ws.stg, ws.partial, tw, img_max, otf, ws.dot_lanes, B, nchunks,
                        grad_img == nullptr ? [] { const char* e = getenv("B200CAM_DISCARD"); return e ? atoi(e) : 1; }() : 0, dot_warps});
    LAUNCH_CHECK();
    // the side-job CTAs (coef[b]) are only needed by the spatial kernels: k_tie_term, and k_tie_term_img of the optional dL/dimg
    const bool side_job = !spectral || grad_img != nullptr;
    launch_k(Pdl{}, k_cols_reduce_inv<N>, 3 * T::NC + (side_job ? B : 0), ReduceInvSmem<N>::THREADS, ReduceInvSmem<N>::BYTES, s, 
        ColsReduceInvParams{ws.partial, ws.stp, tw, nchunks, 1.0f / (static_cast<float>(N) * N),
                            side_job ? ws.dot_lanes : nullptr, img_max, tie_count, ws.coef, B, spectral ? nullptr : img, tie_pos,
                            spectral ? srow : nullptr, dot_warps, dot_count, static_cast<int>(sizeof(Img))});
    LAUNCH_CHECK();
    launch_k(Pdl{}, k_rows_c2r<N>, dim3(tiles, 3), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s,
        RowsC2RParams{ws.stp, grad_psf, tw, nullptr, 1.0f});
    LAUNCH_CHECK();
    if (!spectral) {   // arg-max term of the amax backward (spatial form), ties of channel c handled by the CTAs of row c
        const int per_ch = N * N / 2 / EW_THREADS < 592 ? N * N / 2 / EW_THREADS : 592;   // two adjacent pixels per thread
        launch_k(Pdl{}, k_tie_term<Img>, dim3(per_ch, 3), EW_THREADS, 0, s, TieTermParamsT<Img>{grad_psf, img, tie_count, tie_pos, ws.coef, B, N});
        LAUNCH_CHECK();
    }
    if (grad_img != nullptr) {
        const int cchunks = conv_chunks(N, B);
        launch_k(k_cols_conv<N>, dim3(colgroups, cchunks), ColsSmem<N>::THREADS, ColsSmem<N>::BYTES_CONV, s, 
            ColsConvParams{ws.stg, ws.stg, otf, tw, img_max, B, cchunks, 1, 1.0f});
        LAUNCH_CHECK();
        launch_k(k_rows_c2r<N>, rgrid, RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s, 
            RowsC2RParams{ws.stg, grad_img, tw, nullptr, 1.0f});
        LAUNCH_CHECK();
        const long long tot = static_cast<long long>(planes) * N * N;
        const int grid = static_cast<int>(tot / EW_THREADS < 148 * 8 ? (tot + EW_THREADS - 1) / EW_THREADS : 148 * 8);
        launch_k(k_tie_term_img, grid, EW_THREADS, 0, s, TieTermImgParams{grad_img, psf, tie_count, tie_pos, ws.coef, B, N});
        LAUNCH_CHECK();
    }
    return 0;
}

}  // namespace b200cam

// ==========================================================================================
//                                       C ABI
// ==========================================================================================
using namespace b200cam;

#define DISPATCH_N(N_, CALL)                      \
    switch (N_) {                                 \
        case 64: { constexpr int NN_ = 64; return CALL; }     \
        case 128: { constexpr int NN_ = 128; return CALL; }   \
        case 256: { constexpr int NN_ = 256; return CALL; }   \
        case 512: { constexpr int NN_ = 512; return CALL; }   \
        case 1024: { constexpr int NN_ = 1024; return CALL; } \
        default: return B200CAM_E_BAD_SIZE;       \
    }

namespace b200cam {
// ---- entry points for the other translation units of the library (lens_conv.cu) --------------------------------------
const float2* lens_twiddle(int N) { return b200cam_supported(N) ? twiddle(N) : nullptr; }
// OTF of a centred n x n kernel in the library's layout (rows + columns, sign twist, 1/N^2): psf2otf, Image_Caption/Camera/Utils.py:127-158
int lens_otf(int N, const float* kern, float2* otf, cudaStream_t s) {
    const float2* tw = lens_twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    switch (N) {
        case 128: return otf_impl<128>(kern, otf, tw, 1.0f / (128.f * 128.f), s);
        case 256: return otf_impl<256>(kern, otf, tw, 1.0f / (256.f * 256.f), s);
        case 512: return otf_impl<512>(kern, otf, tw, 1.0f / (512.f * 512.f), s);
        case 1024: return otf_impl<1024>(kern, otf, tw, 1.0f / (1024.f * 1024.f), s);
        default: return B200CAM_E_BAD_SIZE;
    }
}
template <int N>
static int grad_kernel_tail_impl(const float2* partial, float2* stp, float* grad_kern, int nchunks, const float2* tw, cudaStream_t s) {
    using T = Tile<N>;
    launch_k(Pdl{}, k_cols_reduce_inv<N>, 3 * T::NC, ReduceInvSmem<N>::THREADS, ReduceInvSmem<N>::BYTES, s,
        ColsReduceInvParams{partial, stp, tw, nchunks, 1.0f / (static_cast<float>(N) * N), nullptr, nullptr, nullptr, nullptr, 0});
    LAUNCH_CHECK();
    launch_k(Pdl{}, k_rows_c2r<N>, dim3(N / T::ROWS, 3), RowsR2CSmem<N>::THREADS, RowsR2CSmem<N>::BYTES, s,
        RowsC2RParams{stp, grad_kern, tw, nullptr, 1.0f, nullptr, nullptr, 0});
    LAUNCH_CHECK();
    return 0;
}
// chunk partials of sum_b G conj(X) -> dL/dkernel in the centred frame (the tail of conv_bwd_impl)
int lens_grad_kernel_tail(int N, const float2* partial, float2* stp, float* grad_kern, int nchunks, cudaStream_t s) {
    const float2* tw = lens_twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    switch (N) {
        case 128: return grad_kernel_tail_impl<128>(partial, stp, grad_kern, nchunks, tw, s);
        case 256: return grad_kernel_tail_impl<256>(partial, stp, grad_kern, nchunks, tw, s);
        case 512: return grad_kernel_tail_impl<512>(partial, stp, grad_kern, nchunks, tw, s);
        case 1024: return grad_kernel_tail_impl<1024>(partial, stp, grad_kern, nchunks, tw, s);
        default: return B200CAM_E_BAD_SIZE;
    }
}
}  // namespace b200cam

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

extern "C" {

int b200cam_version(void) { return B200CAM_VERSION; }

const char* b200cam_error_string(int code) {
    switch (code) {
        case 0: return "success";
        case B200CAM_E_BAD_SIZE: return "b200cam: unsupported size (N must be 64,128,256,512,1024; B >= 1)";
        case B200CAM_E_NULL: return "b200cam: required pointer is NULL";
        case B200CAM_E_WORKSPACE: return "b200cam: workspace too small";
        case B200CAM_E_NOT_INIT: return "b200cam: b200cam_init(N) was not called on this device";
        case B200CAM_E_ALIGN: return "b200cam: pointer not 16-byte aligned";
        case B200CAM_E_DEVICE: return "b200cam: a kernel gave up waiting (image-max exchange, grid barrier or peer all-reduce); results of that call are invalid";
        default: return code > 0 ? cudaGetErrorString(static_cast<cudaError_t>(code)) : "b200cam: unknown error";
    }
}

unsigned long long b200cam_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
int b200cam_col_chunks(int N, int B, int slots) {
    if (!b200cam_supported(N) || B < 1 || slots < 1) return 0;
    return col_chunks(N, B, slots);
}

int b200cam_device_error(int clear) {
    const DeviceState* st = cur_state();
    if (st == nullptr || st->err_host == nullptr) return 0;
    volatile unsigned* p = st->err_host;
    const int v = static_cast<int>(*p);
    if (clear && v != 0) *p = 0u;
    return v;
}

int b200cam_supported(int N) { return N == 64 || N == 128 || N == 256 || N == 512 || N == 1024; }

int b200cam_init(int N) {
    if (!b200cam_supported(N)) return B200CAM_E_BAD_SIZE;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= MAX_DEV) return B200CAM_E_BAD_SIZE;
    std::lock_guard<std::mutex> lock(g_mutex);
    const int l = log2i(N);
    if (g_state[dev].tw[l] != nullptr) return 0;
    if (g_state[dev].chain_ev == nullptr) CK(cudaEventCreateWithFlags(&g_state[dev].chain_ev, cudaEventDisableTiming));
    {
        const char* e = getenv("B200CAM_PDL_TRIGGER");
        const int trig = e ? atoi(e) : 0;
        CK(cudaMemcpyToSymbol(c_pdl_trigger, &trig, sizeof(int)));
    }
    if (g_state[dev].err_host == nullptr) {
        unsigned* h = nullptr;
        unsigned* d = nullptr;
        CK(cudaHostAlloc(&h, 64, cudaHostAllocMapped));
        *h = 0u;
        CK(cudaHostGetDevicePointer(&d, h, 0));
        g_state[dev].err_host = h;
        g_state[dev].err_dev = d;
    }
    if (g_state[dev].scratch == nullptr) CK(cudaMalloc(&g_state[dev].scratch, sizeof(float) * SCRATCH_FLOATS));
    if (g_state[dev].bar == nullptr) {
        unsigned* bar = nullptr;
        CK(cudaMalloc(&bar, 4 * sizeof(unsigned)));
        CK(cudaMemset(bar, 0, 4 * sizeof(unsigned)));
        g_state[dev].bar = bar;
    }
    float2* tw = nullptr;
    CK(cudaMalloc(&tw, sizeof(float2) * N));
    k_fill_twiddle<<<(N + 255) / 256, 256>>>(tw, N);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    cudaError_t e = cudaSuccess;
    switch (N) {
        case 64: e = init_kernels<64>(); break;
        case 128: e = init_kernels<128>(); break;
        case 256: e = init_kernels<256>(); break;
        case 512: e = init_kernels<512>(); break;
        case 1024: e = init_kernels<1024>(); break;
    }
    if (e == cudaSuccess && N == 256) e = plane_init(dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&g_state[dev].sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) {
        const int sms = g_state[dev].sms;
        switch (N) {
            case 64: e = coop_grid_size<64>(dev, sms, &g_state[dev].coop_grid[l]); break;
            case 128: e = coop_grid_size<128>(dev, sms, &g_state[dev].coop_grid[l]); break;
            case 256: e = coop_grid_size<256>(dev, sms, &g_state[dev].coop_grid[l]); break;
            case 512: e = coop_grid_size<512>(dev, sms, &g_state[dev].coop_grid[l]); break;
            case 1024: e = coop_grid_size<1024>(dev, sms, &g_state[dev].coop_grid[l]); break;
        }
    }
    if (e == cudaSuccess) {
        const int sms = g_state[dev].sms;
        int* cs = &g_state[dev].conv_slots[l];
        int* as = &g_state[dev].accum_slots[l];
        switch (N) {
            case 64: e = column_slots<64>(sms, cs, as); break;
            case 128: e = column_slots<128>(sms, cs, as); break;
            case 256: e = column_slots<256>(sms, cs, as); break;
            case 512: e = column_slots<512>(sms, cs, as); break;
            case 1024: e = column_slots<1024>(sms, cs, as); break;
        }
    }
    if (e == cudaSuccess) {
        int* rf = &g_state[dev].r2c_fit[l];
        int* rf16 = &g_state[dev].r2c16_fit[l];
        int* rf8 = &g_state[dev].r2c8_fit[l];
        int* cf = &g_state[dev].c2r_fit[l];
        switch (N) {
            case 64: e = row_fits<64>(rf, rf16, rf8, cf); break;
            case 128: e = row_fits<128>(rf, rf16, rf8, cf); break;
            case 256: e = row_fits<256>(rf, rf16, rf8, cf); break;
            case 512: e = row_fits<512>(rf, rf16, rf8, cf); break;
            case 1024: e = row_fits<1024>(rf, rf16, rf8, cf); break;
        }
    }
    if (e != cudaSuccess) {
        cudaFree(tw);
        (void)cudaGetLastError();          // do not leave a sticky error behind for later launches
        return static_cast<int>(e);
    }
    g_state[dev].tw[l] = tw;
    return 0;
}

size_t b200cam_otf_bytes(int N) {
    return b200cam_supported(N) ? static_cast<size_t>(3) * (N / 2 + 1) * N * sizeof(float2) : 0;
}

size_t b200cam_psf_workspace_bytes(int N) {
    if (!b200cam_supported(N)) return 0;
    return PsfWs(nullptr, N).bytes;
}

size_t b200cam_sensor_workspace_bytes(int N, int B, int want_img_grad) {
    (void)want_img_grad;
    if (!b200cam_supported(N) || B < 1) return 0;
    return SensorWs(nullptr, N, B, true).bytes;
}

int b200cam_psf_fwd(const float* h, const float* A, const float* Ht, const float* rho, const float* kappa,
                    float* psf, float* field, float* stats, void* workspace, size_t workspace_bytes, int N,
                    void* stream) {
    if (!b200cam_supported(N)) return B200CAM_E_BAD_SIZE;
    if (!h || !A || !Ht || !rho || !kappa || !psf || !field || !stats || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_psf_workspace_bytes(N)) return B200CAM_E_WORKSPACE;
    if (!aligned16(A) || !aligned16(Ht) || !aligned16(field) || !aligned16(workspace)) return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH_N(N, (psf_fwd_impl<NN_>(h, reinterpret_cast<const float2*>(A), reinterpret_cast<const float2*>(Ht), rho,
                                     kappa, psf, reinterpret_cast<float2*>(field), stats, workspace, s)));
}

// ---- Image_Caption sensor epilogue -------------------------------------------------------------------------
static int ew_blocks(long long elems) {
    const long long want = (elems + EW_THREADS - 1) / EW_THREADS;
    return static_cast<int>(want < 148 * 16 ? (want > 0 ? want : 1) : 148 * 16);
}

int b200cam_crop_abs_resize_fwd(const float* conv, float* out, int planes, int n, int P, int off, void* stream) {
    if (planes < 1 || n < 2 || P < 2 || off < 0 || off + P - 1 > n) return B200CAM_E_BAD_SIZE;
    if (!conv || !out) return B200CAM_E_NULL;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    launch_k(k_crop_abs_resize_fwd, ew_blocks(static_cast<long long>(planes) * P * P), EW_THREADS, 0, s, 
        CropAbsResizeParams{conv, out, planes, n, P, off});
    LAUNCH_CHECK();
    return 0;
}

int b200cam_crop_abs_resize_bwd(const float* grad_out, const float* conv, float* grad_conv, int planes, int n, int P, int off,
                                void* stream) {
    if (planes < 1 || n < 2 || P < 2 || off < 0 || off + P - 1 > n) return B200CAM_E_BAD_SIZE;
    if (!grad_out || !conv || !grad_conv) return B200CAM_E_NULL;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    launch_k(k_crop_abs_resize_bwd, ew_blocks(static_cast<long long>(planes) * n * n), EW_THREADS, 0, s, 
        CropAbsResizeBwdParams{grad_out, conv, grad_conv, planes, n, P, off});
    LAUNCH_CHECK();
    return 0;
}

// ---- Zernike projection (SURVEY 8 f1) ----------------------------------------------------------------------
static int zernike_ks(int T, long long NN4) {
    const long long xblocks = (NN4 + EW_THREADS - 1) / EW_THREADS;
    long long ks = (148 * 4 + xblocks - 1) / xblocks;        // about four CTAs per SM in total (twelve: 47 -> 51 us at 300 x 256^2)
    if (ks > T) ks = T;
    if (ks > 32) ks = 32;
    if (ks < 1) ks = 1;
    return static_cast<int>(ks);
}

size_t b200cam_zernike_workspace_bytes(int T, long long NN) {
    if (T < 1 || NN < 4 || NN % 4 != 0) return 0;
    const long long NN4 = NN / 4;
    const long long xblocks = (NN4 + EW_THREADS - 1) / EW_THREADS;
    return static_cast<size_t>(zernike_ks(T, NN4)) * NN4 * sizeof(float4) + static_cast<size_t>(xblocks) * sizeof(int) + 256;
}

int b200cam_zernike_fwd_ex(const float* coef, const float* Z, float* h, void* workspace, size_t workspace_bytes, int T,
                           long long NN, void* stream, const int* active, int nactive) {
    if (T < 1 || NN < 4 || NN % 4 != 0 || NN / 4 > 0x7fffffffLL) return B200CAM_E_BAD_SIZE;
    if (!coef || !Z || !h || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_zernike_workspace_bytes(T, NN)) return B200CAM_E_WORKSPACE;
    if (!aligned16(Z) || !aligned16(h) || !aligned16(workspace)) return B200CAM_E_ALIGN;
    if (active != nullptr && (nactive < 1 || nactive > NN / 4)) return B200CAM_E_BAD_SIZE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int NN4 = static_cast<int>(NN / 4);
    const int nq = active != nullptr ? nactive : NN4;
    const int xblocks = (nq + EW_THREADS - 1) / EW_THREADS, ks = zernike_ks(T, NN4);
    Carver c(workspace);
    int* arrive = c.take<int>((NN4 + EW_THREADS - 1) / EW_THREADS);   // zero on entry (caller zero-fills the workspace once), left zero
    float4* partial = c.take<float4>(static_cast<size_t>(ks) * NN4);
    if (active != nullptr) CK(cudaMemsetAsync(h, 0, sizeof(float) * static_cast<size_t>(NN), s));   // outside the support h = 0
    launch_k(k_zernike_fwd, dim3(xblocks, ks), EW_THREADS, 0, s, 
        ZernikeFwdParams{coef, reinterpret_cast<const float4*>(Z), partial, reinterpret_cast<float4*>(h), arrive, T, NN4, ks, active, nactive});
    LAUNCH_CHECK();
    return 0;
}

int b200cam_zernike_fwd(const float* coef, const float* Z, float* h, void* workspace, size_t workspace_bytes, int T,
                        long long NN, void* stream) {
    return b200cam_zernike_fwd_ex(coef, Z, h, workspace, workspace_bytes, T, NN, stream, nullptr, 0);
}

int b200cam_zernike_bwd_ex(const float* grad_h, const float* Z, float* grad_coef, int T, long long NN, void* stream, const int* active,
                           int nactive) {
    if (T < 1 || NN < 4 || NN % 4 != 0 || NN / 4 > 0x7fffffffLL) return B200CAM_E_BAD_SIZE;
    if (!grad_h || !Z || !grad_coef) return B200CAM_E_NULL;
    if (!aligned16(Z) || !aligned16(grad_h)) return B200CAM_E_ALIGN;
    if (active != nullptr && (nactive < 1 || nactive > NN / 4)) return B200CAM_E_BAD_SIZE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const long long nq = active != nullptr ? nactive : NN / 4;
    // few terms: slice every plane over enough CTAs to fill the device (partials in the per-device scratch, b200cam_init)
    const DeviceState* st = cur_state();
    // A CTA that walks a whole plane alone is a chain of dependent load batches (measured 42 us for 300 x 256^2: 1.6 TB/s):
    // slice every plane so that about eight CTAs per SM are in flight, whatever T is
    int splits = 1;
    if (st != nullptr && st->scratch != nullptr) {
        splits = (8 * 148 + T - 1) / T;
        const int most = static_cast<int>(nq / (8 * EW_THREADS));
        if (splits > most) splits = most;
        if (splits > 64) splits = 64;
        if (splits < 1 || static_cast<long long>(T) * splits > SCRATCH_FLOATS) splits = 1;
    }
    launch_k(k_zernike_bwd, dim3(T, splits), EW_THREADS, 0, s, ZernikeBwdParams{reinterpret_cast<const float4*>(grad_h),
                                                            reinterpret_cast<const float4*>(Z), splits > 1 ? st->scratch : grad_coef,
                                                            static_cast<int>(NN / 4), splits, active, nactive});
    LAUNCH_CHECK();
    if (splits > 1) {
        launch_k(k_zernike_bwd_fin, (T + EW_THREADS - 1) / EW_THREADS, EW_THREADS, 0, s, st->scratch, grad_coef, T, splits);
        LAUNCH_CHECK();
    }
    return 0;
}

int b200cam_zernike_bwd(const float* grad_h, const float* Z, float* grad_coef, int T, long long NN, void* stream) {
    return b200cam_zernike_bwd_ex(grad_h, Z, grad_coef, T, NN, stream, nullptr, 0);
}

int b200cam_psf_field(const float* h, const float* A, const float* Ht, const float* kappa, float* field,
                      void* workspace, size_t workspace_bytes, int N, void* stream, void* dependent_stream,
                      int has_dependent) {
    if (!b200cam_supported(N)) return B200CAM_E_BAD_SIZE;
    if (!h || !A || !Ht || !kappa || !field || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_psf_workspace_bytes(N)) return B200CAM_E_WORKSPACE;
    if (!aligned16(A) || !aligned16(Ht) || !aligned16(field) || !aligned16(workspace)) return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH_N(N, (psf_field_impl<NN_>(h, reinterpret_cast<const float2*>(A), reinterpret_cast<const float2*>(Ht), kappa,
                                       reinterpret_cast<float2*>(field), workspace, s,
                                       static_cast<cudaStream_t>(dependent_stream), has_dependent != 0)));
}

int b200cam_psf_otf_early(float* otf, void* workspace, size_t workspace_bytes, int N, void* stream) {
    if (!b200cam_supported(N)) return B200CAM_E_BAD_SIZE;
    if (!otf || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_psf_workspace_bytes(N)) return B200CAM_E_WORKSPACE;
    if (!aligned16(otf) || !aligned16(workspace)) return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    // |U|^2 / S is the PSF: the OTF does not have to wait for psf_finish to write it out
    if (fuse_otf_rows()) {
        DISPATCH_N(N, (otf_cols_impl<NN_>(PsfWs(workspace, NN_).otf_rows, reinterpret_cast<float2*>(otf), tw,
                                          1.0f / (static_cast<float>(NN_) * NN_), s, PsfWs(workspace, NN_).part_rows,
                                          3 * (NN_ / Tile<NN_>::CROWS))));
    }
    DISPATCH_N(N, (otf_impl<NN_>(PsfWs(workspace, NN_).I, reinterpret_cast<float2*>(otf), tw,
                                 1.0f / (static_cast<float>(NN_) * NN_), s, PsfWs(workspace, NN_).part_rows,
                                 3 * (NN_ / Tile<NN_>::CROWS))));
}

int b200cam_psf_finish(const float* rho, float* psf, float* stats, void* workspace, size_t workspace_bytes, int N,
                       void* stream) {
    if (!b200cam_supported(N)) return B200CAM_E_BAD_SIZE;
    if (!rho || !psf || !stats || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_psf_workspace_bytes(N)) return B200CAM_E_WORKSPACE;
    if (!aligned16(workspace)) return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH_N(N, (psf_finish_impl<NN_>(rho, psf, stats, workspace, s)));
}

int b200cam_psf_bwd(const float* grad_psf, const float* grad_rad, const float* grad_cen, const float* h, const float* A,
                    const float* Ht, const float* rho, const float* kappa, const float* psf, const float* field,
                    float* stats, float* grad_h, void* workspace, size_t workspace_bytes, int N, void* stream) {
    if (!b200cam_supported(N)) return B200CAM_E_BAD_SIZE;
    if (!h || !A || !Ht || !rho || !kappa || !psf || !field || !stats || !grad_h || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_psf_workspace_bytes(N)) return B200CAM_E_WORKSPACE;
    if (!aligned16(A) || !aligned16(Ht) || !aligned16(field) || !aligned16(workspace)) return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH_N(N, (psf_bwd_impl<NN_>(grad_psf, grad_rad, grad_cen, h, reinterpret_cast<const float2*>(A),
                                     reinterpret_cast<const float2*>(Ht), rho, kappa, psf,
                                     reinterpret_cast<const float2*>(field), stats, grad_h, workspace, s)));
}

size_t b200cam_comm_bytes(int N, int world) {
    if (!b200cam_supported(N) || world < 1 || world > COMM_MAX_WORLD) return 0;
    return COMM_HEADER_BYTES + static_cast<size_t>(2) * world * N * N * sizeof(uint2);
}

int b200cam_psf_bwd_allreduce(const float* grad_psf, const float* grad_rad, const float* grad_cen, const float* h, const float* A,
                              const float* Ht, const float* rho, const float* kappa, const float* psf, const float* field,
                              float* stats, float* grad_h, void* workspace, size_t workspace_bytes, int N, void* stream,
                              void* const* peer_bufs, int rank, int world, float scale) {
    if (!b200cam_supported(N) || world < 1 || world > COMM_MAX_WORLD || rank < 0 || rank >= world) return B200CAM_E_BAD_SIZE;
    if (N / 2 > static_cast<int>(COMM_HEADER_BYTES / sizeof(unsigned))) return B200CAM_E_BAD_SIZE;   // one epoch word per tile
    if (!h || !A || !Ht || !rho || !kappa || !psf || !field || !stats || !grad_h || !workspace || !peer_bufs) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_psf_workspace_bytes(N)) return B200CAM_E_WORKSPACE;
    if (!aligned16(A) || !aligned16(Ht) || !aligned16(field) || !aligned16(workspace) || !aligned16(grad_h)) return B200CAM_E_ALIGN;
    CommDev comm;
    for (int r = 0; r < world; ++r) {
        if (!peer_bufs[r] || !aligned16(peer_bufs[r])) return B200CAM_E_NULL;
        comm.buf[r] = static_cast<unsigned char*>(peer_bufs[r]);
    }
    for (int r = world; r < COMM_MAX_WORLD; ++r) comm.buf[r] = nullptr;
    comm.rank = rank; comm.world = world; comm.scale = scale;
    static const double timeout_s = [] { const char* e = getenv("B200CAM_COMM_TIMEOUT_S"); const double v = e ? atof(e) : 30.0; return v > 0 ? v : 30.0; }();
    comm.timeout_clk = static_cast<long long>(timeout_s * 2.0e9);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH_N(N, (psf_bwd_impl<NN_>(grad_psf, grad_rad, grad_cen, h, reinterpret_cast<const float2*>(A),
                                     reinterpret_cast<const float2*>(Ht), rho, kappa, psf,
                                     reinterpret_cast<const float2*>(field), stats, grad_h, workspace, s, &comm)));
}

size_t b200cam_spectrum_bytes(int N, int B) {
    if (!b200cam_supported(N) || B < 1) return 0;
    return static_cast<size_t>(3) * B * (N / 2 + 1) * N * sizeof(float2);
}

int b200cam_sensor_fwd(const float* img, const float* psf, float* sensor, float* img_max, int* tie_count,
                       int* tie_pos, float* otf, float* spectrum, void* workspace, size_t workspace_bytes, int B,
                       int N, void* stream) {
    return b200cam_sensor_fwd_ex(img, psf, sensor, img_max, tie_count, tie_pos, otf, spectrum, workspace, workspace_bytes, B, N,
                                 stream, 0, nullptr, 0.f, 0);
}

int b200cam_sensor_fwd_ex(const float* img, const float* psf, float* sensor, float* img_max, int* tie_count,
                          int* tie_pos, float* otf, float* spectrum, void* workspace, size_t workspace_bytes, int B,
                          int N, void* stream, int flags, const float* noise, float noise_scale, int quant_bits) {
    SensorEpilogue epi;
    if (const int rc = make_epilogue(flags, noise, noise_scale, quant_bits, &epi)) return rc;
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!img || !psf || !sensor || !img_max || !tie_count || !tie_pos || !otf || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, 0)) return B200CAM_E_WORKSPACE;
    if (!aligned16(img) || !aligned16(sensor) || !aligned16(otf) || !aligned16(workspace) || !aligned16(psf))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (spectrum != nullptr && !aligned16(spectrum)) return B200CAM_E_ALIGN;
    DISPATCH_N(N, (sensor_fwd_impl<NN_>(img, psf, sensor, img_max, tie_count, tie_pos,
                                        reinterpret_cast<float2*>(otf), reinterpret_cast<float2*>(spectrum), workspace,
                                        B, s, epi)));
}

int b200cam_sensor_split_supported(int N, int B) {
    return b200cam_supported(N) && B >= 1;
}

int b200cam_sensor_rows(const float* img, float* spectrum, float* img_max, int* tie_count, int B, int N, void* stream) {
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!img || !spectrum || !img_max || !tie_count) return B200CAM_E_NULL;
    if (!aligned16(img) || !aligned16(spectrum)) return B200CAM_E_ALIGN;
    if (!b200cam_sensor_split_supported(N, B)) return B200CAM_E_BAD_SIZE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH_N(N, (sensor_rows_impl<NN_>(img, reinterpret_cast<float2*>(spectrum), img_max, tie_count, B, s)));
}

int b200cam_psf_otf(const float* psf, float* otf, int N, void* stream) {
    if (!b200cam_supported(N)) return B200CAM_E_BAD_SIZE;
    if (!psf || !otf) return B200CAM_E_NULL;
    if (!aligned16(psf) || !aligned16(otf)) return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const float2* tw = twiddle(N);
    if (tw == nullptr) return B200CAM_E_NOT_INIT;
    DISPATCH_N(N, (otf_impl<NN_>(psf, reinterpret_cast<float2*>(otf), tw, 1.0f / (static_cast<float>(NN_) * NN_), s)));
}

int b200cam_sensor_finish(const float* psf, float* sensor, float* img_max, int* tie_count, int* tie_pos, float* otf,
                          const float* spectrum, int otf_ready, void* workspace, size_t workspace_bytes, int B, int N,
                          void* stream) {
    return b200cam_sensor_finish_ex(psf, sensor, img_max, tie_count, tie_pos, otf, spectrum, otf_ready, workspace, workspace_bytes,
                                    B, N, stream, 0, nullptr, 0.f, 0);
}

int b200cam_sensor_finish_ex(const float* psf, float* sensor, float* img_max, int* tie_count, int* tie_pos, float* otf,
                             const float* spectrum, int otf_ready, void* workspace, size_t workspace_bytes, int B, int N,
                             void* stream, int flags, const float* noise, float noise_scale, int quant_bits) {
    SensorEpilogue epi;
    if (const int rc = make_epilogue(flags, noise, noise_scale, quant_bits, &epi)) return rc;
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (epi.seed != nullptr && N == 256 && plane_selected()) return B200CAM_E_BAD_SIZE;   // rows in the plane layout
    if (!psf || !sensor || !img_max || !tie_count || !tie_pos || !otf || !spectrum || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, 0)) return B200CAM_E_WORKSPACE;
    if (!aligned16(sensor) || !aligned16(otf) || !aligned16(workspace) || !aligned16(psf) || !aligned16(spectrum))
        return B200CAM_E_ALIGN;
    if (!b200cam_sensor_split_supported(N, B)) return B200CAM_E_BAD_SIZE;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH_N(N, (sensor_finish_impl<NN_>(psf, sensor, img_max, tie_count, tie_pos, reinterpret_cast<float2*>(otf),
                                           reinterpret_cast<const float2*>(spectrum), SensorWs(workspace, NN_, B, false),
                                           B, otf_ready, s, epi)));
}

// the noise of B200CAM_SENSOR_NOISE_PHILOX, materialised; the seed block is checked as make_epilogue checks it
int b200cam_sensor_noise(const void* seed_block, float* out, long long count, void* stream) {
    if (seed_block == nullptr || out == nullptr) return B200CAM_E_NULL;
    if (count < 0 || count % 4 != 0) return B200CAM_E_BAD_SIZE;
    if (reinterpret_cast<uintptr_t>(seed_block) % 8 != 0 || !aligned16(out)) return B200CAM_E_ALIGN;
    if (count == 0) return 0;
    const long long n4 = count / 4;
    const int grid = static_cast<int>(n4 / EW_THREADS < 148 * 8 ? (n4 + EW_THREADS - 1) / EW_THREADS : 148 * 8);
    launch_k(k_philox_noise, grid, EW_THREADS, 0, static_cast<cudaStream_t>(stream),
             static_cast<const b200cam_noise_seed*>(seed_block), out, n4);
    LAUNCH_CHECK();
    return 0;
}

int b200cam_conv_fwd(const float* img, const float* kernel, float* out, float* otf, float* spectrum, void* workspace,
                     size_t workspace_bytes, int B, int N, void* stream) {
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!img || !kernel || !out || !otf || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, 0)) return B200CAM_E_WORKSPACE;
    if (!aligned16(img) || !aligned16(kernel) || !aligned16(out) || !aligned16(otf) || !aligned16(workspace) ||
        (spectrum && !aligned16(spectrum)))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH_N(N, (conv_fwd_impl<NN_>(img, kernel, out, reinterpret_cast<float2*>(otf), reinterpret_cast<float2*>(spectrum),
                                      workspace, B, s)));
}

int b200cam_conv_bwd(const float* grad_out, const float* img, const float* otf, const float* spectrum, float* grad_kernel,
                     float* grad_img, void* workspace, size_t workspace_bytes, int B, int N, void* stream) {
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!grad_out || !img || !otf || !grad_kernel || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, grad_img != nullptr)) return B200CAM_E_WORKSPACE;
    if (!aligned16(grad_out) || !aligned16(img) || !aligned16(otf) || !aligned16(grad_kernel) || !aligned16(workspace) ||
        (spectrum && !aligned16(spectrum)) || (grad_img && !aligned16(grad_img)))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    DISPATCH_N(N, (conv_bwd_impl<NN_>(grad_out, img, reinterpret_cast<const float2*>(otf),
                                      reinterpret_cast<const float2*>(spectrum), grad_kernel, grad_img, workspace, B, s)));
}

int b200cam_sensor_bwd(const float* grad_sensor, const float* img, const float* sensor, const float* img_max,
                       const int* tie_count, const int* tie_pos, const float* psf, const float* otf,
                       const float* spectrum, float* grad_psf, float* grad_img, void* workspace,
                       size_t workspace_bytes, int B, int N, void* stream) {
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!grad_sensor || !img || !sensor || !img_max || !tie_count || !tie_pos || !psf || !otf || !grad_psf || !workspace)
        return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, grad_img != nullptr)) return B200CAM_E_WORKSPACE;
    if (!aligned16(grad_sensor) || !aligned16(img) || !aligned16(sensor) || !aligned16(otf) || !aligned16(workspace) ||
        !aligned16(grad_psf) || (grad_img && !aligned16(grad_img)))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const float2* spec = reinterpret_cast<const float2*>(spectrum);
    DISPATCH_N(N, (sensor_bwd_impl<NN_>(grad_sensor, img, sensor, img_max, tie_count, tie_pos, psf,
                                        reinterpret_cast<const float2*>(otf), spec, grad_psf, grad_img, workspace,
                                        B, s)));
}

// ---- bf16 sensor image / bf16 upstream gradient ------------------------------------------------------------
// `conv` [B][3][N][N] fp32 scratch (the un-normalised image; free once the call's work has run), `sensor` bf16 bit patterns
int b200cam_sensor_fwd_bf16(const float* img, const float* psf, float* conv, unsigned short* sensor, float* img_max, int* tie_count,
                            int* tie_pos, float* otf, float* spectrum, void* workspace, size_t workspace_bytes, int B, int N,
                            void* stream, int flags, const float* noise, float noise_scale, int quant_bits) {
    SensorEpilogue epi;
    if (const int rc = make_epilogue(flags, noise, noise_scale, quant_bits, &epi)) return rc;
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!img || !psf || !conv || !sensor || !img_max || !tie_count || !tie_pos || !otf || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, 0)) return B200CAM_E_WORKSPACE;
    if (!aligned16(img) || !aligned16(conv) || !aligned16(sensor) || !aligned16(otf) || !aligned16(workspace) || !aligned16(psf) ||
        (spectrum != nullptr && !aligned16(spectrum)))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    bf16* out = reinterpret_cast<bf16*>(sensor);
    DISPATCH_N(N, (sensor_fwd_impl<NN_>(img, psf, conv, img_max, tie_count, tie_pos, reinterpret_cast<float2*>(otf),
                                        reinterpret_cast<float2*>(spectrum), workspace, B, s, epi, out)));
}

int b200cam_sensor_finish_bf16(const float* psf, float* conv, unsigned short* sensor, float* img_max, int* tie_count, int* tie_pos,
                               float* otf, const float* spectrum, int otf_ready, void* workspace, size_t workspace_bytes, int B,
                               int N, void* stream, int flags, const float* noise, float noise_scale, int quant_bits) {
    SensorEpilogue epi;
    if (const int rc = make_epilogue(flags, noise, noise_scale, quant_bits, &epi)) return rc;
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (N == 256 && plane_selected()) return B200CAM_E_BAD_SIZE;     // b200cam_sensor_rows wrote the plane layout
    if (!psf || !conv || !sensor || !img_max || !tie_count || !tie_pos || !otf || !spectrum || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, 0)) return B200CAM_E_WORKSPACE;
    if (!aligned16(conv) || !aligned16(sensor) || !aligned16(otf) || !aligned16(workspace) || !aligned16(psf) || !aligned16(spectrum))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    bf16* out = reinterpret_cast<bf16*>(sensor);
    DISPATCH_N(N, (sensor_finish_impl<NN_>(psf, conv, img_max, tie_count, tie_pos, reinterpret_cast<float2*>(otf),
                                           reinterpret_cast<const float2*>(spectrum), SensorWs(workspace, NN_, B, false),
                                           B, otf_ready, s, epi, out)));
}

int b200cam_sensor_bwd_bf16(const unsigned short* grad_sensor, const float* img, const float* img_max, const int* tie_count,
                            const int* tie_pos, const float* psf, const float* otf, const float* spectrum, float* grad_psf,
                            float* grad_img, void* workspace, size_t workspace_bytes, int B, int N, void* stream) {
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!grad_sensor || !img || !img_max || !tie_count || !tie_pos || !psf || !otf || !grad_psf || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, grad_img != nullptr)) return B200CAM_E_WORKSPACE;
    if (!aligned16(grad_sensor) || !aligned16(img) || !aligned16(otf) || !aligned16(workspace) || !aligned16(grad_psf) ||
        (spectrum && !aligned16(spectrum)) || (grad_img && !aligned16(grad_img)))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bf16* g = reinterpret_cast<const bf16*>(grad_sensor);
    DISPATCH_N(N, (sensor_bwd_impl<NN_, bf16>(g, img, nullptr, img_max, tie_count, tie_pos, psf, reinterpret_cast<const float2*>(otf),
                                              reinterpret_cast<const float2*>(spectrum), grad_psf, grad_img, workspace, B, s)));
}

// ---- uint8 images ------------------------------------------------------------------------------------------
// The same calls with the images as uint8 bytes (what a decoder yields), converted in the kernels as byte * fp32(1/255), i.e.
// exactly torch's u8.float() / 255.0 on the GPU: every output is that of the fp32 call on the converted batch, bit for bit.
// They always run the default two-pass pipeline (the opt-in plane kernels read fp32 images only).
int b200cam_sensor_rows_u8(const unsigned char* img, float* spectrum, float* img_max, int* tie_count, int B, int N, void* stream) {
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (N == 256 && plane_selected()) return B200CAM_E_BAD_SIZE;     // b200cam_sensor_finish would expect the plane layout
    if (!img || !spectrum || !img_max || !tie_count) return B200CAM_E_NULL;
    if (!aligned16(img) || !aligned16(spectrum)) return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const u8* x = reinterpret_cast<const u8*>(img);
    DISPATCH_N(N, (sensor_rows_impl<NN_, u8>(x, reinterpret_cast<float2*>(spectrum), img_max, tie_count, B, s)));
}

int b200cam_sensor_fwd_u8(const unsigned char* img, const float* psf, float* sensor, float* img_max, int* tie_count, int* tie_pos,
                          float* otf, float* spectrum, void* workspace, size_t workspace_bytes, int B, int N, void* stream, int flags,
                          const float* noise, float noise_scale, int quant_bits) {
    SensorEpilogue epi;
    if (const int rc = make_epilogue(flags, noise, noise_scale, quant_bits, &epi)) return rc;
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!img || !psf || !sensor || !img_max || !tie_count || !tie_pos || !otf || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, 0)) return B200CAM_E_WORKSPACE;
    if (!aligned16(img) || !aligned16(sensor) || !aligned16(otf) || !aligned16(workspace) || !aligned16(psf) ||
        (spectrum != nullptr && !aligned16(spectrum)))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const u8* x = reinterpret_cast<const u8*>(img);
    DISPATCH_N(N, (sensor_fwd_impl<NN_, u8>(x, psf, sensor, img_max, tie_count, tie_pos, reinterpret_cast<float2*>(otf),
                                            reinterpret_cast<float2*>(spectrum), workspace, B, s, epi)));
}

int b200cam_sensor_fwd_u8_bf16(const unsigned char* img, const float* psf, float* conv, unsigned short* sensor, float* img_max,
                               int* tie_count, int* tie_pos, float* otf, float* spectrum, void* workspace, size_t workspace_bytes,
                               int B, int N, void* stream, int flags, const float* noise, float noise_scale, int quant_bits) {
    SensorEpilogue epi;
    if (const int rc = make_epilogue(flags, noise, noise_scale, quant_bits, &epi)) return rc;
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!img || !psf || !conv || !sensor || !img_max || !tie_count || !tie_pos || !otf || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, 0)) return B200CAM_E_WORKSPACE;
    if (!aligned16(img) || !aligned16(conv) || !aligned16(sensor) || !aligned16(otf) || !aligned16(workspace) || !aligned16(psf) ||
        (spectrum != nullptr && !aligned16(spectrum)))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const u8* x = reinterpret_cast<const u8*>(img);
    bf16* out = reinterpret_cast<bf16*>(sensor);
    DISPATCH_N(N, (sensor_fwd_impl<NN_, u8>(x, psf, conv, img_max, tie_count, tie_pos, reinterpret_cast<float2*>(otf),
                                            reinterpret_cast<float2*>(spectrum), workspace, B, s, epi, out)));
}

int b200cam_sensor_bwd_u8(const float* grad_sensor, const unsigned char* img, const float* sensor, const float* img_max,
                          const int* tie_count, const int* tie_pos, const float* psf, const float* otf, const float* spectrum,
                          float* grad_psf, float* grad_img, void* workspace, size_t workspace_bytes, int B, int N, void* stream) {
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!grad_sensor || !img || !sensor || !img_max || !tie_count || !tie_pos || !psf || !otf || !grad_psf || !workspace)
        return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, grad_img != nullptr)) return B200CAM_E_WORKSPACE;
    if (!aligned16(grad_sensor) || !aligned16(img) || !aligned16(sensor) || !aligned16(otf) || !aligned16(workspace) ||
        !aligned16(grad_psf) || (spectrum && !aligned16(spectrum)) || (grad_img && !aligned16(grad_img)))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const u8* x = reinterpret_cast<const u8*>(img);
    DISPATCH_N(N, (sensor_bwd_impl<NN_, float, u8>(grad_sensor, x, sensor, img_max, tie_count, tie_pos, psf,
                                                   reinterpret_cast<const float2*>(otf), reinterpret_cast<const float2*>(spectrum),
                                                   grad_psf, grad_img, workspace, B, s)));
}

int b200cam_sensor_bwd_u8_bf16(const unsigned short* grad_sensor, const unsigned char* img, const float* img_max, const int* tie_count,
                               const int* tie_pos, const float* psf, const float* otf, const float* spectrum, float* grad_psf,
                               float* grad_img, void* workspace, size_t workspace_bytes, int B, int N, void* stream) {
    if (!b200cam_supported(N) || B < 1) return B200CAM_E_BAD_SIZE;
    if (!grad_sensor || !img || !img_max || !tie_count || !tie_pos || !psf || !otf || !grad_psf || !workspace) return B200CAM_E_NULL;
    if (workspace_bytes < b200cam_sensor_workspace_bytes(N, B, grad_img != nullptr)) return B200CAM_E_WORKSPACE;
    if (!aligned16(grad_sensor) || !aligned16(img) || !aligned16(otf) || !aligned16(workspace) || !aligned16(grad_psf) ||
        (spectrum && !aligned16(spectrum)) || (grad_img && !aligned16(grad_img)))
        return B200CAM_E_ALIGN;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bf16* g = reinterpret_cast<const bf16*>(grad_sensor);
    const u8* x = reinterpret_cast<const u8*>(img);
    DISPATCH_N(N, (sensor_bwd_impl<NN_, bf16, u8>(g, x, nullptr, img_max, tie_count, tie_pos, psf, reinterpret_cast<const float2*>(otf),
                                                  reinterpret_cast<const float2*>(spectrum), grad_psf, grad_img, workspace, B, s)));
}

}  // extern "C"
