// b200cam: host/device compatibility layer.
//
// The kernel bodies in this directory are written as `B200_HD` function templates split into
// barrier-separated phases (see exec.cuh).  nvcc compiles them for sm_100a; the test-only
// emulator (tests/emu/) compiles the very same bodies with g++ and runs the phases as loops
// over thread ids, which lets the index arithmetic be checked on a machine without a GPU.
// Nothing in the shipped library executes on the CPU.
#pragma once

#include <cmath>
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#define B200_HD __host__ __device__ __forceinline__
#define B200_D __device__ __forceinline__
#else
#define B200_HD inline
struct float2 { float x, y; };
struct alignas(16) float4 { float x, y, z, w; };
static inline float2 make_float2(float x, float y) { return float2{x, y}; }
static inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }
#endif

namespace b200cam {

// ---- complex helpers (float2 = re, im) -------------------------------------------------
// On the device these map to the packed fp32 instructions of sm_100a (one FADD2 / FFMA2 per complex add, two
// per complex multiply; half swap and per-half negation are operand modifiers) - see pkfft.cuh.
#if defined(__CUDA_ARCH__)
B200_HD float2 cadd(float2 a, float2 b) { return __fadd2_rn(a, b); }
B200_HD float2 csub(float2 a, float2 b) { return __ffma2_rn(b, make_float2(-1.f, -1.f), a); }
B200_HD float2 cmul(float2 a, float2 b) {
    return __ffma2_rn(make_float2(a.y, a.x), make_float2(-b.y, b.y), __fmul2_rn(a, make_float2(b.x, b.x)));
}
// a * conj(b)
B200_HD float2 cmulc(float2 a, float2 b) {
    return __ffma2_rn(make_float2(a.y, a.x), make_float2(b.y, -b.y), __fmul2_rn(a, make_float2(b.x, b.x)));
}
#else
B200_HD float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
B200_HD float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
B200_HD float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
// a * conj(b)
B200_HD float2 cmulc(float2 a, float2 b) { return make_float2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); }
#endif
B200_HD float2 cconj(float2 a) { return make_float2(a.x, -a.y); }
B200_HD float2 cscale(float2 a, float s) { return make_float2(a.x * s, a.y * s); }
// multiply by +i / -i
B200_HD float2 cmul_i(float2 a) { return make_float2(-a.y, a.x); }
B200_HD float2 cmul_mi(float2 a) { return make_float2(a.y, -a.x); }

// ---- read-only loads --------------------------------------------------------------------
template <class T>
B200_HD T ld_ro(const T* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

// ---- bf16 sensor images / gradients ---------------------------------------------------------
// A bfloat16 value as its bit pattern (it crosses the C ABI as unsigned short: C has no bf16 type).  Widening to fp32 is
// exact (the 16 bits become the high half of the float); narrowing rounds to nearest-even, as torch's .to(torch.bfloat16).
struct bf16 {
    unsigned short bits;
};
B200_HD float to_float(float v) { return v; }
B200_HD float to_float(bf16 v) {
    const uint32_t u = static_cast<uint32_t>(v.bits) << 16;
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f;
    std::memcpy(&f, &u, 4);
    return f;
#endif
}
// ---- uint8 images ----------------------------------------------------------------------------
// A uint8 image byte, as a decoder yields it.  Its value is byte * fp32(1/255): torch's u8.float() / 255.0 on the GPU
// multiplies by the fp32 reciprocal of the CPU scalar, so this is bit for bit the image the caller would otherwise convert
// (ImgLoadU8 of lens_conv.cu is the same rule).  A tag type of its own, so that no generic unsigned char conversion picks
// it up by accident.
struct u8 {
    unsigned char bits;
};
B200_HD float to_float(u8 v) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(static_cast<float>(v.bits), 1.0f / 255.0f);
#else
    return static_cast<float>(v.bits) * (1.0f / 255.0f);
#endif
}
// element loads through the read-only path (fp32, or bf16 / uint8 widened in registers)
B200_HD float load_elem(const float* p) { return ld_ro(p); }
B200_HD float load_elem(const bf16* p) { return to_float(bf16{ld_ro(reinterpret_cast<const unsigned short*>(p))}); }
B200_HD float load_elem(const u8* p) { return to_float(u8{ld_ro(reinterpret_cast<const unsigned char*>(p))}); }
// fp32 -> bf16, round to nearest-even.  Device: __float2bfloat16_rn (the conversion torch's CUDA cast uses).  Host (emulator):
// the same bit rule - add 0x7fff plus the lowest kept bit, truncate - which gives the identical result for every finite
// value and for the infinities; NaN becomes the canonical quiet NaN of its sign.
B200_HD unsigned short bf16_bits_rn(float v) {
#if defined(__CUDA_ARCH__)
    return __bfloat16_as_ushort(__float2bfloat16_rn(v));
#else
    uint32_t u;
    std::memcpy(&u, &v, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<unsigned short>(((u >> 16) & 0x8000u) | 0x7fc0u);
    return static_cast<unsigned short>((u + 0x7fffu + ((u >> 16) & 1u)) >> 16);
#endif
}
// four outputs of an element-wise pass: fp32 as one float4 store, bf16 as one 8-byte store
B200_HD void store4(float* base, long long i4, float a, float b, float c, float d) {
    reinterpret_cast<float4*>(base)[i4] = make_float4(a, b, c, d);
}
B200_HD void store4(bf16* base, long long i4, float a, float b, float c, float d) {
    const uint32_t lo = static_cast<uint32_t>(bf16_bits_rn(a)) | (static_cast<uint32_t>(bf16_bits_rn(b)) << 16);
    const uint32_t hi = static_cast<uint32_t>(bf16_bits_rn(c)) | (static_cast<uint32_t>(bf16_bits_rn(d)) << 16);
#if defined(__CUDACC__)
    reinterpret_cast<uint2*>(base)[i4] = make_uint2(lo, hi);
#else
    uint32_t* p = reinterpret_cast<uint32_t*>(base) + 2 * i4;
    p[0] = lo;
    p[1] = hi;
#endif
}
// four consecutive gradient values (16-byte fp32 / 8-byte bf16 load)
B200_HD float4 load4(const float* base, long long i4) { return ld_ro(reinterpret_cast<const float4*>(base) + i4); }
B200_HD float4 load4(const bf16* base, long long i4) {
#if defined(__CUDA_ARCH__)
    const uint2 w = __ldg(reinterpret_cast<const uint2*>(base) + i4);
    return make_float4(__uint_as_float(w.x << 16), __uint_as_float(w.x & 0xffff0000u), __uint_as_float(w.y << 16),
                       __uint_as_float(w.y & 0xffff0000u));
#else
    return make_float4(to_float(base[4 * i4]), to_float(base[4 * i4 + 1]), to_float(base[4 * i4 + 2]), to_float(base[4 * i4 + 3]));
#endif
}

// ---- asynchronous global -> shared copies (LDGSTS: no register staging, the warp keeps computing) -----------
// 16 bytes, both addresses 16-byte aligned; L2 only (.cg): the data is consumed once from shared memory.
B200_HD void async_copy16(void* smem_dst, const void* gsrc) {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst))),
                 "l"(gsrc)
                 : "memory");
#else
    std::memcpy(smem_dst, gsrc, 16);
#endif
}
// all copies issued by THIS thread have landed (other lanes' copies: follow with a warp / block barrier)
B200_HD void async_wait_all() {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.wait_all;\n" ::: "memory");
#endif
}

// ---- drop a 128-byte line of DEAD data from L2 without writing it back to HBM --------------------------------
// The spectra between the row and column passes are written by one kernel, read once by the next and never again;
// left alone, every such line is eventually written back (about a quarter of the step's DRAM traffic).
B200_HD void discard_line(const void* p128) {
#if defined(__CUDA_ARCH__)
    asm volatile("discard.global.L2 [%0], 128;\n" ::"l"(p128) : "memory");
#else
    (void)p128;
#endif
}

// ---- pull a 128-byte line into L2 ahead of a later gather (fire and forget) -------------------------------------
B200_HD void prefetch_l2(const void* p128) {
#if defined(__CUDA_ARCH__)
    asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p128) : "memory");
#else
    (void)p128;
#endif
}

// ---- float max through integer atomics (order independent => deterministic) --------------
B200_HD void atomic_max_float(float* addr, float v) {
#if defined(__CUDA_ARCH__)
    if (v >= 0.f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
    else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
#else
    if (v > *addr) *addr = v;
#endif
}

B200_HD int atomic_add_int(int* addr, int v) {
#if defined(__CUDA_ARCH__)
    return atomicAdd(addr, v);
#else
    int old = *addr; *addr = old + v; return old;
#endif
}

B200_HD float neg_inf() {
#if defined(__CUDA_ARCH__)
    return __int_as_float(0xff800000);
#else
    return -INFINITY;
#endif
}

}  // namespace b200cam
