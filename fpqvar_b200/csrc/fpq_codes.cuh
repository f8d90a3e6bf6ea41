// Quantizer -> codes: the element functions that turn a group's values into e4m3 code bytes (include/fpq_b200.h, "Packed
// low-bit operands").  Shared by fpq_pack_codes (fpq_gemm.cu) and the codes output of the fused rotate kernels
// (fpq_rotate.cu), so that both emit the same bytes for the same fp16 values.
#pragma once
#include "fpq_h16.cuh"
#include <cuda_fp8.h>
#include <type_traits>

namespace fpq {

template <typename T> struct Chunk16;
template <> struct Chunk16<__half> {
    static __device__ __forceinline__ void load(const __half* p, float (&v)[16]) {
        const uint4 a = ldg_stream(p), b = ldg_stream(p + 8);
        const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            v[2 * i] = h2f(uint16_t(w[i] & 0xffffu));
            v[2 * i + 1] = h2f(uint16_t(w[i] >> 16));
        }
    }
    static __device__ __forceinline__ float scale(float amax, float vmax) { return __half2float(__float2half_rn(__fdiv_rn(amax, vmax))); }
    static __device__ __forceinline__ float norm(float x, float s) { return __half2float(__float2half_rn(__fdiv_rn(x, s))); }
};
template <> struct Chunk16<float> {
    static __device__ __forceinline__ void load(const float* p, float (&v)[16]) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint4 a = ldg_stream(p + 4 * j);
            v[4 * j] = __uint_as_float(a.x); v[4 * j + 1] = __uint_as_float(a.y);
            v[4 * j + 2] = __uint_as_float(a.z); v[4 * j + 3] = __uint_as_float(a.w);
        }
    }
    static __device__ __forceinline__ float scale(float amax, float vmax) { return __fdiv_rn(amax, vmax); }
    static __device__ __forceinline__ float norm(float x, float s) { return __fdiv_rn(x, s); }
};

__device__ __forceinline__ uint32_t e4m3x4(float a, float b, float c, float d) {
    const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E4M3);
    const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E4M3);
    return lo | (hi << 16);
}
// the same from two fp16 pairs of grid values (exact in both types): four codes, element order lo, hi, lo, hi
__device__ __forceinline__ uint32_t e4m3x4_h2(uint32_t ab, uint32_t cd) {
    __half2_raw r0, r1;
    r0.x = uint16_t(ab & 0xffffu); r0.y = uint16_t(ab >> 16);
    r1.x = uint16_t(cd & 0xffffu); r1.y = uint16_t(cd >> 16);
    const uint32_t lo = __nv_cvt_halfraw2_to_fp8x2(r0, __NV_SATFINITE, __NV_E4M3);
    const uint32_t hi = __nv_cvt_halfraw2_to_fp8x2(r1, __NV_SATFINITE, __NV_E4M3);
    return lo | (hi << 16);
}

// Grid values of 16 elements that share the scale s.  fp16 tensors with a regular scale (normal, finite: everything but zero,
// tiny, inf and NaN groups) take the division-free element function of the packed fp16 quantizers (fpq_h16.cuh: half(x * RN(1/s))
// == half(x / s), tie shift 2^-17, magic-number rounding; checked against the literal sequence for every (x, scale) pair by
// fpq_selftest_f16_flow) -- the grid value is that function's intermediate; everything else takes the literal sequence.
template <typename T, class HG>
__device__ __forceinline__ void grid_values16(const float (&v)[16], float s, float delta, float (&q)[16]) {
    if constexpr (std::is_same<T, __half>::value) {
        if (scale_bits_regular(uint32_t(__half_as_ushort(__float2half_rn(s))))) {
            const float r = rcp_rn_normal(s);
            const uint64_t r2 = pk(r, r);
#pragma unroll
            for (int i = 0; i < 16; i += 2) {
                const uint32_t v2 = pack_h2_u64(fmul2(pk(v[i], v[i + 1]), r2));                      // half(x/s)
                const F2 f = unpk(round_pair_magic(fhadd(uint16_t(v2 & 0xffffu), delta), fhadd(uint16_t(v2 >> 16), delta), Magic<HG>::EM, Magic<HG>::SC));
                q[i] = f.lo;
                q[i + 1] = f.hi;
            }
            return;
        }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) q[i] = round_any_sym<HG, TIE_KERNEL>(Chunk16<T>::norm(v[i], s));
}

// 16 codes of 16 fp16 values (8 packed words, element order) that share the scale s: grid_values16, as fpq_pack_codes runs it.
// Out of line: the fused rotate kernels call it only for groups with an irregular scale (zero, subnormal, inf, NaN), which
// keeps the literal sequence out of their register tile (as literal_sym_h16 does for their fp16 output).
template <class HG>
static __device__ __noinline__ uint4 codes16_h16(const uint32_t* w, float s, float delta) {
    float v[16], q[16];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        v[2 * i] = h2f(uint16_t(w[i] & 0xffffu));
        v[2 * i + 1] = h2f(uint16_t(w[i] >> 16));
    }
    grid_values16<__half, HG>(v, s, delta, q);
    return make_uint4(e4m3x4(q[0], q[1], q[2], q[3]), e4m3x4(q[4], q[5], q[6], q[7]), e4m3x4(q[8], q[9], q[10], q[11]),
                      e4m3x4(q[12], q[13], q[14], q[15]));
}

}  // namespace fpq
