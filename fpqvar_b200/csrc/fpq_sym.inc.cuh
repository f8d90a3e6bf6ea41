// libfpq_b200 -- symmetric fake-quant kernels (reference rows a2, a4, a5, a6 of SURVEY.md section 8)
// Part of the C ABI of include/fpq_b200.h; no torch types here.
#include "fpq_h16.cuh"

namespace fpq {

// ------------------------------------------------------------------------------------------
// Symmetric per-group fake quant, GS = 16*LPG elements per group
// ------------------------------------------------------------------------------------------
template <typename InT, typename OutT, int FMT, int TIE, int LPG>
__global__ void __launch_bounds__(256) fake_quant_group_kernel(const InT* __restrict__ x, OutT* __restrict__ out,
                                                               size_t n_groups, int clamp3) {
    constexpr int GS = 16 * LPG;
    constexpr int IN_VEC = 16 / sizeof(InT);
    constexpr int GROUPS_PER_WARP = 32 / LPG;
    const int lane = threadIdx.x & 31;
    const int lig = lane % LPG;                    // lane in group
    const size_t warp_global = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;

    for (size_t gbase = warp_global * GROUPS_PER_WARP; gbase < n_groups; gbase += n_warps * GROUPS_PER_WARP) {
        const size_t g = gbase + lane / LPG;
        const bool valid = g < n_groups;
        float v[16];
        if (valid) {
            Vec16<InT>::load(x + g * GS, lig, LPG, v);
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = 0.0f;
        }
        if (clamp3) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = clamp3_keep_nan(v[i]);
        }
        sym_quant_tile<InT, FMT, TIE, LPG>(v);
        if (valid) store16<OutT, IN_VEC>(out + g * GS, lig, LPG, v);
    }
}

// ------------------------------------------------------------------------------------------
// Symmetric per-row fake quant (per_token / per_channel), any row length.  One CTA per row
// (grid-stride over rows); pass 1 reduces the absmax, pass 2 re-reads the row (L2-resident,
// it was just streamed) and quantizes.  Scalar accesses unless the row is 16-byte aligned.
// ------------------------------------------------------------------------------------------
template <typename InT, typename OutT, int FMT, int TIE>
__global__ void __launch_bounds__(256) fake_quant_row_kernel(const InT* __restrict__ x, OutT* __restrict__ out,
                                                             size_t n_rows, size_t row_len, int clamp3) {
    using HG = typename SymFmt<FMT>::HG;
    __shared__ float red[32];
    constexpr int VEC = 16 / sizeof(InT);
    for (size_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const InT* xr = x + row * row_len;
        OutT* orow = out + row * row_len;
        const bool vec_ok = (row_len % VEC == 0) && ((reinterpret_cast<uintptr_t>(xr) & 15) == 0);
        float a = 0.0f;
        if (vec_ok) {
            for (size_t i = threadIdx.x; i < row_len / VEC; i += blockDim.x) {
                const uint4 u = *reinterpret_cast<const uint4*>(xr + i * VEC);
                const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if constexpr (sizeof(InT) == 2) {
                        float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[k]));
                        if (clamp3) { f.x = clamp3_keep_nan(f.x); f.y = clamp3_keep_nan(f.y); }
                        a = fmax_nan(a, fmax_nan(fabsf(f.x), fabsf(f.y)));
                    } else {
                        float f = __uint_as_float(w[k]);
                        if (clamp3) f = clamp3_keep_nan(f);
                        a = fmax_nan(a, fabsf(f));
                    }
                }
            }
        } else {
            for (size_t i = threadIdx.x; i < row_len; i += blockDim.x) {
                float f = load_elem(xr + i);
                if (clamp3) f = clamp3_keep_nan(f);
                a = fmax_nan(a, fabsf(f));
            }
        }
        a = block_max_nan(a, red);
        const float s = rnd_in<InT>(__fdiv_rn(a, HG::VMAX));
        const bool regular = scale_regular<InT>(s);
        const float r = regular ? __frcp_rn(s) : 0.0f;
        const GridTable& gt = c_grids[SymFmt<FMT>::GT];
        for (size_t i = threadIdx.x; i < row_len; i += blockDim.x) {
            float f = load_elem(xr + i);
            if (clamp3) f = clamp3_keep_nan(f);
            const float q = regular ? quant_elem_fast<InT, HG, TIE>(f, s, r) : quant_elem_literal<InT, TIE>(f, s, gt);
            store_elem(orow + i, q * s);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Per-row fake quant with the row resident in registers: one CTA per row, V 16-byte vectors per
// thread, ONE pass over HBM (load -> block absmax -> quantize -> store).  Covers the per_token /
// per_channel shapes of the FP6 README configs (rows of 1920 .. 9216) when the row is 16-byte
// aligned and fits V <= 4 vectors x 1024 threads.
// ------------------------------------------------------------------------------------------
// Row scalars are derived once per row by warp 0 and broadcast (measured against the every-thread form, rows of 2304 /
// 7680 / 9216 fp16: 4.77 / 5.00 / 4.80 -> 5.66 / 5.59 / 5.32 TB/s).
template <typename InT, typename OutT, int FMT, int TIE, int V>
__global__ void __launch_bounds__(1024) fake_quant_row_reg_kernel(const InT* __restrict__ x, OutT* __restrict__ out, size_t n_rows,
                                                                  int row_vecs, int clamp3) {
    using HG = typename SymFmt<FMT>::HG;
    constexpr int VEC = 16 / sizeof(InT);
    __shared__ float red[36];
    const int tid = threadIdx.x, nt = blockDim.x;
    const float delta = tie_delta_kernel(uint32_t((size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 40));
    auto load_row = [&](size_t row, uint4 (&dst)[V]) {
        const InT* xr = x + row * size_t(row_vecs) * VEC;
#pragma unroll
        for (int k = 0; k < V; ++k) {
            const int vi = tid + k * nt;
            dst[k] = (row < n_rows && vi < row_vecs) ? ldg_stream(xr + size_t(vi) * VEC) : make_uint4(0u, 0u, 0u, 0u);
        }
    };
    uint4 u[V], un[V];
    load_row(blockIdx.x, un);
    for (size_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
        OutT* orow = out + row * size_t(row_vecs) * VEC;
#pragma unroll
        for (int k = 0; k < V; ++k) u[k] = un[k];
        load_row(row + gridDim.x, un);                 // next row's loads fly while this one reduces and computes
        // absmax over the row (NaN propagates, as torch's abs().max())
        float a = 0.0f;
#pragma unroll
        for (int k = 0; k < V; ++k) {
            const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if constexpr (sizeof(InT) == 2) {
                    float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
                    if (clamp3) { f.x = clamp3_keep_nan(f.x); f.y = clamp3_keep_nan(f.y); }
                    a = fmax_nan(a, fmax_nan(fabsf(f.x), fabsf(f.y)));
                } else {
                    float f = __uint_as_float(w[q]);
                    if (clamp3) f = clamp3_keep_nan(f);
                    a = fmax_nan(a, fabsf(f));
                }
            }
        }
        // row scalars once per row (see signsplit_row_reg_kernel)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a = fmax_nan(a, __shfl_xor_sync(0xffffffffu, a, o));
        __syncthreads();
        if ((tid & 31) == 0) red[tid >> 5] = a;
        __syncthreads();
        if (tid < 32) {
            const int nw = (nt + 31) >> 5;
            float m = tid < nw ? red[tid] : 0.0f;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmax_nan(m, __shfl_xor_sync(0xffffffffu, m, o));
            if (tid == 0) {
                const float s0 = rnd_in<InT>(__fdiv_rn(m, HG::VMAX));
                const bool reg0 = scale_regular<InT>(s0);
                red[32] = s0; red[33] = reg0 ? __frcp_rn(s0) : 0.0f; red[34] = reg0 ? 1.0f : 0.0f;
            }
        }
        __syncthreads();
        const float s = red[32], r = red[33];
        const bool regular = red[34] != 0.0f;
        const GridTable& gt = c_grids[SymFmt<FMT>::GT];
#pragma unroll
        for (int k = 0; k < V; ++k) {
            const int vi = tid + k * nt;
            if (vi >= row_vecs) continue;
            const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
            if constexpr (sizeof(InT) == 2 && sizeof(OutT) == 2 && TIE == TIE_KERNEL) {
                uint32_t o[4];
                if (regular && !clamp3 && scale_bits_regular_for<HG>(f2h(s))) {      // s is an fp16 value here
                    const SymK sk = make_symk<HG>(s, r);
#pragma unroll
                    for (int q = 0; q < 4; ++q) o[q] = sym_pair_h16<HG>(w[q], sk, delta);
                } else {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
                        if (clamp3) { f.x = clamp3_keep_nan(f.x); f.y = clamp3_keep_nan(f.y); }
                        const float q0 = regular ? quant_elem_fast<InT, HG, TIE>(f.x, s, r) : quant_elem_literal<InT, TIE>(f.x, s, gt);
                        const float q1 = regular ? quant_elem_fast<InT, HG, TIE>(f.y, s, r) : quant_elem_literal<InT, TIE>(f.y, s, gt);
                        o[q] = pack_h2(q0 * s, q1 * s);
                    }
                }
                stg_stream(orow + size_t(vi) * VEC, make_uint4(o[0], o[1], o[2], o[3]));
            } else {
                float f[VEC];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if constexpr (sizeof(InT) == 2) {
                        const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
                        f[2 * q] = t.x; f[2 * q + 1] = t.y;
                    } else {
                        f[q] = __uint_as_float(w[q]);
                    }
                }
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    float t = f[e];
                    if (clamp3) t = clamp3_keep_nan(t);
                    f[e] = (regular ? quant_elem_fast<InT, HG, TIE>(t, s, r) : quant_elem_literal<InT, TIE>(t, s, gt)) * s;
                }
                OutT* po = orow + size_t(vi) * VEC;
                if constexpr (sizeof(OutT) == 4) {
#pragma unroll
                    for (int e = 0; e < VEC; e += 4)
                        stg_stream(po + e, make_uint4(__float_as_uint(f[e]), __float_as_uint(f[e + 1]), __float_as_uint(f[e + 2]), __float_as_uint(f[e + 3])));
                } else if constexpr (VEC == 8) {
                    stg_stream(po, make_uint4(pack_h2(f[0], f[1]), pack_h2(f[2], f[3]), pack_h2(f[4], f[5]), pack_h2(f[6], f[7])));
                } else {
                    stg_stream(po, make_uint2(pack_h2(f[0], f[1]), pack_h2(f[2], f[3])));
                }
            }
        }
    }
}

template <typename InT, typename OutT>
static bool sym_row_reg_fits(const InT* xi, OutT* oo, size_t row_len) {
    constexpr int VEC = 16 / sizeof(InT);
    if (row_len % VEC != 0 || row_len < 256) return false;
    if ((reinterpret_cast<uintptr_t>(xi) & 15) || (reinterpret_cast<uintptr_t>(oo) & 15)) return false;
    if ((row_len * sizeof(OutT)) % 16 != 0 && sizeof(OutT) < sizeof(InT)) {
        if ((row_len * sizeof(OutT)) % 8 != 0) return false;
    }
    return row_len / VEC <= 4096;
}

template <typename InT, typename OutT, int FMT, int TIE>
static int launch_sym(const void* x, void* out, size_t n_rows, size_t row_len, int clamp3, cudaStream_t st) {
    const InT* xi = static_cast<const InT*>(x);
    OutT* oo = static_cast<OutT*>(out);
    const bool pow2_group = (row_len == 128 || row_len == 64) &&
                            ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    if constexpr (sizeof(InT) == 2 && sizeof(OutT) == 2 && TIE == TIE_KERNEL) {
        if (pow2_group && row_len == 128 && !clamp3) return launch_sym_h16(FMT, x, out, n_rows, st);
        if (pow2_group && row_len == 64 && !clamp3) return launch_sym_h16_g64(FMT, x, out, n_rows, st);
    }
    if (pow2_group) {
        const int lpg = int(row_len / 16);
        const size_t groups_per_block = (256 / 32) * (32 / lpg);
        const unsigned grid = grid_for(n_rows, groups_per_block, 64);
        if (lpg == 8) fake_quant_group_kernel<InT, OutT, FMT, TIE, 8><<<grid, 256, 0, st>>>(xi, oo, n_rows, clamp3);
        else fake_quant_group_kernel<InT, OutT, FMT, TIE, 4><<<grid, 256, 0, st>>>(xi, oo, n_rows, clamp3);
    } else if (sym_row_reg_fits(xi, oo, row_len)) {
        launch_row_reg([](auto v) { return fake_quant_row_reg_kernel<InT, OutT, FMT, TIE, v.value>; }, false, xi, oo, n_rows, row_len, clamp3, st);
    } else {
        const unsigned grid = grid_for(n_rows, 1, 16);
        fake_quant_row_kernel<InT, OutT, FMT, TIE><<<grid, 256, 0, st>>>(xi, oo, n_rows, row_len, clamp3);
    }
    return finish_launch();
}

template <int TIE>
static int dispatch_sym(int in_dtype, int out_dtype, int format, const void* x, void* out, size_t n_rows, size_t row_len, int clamp3,
                        cudaStream_t st) {
    return with_dtypes(in_dtype, out_dtype, [&](auto in_t, auto out_t) {
        return with_sym_format(format, [&](auto fmt) {
            return launch_sym<typename decltype(in_t)::type, typename decltype(out_t)::type, fmt.value, TIE>(x, out, n_rows, row_len, clamp3, st);
        });
    });
}

// One translation unit per tie rule (FPQ_SYM_TIE_PART = 0 / 1, see fpq_sym_k.cu / fpq_sym_a.cu): the 4 dtype
// pairs x 5 formats x {group, row-in-registers x3, row} instantiations of one rule take ~80 s of nvcc each.
#if FPQ_SYM_TIE_PART == 0
int fake_quant_kernel_tie(int in_dtype, int out_dtype, int format, const void* x, void* out, size_t n_rows, size_t row_len, int clamp3,
                          cudaStream_t st) {
    return dispatch_sym<TIE_KERNEL>(in_dtype, out_dtype, format, x, out, n_rows, row_len, clamp3, st);
}
#else
int fake_quant_argmin_tie(int in_dtype, int out_dtype, int format, const void* x, void* out, size_t n_rows, size_t row_len, int clamp3,
                          cudaStream_t st) {
    return dispatch_sym<TIE_ARGMIN>(in_dtype, out_dtype, format, x, out, n_rows, row_len, clamp3, st);
}
#endif

}  // namespace fpq

#if FPQ_SYM_TIE_PART == 0
using namespace fpq;

extern "C" int fpq_fake_quant(const void* x, void* out, size_t n_rows, size_t row_len, int in_dtype, int out_dtype, int format,
                              int tie_mode, unsigned flags, void* stream) {
    if (row_len == 0 || (n_rows && (!x || !out || x == out))) return FPQ_ERR_ARG;
    if (flags & ~FPQ_FLAG_CLAMP3) return FPQ_ERR_ARG;
    if (n_rows == 0) return FPQ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int clamp3 = (flags & FPQ_FLAG_CLAMP3) ? 1 : 0;
    if (tie_mode == FPQ_TIE_KERNEL) return fake_quant_kernel_tie(in_dtype, out_dtype, format, x, out, n_rows, row_len, clamp3, st);
    if (tie_mode == FPQ_TIE_ARGMIN) return fake_quant_argmin_tie(in_dtype, out_dtype, format, x, out, n_rows, row_len, clamp3, st);
    return FPQ_ERR_ARG;
}
#endif
