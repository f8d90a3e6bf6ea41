// libfpq_b200 -- sign-split fake-quant kernels (reference row a3 of SURVEY.md section 8)
// Part of the C ABI of include/fpq_b200.h; no torch types here.
#include "fpq_h16.cuh"

namespace fpq {

// ------------------------------------------------------------------------------------------
// Sign-split formats
// ------------------------------------------------------------------------------------------
// One element, literal reference sequence (quant_utils.py:428-451 / :404-410).
template <typename InT, typename OutT, int SPLIT, int TIE>
__device__ __forceinline__ float signsplit_elem_literal(float x, float sn, float sp) {
    using SF = SplitFmt<SPLIT>;
    const float xn = (x <= 0.0f) ? x : 0.0f;
    const float xp = (x > 0.0f) ? x : 0.0f;
    const float vn = rnd_in<InT>(__fdiv_rn(xn, sn));
    const float vp = rnd_in<InT>(__fdiv_rn(xp, sp));
    const float qn = scan_rule<TIE>(vn, c_grids[SF::GT_N].v, c_grids[SF::GT_N].k);
    const float qp = scan_rule<TIE>(vp, c_grids[SF::GT_P].v, c_grids[SF::GT_P].k);
    if (TIE == TIE_KERNEL) return __fadd_rn(__fmul_rn(qn, sn), __fmul_rn(qp, sp));
    return __fmul_rn(__fadd_rn(qn, qp), (x <= 0.0f) ? sn : sp);
}

// Eight fp16 elements, literal sequence under the kernel tie rule, out of line (cold path of the row kernel).
template <int SPLIT>
static __device__ __noinline__ uint4 signsplit_vec_literal_h16(uint4 v, float sn, float sp) {
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
        w[q] = pack_h2(signsplit_elem_literal<__half, __half, SPLIT, TIE_KERNEL>(t.x, sn, sp),
                       signsplit_elem_literal<__half, __half, SPLIT, TIE_KERNEL>(t.y, sn, sp));
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// Fast element: only the side the element lives on does any work; the other side
// contributes R(0/s)*s = +0 (s regular or zero) which leaves the sum unchanged.
template <typename InT, int SPLIT, int TIE>
__device__ __forceinline__ float signsplit_elem_fast(float x, float sn, float rn, float sp, float rp) {
    using SF = SplitFmt<SPLIT>;
    if (x > 0.0f) return quant_elem_fast<InT, typename SF::POS, TIE>(x, sp, rp) * sp;
    // x <= 0, or NaN (NaN fails both where() tests and is replaced by 0 on both sides; under the
    // argmin rule its scale is where(x<=0, sn, sp) = sp, but the product is +0 either way)
    const float xn = (x <= 0.0f) ? x : 0.0f;
    return quant_elem_fast<InT, typename SF::NEG, TIE>(xn, sn, rn) * sn;
}

// May a group take the fast path?  A zero scale means "no element on that side": the
// reference then computes 0/0 = NaN for every element of that half.  Under the kernel rule
// NaN rounds to +0 and the half contributes nothing (fast path with r = 0).  Under the argmin
// rule NaN rounds to grid[0]: harmless for the positive grid (grid[0] = 0) but the negative
// grid's grid[0] = -VMAX shifts every positive element, so sn == 0 goes the literal way.
template <typename InT, int TIE> __device__ __forceinline__ bool split_fast_ok(float sn, float sp) {
    const bool n_ok = scale_regular<InT>(sn) || (TIE == TIE_KERNEL && sn == 0.0f);
    const bool p_ok = scale_regular<InT>(sp) || sp == 0.0f;
    return n_ok && p_ok;
}

template <typename InT, typename OutT, int SPLIT, int TIE, int LPG>
__global__ void __launch_bounds__(256) signsplit_group_kernel(const InT* __restrict__ x, OutT* __restrict__ out,
                                                              size_t n_groups, unsigned* __restrict__ nan_flag) {
    using SF = SplitFmt<SPLIT>;
    constexpr int GS = 16 * LPG;
    constexpr int IN_VEC = 16 / sizeof(InT);
    constexpr int GROUPS_PER_WARP = 32 / LPG;
    const int lane = threadIdx.x & 31;
    const int lig = lane % LPG;
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
        // max|x_neg| and max|x_pos|; NaN elements count as 0 on both sides (where() semantics)
        float an = 0.0f, ap = 0.0f;
        bool has_nan = false;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            an = fmaxf(an, (v[i] <= 0.0f) ? -v[i] : 0.0f);
            ap = fmaxf(ap, (v[i] > 0.0f) ? v[i] : 0.0f);
            has_nan |= (v[i] != v[i]);
        }
        an = group_max<LPG>(an);
        ap = group_max<LPG>(ap);
        if (nan_flag != nullptr && has_nan) atomicOr(nan_flag, 1u);
        const float sn = rnd_in<InT>(__fdiv_rn(an, SF::NEG::VMAX));
        const float sp = rnd_in<InT>(__fdiv_rn(ap, SF::POS::VMAX));
        if (split_fast_ok<InT, TIE>(sn, sp)) {
            const float rn = sn == 0.0f ? 0.0f : __frcp_rn(sn);
            const float rp = sp == 0.0f ? 0.0f : __frcp_rn(sp);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = signsplit_elem_fast<InT, SPLIT, TIE>(v[i], sn, rn, sp, rp);
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = signsplit_elem_literal<InT, OutT, SPLIT, TIE>(v[i], sn, sp);
        }
        if (valid) store16<OutT, IN_VEC>(out + g * GS, lig, LPG, v);
    }
}

template <typename InT, typename OutT, int SPLIT, int TIE>
__global__ void __launch_bounds__(256) signsplit_row_kernel(const InT* __restrict__ x, OutT* __restrict__ out,
                                                            size_t n_rows, size_t row_len, unsigned* __restrict__ nan_flag) {
    using SF = SplitFmt<SPLIT>;
    __shared__ float red[32];
    for (size_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const InT* xr = x + row * row_len;
        OutT* orow = out + row * row_len;
        float an = 0.0f, ap = 0.0f;
        bool has_nan = false;
        for (size_t i = threadIdx.x; i < row_len; i += blockDim.x) {
            const float f = load_elem(xr + i);
            an = fmaxf(an, (f <= 0.0f) ? -f : 0.0f);
            ap = fmaxf(ap, (f > 0.0f) ? f : 0.0f);
            has_nan |= (f != f);
        }
        an = block_max_nan(an, red);
        ap = block_max_nan(ap, red);
        if (nan_flag != nullptr && has_nan) atomicOr(nan_flag, 1u);
        const float sn = rnd_in<InT>(__fdiv_rn(an, SF::NEG::VMAX));
        const float sp = rnd_in<InT>(__fdiv_rn(ap, SF::POS::VMAX));
        const bool fast = split_fast_ok<InT, TIE>(sn, sp);
        const float rn = (fast && sn != 0.0f) ? __frcp_rn(sn) : 0.0f;
        const float rp = (fast && sp != 0.0f) ? __frcp_rn(sp) : 0.0f;
        for (size_t i = threadIdx.x; i < row_len; i += blockDim.x) {
            const float f = load_elem(xr + i);
            const float o = fast ? signsplit_elem_fast<InT, SPLIT, TIE>(f, sn, rn, sp, rp)
                                 : signsplit_elem_literal<InT, OutT, SPLIT, TIE>(f, sn, sp);
            store_elem(orow + i, o);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Per-row sign-split with the row resident in registers (per_token variants of the FP6 configs,
// fp6_quant_int_neg_e2m3_pos_per_token_cuda qu.py:614-646): one CTA per row, V 16-byte vectors per
// thread, one HBM pass, the next row's loads in flight during the block reduction.
// ------------------------------------------------------------------------------------------
// Row scalars are derived once per row by warp 0 and broadcast (measured against the every-thread form: rows of 7680 / 9216
// fp16 4.59 / 4.34 -> 5.25 / 5.01 TB/s, rows of 1920 unchanged).
template <typename InT, typename OutT, int SPLIT, int TIE, int V>
__global__ void __launch_bounds__(1024) signsplit_row_reg_kernel(const InT* __restrict__ x, OutT* __restrict__ out, size_t n_rows,
                                                                 int row_vecs, unsigned* __restrict__ nan_flag) {
    using SF = SplitFmt<SPLIT>;
    constexpr int VEC = 16 / sizeof(InT);
    __shared__ float red[104];                        // warp partials (an, ap, NaN flag) + the five row scalars
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
        load_row(row + gridDim.x, un);
        float an = 0.0f, ap = 0.0f;
        bool has_nan = false;
        auto float_maxima = [&]() {                    // where(x<=0, x, 0) / where(x>0, x, 0): a NaN counts as 0 (qu.py:619-620)
            an = 0.0f; ap = 0.0f;
#pragma unroll
            for (int k = 0; k < V; ++k) {
                const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float f[2];
                    int n = 1;
                    if constexpr (sizeof(InT) == 2) {
                        const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
                        f[0] = t.x; f[1] = t.y; n = 2;
                    } else {
                        f[0] = __uint_as_float(w[q]); f[1] = 0.0f;
                    }
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        if (e < n) {
                            an = fmaxf(an, (f[e] <= 0.0f) ? -f[e] : 0.0f);
                            ap = fmaxf(ap, (f[e] > 0.0f) ? f[e] : 0.0f);
                            has_nan |= (f[e] != f[e]);
                        }
                    }
                }
            }
        };
        if constexpr (sizeof(InT) == 2) {
            // both maxima from the integer order of the fp16 bit patterns, two elements per VIMNMX (fpq_h16.cu)
            uint32_t pm = 0u, nm = 0u;
#pragma unroll
            for (int k = 0; k < V; ++k) {
                pm = __vmaxs2(__vmaxs2(pm, u[k].x), __vmaxs2(u[k].y, __vmaxs2(u[k].z, u[k].w)));
                nm = __vmaxu2(__vmaxu2(nm, u[k].x), __vmaxu2(u[k].y, __vmaxu2(u[k].z, u[k].w)));
            }
            const uint32_t pbits = uint32_t(max(int(short(pm & 0xffffu)), int(short(pm >> 16))));
            const uint32_t nraw = max(nm & 0xffffu, nm >> 16);
            const uint32_t nbits = nraw >= 0x8000u ? (nraw & 0x7fffu) : 0u;
            if (pbits > 0x7C00u || nbits > 0x7C00u) float_maxima();          // this thread holds a NaN
            else { an = h2f(uint16_t(nbits)); ap = h2f(uint16_t(pbits)); }
        } else {
            float_maxima();
        }
        if (nan_flag != nullptr && has_nan) atomicOr(nan_flag, 1u);
        // Row scalars once per row: warp partials -> shared, warp 0 finishes the reduction and derives the scales, everybody
        // reads five floats back (instead of every thread redoing the reduction, two IEEE divisions and two reciprocals).
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            an = fmaxf(an, __shfl_xor_sync(0xffffffffu, an, o));
            ap = fmaxf(ap, __shfl_xor_sync(0xffffffffu, ap, o));
        }
        const bool warp_nan = __any_sync(0xffffffffu, has_nan);
        const int wid = tid >> 5, lane = tid & 31, nw = (nt + 31) >> 5;
        __syncthreads();                                   // the previous row's readers of red[] are done
        if (lane == 0) { red[wid] = an; red[32 + wid] = ap; red[64 + wid] = warp_nan ? 1.0f : 0.0f; }
        __syncthreads();
        if (wid == 0) {
            float a = lane < nw ? red[lane] : 0.0f, b = lane < nw ? red[32 + lane] : 0.0f;
            const bool any_nan = __any_sync(0xffffffffu, lane < nw && red[64 + lane] != 0.0f);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                a = fmaxf(a, __shfl_xor_sync(0xffffffffu, a, o));
                b = fmaxf(b, __shfl_xor_sync(0xffffffffu, b, o));
            }
            if (lane == 0) {
                const float sn0 = rnd_in<InT>(__fdiv_rn(a, SF::NEG::VMAX));
                const float sp0 = rnd_in<InT>(__fdiv_rn(b, SF::POS::VMAX));
                const bool fast0 = split_fast_ok<InT, TIE>(sn0, sp0) && !any_nan;      // rows holding a NaN take the literal sequence
                red[96] = sn0; red[97] = sp0;
                red[98] = (fast0 && sn0 != 0.0f) ? __frcp_rn(sn0) : 0.0f;
                red[99] = (fast0 && sp0 != 0.0f) ? __frcp_rn(sp0) : 0.0f;
                red[100] = fast0 ? 1.0f : 0.0f;
            }
        }
        __syncthreads();
        const float sn = red[96], sp = red[97], rn = red[98], rp = red[99];
        const bool fast = red[100] != 0.0f;
        const SplitK sk = make_splitk<typename SF::NEG, typename SF::POS>(sn, rn, sp, rp);
        auto pair = [&](uint32_t w2) { return split_pair_h16<typename SF::NEG, typename SF::POS>(w2, sk, delta); };
#pragma unroll
        for (int k = 0; k < V; ++k) {
            const int vi = tid + k * nt;
            if (vi >= row_vecs) continue;
            const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
            if constexpr (sizeof(InT) == 2 && sizeof(OutT) == 2 && TIE == TIE_KERNEL) {
                // packed path; rows with an irregular scale or a NaN go through the out-of-line literal sequence (by value:
                // registers are not addressable), so the loop the hardware fetches stays small
                uint4 o;
                if (fast) {
                    o.x = pair(w[0]);
                    o.y = pair(w[1]);
                    o.z = pair(w[2]);
                    o.w = pair(w[3]);
                } else {
                    o = signsplit_vec_literal_h16<SPLIT>(u[k], sn, sp);
                }
                stg_stream(orow + size_t(vi) * VEC, o);
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
                for (int e = 0; e < VEC; ++e)
                    f[e] = fast ? signsplit_elem_fast<InT, SPLIT, TIE>(f[e], sn, rn, sp, rp) : signsplit_elem_literal<InT, OutT, SPLIT, TIE>(f[e], sn, sp);
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
static bool split_row_reg_fits(const InT* xi, OutT* oo, size_t row_len) {
    constexpr int VEC = 16 / sizeof(InT);
    if (row_len % VEC != 0 || row_len < 256) return false;
    if ((reinterpret_cast<uintptr_t>(xi) & 15) || (reinterpret_cast<uintptr_t>(oo) & 15)) return false;
    return row_len / VEC <= 4096;
}

// qu.py:421-422 with a NaN in the tensor: clamp(x, -NaN, NaN) makes every element NaN, both
// where() halves become 0, every scale 0, every quotient 0/0 -> q = 0 (kernel rule) or
// grid[0] (argmin rule), and the output is (+0)*0 + (+0)*0 = +0, resp. (g0n + g0p) * 0 = -0.
template <typename OutT>
__global__ void poison_fill_kernel(OutT* __restrict__ out, size_t n, unsigned* __restrict__ ws, float fill) {
    if (*reinterpret_cast<volatile unsigned*>(ws) != 0u)
        for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) store_elem(out + i, fill);
    // leave the workspace {flag, ticket} zeroed for the next call: the last CTA to get here resets it
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(ws + 1, 1u) == gridDim.x - 1) { ws[0] = 0u; ws[1] = 0u; }
}

template <typename InT, typename OutT, int SPLIT, int TIE>
static int launch_split(const void* x, void* out, size_t n_rows, size_t row_len, unsigned* flag, cudaStream_t st) {
    const InT* xi = static_cast<const InT*>(x);
    OutT* oo = static_cast<OutT*>(out);
    const bool pow2_group = (row_len == 128 || row_len == 64) &&
                            ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    bool launched = false;
    if constexpr (sizeof(InT) == 2 && sizeof(OutT) == 2 && TIE == TIE_KERNEL) {
        if (pow2_group && row_len == 128) {
            const int rc0 = launch_split_h16(SPLIT, x, out, n_rows, flag, st);
            if (rc0 != FPQ_OK) return rc0;
            launched = true;
        }
    }
    if (launched) {
    } else if (pow2_group) {
        const int lpg = int(row_len / 16);
        const size_t groups_per_block = (256 / 32) * (32 / lpg);
        const unsigned grid = grid_for(n_rows, groups_per_block, 64);
        if (lpg == 8) signsplit_group_kernel<InT, OutT, SPLIT, TIE, 8><<<grid, 256, 0, st>>>(xi, oo, n_rows, flag);
        else signsplit_group_kernel<InT, OutT, SPLIT, TIE, 4><<<grid, 256, 0, st>>>(xi, oo, n_rows, flag);
    } else if (split_row_reg_fits(xi, oo, row_len)) {
        launch_row_reg([](auto v) { return signsplit_row_reg_kernel<InT, OutT, SPLIT, TIE, v.value>; }, true, xi, oo, n_rows, row_len, flag, st);
    } else {
        const unsigned grid = grid_for(n_rows, 1, 16);
        signsplit_row_kernel<InT, OutT, SPLIT, TIE><<<grid, 256, 0, st>>>(xi, oo, n_rows, row_len, flag);
    }
    if (launched) return FPQ_OK;                      // the packed kernels handle the whole-tensor clip in their epilogue
    int rc = finish_launch();
    if (rc != FPQ_OK || flag == nullptr) return rc;
    // all-NaN tensor after the reference's clamp: kernel rule -> +0 everywhere; argmin rule ->
    // (grid_neg[0] + grid_pos[0]) * 0 = -0 everywhere
    const float fill = TIE == TIE_KERNEL ? 0.0f : -0.0f;
    const size_t n = n_rows * row_len;
    poison_fill_kernel<OutT><<<grid_for(n, 256 * 8, 8), 256, 0, st>>>(oo, n, flag, fill);
    return finish_launch();
}

template <int TIE>
static int dispatch_split(int in_dtype, int out_dtype, int split, const void* x, void* out, size_t n_rows, size_t row_len, unsigned* flag,
                          cudaStream_t st) {
    return with_dtypes(in_dtype, out_dtype, [&](auto in_t, auto out_t) {
        return with_split_format(split, [&](auto sf) {
            return launch_split<typename decltype(in_t)::type, typename decltype(out_t)::type, sf.value, TIE>(x, out, n_rows, row_len, flag, st);
        });
    });
}

// One translation unit per tie rule (FPQ_SPLIT_TIE_PART = 0 / 1: fpq_split_k.cu / fpq_split_a.cu), as for fpq_sym.
#if FPQ_SPLIT_TIE_PART == 0
int signsplit_kernel_tie(int in_dtype, int out_dtype, int split, const void* x, void* out, size_t n_rows, size_t row_len, unsigned* flag,
                         cudaStream_t st) {
    return dispatch_split<TIE_KERNEL>(in_dtype, out_dtype, split, x, out, n_rows, row_len, flag, st);
}
#else
int signsplit_argmin_tie(int in_dtype, int out_dtype, int split, const void* x, void* out, size_t n_rows, size_t row_len, unsigned* flag,
                         cudaStream_t st) {
    return dispatch_split<TIE_ARGMIN>(in_dtype, out_dtype, split, x, out, n_rows, row_len, flag, st);
}
#endif

}  // namespace fpq

#if FPQ_SPLIT_TIE_PART == 0
using namespace fpq;

extern "C" int fpq_fake_quant_signsplit(const void* x, void* out, size_t n_rows, size_t row_len, int in_dtype, int out_dtype,
                                        int split_format, int tie_mode, unsigned flags, void* workspace, void* stream) {
    if (row_len == 0 || (n_rows && (!x || !out || x == out))) return FPQ_ERR_ARG;
    if (flags & ~FPQ_FLAG_GLOBAL_CLIP) return FPQ_ERR_ARG;
    if ((flags & FPQ_FLAG_GLOBAL_CLIP) && !workspace) return FPQ_ERR_ARG;
    if (n_rows == 0) return FPQ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned* flag = (flags & FPQ_FLAG_GLOBAL_CLIP) ? static_cast<unsigned*>(workspace) : nullptr;
    if (tie_mode == FPQ_TIE_KERNEL) return signsplit_kernel_tie(in_dtype, out_dtype, split_format, x, out, n_rows, row_len, flag, st);
    if (tie_mode == FPQ_TIE_ARGMIN) return signsplit_argmin_tie(in_dtype, out_dtype, split_format, x, out, n_rows, row_len, flag, st);
    return FPQ_ERR_ARG;
}
#endif
