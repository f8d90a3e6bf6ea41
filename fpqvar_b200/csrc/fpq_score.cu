// libfpq_b200 -- batched format scoring (reference row a10 of SURVEY.md section 8).
// The search scripts quantize the same tensor once per candidate format and reduce
// mean((x - x_q)^2) each time (search/search_fp4_format.py:340-374,472-476,840-893;
// search/search_fp6_format.py:547-554).  Here x is read ONCE: each 128-group sits in the
// registers of 8 lanes, every candidate is applied to the register tile, and the per-candidate
// squared error is accumulated in fp32 per lane, fp64 per block, one atomicAdd(double) per
// block and candidate.
#include "fpq_h16.cuh"

namespace fpq {

constexpr int MAX_CAND = 8;
struct Candidates { int n; int fmt[MAX_CAND]; };

// squared error of one symmetric candidate over the lane's 16 values
template <typename InT, int FMT, int TIE>
__device__ __forceinline__ float sse_sym(const float (&v)[16], float a) {
    using HG = typename SymFmt<FMT>::HG;
    const float s = rnd_in<InT>(__fdiv_rn(a, HG::VMAX));
    float acc = 0.0f;
    if (scale_regular<InT>(s)) {
        const float r = __frcp_rn(s);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            // output dtype of the reference quantizers: the input dtype for the *_cuda functions
            // (kernel rule), fp32 for the argmin ones
            float o = quant_elem_fast<InT, HG, TIE>(v[i], s, r) * s;
            if (TIE == TIE_KERNEL) o = rnd_in<InT>(o);
            const float d = v[i] - o;
            acc = fmaf(d, d, acc);
        }
    } else {
        const GridTable& gt = c_grids[SymFmt<FMT>::GT];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            float o = quant_elem_literal<InT, TIE>(v[i], s, gt) * s;
            if (TIE == TIE_KERNEL) o = rnd_in<InT>(o);
            const float d = v[i] - o;
            acc = fmaf(d, d, acc);
        }
    }
    return acc;
}

template <typename InT, int SPLIT, int TIE>
__device__ __forceinline__ float sse_split(const float (&v)[16], float an, float ap) {
    using SF = SplitFmt<SPLIT>;
    const float sn = rnd_in<InT>(__fdiv_rn(an, SF::NEG::VMAX));
    const float sp = rnd_in<InT>(__fdiv_rn(ap, SF::POS::VMAX));
    const bool n_ok = scale_regular<InT>(sn) || (TIE == TIE_KERNEL && sn == 0.0f);
    const bool p_ok = scale_regular<InT>(sp) || sp == 0.0f;
    float acc = 0.0f;
    if (n_ok && p_ok) {
        const float rn = sn == 0.0f ? 0.0f : __frcp_rn(sn);
        const float rp = sp == 0.0f ? 0.0f : __frcp_rn(sp);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const float x = v[i];
            float o;
            if (x > 0.0f) o = quant_elem_fast<InT, typename SF::POS, TIE>(x, sp, rp) * sp;
            else o = quant_elem_fast<InT, typename SF::NEG, TIE>((x <= 0.0f) ? x : 0.0f, sn, rn) * sn;
            if (TIE == TIE_KERNEL) o = rnd_in<InT>(o);
            const float d = x - o;
            acc = fmaf(d, d, acc);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const float x = v[i];
            const float xn = (x <= 0.0f) ? x : 0.0f, xp = (x > 0.0f) ? x : 0.0f;
            const float qn = scan_rule<TIE>(rnd_in<InT>(__fdiv_rn(xn, sn)), c_grids[SF::GT_N].v, c_grids[SF::GT_N].k);
            const float qp = scan_rule<TIE>(rnd_in<InT>(__fdiv_rn(xp, sp)), c_grids[SF::GT_P].v, c_grids[SF::GT_P].k);
            float o = TIE == TIE_KERNEL ? rnd_in<InT>(__fadd_rn(__fmul_rn(qn, sn), __fmul_rn(qp, sp)))
                                        : __fmul_rn(__fadd_rn(qn, qp), (x <= 0.0f) ? sn : sp);
            const float d = x - o;
            acc = fmaf(d, d, acc);
        }
    }
    return acc;
}

template <typename InT, int TIE>
__global__ void __launch_bounds__(256) score_formats_kernel(const InT* __restrict__ x, size_t n_groups, Candidates cand,
                                                            double* __restrict__ sse) {
    constexpr int LPG = 8, GS = 128;
    __shared__ double s_acc[MAX_CAND];
    if (threadIdx.x < MAX_CAND) s_acc[threadIdx.x] = 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int lig = lane % LPG;
    const size_t warp_global = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    double acc[MAX_CAND];
#pragma unroll
    for (int c = 0; c < MAX_CAND; ++c) acc[c] = 0.0;

    for (size_t gbase = warp_global * 4; gbase < n_groups; gbase += n_warps * 4) {
        const size_t g = gbase + lane / LPG;
        float v[16];
        if (g < n_groups) {
            Vec16<InT>::load(x + g * GS, lig, LPG, v);
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = 0.0f;
        }
        float a = 0.0f, an = 0.0f, ap = 0.0f;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            a = fmax_nan(a, fabsf(v[i]));
            an = fmaxf(an, (v[i] <= 0.0f) ? -v[i] : 0.0f);
            ap = fmaxf(ap, (v[i] > 0.0f) ? v[i] : 0.0f);
        }
        a = group_max_nan<LPG>(a);
        an = group_max<LPG>(an);
        ap = group_max<LPG>(ap);
#pragma unroll
        for (int c = 0; c < MAX_CAND; ++c) {
            if (c < cand.n) {
                float e;
                switch (cand.fmt[c]) {
                    case FPQ_FMT_E2M1: e = sse_sym<InT, FPQ_FMT_E2M1, TIE>(v, a); break;
                    case FPQ_FMT_E1M2: e = sse_sym<InT, FPQ_FMT_E1M2, TIE>(v, a); break;
                    case FPQ_FMT_E3M0: e = sse_sym<InT, FPQ_FMT_E3M0, TIE>(v, a); break;
                    case FPQ_FMT_E2M3: e = sse_sym<InT, FPQ_FMT_E2M3, TIE>(v, a); break;
                    case FPQ_FMT_E3M2: e = sse_sym<InT, FPQ_FMT_E3M2, TIE>(v, a); break;
                    case 16 + FPQ_SPLIT_E1M2NEG_E2M1POS: e = sse_split<InT, FPQ_SPLIT_E1M2NEG_E2M1POS, TIE>(v, an, ap); break;
                    case 16 + FPQ_SPLIT_INTNEG_E2M3POS: e = sse_split<InT, FPQ_SPLIT_INTNEG_E2M3POS, TIE>(v, an, ap); break;
                    default: e = sse_split<InT, FPQ_SPLIT_AFPQ_E2M1, TIE>(v, an, ap); break;
                }
                acc[c] += double(e);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < MAX_CAND; ++c) {
        if (c < cand.n) {
            double e = acc[c];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
            if (lane == 0) atomicAdd(&s_acc[c], e);
        }
    }
    __syncthreads();
    if (threadIdx.x < cand.n) atomicAdd(&sse[threadIdx.x], s_acc[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------
// Packed variant for fp16 tensors under the kernel tie rule (the proj / fc2 calibration activations):
// the element functions of fpq_h16.cuh (conversion hardware for e2m1 / e1m2 / e2m3 / e3m2), ~5 instructions per
// element and candidate, and an error term that never leaves fp16 / mixed precision:
//     d   = x - o          fp16x2 subtraction, EXACT: o is the grid value next to x, so o/2 <= x <= 2o (or o = 0)
//     acc = d*d + acc      FHFMA (fp16 * fp16 + fp32 -> fp32), one per element
// 4 lanes x 32 halves per group, like the quantizer kernels.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t hsub2(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("sub.rn.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}
__device__ __forceinline__ float fhfma(uint16_t a, uint16_t b, float c) {        // fp32 = fp16 * fp16 + fp32
    float d;
    asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(d) : "h"(a), "h"(b), "f"(c));
    return d;
}
// (acc0, acc1) += (x - o)^2 of the two halves
__device__ __forceinline__ void sq_err_pair(uint32_t x2, uint32_t o2, float& acc0, float& acc1) {
    const uint32_t d2 = hsub2(x2, o2);
    acc0 = fhfma(uint16_t(d2 & 0xffffu), uint16_t(d2 & 0xffffu), acc0);
    acc1 = fhfma(uint16_t(d2 >> 16), uint16_t(d2 >> 16), acc1);
}

template <int FMT>
__device__ __forceinline__ float sse_sym_h16(const uint32_t (&p)[16], const uint64_t (&xf)[16], uint32_t absmax_b, float delta, const __half* src, int lig) {
    using HG = typename SymFmt<FMT>::HG;
    const float a = h2f(uint16_t(absmax_b));
    const __half sh = scale_from_absmax_h16<HG>(a);
    float acc0 = 0.0f, acc1 = 0.0f;
    const uint32_t sb = __half_as_ushort(sh);
    if constexpr (HwCvt<HG>::AVAILABLE) {
        // Formats the FP4 / FP6 conversion hardware knows (e2m1, e2m3, e3m2; e1m2 as the uniform low end of e2m3): the
        // quantizer's element function with the hardware round trip (exhaustively bit-exact, fpq_selftest_f16_flow of the
        // FPQ_HWCVT=1 build), 10 instructions per pair and candidate with the error term.  (Skipping the fp16 rounding of
        // x/s and the tie shift would save three of them, but values that the fp16 rounding carries across a midpoint change
        // the sums by 1e-5 relative -- measured -- which is outside the 2e-6 the scorer promises.)
        if (scale_bits_regular_hw<HG>(sb)) {
            const float s = __half2float(sh);
            const float rr = rcp_rn_normal(s) * HwCvt<HG>::PRE;
            const uint64_t r2 = pk(rr, rr);
            const uint32_t sh2 = dup_h(__float2half_rn(s * (1.0f / HwCvt<HG>::PRE)));
#pragma unroll
            for (int i = 0; i < 16; ++i) sq_err_pair(p[i], sym_pair_h16_hw<HG>(xf[i], r2, sh2, delta), acc0, acc1);
            return acc0 + acc1;
        }
    } else {
        if (scale_bits_regular(sb)) {
            const float s = __half2float(sh);
            const float r = rcp_rn_normal(s);
            const uint64_t r2 = pk(r, r), s2 = pk(s, s);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const uint32_t v2 = pack_h2_u64(fmul2(xf[i], r2));                            // half(x/s)
                const uint64_t q = round_pair_magic(fhadd(uint16_t(v2 & 0xffffu), delta), fhadd(uint16_t(v2 >> 16), delta), Magic<HG>::EM, Magic<HG>::SC);
                sq_err_pair(p[i], pack_h2_u64(fmul2(q, s2)), acc0, acc1);
            }
            return acc0 + acc1;
        }
    }
    {
        // irregular scale (zero / subnormal / inf / NaN): the literal reference sequence, element by element FROM MEMORY (indexing
        // the register tile with a loop counter would push it into local memory for the whole kernel)
        const float s = rnd_in<__half>(__fdiv_rn(a, HG::VMAX));
        const GridTable& gt = c_grids[SymFmt<FMT>::GT];
#pragma unroll 1
        for (int k = 0; k < 32; ++k) {
            const float f = __half2float(src[((k >> 3) * 4 + lig) * 8 + (k & 7)]);
            const float d = f - rnd_in<__half>(quant_elem_literal<__half, TIE_KERNEL>(f, s, gt) * s);
            acc0 = fmaf(d, d, acc0);
        }
    }
    return acc0 + acc1;
}

template <int SPLIT>
__device__ __forceinline__ float sse_split_h16(const uint32_t (&p)[16], const uint64_t (&xf)[16], uint32_t pbits, uint32_t nbits, float delta, const __half* src, int lig) {
    using SF = SplitFmt<SPLIT>;
    const float an = h2f(uint16_t(nbits)), ap = h2f(uint16_t(pbits));
    const __half snh = scale_from_absmax_h16<typename SF::NEG>(an), sph = scale_from_absmax_h16<typename SF::POS>(ap);
    const bool fast = (scale_bits_regular(__half_as_ushort(snh)) || nbits == 0u) && (scale_bits_regular(__half_as_ushort(sph)) || pbits == 0u);
    float acc0 = 0.0f, acc1 = 0.0f;
    if (fast) {
        const float sn = __half2float(snh), sp = __half2float(sph);
        const SplitK k = make_splitk<typename SF::NEG, typename SF::POS>(sn, nbits == 0u ? 0.0f : rcp_rn_normal(sn), sp, pbits == 0u ? 0.0f : rcp_rn_normal(sp));
#pragma unroll
        for (int i = 0; i < 16; ++i) sq_err_pair(p[i], split_pair_h16_w<typename SF::NEG, typename SF::POS>(xf[i], p[i], k, delta), acc0, acc1);
    } else {
        const float sn = rnd_in<__half>(__fdiv_rn(an, SF::NEG::VMAX)), sp = rnd_in<__half>(__fdiv_rn(ap, SF::POS::VMAX));
        auto lit = [&](float xv) {
            const float xn = (xv <= 0.0f) ? xv : 0.0f, xp = (xv > 0.0f) ? xv : 0.0f;
            const float qn = scan_kernel_rule(rnd_in<__half>(__fdiv_rn(xn, sn)), c_grids[SF::GT_N].v, c_grids[SF::GT_N].k);
            const float qp = scan_kernel_rule(rnd_in<__half>(__fdiv_rn(xp, sp)), c_grids[SF::GT_P].v, c_grids[SF::GT_P].k);
            return rnd_in<__half>(__fadd_rn(__fmul_rn(qn, sn), __fmul_rn(qp, sp)));
        };
#pragma unroll 1
        for (int k = 0; k < 32; ++k) {
            const float f = __half2float(src[((k >> 3) * 4 + lig) * 8 + (k & 7)]);
            const float d = f - lit(f);
            acc0 = fmaf(d, d, acc0);
        }
    }
    return acc0 + acc1;
}

__global__ void __launch_bounds__(256) score_formats_h16_kernel(const __half* __restrict__ x, size_t n_groups, Candidates cand, double* __restrict__ sse) {
    constexpr int LPG = 4, GPW = 8;
    __shared__ double s_acc[MAX_CAND];
    if (threadIdx.x < MAX_CAND) s_acc[threadIdx.x] = 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int lig = lane % LPG;
    const size_t warp_global = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    const float delta = tie_delta_kernel(uint32_t(warp_global >> 33));
    for (size_t gbase = warp_global * GPW; gbase < n_groups; gbase += n_warps * GPW) {
        const size_t g = gbase + lane / LPG;
        uint32_t p[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint4 u = make_uint4(0u, 0u, 0u, 0u);
            if (g < n_groups) u = ldg_stream(x + g * 128 + (j * LPG + lig) * 8);
            p[4 * j] = u.x; p[4 * j + 1] = u.y; p[4 * j + 2] = u.z; p[4 * j + 3] = u.w;
        }
        // the three group maxima as fp16 bit patterns (NaN patterns are extreme in every order)
        uint32_t am = 0u, pm = 0u, nm = 0u;
#pragma unroll
        for (int i = 0; i < 16; ++i) { am = __vmaxu2(am, p[i] & 0x7FFF7FFFu); pm = __vmaxs2(pm, p[i]); nm = __vmaxu2(nm, p[i]); }
        uint32_t amax = max(am & 0xffffu, am >> 16), nmax = max(nm & 0xffffu, nm >> 16);
        int pmax = max(int(short(pm & 0xffffu)), int(short(pm >> 16)));
#pragma unroll
        for (int o = LPG / 2; o > 0; o >>= 1) {
            amax = max(amax, __shfl_xor_sync(0xffffffffu, amax, o));
            nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o));
            pmax = max(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
        }
        uint32_t pbits = uint32_t(pmax), nbits = nmax >= 0x8000u ? (nmax & 0x7fffu) : 0u;
        if (amax > 0x7C00u) {
            // a NaN in the group: where() turns it into 0 on both sides of a sign-split format; redo those two maxima
            float an = 0.0f, ap = 0.0f;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&p[i]));
                an = fmaxf(an, fmaxf((f.x <= 0.0f) ? -f.x : 0.0f, (f.y <= 0.0f) ? -f.y : 0.0f));
                ap = fmaxf(ap, fmaxf((f.x > 0.0f) ? f.x : 0.0f, (f.y > 0.0f) ? f.y : 0.0f));
            }
            nbits = f2h(group_max<LPG>(an));
            pbits = f2h(group_max<LPG>(ap));
        }
        uint64_t xf[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) xf[i] = widen_h2(p[i]);
        const bool live = g < n_groups;
        const __half* src = x + (live ? g : 0) * 128;                // the literal fallbacks read the group from memory; a dead lane set's result is dropped
#pragma unroll 1
        for (int c = 0; c < cand.n; ++c) {
            float e;
            switch (cand.fmt[c]) {
                case FPQ_FMT_E2M1: e = sse_sym_h16<FPQ_FMT_E2M1>(p, xf, amax, delta, src, lig); break;
                case FPQ_FMT_E1M2: e = sse_sym_h16<FPQ_FMT_E1M2>(p, xf, amax, delta, src, lig); break;
                case FPQ_FMT_E3M0: e = sse_sym_h16<FPQ_FMT_E3M0>(p, xf, amax, delta, src, lig); break;
                case FPQ_FMT_E2M3: e = sse_sym_h16<FPQ_FMT_E2M3>(p, xf, amax, delta, src, lig); break;
                case FPQ_FMT_E3M2: e = sse_sym_h16<FPQ_FMT_E3M2>(p, xf, amax, delta, src, lig); break;
                case 16 + FPQ_SPLIT_E1M2NEG_E2M1POS: e = sse_split_h16<FPQ_SPLIT_E1M2NEG_E2M1POS>(p, xf, pbits, nbits, delta, src, lig); break;
                case 16 + FPQ_SPLIT_INTNEG_E2M3POS: e = sse_split_h16<FPQ_SPLIT_INTNEG_E2M3POS>(p, xf, pbits, nbits, delta, src, lig); break;
                default: e = sse_split_h16<FPQ_SPLIT_AFPQ_E2M1>(p, xf, pbits, nbits, delta, src, lig); break;
            }
            if (!live) e = 0.0f;
            // 32 lanes x 32 elements in fp32, then one fp64 add per warp, trip and candidate
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
            if (lane == 0) atomicAdd(&s_acc[c], double(e));
        }
    }
    __syncthreads();
    if (threadIdx.x < cand.n) atomicAdd(&sse[threadIdx.x], s_acc[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------
// Output-level loss of the search (search_fp4_format.py:472-476 `compute_quant_error(y_fp, y_q)` inside the loop :798-816):
//     out += sum_r w[r] * sum_c (a[r, c] - b[r, c])^2
// in ONE read of the two matrices: no difference tensor, no squared tensor, no per-row partial tensor (the ATen sequence
// sub_ -> float -> square_ -> sum(dim=1) -> dot moves the [rows, C_out] matrix through HBM nine times).  w[r] carries
// the 1 / (rows_j * C_out * J) of the per-tensor means when the calibration set is row-stacked (search_layer_batched);
// NULL = 1.  One warp per row slice, 128-bit loads, fp32 within a lane's 8..16 products, fp64 from there on.
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) sse_rows_kernel(const T* __restrict__ a, const T* __restrict__ b, size_t n_rows, size_t n_cols,
                                                       const double* __restrict__ w, double* __restrict__ out) {
    constexpr int VEC = 16 / sizeof(T);
    __shared__ double s_acc;
    if (threadIdx.x == 0) s_acc = 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const size_t warp_global = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    const size_t vecs_per_row = n_cols / VEC;
    double acc = 0.0;
    for (size_t r = warp_global; r < n_rows; r += n_warps) {
        const T* ar = a + r * n_cols;
        const T* br = b + r * n_cols;
        double row = 0.0;
        for (size_t v0 = 0; v0 < vecs_per_row; v0 += 64) {             // two independent 128-bit loads per lane and matrix in flight
            float part = 0.0f;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const size_t v = v0 + size_t(k) * 32 + lane;
                if (v < vecs_per_row) {
                    const uint4 ua = ldg_stream(ar + v * VEC), ub = ldg_stream(br + v * VEC);
                    if constexpr (sizeof(T) == 2) {
                        const uint32_t wa[4] = {ua.x, ua.y, ua.z, ua.w}, wb[4] = {ub.x, ub.y, ub.z, ub.w};
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float2 fa = __half22float2(*reinterpret_cast<const __half2*>(&wa[i]));
                            const float2 fb = __half22float2(*reinterpret_cast<const __half2*>(&wb[i]));
                            const float d0 = fa.x - fb.x, d1 = fa.y - fb.y;
                            part = fmaf(d0, d0, part);
                            part = fmaf(d1, d1, part);
                        }
                    } else {
                        const float fa[4] = {__uint_as_float(ua.x), __uint_as_float(ua.y), __uint_as_float(ua.z), __uint_as_float(ua.w)};
                        const float fb[4] = {__uint_as_float(ub.x), __uint_as_float(ub.y), __uint_as_float(ub.z), __uint_as_float(ub.w)};
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float d = fa[i] - fb[i];
                            part = fmaf(d, d, part);
                        }
                    }
                }
            }
            row += double(part);
        }
        acc += row * (w != nullptr ? w[r] : 1.0);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) atomicAdd(&s_acc, acc);
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(out, s_acc);
}

}  // namespace fpq

using namespace fpq;

extern "C" int fpq_sse_rows(const void* a, const void* b, size_t n_rows, size_t n_cols, int dtype, const double* row_weight, double* out, void* stream) {
    if (!out || (n_rows && n_cols && (!a || !b))) return FPQ_ERR_ARG;
    if (dtype != FPQ_F32 && dtype != FPQ_F16) return FPQ_ERR_ARG;
    const size_t vec = dtype == FPQ_F16 ? 8 : 4;
    if (n_cols % vec) return FPQ_ERR_UNSUPPORTED;                  // whole 16-byte vectors per row (every C_out of the search is a multiple of 128)
    if ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) return FPQ_ERR_ARG;
    if (n_rows == 0 || n_cols == 0) return FPQ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned grid = grid_for(n_rows, 8, 8);
    if (dtype == FPQ_F16) sse_rows_kernel<__half><<<grid, 256, 0, st>>>(static_cast<const __half*>(a), static_cast<const __half*>(b), n_rows, n_cols, row_weight, out);
    else sse_rows_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(a), static_cast<const float*>(b), n_rows, n_cols, row_weight, out);
    return finish_launch();
}

extern "C" int fpq_score_formats(const void* x, size_t n_rows, size_t row_len, int in_dtype, const int* formats_host, int n_formats,
                                 int tie_mode, double* sse, void* stream) {
    if (!formats_host || n_formats < 1 || n_formats > MAX_CAND || !sse || (n_rows && !x)) return FPQ_ERR_ARG;
    if (row_len != 128) return FPQ_ERR_UNSUPPORTED;       // the search scripts use group_size 128 throughout
    if (reinterpret_cast<uintptr_t>(x) & 15) return FPQ_ERR_ARG;
    Candidates cand;
    cand.n = n_formats;
    for (int i = 0; i < MAX_CAND; ++i) cand.fmt[i] = 0;
    for (int i = 0; i < n_formats; ++i) {
        const int f = formats_host[i];
        const bool ok = (f >= 0 && f < FPQ_NUM_SYM_FORMATS) || (f >= 16 && f < 16 + FPQ_NUM_SPLIT_FORMATS);
        if (!ok) return FPQ_ERR_ARG;
        cand.fmt[i] = f;
    }
    if (n_rows == 0) return FPQ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned grid = grid_for(n_rows, 32, 8);
    if (in_dtype == FPQ_F32 && tie_mode == FPQ_TIE_KERNEL) score_formats_kernel<float, TIE_KERNEL><<<grid, 256, 0, st>>>(static_cast<const float*>(x), n_rows, cand, sse);
    else if (in_dtype == FPQ_F32 && tie_mode == FPQ_TIE_ARGMIN) score_formats_kernel<float, TIE_ARGMIN><<<grid, 256, 0, st>>>(static_cast<const float*>(x), n_rows, cand, sse);
    else if (in_dtype == FPQ_F16 && tie_mode == FPQ_TIE_KERNEL)
        score_formats_h16_kernel<<<grid_for(n_rows, 64, 4), 256, 0, st>>>(static_cast<const __half*>(x), n_rows, cand, sse);
    else if (in_dtype == FPQ_F16 && tie_mode == FPQ_TIE_ARGMIN) score_formats_kernel<__half, TIE_ARGMIN><<<grid, 256, 0, st>>>(static_cast<const __half*>(x), n_rows, cand, sse);
    else return FPQ_ERR_ARG;
    return finish_launch();
}
