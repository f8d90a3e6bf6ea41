// Shared device helpers of libfpq_b200 (constant grid tables, streaming loads/stores, the
// 16-elements-per-lane register tile, group reductions, launch bookkeeping) and the format
// traits and run-time format / dtype dispatchers of every launcher.
//
// Thread mapping of the group kernels: a group of GS contiguous elements is owned by
// LPG = GS/16 adjacent lanes; lane l holds 16 elements as 16-byte vectors, vector j of lane l
// covering elements [j*VEC*LPG + l*VEC, +VEC).  One warp-wide 128-bit load therefore touches
// 32/LPG groups x (16*LPG) contiguous bytes: whole 128-byte lines for the reference's GS=128.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>
#include <math.h>
#include <type_traits>

#include "../../include/fpq_b200.h"
#include "fpq_round.cuh"

namespace fpq {

// ------------------------------------------------------------------------------------------
// constant tables: the reference's grids spelled out (one private copy per translation unit)
// ------------------------------------------------------------------------------------------
#define E2M1_POS_ 0.5f, 1.0f, 1.5f, 2.0f, 3.0f, 4.0f, 6.0f
#define E2M1_NEG_ -6.0f, -4.0f, -3.0f, -2.0f, -1.5f, -1.0f, -0.5f
#define E1M2_POS_ 0.25f, 0.5f, 0.75f, 1.0f, 1.25f, 1.5f, 1.75f
#define E1M2_NEG_ -1.75f, -1.5f, -1.25f, -1.0f, -0.75f, -0.5f, -0.25f
#define E3M0_POS_ 0.25f, 0.5f, 1.0f, 2.0f, 4.0f, 8.0f, 16.0f
#define E3M0_NEG_ -16.0f, -8.0f, -4.0f, -2.0f, -1.0f, -0.5f, -0.25f
#define E2M3_POS_ 0.125f, 0.25f, 0.375f, 0.5f, 0.625f, 0.75f, 0.875f, 1.0f, 1.125f, 1.25f, 1.375f, 1.5f, 1.625f, 1.75f, 1.875f, \
                  2.0f, 2.25f, 2.5f, 2.75f, 3.0f, 3.25f, 3.5f, 3.75f, 4.0f, 4.5f, 5.0f, 5.5f, 6.0f, 6.5f, 7.0f, 7.5f
#define E2M3_NEG_ -7.5f, -7.0f, -6.5f, -6.0f, -5.5f, -5.0f, -4.5f, -4.0f, -3.75f, -3.5f, -3.25f, -3.0f, -2.75f, -2.5f, -2.25f, -2.0f, \
                  -1.875f, -1.75f, -1.625f, -1.5f, -1.375f, -1.25f, -1.125f, -1.0f, -0.875f, -0.75f, -0.625f, -0.5f, -0.375f, -0.25f, -0.125f
#define E3M2_POS_ 0.0625f, 0.125f, 0.1875f, 0.25f, 0.3125f, 0.375f, 0.4375f, 0.5f, 0.625f, 0.75f, 0.875f, 1.0f, 1.25f, 1.5f, 1.75f, \
                  2.0f, 2.5f, 3.0f, 3.5f, 4.0f, 5.0f, 6.0f, 7.0f, 8.0f, 10.0f, 12.0f, 14.0f, 16.0f, 20.0f, 24.0f, 28.0f
#define E3M2_NEG_ -28.0f, -24.0f, -20.0f, -16.0f, -14.0f, -12.0f, -10.0f, -8.0f, -7.0f, -6.0f, -5.0f, -4.0f, -3.5f, -3.0f, -2.5f, -2.0f, \
                  -1.75f, -1.5f, -1.25f, -1.0f, -0.875f, -0.75f, -0.625f, -0.5f, -0.4375f, -0.375f, -0.3125f, -0.25f, -0.1875f, -0.125f, -0.0625f
#define INT_NEG_ -32.f, -31.f, -30.f, -29.f, -28.f, -27.f, -26.f, -25.f, -24.f, -23.f, -22.f, -21.f, -20.f, -19.f, -18.f, -17.f, \
                 -16.f, -15.f, -14.f, -13.f, -12.f, -11.f, -10.f, -9.f, -8.f, -7.f, -6.f, -5.f, -4.f, -3.f, -2.f, -1.f

static __constant__ GridTable c_grids[GT_COUNT] = {
    {15, {E2M1_NEG_, 0.0f, E2M1_POS_}},
    {15, {E1M2_NEG_, 0.0f, E1M2_POS_}},
    {15, {E3M0_NEG_, 0.0f, E3M0_POS_}},
    {64, {E2M3_NEG_, 0.0f, 0.0f, E2M3_POS_}},
    {64, {E3M2_NEG_, 0.0f, 0.0f, E3M2_POS_}},
    {33, {INT_NEG_, 0.0f}},
    {32, {0.0f, E2M3_POS_}},
    {8, {E1M2_NEG_, 0.0f}},
    {8, {0.0f, E2M1_POS_}},
    {8, {E2M1_NEG_, 0.0f}},
};


// launch bookkeeping (defined in fpq_grid.cu)
int finish_launch();
int sm_count();
// Launch-geometry choices that were made from measurements and that the measurement tools (tools/rowbench.py,
// tools/abbench.py) and the GPU tests move at run time through fpq_set_tunable() -- not through the environment.
struct Tunables {
    int pdl = 1;                               // programmatic dependent launch on (0: plain stream-ordered launches)
    int row_v = 0;                             // values-per-thread of the per-token kernels: 0 = chosen by row_reg_vectors, else 1 | 2 | 4
    long long rot_small_max_chunks = 40000;    // rotate launches up to this many 128-chunks take the small-launch kernel (measured: VAR-d30 stage 4, 37 500 chunks, 9.95 vs 11.0 us)
    int smem_kb = 0;                           // shared-memory carveout (KB per SM) every activation kernel asks for; 0 = leave it to the driver
    int gemm_stages = 6;                       // shared-memory ring depth of the low-bit GEMM (2..6 stages of 32 KB, 2..4 of 48 KB with 256-column tiles)
    int gemm_pair = -1;                        // CTA pairs with cta_group::2 MMAs (default tile shape only): 1 on | 0 off | -1 (default) on for row scales and >= 4 row tiles
    int gemm_tile_n = 256;                     // C tile columns of the low-bit GEMM: 128 | 256
    int gemm_epi_cols = 128;                   // columns per epilogue warp: 32 (128-column tiles only) | 64 | 128; fewer = more epilogue warps per scheduler (measured: no faster)
};
extern Tunables g_tun;
// symmetric fake quant, one translation unit per tie rule (fpq_sym_k.cu / fpq_sym_a.cu)
int fake_quant_kernel_tie(int in_dtype, int out_dtype, int format, const void* x, void* out, size_t n_rows, size_t row_len, int clamp3, cudaStream_t st);
int fake_quant_argmin_tie(int in_dtype, int out_dtype, int format, const void* x, void* out, size_t n_rows, size_t row_len, int clamp3, cudaStream_t st);
int signsplit_kernel_tie(int in_dtype, int out_dtype, int split, const void* x, void* out, size_t n_rows, size_t row_len, unsigned* flag, cudaStream_t st);
int signsplit_argmin_tie(int in_dtype, int out_dtype, int split, const void* x, void* out, size_t n_rows, size_t row_len, unsigned* flag, cudaStream_t st);
// packed fp16 -> fp16 group-of-128 kernels, kernel tie rule (fpq_h16.cu)
int launch_sym_h16(int format, const void* x, void* out, size_t n_groups, cudaStream_t st);
int launch_sym_h16_g64(int format, const void* x, void* out, size_t n_groups, cudaStream_t st);   // groups / rows of 64 (KV cache)
int launch_split_h16(int split, const void* x, void* out, size_t n_groups, unsigned* nan_flag, cudaStream_t st);
static inline unsigned grid_for(size_t work_items, size_t items_per_block, int blocks_per_sm) {
    size_t need = (work_items + items_per_block - 1) / items_per_block;
    size_t cap = size_t(sm_count()) * blocks_per_sm;
    if (need < 1) need = 1;
    return unsigned(need < cap ? need : cap);
}

// Row-per-CTA persistent kernels (per_token / per_channel): how many values each thread keeps of its row (V uint4
// vectors) and how many CTAs are REALLY resident per SM.  The grid must not exceed the resident CTAs: a persistent
// CTA that only starts when another one has finished all of its rows runs a second, half-empty wave.
// The tunable row_v = 1|2|4 overrides the choice (measurement aid).
static inline int row_reg_vectors(size_t row_vecs, bool heavy_loop) {
    // Measured with tools/rowbench.py (profiles/r1_rowbench.txt).  Sign-split (heavy_loop): the smallest CTA wins at every
    // row length (V = 1 / 2 / 4 at 0.6 / 0.8 / 1.0), weighed against the lanes the last warp wastes.  Symmetric: CTAs of
    // 128-288 threads win (rows of 1920: V=2, 7680 / 9216: V=4); larger V on ties.
    int v = 1;
    float best = 0.0f;
    for (int c = 1; c <= 4; c *= 2) {
        const size_t thr = (row_vecs + c - 1) / c;
        if (thr > 1024) continue;
        const float padded = float((thr + 31) / 32 * 32);
        float score = float(thr) / padded;
        if (heavy_loop) score *= (c == 1 ? 0.6f : c == 2 ? 0.8f : 1.0f);
        else score /= 1.0f + fabsf(log2f(padded / 181.0f));
        if (score >= best) { best = score; v = c; }
    }
    if (const int f = g_tun.row_v; (f == 1 || f == 2 || f == 4) && (row_vecs + f - 1) / f <= 1024) v = f;
    while ((row_vecs + v - 1) / v > 1024) v *= 2;
    return v;
}
template <typename KernelT>
static inline unsigned resident_row_grid(KernelT kernel, int threads, size_t n_rows, int* cache) {
    int per_sm = cache[threads / 32];
    if (per_sm == 0) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
        cache[threads / 32] = per_sm;
    }
    const size_t cap = size_t(sm_count()) * per_sm;
    return unsigned(n_rows < cap ? n_rows : cap);
}
// Launches a row-in-registers kernel (x, out, n_rows, row_vecs, last) on rows the caller has found eligible;
// kernel_for(std::integral_constant<int, V>{}) returns the kernel for V = 1 | 2 | 4.  The occupancy cache is a static of
// this template, so it stays per kernel family as long as each caller instantiation passes its own lambda type: residency
// depends on each kernel's registers.
template <typename KernelFor, typename InT, typename OutT, typename Last>
static inline void launch_row_reg(KernelFor kernel_for, bool heavy_loop, const InT* x, OutT* out, size_t n_rows, size_t row_len, Last last,
                                  cudaStream_t st) {
    const size_t row_vecs = row_len / (16 / sizeof(InT));
    const int v = row_reg_vectors(row_vecs, heavy_loop);
    int threads = int((row_vecs + v - 1) / v);
    threads = (threads + 31) / 32 * 32;
    static int occ[3][33];                            // resident CTAs per SM, per (V, threads / 32); 0 = not asked yet
    auto launch = [&](auto vc, int* cache) {
        const auto k = kernel_for(vc);
        k<<<resident_row_grid(k, threads, n_rows, cache), threads, 0, st>>>(x, out, n_rows, int(row_vecs), last);
    };
    if (v == 1) launch(std::integral_constant<int, 1>{}, occ[0]);
    else if (v == 2) launch(std::integral_constant<int, 2>{}, occ[1]);
    else launch(std::integral_constant<int, 4>{}, occ[2]);
}

// ------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL).  The activation kernels are short (2-130 us) and a VAR pass
// issues 1200 of them back to back; a kernel launched with the programmatic-serialization attribute may
// have its CTAs scheduled while the previous kernel in the stream is still draining, and runs its
// prologue (index math, shared-memory tables built from PARAMETER tensors) until pdl_wait(), which
// returns once the previous kernel has completed and its writes are visible.  Nothing that a previous
// kernel may have produced (x) is read, and nothing is written, before pdl_wait().
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }


// Every activation kernel asks for the SAME L1 / shared-memory split (tunable smem_kb): an SM only changes its split when
// it is idle, so kernels that alternate between two splits (rotate -> group -> rotate -> sign-split ... in a VAR pass)
// cannot overlap their tails and pay a drain per launch (measured: 28.1 ms instead of 24.7 ms per step when only the
// streaming rotate kernel asked for shared memory).  The split is a trade: the streaming rotate kernel keeps its bytes in
// flight in shared memory, the register-tile kernels keep theirs in L1 lines (a pending ld.global holds a line of the L1
// data array even with L1::no_allocate), so shrinking L1 to the minimum costs them a quarter of their bandwidth
// (6.4 -> 4.8 TB/s with the 228 KB carveout).  Set once per (kernel, device, value); defined in fpq_grid.cu.
void prefer_carveout(const void* kernel);

template <typename... KArgs, typename... Args>
static inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, unsigned block, size_t smem, cudaStream_t st, Args... args) {
    prefer_carveout(reinterpret_cast<const void*>(kernel));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_tun.pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float fmax_nan(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}

__device__ __forceinline__ uint4 ldg_stream(const void* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void stg_stream(void* p, uint4 v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void stg_stream(void* p, uint2 v) {
    asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" :: "l"(p), "r"(v.x), "r"(v.y) : "memory");
}

__device__ __forceinline__ float h2f(uint16_t b) { return __half2float(__ushort_as_half(b)); }
__device__ __forceinline__ uint16_t f2h(float f) { return __half_as_ushort(__float2half_rn(f)); }
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
    __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}

// 16 elements per lane, as floats, whatever the storage type
template <typename T> struct Vec16;
template <> struct Vec16<float> {
    static constexpr int NV = 4, VEC = 4;
    static __device__ __forceinline__ void load(const float* base, int lane_in_group, int lpg, float (&v)[16]) {
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            uint4 u = ldg_stream(base + (j * lpg + lane_in_group) * VEC);
            v[4 * j + 0] = __uint_as_float(u.x); v[4 * j + 1] = __uint_as_float(u.y);
            v[4 * j + 2] = __uint_as_float(u.z); v[4 * j + 3] = __uint_as_float(u.w);
        }
    }
    static __device__ __forceinline__ void store(float* base, int lane_in_group, int lpg, const float (&v)[16]) {
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            uint4 u = make_uint4(__float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]), __float_as_uint(v[4 * j + 3]));
            stg_stream(base + (j * lpg + lane_in_group) * VEC, u);
        }
    }
};
template <> struct Vec16<__half> {
    static constexpr int NV = 2, VEC = 8;
    static __device__ __forceinline__ void load(const __half* base, int lane_in_group, int lpg, float (&v)[16]) {
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            uint4 u = ldg_stream(base + (j * lpg + lane_in_group) * VEC);
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[k]));
                v[8 * j + 2 * k] = f.x; v[8 * j + 2 * k + 1] = f.y;
            }
        }
    }
    // element order of a lane's 16 values depends on the INPUT type's vector width; the
    // store helpers below take the input VEC so that in/out types may differ.
};

// store 16 per-lane values (laid out for an input type with IN_VEC elements per 16-byte vector)
template <typename OutT, int IN_VEC>
__device__ __forceinline__ void store16(OutT* base, int lane_in_group, int lpg, const float (&v)[16]) {
    constexpr int NV = 16 / IN_VEC;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        OutT* p = base + (j * lpg + lane_in_group) * IN_VEC;
        if constexpr (sizeof(OutT) == 4) {
#pragma unroll
            for (int k = 0; k < IN_VEC; k += 4) {
                uint4 u = make_uint4(__float_as_uint(v[IN_VEC * j + k]), __float_as_uint(v[IN_VEC * j + k + 1]),
                                     __float_as_uint(v[IN_VEC * j + k + 2]), __float_as_uint(v[IN_VEC * j + k + 3]));
                stg_stream(p + k, u);
            }
        } else {
            if constexpr (IN_VEC == 8) {
                uint4 u = make_uint4(pack_h2(v[8 * j], v[8 * j + 1]), pack_h2(v[8 * j + 2], v[8 * j + 3]),
                                     pack_h2(v[8 * j + 4], v[8 * j + 5]), pack_h2(v[8 * j + 6], v[8 * j + 7]));
                stg_stream(p, u);
            } else {
                uint2 u = make_uint2(pack_h2(v[4 * j], v[4 * j + 1]), pack_h2(v[4 * j + 2], v[4 * j + 3]));
                stg_stream(p, u);
            }
        }
    }
}

template <typename T> __device__ __forceinline__ float to_out(float f);
template <> __device__ __forceinline__ float to_out<float>(float f) { return f; }
template <> __device__ __forceinline__ float to_out<__half>(float f) { return f; }   // rounding happens in store16

// reference arithmetic "in the input dtype": round to fp16 when the tensor is fp16
template <typename InT> __device__ __forceinline__ float rnd_in(float f) {
    if constexpr (sizeof(InT) == 2) return __half2float(__float2half_rn(f));
    else return f;
}

template <int LPG>
__device__ __forceinline__ float group_max_nan(float a) {
#pragma unroll
    for (int o = LPG / 2; o > 0; o >>= 1) a = fmax_nan(a, __shfl_xor_sync(0xffffffffu, a, o));
    return a;
}
template <int LPG>
__device__ __forceinline__ float group_max(float a) {      // NaN-ignoring (inputs already sanitised)
#pragma unroll
    for (int o = LPG / 2; o > 0; o >>= 1) a = fmaxf(a, __shfl_xor_sync(0xffffffffu, a, o));
    return a;
}

// ------------------------------------------------------------------------------------------
// The quantizer formats: the half grid and grid table of each symmetric format, the negative and
// positive halves of each sign-split format, and the dispatchers that turn a run-time FPQ_FMT_* /
// FPQ_SPLIT_* / dtype code into a template argument.  f receives a std::integral_constant (read
// fmt.value) or a DType tag (read typename decltype(t)::type); a code outside the set is FPQ_ERR_ARG.
// ------------------------------------------------------------------------------------------
template <int FMT> struct SymFmt;
template <> struct SymFmt<FPQ_FMT_E2M1> { using HG = HG_E2M1; static constexpr int GT = GT_E2M1; };
template <> struct SymFmt<FPQ_FMT_E1M2> { using HG = HG_E1M2; static constexpr int GT = GT_E1M2; };
template <> struct SymFmt<FPQ_FMT_E3M0> { using HG = HG_E3M0; static constexpr int GT = GT_E3M0; };
template <> struct SymFmt<FPQ_FMT_E2M3> { using HG = HG_E2M3; static constexpr int GT = GT_E2M3; };
template <> struct SymFmt<FPQ_FMT_E3M2> { using HG = HG_E3M2; static constexpr int GT = GT_E3M2; };

template <int SPLIT> struct SplitFmt;
template <> struct SplitFmt<FPQ_SPLIT_E1M2NEG_E2M1POS> { using NEG = HG_E1M2; using POS = HG_E2M1; static constexpr int GT_N = GT_E1M2_NEG, GT_P = GT_E2M1_POS; };
template <> struct SplitFmt<FPQ_SPLIT_INTNEG_E2M3POS> { using NEG = HG_INT32; using POS = HG_E2M3; static constexpr int GT_N = GT_INT_NEG, GT_P = GT_E2M3_POS; };
template <> struct SplitFmt<FPQ_SPLIT_AFPQ_E2M1> { using NEG = HG_E2M1; using POS = HG_E2M1; static constexpr int GT_N = GT_E2M1_NEG, GT_P = GT_E2M1_POS; };

template <typename F>
static inline int with_sym_format(int format, F&& f) {
    switch (format) {
        case FPQ_FMT_E2M1: return f(std::integral_constant<int, FPQ_FMT_E2M1>{});
        case FPQ_FMT_E1M2: return f(std::integral_constant<int, FPQ_FMT_E1M2>{});
        case FPQ_FMT_E3M0: return f(std::integral_constant<int, FPQ_FMT_E3M0>{});
        case FPQ_FMT_E2M3: return f(std::integral_constant<int, FPQ_FMT_E2M3>{});
        case FPQ_FMT_E3M2: return f(std::integral_constant<int, FPQ_FMT_E3M2>{});
        default: return FPQ_ERR_ARG;
    }
}

template <typename F>
static inline int with_split_format(int split, F&& f) {
    switch (split) {
        case FPQ_SPLIT_E1M2NEG_E2M1POS: return f(std::integral_constant<int, FPQ_SPLIT_E1M2NEG_E2M1POS>{});
        case FPQ_SPLIT_INTNEG_E2M3POS: return f(std::integral_constant<int, FPQ_SPLIT_INTNEG_E2M3POS>{});
        case FPQ_SPLIT_AFPQ_E2M1: return f(std::integral_constant<int, FPQ_SPLIT_AFPQ_E2M1>{});
        default: return FPQ_ERR_ARG;
    }
}

template <typename T> struct DType { using type = T; };
template <typename F>
static inline int with_dtypes(int in_dtype, int out_dtype, F&& f) {
    if (in_dtype == FPQ_F32 && out_dtype == FPQ_F32) return f(DType<float>{}, DType<float>{});
    if (in_dtype == FPQ_F32 && out_dtype == FPQ_F16) return f(DType<float>{}, DType<__half>{});
    if (in_dtype == FPQ_F16 && out_dtype == FPQ_F16) return f(DType<__half>{}, DType<__half>{});
    if (in_dtype == FPQ_F16 && out_dtype == FPQ_F32) return f(DType<__half>{}, DType<float>{});
    return FPQ_ERR_ARG;
}

// Is the scale "regular", i.e. may the reciprocal-multiply fast path be used?
//   fp32 tensors: 2^-100 <= s <= 2^100 (1/s and x*(1/s) stay normal)
//   fp16 tensors: s is a normal, finite fp16 number
template <typename InT> __device__ __forceinline__ bool scale_regular(float s) {
    if constexpr (sizeof(InT) == 2) return s >= 6.103515625e-05f && s <= 65504.0f;
    else return s >= 7.888609052210118e-31f && s <= 1.2676506002282294e30f;
}

// ------------------------------------------------------------------------------------------
// One element of the symmetric path, given the group's scale s (already rounded to the input
// dtype) and r = RN(1/s).
//
// fp16 tensors: the reference computes v = half(float(x)/float(s)).  For 11-bit operands
//   x*RN(1/s) is within 2^-23 (relative) of x/s, while a quotient of two 11-bit integers cannot sit
//   closer than 1/(2^11 * 2^12) (relative) to a 12-bit rounding boundary without being equal to it,
//   and it cannot be equal -- so half(x*r) == half(x/s) whenever the quotient is a NORMAL fp16
//   number.  Among subnormal quotients (|v| < 2^-14) x/s can be an exact tie (3*2^-24 / 6 = 2^-25)
//   and the two may round to neighbouring subnormals; both lie far below the first grid midpoint of
//   every format, so the grid value is the same.  fpq_selftest_f16_flow (fpq_h16.cu) compares the
//   final outputs of this path with the literal sequence for EVERY (x, scale) pair of fp16 values.
// fp32 tensors: v = x/s in fp32.  x*r is within 2 ulp of it; the closed-form rounding reports
//   when its argument is within 32 ulp of a decision boundary and only those elements pay for
//   an IEEE division.
// ------------------------------------------------------------------------------------------
template <typename InT, class HG, int TIE>
__device__ __forceinline__ float quant_elem_fast(float x, float s, float r) {
    if constexpr (sizeof(InT) == 2) {
        const float v = __half2float(__float2half_rn(x * r));
        return round_closed<HG, TIE, false>(v);
    } else {
        bool near;
        float q = round_closed_near<HG, TIE>(x * r, near);
        if (near) q = round_closed<HG, TIE, false>(__fdiv_rn(x, s));
        return q;
    }
}

// the literal reference sequence for one element (irregular groups only)
template <typename InT, int TIE>
__device__ __forceinline__ float quant_elem_literal(float x, float s, const GridTable& g) {
    const float v = rnd_in<InT>(__fdiv_rn(x, s));
    return scan_rule<TIE>(v, g.v, g.k);
}

__device__ __forceinline__ float clamp3_keep_nan(float x) { return x < -3.0f ? -3.0f : (x > 3.0f ? 3.0f : x); }

// ------------------------------------------------------------------------------------------
// Fake-quantize one group held in registers (16 values per lane, LPG lanes per group), in place:
// absmax -> scale -> round -> rescale.  Values are the INPUT-dtype values widened to fp32; the
// result is q*s in fp32 (the caller's store rounds it to the output dtype).
// ------------------------------------------------------------------------------------------
template <typename InT, int FMT, int TIE, int LPG>
__device__ __forceinline__ void sym_quant_tile(float (&v)[16]) {
    using HG = typename SymFmt<FMT>::HG;
    float a = 0.0f;
#pragma unroll
    for (int i = 0; i < 16; ++i) a = fmax_nan(a, fabsf(v[i]));
    a = group_max_nan<LPG>(a);
    const float s = rnd_in<InT>(__fdiv_rn(a, HG::VMAX));      // quant_utils.py:320
    if (scale_regular<InT>(s)) {
        const float r = __frcp_rn(s);
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = quant_elem_fast<InT, HG, TIE>(v[i], s, r) * s;
    } else {
        // zero, subnormal, huge, inf or NaN scale: follow the reference literally
        const GridTable& gt = c_grids[SymFmt<FMT>::GT];
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = quant_elem_literal<InT, TIE>(v[i], s, gt) * s;
    }
}


template <typename InT> __device__ __forceinline__ float load_elem(const InT* p) {
    if constexpr (sizeof(InT) == 2) return __half2float(*p); else return *p;
}
template <typename OutT> __device__ __forceinline__ void store_elem(OutT* p, float f) {
    if constexpr (sizeof(OutT) == 2) *p = __float2half_rn(f); else *p = f;
}

__device__ __forceinline__ float block_max_nan(float a, float* smem) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a = fmax_nan(a, __shfl_xor_sync(0xffffffffu, a, o));
    const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) smem[w] = a;
    __syncthreads();
    float r = smem[0];
    for (int i = 1; i < nw; ++i) r = fmax_nan(r, smem[i]);
    return r;
}

// (Measured and rejected: one-barrier reductions with parity-double-buffered scratch for the persistent row kernels ran
// 5-10 % SLOWER than the two-barrier form -- rows of 1920 / 7680 fp16, sym 5302 -> 5030, sign-split 4093 -> 3764 GB/s.)

}  // namespace fpq
