// libfpq_b200 -- packed fp16 -> fp16 kernels (kernel tie rule, groups of 128): the activation
// quantizers of the hot path (reference rows a2, a3 of SURVEY.md section 8) at low instruction
// count, see fpq_h16.cuh.  Part of the C ABI of include/fpq_b200.h; no torch types here.
#include "fpq_h16.cuh"

namespace fpq {

// Software pipelining (two register tiles in ping-pong).  Measured on B200 (tools/kbench.py, profiles/r1_kbench.txt, the
// "variant" sections): +3 % for the symmetric kernel (42 -> 70 registers), -8 % for the sign-split kernel (52 -> 84
// registers, occupancy drops to 3 CTAs), so only the former uses it.
// Occupancy of the sign-split kernel, measured (profiles/r1_kbench.txt, kbench_11): as compiled (56 registers, 4 CTAs/SM)
// 6.31 TB/s burst / 5.67 sustained; forced to 5 CTAs (48 registers, spills) 5.75 / 5.35; 6 CTAs (40 registers) 5.48 / 5.49;
// 2 CTAs (90 registers) 5.26 / 5.20.  Plain __launch_bounds__(256) it stays.
// lanes per 128-group.  Measured: 2 lanes x 64 halves is slower (sign-split 5.36 vs 6.40 TB/s burst, 5.30 vs 5.66 sustained;
// symmetric 5.59 vs 6.34): a warp-wide load then touches 16 groups x 32 bytes instead of 8 x 64.
constexpr int H16_LPG = 4;             // lanes per 128-group
constexpr int H16_NV = 16 / H16_LPG;   // 16-byte vectors per lane and group (4 lanes: 32 halves = 16 packed words per lane)
constexpr int H16_NW = 4 * H16_NV;
constexpr int H16_GPW = 32 / H16_LPG;   // groups per warp and loop trip

// vector j of lane l covers halves [(j*LPG + l)*8, +8) of the group: a warp-wide 128-bit load touches
// 8 groups x 64 contiguous bytes (whole 32-byte sectors; the other half of each 128-byte line follows
// with the next j)
__device__ __forceinline__ void load_tile_h16(const __half* base, int lig, uint32_t (&p)[H16_NW]) {
#pragma unroll
    for (int j = 0; j < H16_NV; ++j) {
        const uint4 u = ldg_stream(base + (j * H16_LPG + lig) * 8);
        p[4 * j] = u.x; p[4 * j + 1] = u.y; p[4 * j + 2] = u.z; p[4 * j + 3] = u.w;
    }
}
__device__ __forceinline__ void store_tile_h16(__half* base, int lig, const uint32_t (&p)[H16_NW]) {
#pragma unroll
    for (int j = 0; j < H16_NV; ++j) stg_stream(base + (j * H16_LPG + lig) * 8, make_uint4(p[4 * j], p[4 * j + 1], p[4 * j + 2], p[4 * j + 3]));
}

template <int FMT>
__global__ void __launch_bounds__(256) fake_quant_group_h16_kernel(const __half* __restrict__ x, __half* __restrict__ out, size_t n_groups) {
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31;
    const int lig = lane % H16_LPG;
    const size_t warp_global = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    const float delta = tie_delta_kernel(uint32_t(warp_global >> 33));
    const size_t stride = n_warps * H16_GPW;
    pdl_wait();
    auto load = [&](size_t gbase, uint32_t (&p)[H16_NW]) {
        const size_t g = gbase + lane / H16_LPG;
        if (g < n_groups) {
            load_tile_h16(x + g * 128, lig, p);
        } else {
#pragma unroll
            for (int i = 0; i < H16_NW; ++i) p[i] = 0u;
        }
    };
    auto work = [&](size_t gbase, uint32_t (&p)[H16_NW]) {
        const size_t g = gbase + lane / H16_LPG;
        float s;
        const bool ok = sym_quant_tile_h16<FMT, H16_LPG, H16_NW>(p, s, delta);
        if (g < n_groups) {
            if (ok) store_tile_h16(out + g * 128, lig, p);
            else literal_sym_h16(x + g * 128, out + g * 128, lig, H16_LPG, 8, H16_NV, s, SymFmt<FMT>::GT);
        }
    };
    // two register tiles in ping-pong: the loads of the next trip are in flight while this one computes
    uint32_t A[H16_NW], B[H16_NW];
    size_t g0 = warp_global * H16_GPW;
    if (g0 < n_groups) load(g0, A);
    for (; g0 < n_groups; g0 += 2 * stride) {
        const size_t g1 = g0 + stride, g2 = g1 + stride;
        if (g1 < n_groups) load(g1, B);
        work(g0, A);
        if (g2 < n_groups) load(g2, A);
        if (g1 < n_groups) work(g1, B);
    }
}

// ------------------------------------------------------------------------------------------
// Groups / rows of 64 (the KV cache: fp6_quant_e2m3_per_token_cuda on [B, L, H, 64], basic_var.py:193-194).
// Same packed element path; 4 lanes x 2 vectors x 8 halves per group, so a warp-wide 128-bit load still touches
// 8 groups x 64 contiguous bytes.  Two independent tiles per trip keep four loads in flight per lane.  (The generic
// kernel these rows used to take ran at 20.4 instructions per element, 81 % issue utilisation: profiles/r1e.)
// ------------------------------------------------------------------------------------------
template <int FMT>
__global__ void __launch_bounds__(256) fake_quant_group64_h16_kernel(const __half* __restrict__ x, __half* __restrict__ out, size_t n_groups) {
    constexpr int LPG = 4, NV = 2, NW = 4 * NV, GPW = 32 / LPG;
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31;
    const int lig = lane % LPG;
    const size_t warp_global = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    const float delta = tie_delta_kernel(uint32_t(warp_global >> 33));
    const size_t stride = n_warps * GPW;
    pdl_wait();
    auto load = [&](size_t g, uint32_t (&p)[NW]) {
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            uint4 u = make_uint4(0u, 0u, 0u, 0u);
            if (g < n_groups) u = ldg_stream(x + g * 64 + (j * LPG + lig) * 8);
            p[4 * j] = u.x; p[4 * j + 1] = u.y; p[4 * j + 2] = u.z; p[4 * j + 3] = u.w;
        }
    };
    auto finish = [&](size_t g, uint32_t (&p)[NW]) {
        float s;
        const bool ok = sym_quant_tile_h16<FMT, LPG, NW>(p, s, delta);
        if (g < n_groups) {
            if (ok) {
#pragma unroll
                for (int j = 0; j < NV; ++j)
                    stg_stream(out + g * 64 + (j * LPG + lig) * 8, make_uint4(p[4 * j], p[4 * j + 1], p[4 * j + 2], p[4 * j + 3]));
            } else {
                literal_sym_h16(x + g * 64, out + g * 64, lig, LPG, 8, NV, s, SymFmt<FMT>::GT);
            }
        }
    };
    for (size_t g0 = warp_global * GPW; g0 < n_groups; g0 += 2 * stride) {
        const size_t ga = g0 + lane / LPG, gb = ga + stride;
        uint32_t A[NW], B[NW];
        load(ga, A);
        load(gb, B);
        finish(ga, A);
        finish(gb, B);
    }
}

// ------------------------------------------------------------------------------------------
// Segments with a pitch, optionally IN PLACE (fpq_fake_quant_segments): the appended slice [B, lo:cur, H, head_dim] of a
// KV cache [B, L_max, H, head_dim] is B contiguous segments `pitch` elements apart.  blockIdx.y walks the segments; inside
// a segment the groups (GS = 64 or 128 halves) are contiguous.  No __restrict__ and plain (coherent) loads: out may be x,
// every element is read by the lane that later writes it, and nothing is read twice.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_plain(const void* p) {
    uint4 v;
    asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
template <int FMT, int GS>
__global__ void __launch_bounds__(256) fake_quant_segments_h16_kernel(const __half* x, __half* out, size_t groups_per_segment, size_t pitch_x,
                                                                      size_t pitch_out) {
    constexpr int LPG = 4, NV = GS / 32, NW = 4 * NV, GPW = 32 / LPG;
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31;
    const int lig = lane % LPG;
    const size_t warp_in_seg = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    const float delta = tie_delta_kernel(uint32_t(warp_in_seg >> 33));
    x += size_t(blockIdx.y) * pitch_x;
    out += size_t(blockIdx.y) * pitch_out;
    pdl_wait();
    for (size_t g0 = warp_in_seg * GPW; g0 < groups_per_segment; g0 += n_warps * GPW) {
        const size_t g = g0 + lane / LPG;
        const bool live = g < groups_per_segment;
        uint32_t p[NW];
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            uint4 u = make_uint4(0u, 0u, 0u, 0u);
            if (live) u = ldg_plain(x + g * GS + (j * LPG + lig) * 8);
            p[4 * j] = u.x; p[4 * j + 1] = u.y; p[4 * j + 2] = u.z; p[4 * j + 3] = u.w;
        }
        float s;
        const bool ok = sym_quant_tile_h16<FMT, LPG, NW>(p, s, delta);
        if (live) {
            if (ok) {
#pragma unroll
                for (int j = 0; j < NV; ++j) stg_stream(out + g * GS + (j * LPG + lig) * 8, make_uint4(p[4 * j], p[4 * j + 1], p[4 * j + 2], p[4 * j + 3]));
            } else {
                literal_sym_h16(x + g * GS, out + g * GS, lig, LPG, 8, NV, s, SymFmt<FMT>::GT);      // element-wise: safe in place
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// sign-split
// ------------------------------------------------------------------------------------------
// Group maxima by integer order of the fp16 bit patterns (two elements per VIMNMX):
//   signed 16-bit max   -> the largest positive value (bits < 0x8000 order like the values)
//   unsigned 16-bit max -> 0x8000 | largest negative magnitude, if any element is negative
// NaN patterns are the extreme of either order, so they surface in the result.
// returns 0: handled; 1: irregular scale (sn, sp valid) -> literal_split_h16; 2: the group holds a NaN
// -> literal_split_nan_group_h16
template <int SPLIT, int LPG, int NW>
__device__ __forceinline__ int split_quant_tile_h16(uint32_t (&p)[NW], float& sn, float& sp, float delta) {
    using SF = SplitFmt<SPLIT>;
    uint32_t pm = 0u, nm = 0u;
#pragma unroll
    for (int i = 0; i < NW; ++i) { pm = __vmaxs2(pm, p[i]); nm = __vmaxu2(nm, p[i]); }
    int pmax = max(int(short(pm & 0xffffu)), int(short(pm >> 16)));          // >= 0
    uint32_t nmax = max(nm & 0xffffu, nm >> 16);
#pragma unroll
    for (int o = LPG / 2; o > 0; o >>= 1) {
        pmax = max(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
        nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o));
    }
    const uint32_t pbits = uint32_t(pmax);
    const uint32_t nbits = nmax >= 0x8000u ? (nmax & 0x7fffu) : 0u;
    if (pbits > 0x7C00u || nbits > 0x7C00u) return 2;
    const float an = h2f(uint16_t(nbits)), ap = h2f(uint16_t(pbits));
    const __half snh = scale_from_absmax_h16<typename SF::NEG>(an);           // quant_utils.py:432
    const __half sph = scale_from_absmax_h16<typename SF::POS>(ap);           // quant_utils.py:433
    sn = __half2float(snh);
    sp = __half2float(sph);
    // a side without elements has absmax 0 and scale 0 exactly (nbits / pbits == 0)
    const uint32_t snb = __half_as_ushort(snh), spb = __half_as_ushort(sph);
    if (!((scale_bits_regular(snb) || nbits == 0u) && (scale_bits_regular(spb) || pbits == 0u))) {
        sn = rnd_in<__half>(__fdiv_rn(an, SF::NEG::VMAX));                    // literal scales for the literal path
        sp = rnd_in<__half>(__fdiv_rn(ap, SF::POS::VMAX));
        return 1;
    }
    const SplitK k = make_splitk<typename SF::NEG, typename SF::POS>(sn, nbits == 0u ? 0.0f : rcp_rn_normal(sn), sp, pbits == 0u ? 0.0f : rcp_rn_normal(sp));
#pragma unroll
    for (int i = 0; i < NW; ++i) p[i] = split_pair_h16<typename SF::NEG, typename SF::POS>(p[i], k, delta);
    return 0;
}

// Whole-tensor clip of the reference (qu.py:421-422) when the tensor holds a NaN: every output becomes +0.
// workspace = {flag, ticket}, zero between calls.  The common path must not wait for anything: a CTA whose stores are
// issued fences them and bumps the ticket with a fire-and-forget wrapping increment (atomicInc modulo the grid size: after
// gridDim.x increments the ticket is 0 again by itself -- no reset, no memset between calls, and no CTA ever waits for the
// value).  The rare path: the ONE thread whose atomicOr turned the flag from 0 to 1 makes its CTA the owner of the
// rewrite; the owner waits until every other CTA has bumped the ticket (they are all resident or done: the grid calls
// launch_dependents first thing, and a single spinning CTA cannot starve the others), rewrites `out`, clears the flag and
// bumps the ticket last.  (Round 1 had every CTA take a RETURNING ticket and the last one look at the flag: one more
// atomic round trip and a second barrier at the end of every CTA, ~2 us on the launch-bound early stages.)
__device__ __forceinline__ void poison_epilogue(__half* out, size_t n, unsigned* ws, bool owner) {
    const int own = __syncthreads_or(owner ? 1 : 0);            // also: every warp of the CTA has issued its stores
    if (!own) {
        if (threadIdx.x == 0)               // release: this CTA's stores (made visible to this thread by the barrier) before the ticket
            asm volatile("red.release.gpu.global.inc.u32 [%0], %1;" ::"l"(ws + 1), "r"(gridDim.x - 1) : "memory");
        return;
    }
    if (threadIdx.x == 0) {
        while (*reinterpret_cast<volatile unsigned*>(ws + 1) != gridDim.x - 1) {}
        __threadfence();
    }
    __syncthreads();
    for (size_t i = threadIdx.x; i < n / 8; i += blockDim.x) reinterpret_cast<uint4*>(out)[i] = make_uint4(0u, 0u, 0u, 0u);
    for (size_t i = (n / 8) * 8 + threadIdx.x; i < n; i += blockDim.x) out[i] = __ushort_as_half(0);
    __syncthreads();
    if (threadIdx.x == 0) {
        ws[0] = 0u;
        __threadfence();
        atomicInc(ws + 1, gridDim.x - 1);
    }
}

// GELU(tanh) of an fp16 value the way ATen's CUDA kernel computes it for a Half tensor (ActivationGeluKernel.cu,
// GeluCUDAKernelImpl, approximate = "tanh": opmath float, the constants below, libdevice tanhf, one rounding to fp16 at the
// end) -- what `self.act(self.fc1(x))` produces under the reference's fp16 autocast (basic_var.py:108,120).  The expression
// is written like ATen's so that nvcc contracts it the same way; fpq_selftest_gelu compares it with a tensor of torch's own
// outputs for all 65 536 fp16 inputs.
__device__ __forceinline__ float gelu_tanh_f32(float x) {
    constexpr float kBeta = float(1.4142135623730951 * 1.1283791670955126 * 0.5);     // M_SQRT2 * M_2_SQRTPI * 0.5
    constexpr float kKappa = 0.044715f;
    const float x_cube = x * x * x;
    const float inner = kBeta * (x + kKappa * x_cube);
    return 0.5f * x * (1.0f + tanhf(inner));
}
__device__ __forceinline__ uint32_t gelu_tanh_h2(uint32_t x2) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&x2));
    return pack_h2(gelu_tanh_f32(f.x), gelu_tanh_f32(f.y));
}

// GELU = true: out = signsplit_quant(gelu_tanh(x)) in one pass (fpq_gelu_fake_quant_signsplit): the fc2 input of the
// reference, `fc2.act_quant(self.act(self.fc1(x)))`, without the round trip of the activation tensor through HBM.
template <int SPLIT, bool GELU>
__global__ void __launch_bounds__(256) signsplit_group_h16_kernel(const __half* __restrict__ x, __half* __restrict__ out, size_t n_groups,
                                                                  unsigned* __restrict__ nan_flag) {
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31;
    const int lig = lane % H16_LPG;
    const size_t warp_global = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    const float delta = tie_delta_kernel(uint32_t(warp_global >> 33));
    const size_t stride = n_warps * H16_GPW;
    bool owner = false;                     // this thread turned the NaN flag from 0 to 1 (poison_epilogue)
    pdl_wait();
    auto load = [&](size_t gbase, uint32_t (&p)[H16_NW]) {
        const size_t g = gbase + lane / H16_LPG;
        if (g < n_groups) {
            load_tile_h16(x + g * 128, lig, p);
            if constexpr (GELU) {
#pragma unroll
                for (int i = 0; i < H16_NW; ++i) p[i] = gelu_tanh_h2(p[i]);
            }
        } else {
#pragma unroll
            for (int i = 0; i < H16_NW; ++i) p[i] = 0u;
        }
    };
    auto work = [&](size_t gbase, uint32_t (&p)[H16_NW]) {
        using SF = SplitFmt<SPLIT>;
        const size_t g = gbase + lane / H16_LPG;
        float sn, sp;
        const int rc = split_quant_tile_h16<SPLIT, H16_LPG, H16_NW>(p, sn, sp, delta);
        if (rc == 2 && nan_flag != nullptr) owner |= (atomicOr(nan_flag, 1u) == 0u);     // exactly one thread of the grid sees the 0
        if (g < n_groups) {
            // rc != 0 leaves p untouched.  The literal sequences work from memory: with GELU fused in, the activated tile goes
            // to `out` first and is quantized there in place (all lanes of the group store before any of them rescans it)
            const __half* src = x + g * 128;
            if (GELU || rc == 0) store_tile_h16(out + g * 128, lig, p);
            if (GELU && rc != 0) { __syncwarp(0xFu << (lane & ~3)); src = out + g * 128; }      // rc is uniform over the 4 lanes of a group, not over the warp
            if (rc == 1) literal_split_h16(src, out + g * 128, lig, H16_LPG, 8, H16_NV, sn, sp, SF::GT_N, SF::GT_P);
            else if (rc == 2) literal_split_nan_group_h16(src, out + g * 128, lig, H16_LPG, 8, H16_NV, SF::NEG::VMAX, SF::POS::VMAX, SF::GT_N, SF::GT_P);
        }
    };
    for (size_t gbase = warp_global * H16_GPW; gbase < n_groups; gbase += stride) {
        uint32_t p[H16_NW];
        load(gbase, p);
        work(gbase, p);
    }
    if (nan_flag != nullptr) poison_epilogue(out, n_groups * 128, nan_flag, owner);
}

static unsigned grid_h16(size_t n_groups) {
    // 8 warps x 8 groups per block and trip; enough blocks to fill every SM's thread slots
    return grid_for(n_groups, 8 * H16_GPW, 8);
}

int launch_sym_h16(int format, const void* x, void* out, size_t n_groups, cudaStream_t st) {
    const __half* xi = static_cast<const __half*>(x);
    __half* oo = static_cast<__half*>(out);
    const unsigned grid = grid_h16(n_groups);
    return with_sym_format(format, [&](auto fmt) {
        launch_pdl(fake_quant_group_h16_kernel<fmt.value>, grid, 256, 0, st, xi, oo, n_groups);
        return finish_launch();
    });
}

int launch_sym_h16_g64(int format, const void* x, void* out, size_t n_groups, cudaStream_t st) {
    const __half* xi = static_cast<const __half*>(x);
    __half* oo = static_cast<__half*>(out);
    const unsigned grid = grid_for(n_groups, 8 * 8 * 2, 8);       // 8 warps x 8 groups x 2 tiles per block and trip
    return with_sym_format(format, [&](auto fmt) {
        launch_pdl(fake_quant_group64_h16_kernel<fmt.value>, grid, 256, 0, st, xi, oo, n_groups);
        return finish_launch();
    });
}

template <bool GELU>
static int launch_split_h16_t(int split, const void* x, void* out, size_t n_groups, unsigned* nan_flag, cudaStream_t st) {
    const __half* xi = static_cast<const __half*>(x);
    __half* oo = static_cast<__half*>(out);
    const unsigned grid = grid_h16(n_groups);
    return with_split_format(split, [&](auto sf) {
        launch_pdl(signsplit_group_h16_kernel<sf.value, GELU>, grid, 256, 0, st, xi, oo, n_groups, nan_flag);
        return finish_launch();
    });
}
int launch_split_h16(int split, const void* x, void* out, size_t n_groups, unsigned* nan_flag, cudaStream_t st) {
    return launch_split_h16_t<false>(split, x, out, n_groups, nan_flag, st);
}

// all 65 536 fp16 inputs through gelu_tanh_f32 -> fp16 (the table the GPU test compares with torch's own GELU output)
__global__ void gelu_table_kernel(__half* __restrict__ out) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 65536u) out[i] = __float2half_rn(gelu_tanh_f32(__half2float(__ushort_as_half(uint16_t(i)))));
}

// ------------------------------------------------------------------------------------------
// Exhaustive self-test of the packed element functions: every (x, scale) pair of fp16 values
// that can meet in a regular group, against the literal reference sequence
// (divide -> half -> scan -> multiply -> half).
// ------------------------------------------------------------------------------------------
template <class HG>
__device__ __forceinline__ bool pair_possible(float x, float s) {
    // x can share a group with scale s only if |x| <= absmax and half(absmax/VMAX) == s, which
    // implies half(|x|/VMAX) <= s
    return rnd_in<__half>(__fdiv_rn(fabsf(x), HG::VMAX)) <= s;
}

template <int CODE>
__global__ void selftest_f16_flow_kernel(unsigned long long* result) {
    unsigned long long bad = 0, first = ~0ull;
    // s: every regular fp16 scale 0x0400..0x7BFF; x: every fp16 bit pattern that is finite
    const unsigned long long total = (0x7C00ull - 0x0400ull) << 16;
    for (unsigned long long idx = size_t(blockIdx.x) * blockDim.x + threadIdx.x; idx < total; idx += size_t(gridDim.x) * blockDim.x) {
        const uint16_t sb = uint16_t(0x0400u + (idx >> 16));
        const uint16_t xb = uint16_t(idx & 0xffffu);
        if ((xb & 0x7fffu) >= 0x7C00u) continue;
        const float s = h2f(sb), x = h2f(xb);
        const float r = rcp_rn_normal(s);
        const float delta = tie_delta_kernel(0u);
        if (xb == 0 && __float_as_uint(r) != __float_as_uint(__frcp_rn(s))) { ++bad; if (idx < first) first = idx; }
        // The pair under test holds x in its low half and -x in its high half (both halves and both signs of the packed
        // instructions at once); a half whose value cannot occur next to this scale is not compared.
        const uint32_t x2 = uint32_t(xb) | (uint32_t(xb ^ 0x8000u) << 16);
        uint32_t got, want[2];
        bool check[2];
        if constexpr (CODE >= 32) {                              // the conversion-hardware element function (scorer; FPQ_HWCVT builds)
            using HG = typename SymFmt<CODE - 32>::HG;
            static_assert(HwCvt<HG>::AVAILABLE, "no conversion hardware for this format");
            if (!scale_bits_regular_hw<HG>(sb)) continue;
            check[0] = check[1] = pair_possible<HG>(x, s);
            const float rr = r * HwCvt<HG>::PRE;
            got = sym_pair_h16_hw<HG>(widen_h2(x2), pk(rr, rr), dup_h(__float2half_rn(s * (1.0f / HwCvt<HG>::PRE))), delta);
            want[0] = f2h(quant_elem_literal<__half, TIE_KERNEL>(x, s, c_grids[SymFmt<CODE - 32>::GT]) * s);
            want[1] = f2h(quant_elem_literal<__half, TIE_KERNEL>(-x, s, c_grids[SymFmt<CODE - 32>::GT]) * s);
        } else if constexpr (CODE < 16) {
            using HG = typename SymFmt<CODE>::HG;
            if (!scale_bits_regular_for<HG>(sb)) continue;      // scales the kernels send down the literal path
            check[0] = check[1] = pair_possible<HG>(x, s);
            got = sym_pair_h16<HG>(x2, make_symk<HG>(s, r), delta);
            want[0] = f2h(quant_elem_literal<__half, TIE_KERNEL>(x, s, c_grids[SymFmt<CODE>::GT]) * s);
            want[1] = f2h(quant_elem_literal<__half, TIE_KERNEL>(-x, s, c_grids[SymFmt<CODE>::GT]) * s);
        } else {
            using SF = SplitFmt<CODE - 16>;
            // the other side's scale does not influence an element: use the same s on both sides
            got = split_pair_h16<typename SF::NEG, typename SF::POS>(x2, make_splitk<typename SF::NEG, typename SF::POS>(s, r, s, r), delta);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float xv = h ? -x : x;
                const bool pos = xv > 0.0f;
                check[h] = pos ? pair_possible<typename SF::POS>(xv, s) : pair_possible<typename SF::NEG>(xv, s);
                const float xn = (xv <= 0.0f) ? xv : 0.0f, xp = pos ? xv : 0.0f;
                const float qn = scan_kernel_rule(rnd_in<__half>(__fdiv_rn(xn, s)), c_grids[SF::GT_N].v, c_grids[SF::GT_N].k);
                const float qp = scan_kernel_rule(rnd_in<__half>(__fdiv_rn(xp, s)), c_grids[SF::GT_P].v, c_grids[SF::GT_P].k);
                want[h] = f2h(__fadd_rn(__fmul_rn(qn, s), __fmul_rn(qp, s)));
            }
        }
        if ((check[0] && (got & 0xffffu) != want[0]) || (check[1] && (got >> 16) != want[1])) { ++bad; if (idx < first) first = idx; }
    }
    // scale: half(a * RN(1/VMAX)) == half(a / VMAX) for every fp16 absmax a whose scale is regular by
    // either formula (irregular scales are recomputed with the true division)
    for (unsigned ab = blockIdx.x * blockDim.x + threadIdx.x; ab <= 0x7C00u; ab += gridDim.x * blockDim.x) {
        const float a = h2f(uint16_t(ab));
        auto same = [&](uint32_t fast, uint32_t exact) {
            return fast == exact || (!scale_bits_regular(fast) && !scale_bits_regular(exact));
        };
        bool ok;
        if constexpr (CODE >= 32 || CODE < 16) {
            using HG = typename SymFmt<(CODE >= 32 ? CODE - 32 : CODE)>::HG;
            ok = same(__half_as_ushort(scale_from_absmax_h16<HG>(a)), f2h(__fdiv_rn(a, HG::VMAX)));
        } else {
            using SF = SplitFmt<CODE - 16>;
            ok = same(__half_as_ushort(scale_from_absmax_h16<typename SF::NEG>(a)), f2h(__fdiv_rn(a, SF::NEG::VMAX))) &&
                 same(__half_as_ushort(scale_from_absmax_h16<typename SF::POS>(a)), f2h(__fdiv_rn(a, SF::POS::VMAX)));
        }
        if (!ok) { ++bad; first = 0; }
    }
    if (bad) { atomicAdd(result, bad); atomicMin(result + 1, first); }
}

}  // namespace fpq

using namespace fpq;

extern "C" int fpq_selftest_f16_flow(int format, unsigned long long* result, void* stream) {
    if (!result) return FPQ_ERR_ARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaMemsetAsync(result, 0, sizeof(unsigned long long), st);
    cudaMemsetAsync(result + 1, 0xff, sizeof(unsigned long long), st);
    const unsigned grid = unsigned(sm_count()) * 16;
    switch (format) {
        case 0: selftest_f16_flow_kernel<0><<<grid, 256, 0, st>>>(result); break;
        case 1: selftest_f16_flow_kernel<1><<<grid, 256, 0, st>>>(result); break;
        case 2: selftest_f16_flow_kernel<2><<<grid, 256, 0, st>>>(result); break;
        case 3: selftest_f16_flow_kernel<3><<<grid, 256, 0, st>>>(result); break;
        case 4: selftest_f16_flow_kernel<4><<<grid, 256, 0, st>>>(result); break;
        case 16: selftest_f16_flow_kernel<16><<<grid, 256, 0, st>>>(result); break;
        case 17: selftest_f16_flow_kernel<17><<<grid, 256, 0, st>>>(result); break;
        case 18: selftest_f16_flow_kernel<18><<<grid, 256, 0, st>>>(result); break;
        case 32 + FPQ_FMT_E2M1: selftest_f16_flow_kernel<32 + FPQ_FMT_E2M1><<<grid, 256, 0, st>>>(result); break;
        case 32 + FPQ_FMT_E1M2: selftest_f16_flow_kernel<32 + FPQ_FMT_E1M2><<<grid, 256, 0, st>>>(result); break;
        case 32 + FPQ_FMT_E2M3: selftest_f16_flow_kernel<32 + FPQ_FMT_E2M3><<<grid, 256, 0, st>>>(result); break;
        case 32 + FPQ_FMT_E3M2: selftest_f16_flow_kernel<32 + FPQ_FMT_E3M2><<<grid, 256, 0, st>>>(result); break;
        default: return FPQ_ERR_ARG;
    }
    return finish_launch();
}

template <int GS>
static int launch_segments_h16(int format, const __half* x, __half* out, size_t n_segments, size_t groups_per_segment, size_t pitch_x,
                               size_t pitch_out, cudaStream_t st) {
    // per segment: 8 warps x 8 groups per block and trip; the whole grid fills the SMs' thread slots
    size_t per_seg = (groups_per_segment + 63) / 64;
    const size_t cap = (size_t(sm_count()) * 8 + n_segments - 1) / n_segments;
    if (per_seg > cap) per_seg = cap;
    if (per_seg < 1) per_seg = 1;
    const dim3 grid(unsigned(per_seg), unsigned(n_segments), 1);
    return with_sym_format(format, [&](auto fmt) {
        launch_pdl(fake_quant_segments_h16_kernel<fmt.value, GS>, grid, 256, 0, st, x, out, groups_per_segment, pitch_x, pitch_out);
        return finish_launch();
    });
}

extern "C" int fpq_fake_quant_segments(const void* x, void* out, size_t n_segments, size_t rows_per_segment, size_t row_len, size_t pitch_x,
                                       size_t pitch_out, int format, void* stream) {
    if (n_segments && rows_per_segment && (!x || !out)) return FPQ_ERR_ARG;
    if (row_len != 64 && row_len != 128) return FPQ_ERR_UNSUPPORTED;
    if (format < 0 || format >= FPQ_NUM_SYM_FORMATS) return FPQ_ERR_ARG;
    const size_t seg_elems = rows_per_segment * row_len;
    if (pitch_x < seg_elems || pitch_out < seg_elems || (pitch_x % 8) || (pitch_out % 8)) return FPQ_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15) return FPQ_ERR_ARG;
    if (n_segments > 65535) return FPQ_ERR_UNSUPPORTED;
    // out == x (in place, same pitch) is allowed; any other overlap is not
    if (x != out || pitch_x != pitch_out) {
        const char* a = static_cast<const char*>(x);
        const char* b = static_cast<const char*>(out);
        const size_t ea = ((n_segments ? n_segments - 1 : 0) * pitch_x + seg_elems) * 2, eb = ((n_segments ? n_segments - 1 : 0) * pitch_out + seg_elems) * 2;
        if (a < b + eb && b < a + ea) return FPQ_ERR_ARG;
    }
    if (n_segments == 0 || rows_per_segment == 0) return FPQ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const __half* xi = static_cast<const __half*>(x);
    __half* oo = static_cast<__half*>(out);
    if (row_len == 64) return launch_segments_h16<64>(format, xi, oo, n_segments, rows_per_segment, pitch_x, pitch_out, st);
    return launch_segments_h16<128>(format, xi, oo, n_segments, rows_per_segment, pitch_x, pitch_out, st);
}

extern "C" int fpq_gelu_fake_quant_signsplit(const void* x, void* out, size_t n_groups, int split_format, unsigned flags, void* workspace, void* stream) {
    if (n_groups && (!x || !out || x == out)) return FPQ_ERR_ARG;
    if (flags & ~FPQ_FLAG_GLOBAL_CLIP) return FPQ_ERR_ARG;
    if ((flags & FPQ_FLAG_GLOBAL_CLIP) && !workspace) return FPQ_ERR_ARG;
    if (split_format < 0 || split_format >= FPQ_NUM_SPLIT_FORMATS) return FPQ_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15) return FPQ_ERR_ARG;
    if (n_groups == 0) return FPQ_OK;
    unsigned* flag = (flags & FPQ_FLAG_GLOBAL_CLIP) ? static_cast<unsigned*>(workspace) : nullptr;
    return launch_split_h16_t<true>(split_format, x, out, n_groups, flag, static_cast<cudaStream_t>(stream));
}

extern "C" int fpq_selftest_gelu(void* table_65536_halves, void* stream) {
    if (!table_65536_halves) return FPQ_ERR_ARG;
    gelu_table_kernel<<<256, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<__half*>(table_65536_halves));
    return finish_launch();
}
