// Packed low-bit operands and the REAL low-bit GEMM on the 5th-generation tensor cores (SURVEY.md section 8 f4; not in the
// reference, which fake-quantizes and then calls F.linear on fp16 tensors: models_fp_quant_transform_rotate/quant_utils.py:764-769).
//
// Operand format ("codes"): the quantizer's grid value q of every element as ONE e4m3 byte -- every FP4 / FP6 grid of the
// reference (e2m1, e1m2, e3m0, e2m3, e3m2) is a subset of e4m3, so the byte holds q exactly -- plus the fp32 scale of every
// (row, 128-group).  The bytes lie in the order the tensor core reads them, so that a (128 rows x 128 K) operand tile is 16 KB
// of CONTIGUOUS memory that one 1-D bulk copy (cp.async.bulk, the TMA engine; no tensor map) lands in shared memory as the
// canonical K-major no-swizzle UMMA layout:
//     codes [K/128 slabs][rows_pad/8 row blocks][8 chunks of 16 K][8 rows][16 bytes]        rows_pad = rows rounded up to 128
//     scales[K/128 slabs][rows_pad]                                                        fp32, 0 for the padding rows
// At rest the FP4 formats shrink to 4 bits per element (fpq_codes_to_nibbles / fpq_nibbles_to_codes), same order.
//
// GEMM: C[m, n] = sum over slabs t of  sa[t, m] * sw[t, n] * P_t[m, n],   P_t = sum over the slab's 128 k of qa * qw,
// P_t by tcgen05.mma kind::f8f6f4 (e4m3 x e4m3, fp32 accumulate in tensor memory; exact while every partial sum fits fp32's 24
// bits: k_acc * max|q_a| * max|q_w| / (u_a * u_w) <= 2^24, u the grid's resolution, k_acc = 128 with groups of 128 (every pair but
// e3m2 x e3m2) and K with row scales (oracle/lowbit.py exact_accumulation); outside it P_t is within (k_acc - 1) * 2^-24 *
// sum |qa * qw|), the scale product by the epilogue warps on the CUDA cores while the tensor core
// works on the next slabs (512 columns of tensor memory: four 128-column or two 256-column accumulators).  The fp32 operation
// order is fixed -- acc = fma(P*sa, sw, acc), slabs ascending -- so that oracle/gemm_codes.c reproduces C bit for bit inside the
// envelope.
//
// Persistent kernel, one CTA per SM, 128 x 256 (or 128 x 128) tiles of C: warp 0 = bulk-copy producer, warp 1 = MMA issuer (one
// lane), warps 4.. = epilogue (each owns 32 tensor-memory lanes -- its warp-id quarter -- and EC columns, read as 16 x 8
// fragments).  Ring of shared-memory stages {A tile, B tile} and a ring of scale sets {sa, sw}, full / empty mbarriers;
// tcgen05.commit hands a stage back and publishes an accumulator; the epilogue hands the accumulator back as soon as it is in
// registers.  With one scale per row (per_token x per_channel) the whole K accumulates in tensor memory and the epilogue runs
// once per tile.  fp16 C tiles leave through a per-warp staging buffer in shared memory (whole-line stores).
// Measured (B200, profiles/r2_gemm_codes.txt; the fp16 library GEMM on the fake-quantized tensors: 1.44-1.48 PFLOP/s):
//   row scales 2.1-2.55 PFLOP/s: the SM's shared-memory pipe (48 KB in + 48 KB out per 128 x 256 slab at 128 B/clk = 768 clk; CTA
//   pairs sharing B by multicast were no faster, cta_group::2 MMAs -- PAIR below -- gain 3-4 %; the operand layout feeds the MMAs at
//   full rate (tools/umma_bench.cu): what is left is bytes in flight over the stage-recycle latency, ~2400 clk under a loaded L2);
//   groups of 128 1.04-1.49 PFLOP/s: the epilogue's 2 flops per element (512 clk of the fp32 pipe per 128 x 256 slab, as long as
//   the slab's MMAs) and its tensor-memory loads do not fully overlap with a memory-bound main loop; DESIGN.md 3.6 has the
//   experiments (tcgen05.ld alone: ~1 KB/clk per SM, tools/tmem_ldbench.cu; epilogue compiled out; per-tile overhead).
#include "fpq_codes.cuh"
#include "fpq_stream.cuh"

namespace fpq {

namespace {

constexpr int GK = 128;                      // K slab: the reference's quantization group
constexpr int TM = 128;                      // C tile rows (columns: 128 or 256, GemmCfg)
constexpr uint32_t BLK_BYTES = 1024;         // one (8 rows x 128 K) block of codes
constexpr uint32_t A_BYTES = TM * GK, SA_BYTES = TM * 4;

// ---------------------------------------------------------------------------------------------------------------------
// quantizer -> codes.  One warp per (8 rows x 128 K) block: lane = (row & 7) + 8 * (chunk & 3), two chunks of 16 elements per
// lane, so that a warp reads 8 x 128 contiguous bytes (fp16) per instruction pair and writes 512 contiguous bytes per store.
// Arithmetic: the reference's own sequence (qu.py:313-330 and Appendix A of SURVEY.md); see grid_values16 (fpq_codes.cuh).
// ---------------------------------------------------------------------------------------------------------------------
template <typename T, class HG>
__global__ void __launch_bounds__(256) pack_codes_kernel(const T* __restrict__ x, size_t rows, size_t rows_pad, size_t k,
                                                         uint8_t* __restrict__ codes, float* __restrict__ scales) {
    const int lane = threadIdx.x & 31;
    const int r = lane & 7, kq = lane >> 3;
    const size_t slabs = k / GK, row_blocks = rows_pad / 8;
    const size_t n_tasks = slabs * row_blocks;
    const size_t warp0 = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5, n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    for (size_t task = warp0; task < n_tasks; task += n_warps) {
        const size_t rb = task / slabs, slab = task % slabs;         // consecutive warps: consecutive slabs of the same rows
        const size_t row = rb * 8 + r;
        const bool live = row < rows;
        float v[2][16];
        float amax = 0.0f;
        bool nan = false;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (live) Chunk16<T>::load(x + row * k + slab * GK + size_t(kq + 4 * j) * 16, v[j]);
            else {
#pragma unroll
                for (int i = 0; i < 16; ++i) v[j][i] = 0.0f;
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                amax = fmaxf(amax, fabsf(v[j][i]));
                nan |= v[j][i] != v[j][i];
            }
        }
        // the row's group lives in the lanes with the same (lane & 7)
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 8));
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 16));
        unsigned nanmask = __ballot_sync(0xffffffffu, nan);
        nanmask |= nanmask >> 16;
        nanmask |= nanmask >> 8;
        if ((nanmask >> r) & 1u) amax = __int_as_float(0x7fc00000);          // torch's max propagates NaN
        const float s = Chunk16<T>::scale(amax, HG::VMAX);
        uint8_t* blk = codes + (slab * row_blocks + rb) * BLK_BYTES;
        const float delta = tie_delta_kernel(uint32_t(uint64_t(task) >> 40));
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            float q[16];
            grid_values16<T, HG>(v[j], s, delta, q);
            uint4 o;
            o.x = e4m3x4(q[0], q[1], q[2], q[3]);
            o.y = e4m3x4(q[4], q[5], q[6], q[7]);
            o.z = e4m3x4(q[8], q[9], q[10], q[11]);
            o.w = e4m3x4(q[12], q[13], q[14], q[15]);
            *reinterpret_cast<uint4*>(blk + (kq + 4 * j) * 128 + r * 16) = o;
        }
        if (kq == 0) scales[slab * rows_pad + row] = live ? s : 0.0f;
    }
}

// Row-wise scales (the reference's per_token / per_channel functions, qu.py:503-534: absmax over the whole last dim): one warp
// per 8-row block, two passes over the rows (absmax, then quantize; the second pass reads what the first left in L1 / L2).
// scales: [1][rows_pad].
template <typename T, class HG>
__global__ void __launch_bounds__(256) pack_codes_row_kernel(const T* __restrict__ x, size_t rows, size_t rows_pad, size_t k,
                                                             uint8_t* __restrict__ codes, float* __restrict__ scales) {
    const int lane = threadIdx.x & 31;
    const int r = lane & 7, kq = lane >> 3;
    const size_t slabs = k / GK, row_blocks = rows_pad / 8;
    const size_t warp0 = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5, n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    for (size_t rb = warp0; rb < row_blocks; rb += n_warps) {
        const size_t row = rb * 8 + r;
        const bool live = row < rows;
        float amax = 0.0f;
        bool nan = false;
        if (live) {
            for (size_t c = kq; c < slabs * 8; c += 4) {
                float v[16];
                Chunk16<T>::load(x + row * k + c * 16, v);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    amax = fmaxf(amax, fabsf(v[i]));
                    nan |= v[i] != v[i];
                }
            }
        }
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 8));
        amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 16));
        unsigned nanmask = __ballot_sync(0xffffffffu, nan);
        nanmask |= nanmask >> 16;
        nanmask |= nanmask >> 8;
        if ((nanmask >> r) & 1u) amax = __int_as_float(0x7fc00000);
        const float s = Chunk16<T>::scale(amax, HG::VMAX);
        const float delta = tie_delta_kernel(uint32_t(uint64_t(rb) >> 40));
        for (size_t c = kq; c < slabs * 8; c += 4) {
            float v[16], q[16];
            if (live) Chunk16<T>::load(x + row * k + c * 16, v);
            else {
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = 0.0f;
            }
            grid_values16<T, HG>(v, s, delta, q);
            uint4 o;
            o.x = e4m3x4(q[0], q[1], q[2], q[3]);
            o.y = e4m3x4(q[4], q[5], q[6], q[7]);
            o.z = e4m3x4(q[8], q[9], q[10], q[11]);
            o.w = e4m3x4(q[12], q[13], q[14], q[15]);
            *reinterpret_cast<uint4*>(codes + ((c >> 3) * row_blocks + rb) * BLK_BYTES + (c & 7) * 128 + r * 16) = o;
        }
        if (kq == 0) scales[row] = live ? s : 0.0f;
    }
}

// codes -> values: out[row, c] = T( fl32(q) * scale ), the reference's last step (qu.py:328-329).  One thread per 16-byte chunk.
template <typename T>
__global__ void __launch_bounds__(256) unpack_codes_kernel(const uint8_t* __restrict__ codes, const float* __restrict__ scales, size_t rows,
                                                           size_t rows_pad, size_t k, bool row_scale, T* __restrict__ out) {
    const size_t slabs = k / GK, row_blocks = rows_pad / 8;
    const size_t n_chunks = slabs * row_blocks * 64;
    for (size_t c = size_t(blockIdx.x) * blockDim.x + threadIdx.x; c < n_chunks; c += size_t(gridDim.x) * blockDim.x) {
        const size_t blk = c >> 6;
        const int kc = int(c >> 3) & 7, r = int(c) & 7;
        const size_t slab = blk / row_blocks, rb = blk % row_blocks;
        const size_t row = rb * 8 + r;
        if (row >= rows) continue;
        const uint4 u = *reinterpret_cast<const uint4*>(codes + c * 16);
        const float s = scales[(row_scale ? 0 : slab) * rows_pad + row];
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
        T* o = out + row * k + slab * GK + kc * 16;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
            for (int b = 0; b < 4; b += 2) {
                const __half2_raw hr = __nv_cvt_fp8x2_to_halfraw2(__nv_fp8x2_storage_t((w[i] >> (8 * b)) & 0xffffu), __NV_E4M3);
                const float q0 = __half2float(__ushort_as_half(hr.x)), q1 = __half2float(__ushort_as_half(hr.y));
                o[4 * i + b] = T(__fmul_rn(q0, s));
                o[4 * i + b + 1] = T(__fmul_rn(q1, s));
            }
        }
    }
}

// 4-bit storage of the FP4 formats: nibble = sign << 3 | index of |q| in the format's non-negative half grid (ascending);
// byte i holds elements 2i (low nibble) and 2i + 1 of the codes array, whatever its order.
struct NibbleLut { uint8_t e4m3[16]; };

__global__ void __launch_bounds__(256) codes_to_nibbles_kernel(const uint8_t* __restrict__ codes, size_t n_words, NibbleLut lut,
                                                               uint8_t* __restrict__ nib) {
    for (size_t w = size_t(blockIdx.x) * blockDim.x + threadIdx.x; w < n_words; w += size_t(gridDim.x) * blockDim.x) {
        const uint2 u = reinterpret_cast<const uint2*>(codes)[w];
        const uint32_t in[2] = {u.x, u.y};
        uint32_t out = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint8_t b = uint8_t(in[i >> 2] >> (8 * (i & 3)));
            uint32_t idx = 0;
#pragma unroll
            for (int j = 1; j < 8; ++j) idx = (b & 0x7f) == lut.e4m3[j] ? j : idx;
            out |= (idx | ((b >> 7) << 3)) << (4 * i);
        }
        reinterpret_cast<uint32_t*>(nib)[w] = out;
    }
}

__global__ void __launch_bounds__(256) nibbles_to_codes_kernel(const uint8_t* __restrict__ nib, size_t n_words, NibbleLut lut,
                                                               uint8_t* __restrict__ codes) {
    for (size_t w = size_t(blockIdx.x) * blockDim.x + threadIdx.x; w < n_words; w += size_t(gridDim.x) * blockDim.x) {
        const uint32_t in = reinterpret_cast<const uint32_t*>(nib)[w];
        uint32_t out[2] = {0, 0};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t n = (in >> (4 * i)) & 0xfu;
            out[i >> 2] |= uint32_t(lut.e4m3[n]) << (8 * (i & 3));
        }
        reinterpret_cast<uint2*>(codes)[w] = make_uint2(out[0], out[1]);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// tcgen05 primitives
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// cta_group::2: one MMA over a CTA pair, 256 x N x 32: each CTA supplies its 128 rows of A and its half (N/2 rows) of B from its own
// shared memory (same offsets in both), each CTA's tensor memory receives its 128 rows of D.  Issued by the pair's leader only.
__device__ __forceinline__ void tc_mma_f8_duo(uint32_t d_tmem, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_commit_duo(uint64_t* bar) {          // arrives on the barrier at this offset in BOTH CTAs
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(uint16_t(3))
                 : "memory");
}
// arrive on the barrier at this offset in CTA `rank` of the cluster.  Default semantics (release at CTA scope), as CUTLASS's
// ClusterBarrier does: `.release.cluster` compiles to a cluster-wide fence (ERRBAR) in front of every arrive, and the forwarding
// warp then hands over one stage per fence latency (~1400 clk: the whole kernel ran at that pace, profiles/r2_gemm_codes.txt)
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
    asm volatile(
        "{\n"
        ".reg .b32 ra;\n"
        "mapa.shared::cluster.u32 ra, %0, %1;\n"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(rank)
        : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_cta_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// D[tmem] (+)= A[smem] * B[smem]^T, 128 x 128 x 32, e4m3 operands, fp32 accumulate
__device__ __forceinline__ void tc_mma_f8(uint32_t d_tmem, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, no swizzle: core matrix = 8 rows x 16 bytes (128 contiguous bytes); `lbo` = byte step between the two core
// matrices one MMA reads along K, `sbo` = byte step between 8-row groups; descriptor version 1 (Blackwell), layout type 0.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
    return uint64_t((smem_addr >> 4) & 0x3fffu) | (uint64_t((lbo >> 4) & 0x3fffu) << 16) | (uint64_t((sbo >> 4) & 0x3fffu) << 32) |
           (uint64_t(1) << 46);
}
// instruction descriptor (GemmCfg::IDESC): D fp32 (bits 4-5 = 1), A / B e4m3 (format 0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24

// 16 lanes x 16 consecutive fp32 columns in the layout of the classic 16 x 8 accumulator fragment, two 8-column blocks i:
// thread t gets v[4i], v[4i+1] = (lane t/4, columns 8i + 2(t%4), +1) and v[4i+2], v[4i+3] = (lane t/4 + 8, same columns)
// (profiles/r2_tmem_layout.txt: the mapping as measured)
__device__ __forceinline__ void tc_ld_16x256b_x2(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr));
}

enum : int { OUT_F16 = 0, OUT_F32 = 1, OUT_SSE_F16 = 2, OUT_SSE_F32 = 3 };

struct GemmArgs {
    const uint8_t* a_codes;
    const float* a_scales;
    const uint8_t* b_codes;
    const float* b_scales;
    const float* bias;       // fp32 [n] or null
    void* c;                 // output matrix, or the reference matrix of the SSE modes
    double* sse;             // SSE modes: one accumulator
    const double* row_weight;  // SSE modes: weight of every row's squared error, or null (= 1)
    size_t ldc;              // elements
    size_t m, n;             // valid rows / columns of C
    size_t m_pad, n_pad;     // padded row counts of the two code arrays (multiples of 128)
    uint32_t slabs;          // K / 128
    uint32_t group_slabs;    // slabs that share one scale pair: 1 (groups of 128) or `slabs` (per_token x per_channel)
    uint32_t stages;
    uint32_t n_tiles, tiles_n;
};

template <int TN_, int EC_>
struct GemmCfg {
    static constexpr int TN = TN_;
    static constexpr int EC = EC_;                                // columns of C per epilogue warp (x 32 rows: its tensor-memory lanes)
    static constexpr int EPI_WARPS = 4 * (TN / EC);               // each: 32 rows x EC columns
    static constexpr int THREADS = 128 + 32 * EPI_WARPS;          // warps 0..3: producer, MMA issuer, two idle (one warpgroup)
    // (tried: setmaxnreg.dec / .inc between the control warpgroup and the epilogue warps -- ptxas keeps compiling the epilogue for the
    // launch bound and spills more; removed)
    static constexpr uint32_t B_BYTES = TN * GK;
    static constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;    // 32 KB | 48 KB
    // fp16 output: the C tile leaves through a per-warp shared-memory staging buffer (32 rows x 64 columns, rows padded to 144 bytes)
    // so that a warp store covers whole 128-byte lines; from the fragment layout a store instruction touches 8 lines for 128 bytes
    // and the tile's stores alone occupy the load/store pipe for ~4000 clk (profiles/r2_gemm_codes.txt)
    static constexpr bool STAGED_STORE = EPI_WARPS <= 8 && EC >= 64;
    static constexpr uint32_t ST_ROW = 144, ST_WARP = 32 * ST_ROW;
    static constexpr uint32_t ST_BYTES = STAGED_STORE ? EPI_WARPS * ST_WARP : 0;
    static constexpr int MAX_STAGES_FIT = int((227u * 1024u - 2048u - 8u * (SA_BYTES + TN * 4) - ST_BYTES) / (A_BYTES + TN * GK));
    static constexpr int MAX_STAGES = MAX_STAGES_FIT < 6 ? MAX_STAGES_FIT : 6;
    static constexpr uint32_t SC_BYTES = SA_BYTES + TN * 4;       // one scale pair set: sa[128], sw[TN]
    static constexpr int SC_DEPTH = 8;                            // >= stages + 2: the producer never waits on the scale ring first
    static constexpr int ACC = 512 / TN;                          // accumulators in tensor memory: 4 x 128 or 2 x 256 columns
    static constexpr uint32_t TMEM_COLS = 512;
    static constexpr uint32_t IDESC = (1u << 4) | (uint32_t(TN >> 3) << 17) | (uint32_t(TM >> 4) << 24);
    static constexpr size_t smem_bytes(int stages) { return size_t(stages) * STAGE_BYTES + SC_DEPTH * SC_BYTES + ST_BYTES + 1024; }
    // CTA pairs: a stage holds the A tile and HALF of the B tile
    static constexpr uint32_t STAGE_BYTES_PAIR = A_BYTES + B_BYTES / 2;
    static constexpr int MAX_STAGES_PAIR_FIT = int((227u * 1024u - 2048u - 8u * (SA_BYTES + TN * 4) - ST_BYTES) / STAGE_BYTES_PAIR);
    static constexpr int MAX_STAGES_PAIR = MAX_STAGES_PAIR_FIT < 6 ? MAX_STAGES_PAIR_FIT : 6;
    static constexpr size_t smem_bytes_pair(int stages) { return size_t(stages) * STAGE_BYTES_PAIR + SC_DEPTH * SC_BYTES + ST_BYTES + 1024; }
};

// Persistent: CTA b works on tiles b, b + gridDim.x, ...; tile t = (t / tiles_n, t % tiles_n), so that the CTAs running at the same
// time share A panels and the whole of B through L2.  Warp 0 = producer, warp 1 = MMA issuer, warps 4.. = epilogue.
// PAIR: launched as clusters of two CTAs that work on two row tiles of the same tile column (tm = 2 p + rank) with cta_group::2 MMAs:
// each CTA copies its own A tile and only ITS HALF of the B tile into its own shared memory, the pair's leader issues one
// 256 x TN x 32 MMA per K step that reads both CTAs' shared memory, each CTA's tensor memory receives its 128 rows.  Per slab an SM
// takes 32 KB in and 32 KB out of shared memory instead of 48 + 48: the pipe that bounds the single-CTA kernel.  The peer's MMA warp
// forwards "my stage is full" to the leader; the epilogue warps of both CTAs hand accumulators back to the leader.
// Measured (profiles/r2_gemm_codes.txt): bit-exact; row scales 2.42 / 2.63 PFLOP/s against 2.36 / 2.52 for single CTAs, groups of 128
// 1.31 / 1.44 against 1.40 / 1.52 -- so pairs are the default for row scales only.
template <int TN_, int EC_, int OUT, bool PAIR = false>
__global__ void __launch_bounds__(GemmCfg<TN_, EC_>::THREADS, 1) gemm_codes_kernel(const GemmArgs g) {
    using Cfg = GemmCfg<TN_, EC_>;
    constexpr int TN = Cfg::TN, EC = Cfg::EC;
    const uint32_t pair_rank = PAIR ? cluster_cta_rank() : 0u;
    // work items of this CTA: tiles (or tile pairs) first, first + step, ...; item w -> tile column w % tiles_n, tile row w / tiles_n
    // (x 2 + rank for pairs; a pair's second row tile may lie past the end: its loads are clamped, its stores masked by row < m)
    const uint32_t w_first = PAIR ? blockIdx.x / 2 : blockIdx.x, w_step = PAIR ? gridDim.x / 2 : gridDim.x;
    const uint32_t tiles_m = uint32_t(g.m_pad / TM);
    const uint32_t w_count = PAIR ? ((tiles_m + 1) / 2) * g.tiles_n : g.n_tiles;
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_full[6], bar_empty[6], bar_pfull[6], bar_tfull[Cfg::ACC], bar_tempty[Cfg::ACC];
    __shared__ uint64_t bar_sfull[Cfg::SC_DEPTH], bar_sempty[Cfg::SC_DEPTH];
    __shared__ uint32_t tmem_base_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;                 // stage bases on 1 KB
    uint8_t* const stage0 = smem_raw + (smem0 - smem_u32(smem_raw));
    const uint32_t stages = g.stages, slabs = g.slabs, gs = g.group_slabs;
    constexpr uint32_t STAGE = PAIR ? Cfg::STAGE_BYTES_PAIR : Cfg::STAGE_BYTES;
    uint8_t* const sc0 = stage0 + size_t(stages) * STAGE;

    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < stages; ++s) {
            mbar_init(&bar_full[s], 1);
            mbar_init(&bar_empty[s], 1);               // the MMA's commit (pairs: the leader's, multicast)
            mbar_init(&bar_pfull[s], 1);               // pairs, leader: the peer's stage is full
        }
        for (int a = 0; a < Cfg::ACC; ++a) {
            mbar_init(&bar_tfull[a], 1);
            mbar_init(&bar_tempty[a], PAIR ? 2 * Cfg::EPI_WARPS : Cfg::EPI_WARPS);    // pairs: both CTAs' epilogue warps, on the leader
        }
        for (int q = 0; q < Cfg::SC_DEPTH; ++q) {
            mbar_init(&bar_sfull[q], 1);
            mbar_init(&bar_sempty[q], Cfg::EPI_WARPS);
        }
        mbar_fence_init();
    }
    if (warp == 0) {
        if constexpr (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(Cfg::TMEM_COLS)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(Cfg::TMEM_COLS)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();            // the peer's barriers are initialised before anything is sent to them
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;

    if (warp == 0) {
        // ===== producer: two operand copies per slab, two scale copies per scale group =====
        if (lane == 0) {
            const size_t a_blocks = g.m_pad / 8, b_blocks = g.n_pad / 8;
            uint32_t it = 0, gi = 0;
            for (uint32_t w = w_first; w < w_count; w += w_step) {
                const uint32_t tm_raw = PAIR ? 2 * (w / g.tiles_n) + pair_rank : w / g.tiles_n;
                const size_t tm = tm_raw < tiles_m ? tm_raw : tiles_m - 1, tn = w % g.tiles_n;
                const size_t b_left = g.n_pad - tn * TN;
                const uint32_t b_rows = b_left < size_t(TN) ? uint32_t(b_left) : uint32_t(TN);        // last tile column may be half
                for (uint32_t i = 0; i < slabs; ++i, ++it) {
                    if (i % gs == 0) {
                        const uint32_t q = gi % Cfg::SC_DEPTH, qn = gi / Cfg::SC_DEPTH;
                        if (qn > 0) mbar_wait(&bar_sempty[q], (qn - 1) & 1);
                        uint8_t* sc = sc0 + size_t(q) * Cfg::SC_BYTES;
                        mbar_arrive_expect_tx(&bar_sfull[q], SA_BYTES + b_rows * 4);
                        bulk_load(sc, g.a_scales + size_t(i / gs) * g.m_pad + tm * TM, SA_BYTES, &bar_sfull[q]);
                        bulk_load(sc + SA_BYTES, g.b_scales + size_t(i / gs) * g.n_pad + tn * TN, b_rows * 4, &bar_sfull[q]);
                        ++gi;
                    }
                    const uint32_t s = it % stages, n = it / stages;
                    if (n > 0) mbar_wait(&bar_empty[s], (n - 1) & 1);
                    uint8_t* st = stage0 + size_t(s) * STAGE;
                    if constexpr (PAIR) {
                        const uint32_t half = b_rows / 2 * GK;             // b_rows is 128 or 256: halves of whole 8-row blocks
                        mbar_arrive_expect_tx(&bar_full[s], A_BYTES + half);
                        bulk_load(st, g.a_codes + (size_t(i) * a_blocks + tm * (TM / 8)) * BLK_BYTES, A_BYTES, &bar_full[s]);
                        bulk_load(st + A_BYTES, g.b_codes + (size_t(i) * b_blocks + tn * (TN / 8)) * BLK_BYTES + pair_rank * half, half, &bar_full[s]);
                    } else {
                        mbar_arrive_expect_tx(&bar_full[s], A_BYTES + b_rows * GK);
                        bulk_load(st, g.a_codes + (size_t(i) * a_blocks + tm * (TM / 8)) * BLK_BYTES, A_BYTES, &bar_full[s]);
                        bulk_load(st + A_BYTES, g.b_codes + (size_t(i) * b_blocks + tn * (TN / 8)) * BLK_BYTES, b_rows * GK, &bar_full[s]);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===== MMA issuer: four 128 x TN x 32 MMAs per slab; a scale group accumulates in tensor memory =====
        uint32_t it = 0, gi = 0;
        if (PAIR && pair_rank != 0) {
            // the pair's second CTA issues no MMA: tell the leader when this CTA's stage is full
            for (uint32_t w = w_first; w < w_count; w += w_step)
                for (uint32_t i = 0; i < slabs; ++i, ++it) {
                    mbar_wait(&bar_full[it % stages], (it / stages) & 1);
                    if (lane == 0) mbar_arrive_remote(&bar_pfull[it % stages], 0u);
                    __syncwarp();
                }
        } else {
            for (uint32_t w = w_first; w < w_count; w += w_step) {
                const size_t b_left = g.n_pad - size_t(w % g.tiles_n) * TN;
                const uint32_t b_rows = b_left < size_t(TN) ? uint32_t(b_left) : uint32_t(TN);
                // pairs: M = 256 over both CTAs, N = the tile's columns (each CTA holds half of the B rows)
                const uint32_t idesc = PAIR ? ((1u << 4) | ((b_rows >> 3) << 17) | (uint32_t(256 >> 4) << 24)) : Cfg::IDESC;
                for (uint32_t i = 0; i < slabs; ++i, ++it) {
                    const uint32_t s = it % stages, n = it / stages, a = gi % Cfg::ACC, u = gi / Cfg::ACC;
                    const bool first = i % gs == 0, last = i % gs == gs - 1;
                    if (first && u > 0) {
                        mbar_wait(&bar_tempty[a], (u - 1) & 1);
                    }
                    mbar_wait(&bar_full[s], n & 1);
                    if constexpr (PAIR) mbar_wait(&bar_pfull[s], n & 1);       // arrived on from the peer CTA (release.cluster)
                    tc_fence_after();
                    if (lane == 0) {
                        const uint32_t st_addr = smem0 + s * STAGE;
                        const uint64_t da = umma_desc(st_addr, 128u, 1024u), db = umma_desc(st_addr + A_BYTES, 128u, 1024u);
#pragma unroll
                        for (uint32_t kk = 0; kk < GK / 32; ++kk) {     // 32 K = two core matrices = 256 bytes further on
                            if constexpr (PAIR) tc_mma_f8_duo(tmem_base + a * TN, da + kk * (256u >> 4), db + kk * (256u >> 4), idesc, (first && kk == 0) ? 0u : 1u);
                            else tc_mma_f8(tmem_base + a * TN, da + kk * (256u >> 4), db + kk * (256u >> 4), idesc, (first && kk == 0) ? 0u : 1u);
                        }
                        if constexpr (PAIR) {
                            tc_commit_duo(&bar_empty[s]);
                            if (last) tc_commit_duo(&bar_tfull[a]);
                        } else {
                            tc_commit(&bar_empty[s]);
                            if (last) tc_commit(&bar_tfull[a]);
                        }
                    }
                    __syncwarp();
                    if (last) ++gi;
                }
            }
        }
    } else if (warp >= 4) {
        // ===== epilogue: acc = fma(P * sa, sw, acc) per scale group.  A warp owns 32 rows (its tensor-memory lane quarter) x EC
        // columns and reads them as 16 x 8 fragments: a thread holds FOUR rows (tr, tr+8, tr+16, tr+24) x EC/4 columns (the pair
        // 2 tq, 2 tq + 1 of every 8-column block), so that per 128-K slab it needs 4 row scales and EC/4 column scales from shared
        // memory instead of 1 + EC with one row per thread: the column-scale loads (a 16-byte load per lane costs the full 512
        // bytes of return bandwidth even when every lane reads the same address) were what bounded the first version, on the
        // same 128 B/clk shared-memory pipe that carries the operand tiles in and out. =====
        const int quarter = warp & 3;                         // the tensor-memory lanes this warp may touch
        const int col_off = ((warp - 4) >> 2) * EC;           // its columns of the tile
        const int tq = lane & 3, tr = lane >> 2;
        constexpr int NB = EC / 8;                            // 8-column blocks per thread row
        const uint32_t n_groups = slabs / gs;
        uint32_t gi = 0;
        double sse_thread = 0.0;
        for (uint32_t w = w_first; w < w_count; w += w_step) {
            const uint32_t tile_m = PAIR ? 2 * (w / g.tiles_n) + pair_rank : w / g.tiles_n, tile_n = w % g.tiles_n;
            uint64_t acc[4 * NB];                              // [row slot rr][block b]: columns (8 b + 2 tq, + 1) of row tr + 8 rr
#pragma unroll
            for (int j = 0; j < 4 * NB; ++j) acc[j] = 0ull;
            for (uint32_t grp = 0; grp < n_groups; ++grp, ++gi) {
                const uint32_t q = gi % Cfg::SC_DEPTH, a = gi % Cfg::ACC;
                const uint8_t* sc = sc0 + size_t(q) * Cfg::SC_BYTES;
                mbar_wait(&bar_sfull[q], (gi / Cfg::SC_DEPTH) & 1);
                uint64_t sa2[4];
#pragma unroll
                for (int rr = 0; rr < 4; ++rr) {
                    const float sa = reinterpret_cast<const float*>(sc)[quarter * 32 + tr + 8 * rr];
                    sa2[rr] = pk(sa, sa);
                }
                const uint64_t* swp = reinterpret_cast<const uint64_t*>(sc + SA_BYTES + col_off * 4) + tq;     // block b: swp[4 b]
                mbar_wait(&bar_tfull[a], (gi / Cfg::ACC) & 1);
                tc_fence_after();
                const uint32_t t0 = tmem_base + (uint32_t(quarter * 32) << 16) + a * TN + col_off;
                // 16 columns (two blocks, both 16-lane halves) at a time, the next piece's loads in flight under this piece's arithmetic
                uint32_t v[2][2][8];
                tc_ld_16x256b_x2(t0, v[0][0]);
                tc_ld_16x256b_x2(t0 + (16u << 16), v[0][1]);
                tc_wait_ld();
#pragma unroll
                for (int c = 0; c < EC / 16; ++c) {
                    constexpr int LAST = EC / 16 - 1;
                    if (c < LAST) {
                        tc_ld_16x256b_x2(t0 + (c + 1) * 16, v[(c + 1) & 1][0]);
                        tc_ld_16x256b_x2(t0 + (16u << 16) + (c + 1) * 16, v[(c + 1) & 1][1]);
                    } else {
                        // every column of this accumulator is in registers: hand it back before the arithmetic
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            if (PAIR && pair_rank != 0) mbar_arrive_remote(&bar_tempty[a], 0u);       // the leader issues the MMAs
                            else mbar_arrive(&bar_tempty[a]);
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const int bl = c * 2 + i;
                        const uint64_t w = swp[4 * bl];
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const uint32_t* vv = v[c & 1][h];
                            acc[(2 * h) * NB + bl] = ffma2(fmul2(pk(__uint_as_float(vv[4 * i]), __uint_as_float(vv[4 * i + 1])), sa2[2 * h]), w, acc[(2 * h) * NB + bl]);
                            acc[(2 * h + 1) * NB + bl] = ffma2(fmul2(pk(__uint_as_float(vv[4 * i + 2]), __uint_as_float(vv[4 * i + 3])), sa2[2 * h + 1]), w, acc[(2 * h + 1) * NB + bl]);
                        }
                    }
                    if (c < LAST) tc_wait_ld();
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_sempty[q]);
            }
            const size_t row0 = size_t(tile_m) * TM + quarter * 32 + tr, col0 = size_t(tile_n) * TN + col_off + 2 * tq;
            float part[4] = {0.0f, 0.0f, 0.0f, 0.0f};          // SSE modes: squared error of this thread's piece of each of its rows
            if constexpr (OUT == OUT_F16 && Cfg::STAGED_STORE) {
                uint8_t* stg = sc0 + Cfg::SC_DEPTH * Cfg::SC_BYTES + size_t(warp - 4) * Cfg::ST_WARP;
                const size_t trow0 = size_t(tile_m) * TM + quarter * 32, tcol0 = size_t(tile_n) * TN + col_off;
#pragma unroll
                for (int ch = 0; ch < EC / 64; ++ch) {
#pragma unroll
                    for (int bi = 0; bi < 8; ++bi) {
                        const int bl = ch * 8 + bi;
                        uint64_t bias2 = 0ull;
                        if (g.bias && tcol0 + 8 * bl < g.n) { const float2 bb = __ldg(reinterpret_cast<const float2*>(g.bias + tcol0 + 8 * bl + 2 * tq)); bias2 = pk(bb.x, bb.y); }
#pragma unroll
                        for (int rr = 0; rr < 4; ++rr) {
                            const F2 o = unpk(g.bias ? fadd2(acc[rr * NB + bl], bias2) : acc[rr * NB + bl]);
                            *reinterpret_cast<uint32_t*>(stg + (tr + 8 * rr) * Cfg::ST_ROW + bi * 16 + tq * 4) = pack_h2(o.lo, o.hi);
                        }
                    }
                    __syncwarp();
                    const size_t col = tcol0 + ch * 64 + (lane & 7) * 8;
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int rl = it * 4 + (lane >> 3);
                        const uint4 u = *reinterpret_cast<const uint4*>(stg + rl * Cfg::ST_ROW + (lane & 7) * 16);
                        if (trow0 + rl < g.m && col < g.n) *reinterpret_cast<uint4*>(static_cast<__half*>(g.c) + (trow0 + rl) * g.ldc + col) = u;
                    }
                    __syncwarp();
                }
                continue;
            }
#pragma unroll
            for (int bl = 0; bl < NB; ++bl) {
                const size_t col = col0 + 8 * bl;
                if (col >= g.n) break;                         // n is a multiple of 8: whole blocks
                uint64_t bias2 = 0ull;
                if (g.bias) { const float2 bb = __ldg(reinterpret_cast<const float2*>(g.bias + col)); bias2 = pk(bb.x, bb.y); }
#pragma unroll
                for (int rr = 0; rr < 4; ++rr) {
                    const size_t row = row0 + 8 * rr;
                    if (row >= g.m) continue;
                    const F2 o = unpk(g.bias ? fadd2(acc[rr * NB + bl], bias2) : acc[rr * NB + bl]);
                    if constexpr (OUT == OUT_F16) {
                        *reinterpret_cast<uint32_t*>(static_cast<__half*>(g.c) + row * g.ldc + col) = pack_h2(o.lo, o.hi);
                    } else if constexpr (OUT == OUT_F32) {
                        *reinterpret_cast<float2*>(static_cast<float*>(g.c) + row * g.ldc + col) = make_float2(o.lo, o.hi);
                    } else {
                        // squared distance to the reference matrix: fp32 differences and row pieces, float64 across rows
                        float r0, r1;
                        if constexpr (OUT == OUT_SSE_F16) {
                            const uint32_t u = *reinterpret_cast<const uint32_t*>(static_cast<const __half*>(g.c) + row * g.ldc + col);
                            r0 = h2f(uint16_t(u & 0xffffu));
                            r1 = h2f(uint16_t(u >> 16));
                        } else {
                            const float2 u = *reinterpret_cast<const float2*>(static_cast<const float*>(g.c) + row * g.ldc + col);
                            r0 = u.x;
                            r1 = u.y;
                        }
                        const float d0 = r0 - o.lo, d1 = r1 - o.hi;
                        part[rr] = __fmaf_rn(d1, d1, __fmaf_rn(d0, d0, part[rr]));
                    }
                }
            }
            if constexpr (OUT == OUT_SSE_F16 || OUT == OUT_SSE_F32) {
#pragma unroll
                for (int rr = 0; rr < 4; ++rr) {
                    const size_t row = row0 + 8 * rr;
                    if (row < g.m) sse_thread += double(part[rr]) * (g.row_weight ? g.row_weight[row] : 1.0);
                }
            }
        }
        if constexpr (OUT == OUT_SSE_F16 || OUT == OUT_SSE_F32) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) sse_thread += __shfl_xor_sync(0xffffffffu, sse_thread, off);
            if (lane == 0) atomicAdd(g.sse, sse_thread);
        }
    }

    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();            // nothing of the peer is in flight towards this CTA's shared memory any more
    if (warp == 0) {
        tc_fence_after();
        if constexpr (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::TMEM_COLS) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::TMEM_COLS) : "memory");
    }
}

bool half_grid_e4m3(int format, NibbleLut& lut) {
    // |q| of the three FP4 formats as e4m3 bytes (bias 7, 3 mantissa bits), ascending; entries 8..15 = the same with the sign bit
    static const uint8_t e2m1[8] = {0x00, 0x30, 0x38, 0x3c, 0x40, 0x44, 0x48, 0x4c};      // 0 .5 1 1.5 2 3 4 6
    static const uint8_t e1m2[8] = {0x00, 0x28, 0x30, 0x34, 0x38, 0x3a, 0x3c, 0x3e};      // 0 .25 .5 .75 1 1.25 1.5 1.75
    static const uint8_t e3m0[8] = {0x00, 0x28, 0x30, 0x38, 0x40, 0x48, 0x50, 0x58};      // 0 .25 .5 1 2 4 8 16
    const uint8_t* t = format == FPQ_FMT_E2M1 ? e2m1 : format == FPQ_FMT_E1M2 ? e1m2 : format == FPQ_FMT_E3M0 ? e3m0 : nullptr;
    if (!t) return false;
    for (int i = 0; i < 8; ++i) {
        lut.e4m3[i] = t[i];
        lut.e4m3[8 + i] = uint8_t(t[i] | 0x80);
    }
    lut.e4m3[8] = 0x00;           // the quantizer never produces -0 (the grids' zero is +0.0); decode nibble 8 as +0 too
    return true;
}

template <typename T>
int launch_pack_rows(int format, const T* x, size_t rows, size_t rows_pad, size_t k, uint8_t* codes, float* scales, cudaStream_t st) {
    const unsigned grid = grid_for(rows_pad / 8, 8, 8);
    return with_sym_format(format, [&](auto fmt) {
        pack_codes_row_kernel<T, typename SymFmt<fmt.value>::HG><<<grid, 256, 0, st>>>(x, rows, rows_pad, k, codes, scales);
        return finish_launch();
    });
}

template <typename T>
int launch_pack(int format, const T* x, size_t rows, size_t rows_pad, size_t k, uint8_t* codes, float* scales, cudaStream_t st) {
    const size_t tasks = (k / GK) * (rows_pad / 8);
    const unsigned grid = grid_for(tasks, 8, 8);
    return with_sym_format(format, [&](auto fmt) {
        pack_codes_kernel<T, typename SymFmt<fmt.value>::HG><<<grid, 256, 0, st>>>(x, rows, rows_pad, k, codes, scales);
        return finish_launch();
    });
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

}  // namespace fpq

using namespace fpq;

extern "C" size_t fpq_codes_rows_padded(size_t rows) { return (rows + TM - 1) / TM * TM; }

extern "C" int fpq_pack_codes(const void* x, size_t rows, size_t k, size_t scale_group, int in_dtype, int format, uint8_t* codes, float* scales,
                              void* stream) {
    if (k == 0 || k % GK != 0 || (scale_group != GK && scale_group != k)) return FPQ_ERR_ARG;
    if ((rows && (!x || !codes || !scales)) || !aligned16(x) || !aligned16(codes) || !aligned16(scales)) return FPQ_ERR_ARG;
    if (rows == 0) return FPQ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t rows_pad = fpq_codes_rows_padded(rows);
    if (scale_group == GK) {
        if (in_dtype == FPQ_F16) return launch_pack<__half>(format, static_cast<const __half*>(x), rows, rows_pad, k, codes, scales, st);
        if (in_dtype == FPQ_F32) return launch_pack<float>(format, static_cast<const float*>(x), rows, rows_pad, k, codes, scales, st);
    } else {
        if (in_dtype == FPQ_F16) return launch_pack_rows<__half>(format, static_cast<const __half*>(x), rows, rows_pad, k, codes, scales, st);
        if (in_dtype == FPQ_F32) return launch_pack_rows<float>(format, static_cast<const float*>(x), rows, rows_pad, k, codes, scales, st);
    }
    return FPQ_ERR_ARG;
}

extern "C" int fpq_unpack_codes(const uint8_t* codes, const float* scales, size_t rows, size_t k, size_t scale_group, int out_dtype, void* out,
                                void* stream) {
    if (k == 0 || k % GK != 0 || (scale_group != GK && scale_group != k)) return FPQ_ERR_ARG;
    if ((rows && (!out || !codes || !scales)) || !aligned16(codes)) return FPQ_ERR_ARG;
    if (rows == 0) return FPQ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t rows_pad = fpq_codes_rows_padded(rows);
    const unsigned grid = grid_for(rows_pad * k / 16, 256, 8);
    const bool row_scale = scale_group != GK;
    if (out_dtype == FPQ_F16) unpack_codes_kernel<__half><<<grid, 256, 0, st>>>(codes, scales, rows, rows_pad, k, row_scale, static_cast<__half*>(out));
    else if (out_dtype == FPQ_F32) unpack_codes_kernel<float><<<grid, 256, 0, st>>>(codes, scales, rows, rows_pad, k, row_scale, static_cast<float*>(out));
    else return FPQ_ERR_ARG;
    return finish_launch();
}

extern "C" int fpq_codes_to_nibbles(const uint8_t* codes, size_t n_codes, int format, uint8_t* nibbles, void* stream) {
    NibbleLut lut;
    if (!half_grid_e4m3(format, lut)) return FPQ_ERR_UNSUPPORTED;
    if (n_codes % 8 != 0 || (n_codes && (!codes || !nibbles)) || !aligned16(codes) || !aligned16(nibbles)) return FPQ_ERR_ARG;
    if (n_codes == 0) return FPQ_OK;
    codes_to_nibbles_kernel<<<grid_for(n_codes / 8, 256, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(codes, n_codes / 8, lut, nibbles);
    return finish_launch();
}

extern "C" int fpq_nibbles_to_codes(const uint8_t* nibbles, size_t n_codes, int format, uint8_t* codes, void* stream) {
    NibbleLut lut;
    if (!half_grid_e4m3(format, lut)) return FPQ_ERR_UNSUPPORTED;
    if (n_codes % 8 != 0 || (n_codes && (!codes || !nibbles)) || !aligned16(codes) || !aligned16(nibbles)) return FPQ_ERR_ARG;
    if (n_codes == 0) return FPQ_OK;
    nibbles_to_codes_kernel<<<grid_for(n_codes / 8, 256, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(nibbles, n_codes / 8, lut, codes);
    return finish_launch();
}

namespace {

template <int TN_, int EC_, int OUT>
int launch_gemm(GemmArgs& g, cudaStream_t st) {
    using Cfg = GemmCfg<TN_, EC_>;
    if (int(g.stages) > Cfg::MAX_STAGES) g.stages = Cfg::MAX_STAGES;
    const size_t tiles_n = (g.n_pad + TN_ - 1) / TN_;
    const size_t tiles = (g.m_pad / TM) * tiles_n;
    if (tiles > 0x7fffffffull) return FPQ_ERR_UNSUPPORTED;
    g.n_tiles = uint32_t(tiles);
    g.tiles_n = uint32_t(tiles_n);
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev & 63]) {
        if (cudaFuncSetAttribute(gemm_codes_kernel<TN_, EC_, OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(Cfg::smem_bytes(Cfg::MAX_STAGES))) != cudaSuccess)
            return finish_launch();
        attr_set[dev & 63] = true;
    }
    const size_t resident = size_t(sm_count());
    const unsigned grid = unsigned(tiles < resident ? tiles : resident);
    gemm_codes_kernel<TN_, EC_, OUT><<<grid, Cfg::THREADS, Cfg::smem_bytes(int(g.stages)), st>>>(g);
    return finish_launch();
}

// CTA pairs (clusters of two): instantiated for the default tile shape only
template <int TN_, int EC_, int OUT>
int launch_gemm_pair(GemmArgs& g, cudaStream_t st) {
    using Cfg = GemmCfg<TN_, EC_>;
    if (g_tun.gemm_stages >= 6 || int(g.stages) > Cfg::MAX_STAGES_PAIR) g.stages = Cfg::MAX_STAGES_PAIR;     // default: as deep as fits
    const size_t tiles_n = (g.n_pad + TN_ - 1) / TN_, tiles_m = g.m_pad / TM;
    const size_t pairs = (tiles_m + 1) / 2 * tiles_n;
    if (tiles_m * tiles_n > 0x7fffffffull) return FPQ_ERR_UNSUPPORTED;
    g.n_tiles = uint32_t(tiles_m * tiles_n);
    g.tiles_n = uint32_t(tiles_n);
    auto kernel = gemm_codes_kernel<TN_, EC_, OUT, true>;
    static bool attr_set[64] = {};
    static int max_clusters[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(Cfg::THREADS);
    cfg.dynamicSmemBytes = Cfg::smem_bytes_pair(int(g.stages));
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (!attr_set[dev & 63]) {
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(Cfg::smem_bytes_pair(Cfg::MAX_STAGES_PAIR))) != cudaSuccess) return finish_launch();
        cfg.gridDim = dim3(unsigned(sm_count()) / 2 * 2);
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess || n < 1) { cudaGetLastError(); n = sm_count() / 2 - 4; }
        max_clusters[dev & 63] = n;
        attr_set[dev & 63] = true;
    }
    const size_t clusters = pairs < size_t(max_clusters[dev & 63]) ? pairs : size_t(max_clusters[dev & 63]);
    cfg.gridDim = dim3(unsigned(2 * clusters));
    cudaLaunchKernelEx(&cfg, kernel, g);
    return finish_launch();
}

template <int OUT>
int launch_gemm_tn(GemmArgs& g, cudaStream_t st) {
    const int ec = g_tun.gemm_epi_cols;
    if (g_tun.gemm_tile_n == 128) {
        if (ec == 32) return launch_gemm<128, 32, OUT>(g, st);
        if (ec == 64) return launch_gemm<128, 64, OUT>(g, st);
        return launch_gemm<128, 128, OUT>(g, st);
    }
    if (ec == 64) return launch_gemm<256, 64, OUT>(g, st);
    // default (-1): CTA pairs where they were measured faster -- row scales (+3-4 %), not groups of 128 (-6 %)
    const bool pair = g_tun.gemm_pair == 1 || (g_tun.gemm_pair < 0 && g.group_slabs != 1 && g.slabs > 1 && g.m_pad / TM >= 4);
    return pair ? launch_gemm_pair<256, 128, OUT>(g, st) : launch_gemm<256, 128, OUT>(g, st);
}

int gemm_common(GemmArgs& g, const uint8_t* a_codes, const float* a_scales, size_t m, const uint8_t* b_codes, const float* b_scales, size_t n,
                size_t k, size_t scale_group, const float* bias, void* c, size_t ldc) {
    if (k == 0 || k % GK != 0 || k / GK > 0xffffffffull || (scale_group != GK && scale_group != k)) return FPQ_ERR_ARG;
    if (!a_codes || !a_scales || !b_codes || !b_scales || !c) return FPQ_ERR_ARG;
    if (!aligned16(a_codes) || !aligned16(a_scales) || !aligned16(b_codes) || !aligned16(b_scales) || !aligned16(c)) return FPQ_ERR_ARG;
    if (n % 8 != 0 || ldc % 8 != 0 || ldc < n || (reinterpret_cast<uintptr_t>(bias) & 7u)) return FPQ_ERR_ARG;
    g.a_codes = a_codes; g.a_scales = a_scales; g.b_codes = b_codes; g.b_scales = b_scales; g.bias = bias;
    g.c = c; g.sse = nullptr; g.row_weight = nullptr; g.ldc = ldc; g.m = m; g.n = n;
    g.m_pad = fpq_codes_rows_padded(m); g.n_pad = fpq_codes_rows_padded(n);
    g.slabs = uint32_t(k / GK);
    g.group_slabs = scale_group == GK ? 1u : g.slabs;
    g.stages = uint32_t(g_tun.gemm_stages);
    return FPQ_OK;
}

}  // namespace

extern "C" int fpq_gemm_codes(const uint8_t* a_codes, const float* a_scales, size_t m, const uint8_t* b_codes, const float* b_scales,
                              size_t n, size_t k, size_t scale_group, const float* bias, int out_dtype, void* c, size_t ldc, void* stream) {
    if (m == 0 || n == 0) return FPQ_OK;
    if (out_dtype != FPQ_F16 && out_dtype != FPQ_F32) return FPQ_ERR_ARG;
    GemmArgs g;
    if (int rc = gemm_common(g, a_codes, a_scales, m, b_codes, b_scales, n, k, scale_group, bias, c, ldc)) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return out_dtype == FPQ_F16 ? launch_gemm_tn<OUT_F16>(g, st) : launch_gemm_tn<OUT_F32>(g, st);
}

extern "C" int fpq_gemm_codes_sse(const uint8_t* a_codes, const float* a_scales, size_t m, const uint8_t* b_codes, const float* b_scales,
                                  size_t n, size_t k, size_t scale_group, const float* bias, int ref_dtype, const void* ref, size_t ldr,
                                  const double* row_weight, double* sse, void* stream) {
    if (m == 0 || n == 0) return FPQ_OK;
    if ((ref_dtype != FPQ_F16 && ref_dtype != FPQ_F32) || !sse) return FPQ_ERR_ARG;
    GemmArgs g;
    if (int rc = gemm_common(g, a_codes, a_scales, m, b_codes, b_scales, n, k, scale_group, bias, const_cast<void*>(ref), ldr)) return rc;
    g.sse = sse;
    g.row_weight = row_weight;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return ref_dtype == FPQ_F16 ? launch_gemm_tn<OUT_SSE_F16>(g, st) : launch_gemm_tn<OUT_SSE_F32>(g, st);
}
