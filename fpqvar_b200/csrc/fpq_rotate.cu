// libfpq_b200 -- fused GALT transform + 128-block random-Hadamard rotation (+ fake quant).
// Replaces (reference rows a8, a9 of SURVEY.md section 8):
//   activations  basic_var.py:263,266   matmul(x.mul(s), Q)  -> QuantizedLinear.forward act_quant
//   weights      transform_model_utils.py:8-28 (W / s) then rotation_utils.py:129-154 (W.double() @ Q)
// Q = I (x) diag(sigma) H_128 / fl32(sqrt(128)) (rotation_utils.py:69-104, hadamard_utils.py:63-99),
// so (x @ Q) on an aligned 128-chunk is FWHT_128(x * sigma) / c: 7 butterfly stages instead of a
// dense C x C GEMM.
// Both activation kernels write either fp16 (fake-quantized, or rotated only) or, with CODES, the packed operand of the low-bit
// GEMM (fpq_*transform_rotate_pack_codes: e4m3 grid value per element + scale per (row, 128-chunk), fpq_gemm.cu's layout).
//
// Numerics shared by the two activation kernels below (so that a row rotates to the same bits whichever
// kernel the launcher picks for the tensor's size; test_rotation_bits_do_not_depend_on_the_launch_size):
//   * the per-column multiplier is m[c] = RN(smooth[c] * fl32(1/sqrt(128))) * sigma[c % 128] (the sign flip is
//     exact), so every element costs ONE multiply in front of the butterflies and none behind them;
//   * a Sylvester Hadamard transform is the tensor product of a 2-point butterfly (a + b, a - b) over every
//     index bit of the chunk position, in any order; the order fixes the fp32 summation tree and is
//     0, 1, 5, 6, 2, 3, 4 in both kernels.
#include "fpq_codes.cuh"
#include "fpq_stream.cuh"

namespace fpq {

struct SignMask { uint32_t w[4]; };    // bit e of the 128-bit mask set  <=>  sigma[e] = +1

// adaLN modulate operands (fpq_modulate_transform_rotate_quant): t = (x * (scale[b, c] + 1) + shift[b, c]) * smooth[c]
struct Modulate { const float* scale; const float* shift; size_t rows_per_batch; float one; };   // one: 1.0f, or -0.0f (the exact additive identity) under FPQ_MOD_GAIN

// Codes output (fpq_*transform_rotate_pack_codes): the layout of include/fpq_b200.h, rows_pad = fpq_codes_rows_padded(n_rows).
// The kernels that write it store, per element, the grid value the fp16 output would have multiplied by the group's scale, and
// per (row, 128-chunk) that scale: the bytes fpq_pack_codes writes for the fp16 rotated tensor.
struct CodesOut { uint8_t* codes; float* scales; size_t rows_pad; };
constexpr uint32_t CODES_BLOCK_BYTES = 1024;          // 8 rows x 128 K: one row block of a slab

// Codes output: the padding rows n_rows .. rows_pad - 1 of every slab get code 0 and scale 0 from the same launch, spread over
// all of its threads (fewer than 128 rows per slab: one 16-byte store per thread or less at the sizes of a VAR pass).
__device__ __forceinline__ void zero_codes_padding(const CodesOut& co, size_t n_rows, int cpr) {
    const size_t pad = co.rows_pad - n_rows;
    const size_t per_slab = pad * 9;                   // eight 16-byte code pieces and one scale per padding row
    const size_t total = per_slab * size_t(cpr);
    for (size_t u = size_t(blockIdx.x) * blockDim.x + threadIdx.x; u < total; u += size_t(gridDim.x) * blockDim.x) {
        const size_t slab = u / per_slab, v = u % per_slab;
        if (v < pad * 8) {
            const size_t row = n_rows + v / 8;
            *reinterpret_cast<uint4*>(co.codes + (slab * (co.rows_pad / 8) + row / 8) * CODES_BLOCK_BYTES + (v & 7) * 128 + (row & 7) * 16) =
                make_uint4(0u, 0u, 0u, 0u);
        } else {
            co.scales[slab * co.rows_pad + n_rows + (v - pad * 8)] = 0.0f;
        }
    }
}

// Codes of 16 fp16 values of a group with an irregular scale (the literal sequence, out of line).  The values go through a
// copy, so that the caller's register tile itself never needs an address.
template <class HG>
__device__ __forceinline__ uint4 irregular_codes16(const uint32_t* w, float s, float delta) {
    uint32_t t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t[i] = w[i];
    return codes16_h16<HG>(t, s, delta);
}
// The same for a streaming lane's 32 values, stored as its two K pieces (dst, dst + 128) by the out-of-line function itself,
// so that nothing of the caller's but the loop state is live across the call.
template <class HG>
static __device__ __noinline__ void codes32_store_h16(const uint32_t* w, float s, float delta, uint8_t* dst) {
    stg_stream(dst, codes16_h16<HG>(w, s, delta));
    stg_stream(dst + 128, codes16_h16<HG>(w + 8, s, delta));
}
template <class HG>
__device__ __forceinline__ void irregular_codes32(const uint32_t* w, float s, float delta, uint8_t* dst) {
    uint32_t t[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) t[i] = w[i];
    codes32_store_h16<HG>(t, s, delta, dst);
}

// 1 / fl32(sqrt(128)), rounded to fp32 (SURVEY.md section 7: 0x3DB504F3)
__device__ __forceinline__ float inv_sqrt128() { return __uint_as_float(0x3DB504F3u); }

// multipliers of the four columns col0 .. col0 + 3 (col0 % 4 == 0), chunk positions e0 .. e0 + 3
__device__ __forceinline__ void load_mult4(const float* __restrict__ smooth, const SignMask& sm, size_t col0, int e0, uint64_t& m01, uint64_t& m23) {
    float4 s4 = make_float4(1.0f, 1.0f, 1.0f, 1.0f);
    if (smooth != nullptr) s4 = __ldg(reinterpret_cast<const float4*>(smooth + col0));
    float f[4] = {s4.x, s4.y, s4.z, s4.w};
    const uint32_t bits = sm.w[e0 >> 5] >> (e0 & 31);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        f[k] = __fmul_rn(f[k], inv_sqrt128());
        if (!((bits >> k) & 1u)) f[k] = -f[k];
    }
    m01 = pk(f[0], f[1]);
    m23 = pk(f[2], f[3]);
}

// (scale + 1) and shift of four columns of batch row b
__device__ __forceinline__ void load_mod4(const Modulate& mod, size_t off, uint64_t& a01, uint64_t& a23, uint64_t& s01, uint64_t& s23) {
    const float4 sc = __ldg(reinterpret_cast<const float4*>(mod.scale + off));
    const float4 sh = __ldg(reinterpret_cast<const float4*>(mod.shift + off));
    const uint64_t one2 = pk(mod.one, mod.one);
    a01 = fadd2(pk(sc.x, sc.y), one2);               // scale.add(1)
    a23 = fadd2(pk(sc.z, sc.w), one2);
    s01 = pk(sh.x, sh.y);
    s23 = pk(sh.z, sh.w);
}
// .mul(scale.add(1)).add_(shift): the product with the SCALAR mul.rn.f32 (never contracted; ptxas fuses
// mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 -- even through a *1, and even when the product is written as
// fma(x, a, -0.0): measured, the parity tests fail -- which would skip the rounding of the product that the reference's
// separate ATen kernels perform)
__device__ __forceinline__ uint64_t modulate2(uint64_t x, uint64_t a, uint64_t sh) {
    const F2 xv = unpk(x), av = unpk(a);
    return fadd2(pk(__fmul_rn(xv.lo, av.lo), __fmul_rn(xv.hi, av.hi)), sh);
}

// butterfly between packed registers at distance h of P[0..N)
template <int N>
__device__ __forceinline__ void reg_stage(uint64_t (&P)[N], int h) {
    const uint64_t neg1 = pk(-1.0f, -1.0f);
#pragma unroll
    for (int i = 0; i < N; ++i) {
        if ((i & h) == 0) {
            const uint64_t a = P[i], b = P[i + h];
            P[i] = fadd2(a, b);
            P[i + h] = ffma2(b, neg1, a);
        }
    }
}
// butterfly inside every packed pair (index bit 0)
template <int N>
__device__ __forceinline__ void pair_stage(uint64_t (&P)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const F2 f = unpk(P[i]);
        P[i] = pk(f.lo + f.hi, f.lo - f.hi);
    }
}

// ------------------------------------------------------------------------------------------------------------
// Small launches (the first stages of a VAR pass: a few thousand chunks, latency-bound): 8 lanes x 16 values per
// chunk straight from global memory, every 8-lane set bound to ONE column chunk cc so that its 16 multipliers live in
// registers, walking down the rows k, k+K, k+2K, ... of that column.  With fp32 input, value v[4j+k] of lane l is
// element e = 32j + 4l + k of the chunk: index bits 0,1 (k) and 5,6 (j) are in registers, bits 2,3,4 (l) across
// lanes (shfl.xor 1,2,4).  Arithmetic is two elements per instruction where the ISA allows (FMUL2/FFMA2/FADD2 packed
// fp32, sm_100): P[2j] = (v[4j], v[4j+1]), P[2j+1] = (v[4j+2], v[4j+3]).
// MOD (adaLN modulate fused in): a lane set walks CONTIGUOUS rows (k0*R .. k0*R + R - 1) instead of strided ones, so
// the (scale+1) and shift values of its column change only when the batch index does and live in registers in between.
// CODES (codes output instead of `out` / `rotated`): lane l's four 4-element pieces are 4-byte pieces of codes, 256 B apart.
// ------------------------------------------------------------------------------------------------------------
template <int FMT, bool QUANT, bool MOD, bool CODES>
__global__ void __launch_bounds__(256, MOD ? 1 : 0) transform_rotate_quant_small_kernel(const float* __restrict__ x, const float* __restrict__ smooth,
                                                                                       SignMask sm, __half* __restrict__ out, __half* __restrict__ rotated,
                                                                                       size_t n_rows, int cpr, size_t sets_per_col, Modulate mod,
                                                                                       CodesOut co) {
    constexpr int LPG = 8;
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31;
    const int lig = lane % LPG;
    const size_t ls = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) / LPG;       // lane-set id
    const int cc = int(ls % size_t(cpr));
    const size_t k0 = ls / size_t(cpr);
    const bool active = k0 < sets_per_col;
    const size_t row_stride = size_t(cpr) * 128;
    const float delta = tie_delta_kernel(uint32_t(ls >> 36));
    // uniform trip count across the warp (the shuffles need every lane)
    const size_t trips = (n_rows + sets_per_col - 1) / sets_per_col;
    // Nothing is read before pdl_wait(): `smooth` may have been produced (cast, sliced) by the kernel in front of this one.
    pdl_wait();
    uint64_t ms[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) load_mult4(smooth, sm, size_t(cc) * 128 + 32 * j + 4 * lig, 32 * j + 4 * lig, ms[2 * j], ms[2 * j + 1]);
    uint64_t A[MOD ? 8 : 1], SH[MOD ? 8 : 1];         // (scale + 1) and shift of this lane's 16 columns for batch cur_b
    size_t cur_b = ~size_t(0);
    for (size_t t = 0; t < trips; ++t) {
        const size_t row = MOD ? k0 * trips + t : k0 + t * sets_per_col;
        const bool valid = active && row < n_rows;
        const size_t off = row * row_stride + size_t(cc) * 128;
        uint64_t P[8];
        if (valid) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint4 u = ldg_stream(x + off + (j * LPG + lig) * 4);
                P[2 * j] = (uint64_t(u.y) << 32) | u.x;
                P[2 * j + 1] = (uint64_t(u.w) << 32) | u.z;
            }
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) P[i] = 0ull;
        }
        if constexpr (MOD) {
            const size_t b = valid ? row / mod.rows_per_batch : cur_b;
            if (b != cur_b) {
                cur_b = b;
                const size_t mo = b * row_stride + size_t(cc) * 128;
#pragma unroll
                for (int j = 0; j < 4; ++j) load_mod4(mod, mo + (j * LPG + lig) * 4, A[2 * j], A[2 * j + 1], SH[2 * j], SH[2 * j + 1]);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) P[i] = modulate2(P[i], A[i], SH[i]);
        }
        // x * m: basic_var.py:263 `.mul(s)` in fp32, the sign row of Q and the 1/sqrt(128) of the Hadamard matrix
#pragma unroll
        for (int i = 0; i < 8; ++i) P[i] = fmul2(P[i], ms[i]);
        pair_stage(P);          // index bit 0
        reg_stage(P, 1);        // index bit 1
        reg_stage(P, 2);        // index bit 5
        reg_stage(P, 4);        // index bit 6
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {             // index bits 2, 3, 4: across the lanes of the set
            const float sg = (lig & o) ? -1.0f : 1.0f;
            const uint64_t sg2 = pk(sg, sg);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const F2 f = unpk(P[i]);
                const uint64_t q = pk(__shfl_xor_sync(0xffffffffu, f.lo, o), __shfl_xor_sync(0xffffffffu, f.hi, o));
                P[i] = ffma2(P[i], sg2, q);            // upper lane: partner - mine ; lower lane: mine + partner (exact: * +-1)
            }
        }
        // rounded to fp16: the fp16 GEMM output of the reference
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = pack_h2_u64(P[i]);
        if constexpr (CODES) {
            float s;
            const bool ok = sym_quant_tile_h16<FMT, LPG, 8, true, true>(w, s, delta);
            if (valid) {
                const uint4 c = ok ? make_uint4(e4m3x4_h2(w[0], w[1]), e4m3x4_h2(w[2], w[3]), e4m3x4_h2(w[4], w[5]), e4m3x4_h2(w[6], w[7]))
                                   : irregular_codes16<typename SymFmt<FMT>::HG>(w, s, delta);
                // element 32 j + 4 lig + k: K piece 2 j + lig / 4, byte 4 (lig % 4) + k
                uint8_t* cb = co.codes + (size_t(cc) * (co.rows_pad / 8) + row / 8) * CODES_BLOCK_BYTES + (row & 7) * 16 + (lig >> 2) * 128 + (lig & 3) * 4;
                *reinterpret_cast<uint32_t*>(cb) = c.x;
                *reinterpret_cast<uint32_t*>(cb + 256) = c.y;
                *reinterpret_cast<uint32_t*>(cb + 512) = c.z;
                *reinterpret_cast<uint32_t*>(cb + 768) = c.w;
                if (lig == 0) co.scales[size_t(cc) * co.rows_pad + row] = s;
            }
            continue;
        }
        if (valid && rotated != nullptr) {
#pragma unroll
            for (int j = 0; j < 4; ++j) stg_stream(rotated + off + (j * LPG + lig) * 4, make_uint2(w[2 * j], w[2 * j + 1]));
        }
        bool ok = true;
        float s = 0.0f;
        if constexpr (QUANT) ok = sym_quant_tile_h16<FMT, LPG, 8>(w, s, delta);
        if (valid) {
#pragma unroll
            for (int j = 0; j < 4; ++j) stg_stream(out + off + (j * LPG + lig) * 4, make_uint2(w[2 * j], w[2 * j + 1]));
            // irregular scale (zero / subnormal / inf / NaN): `out` now holds this lane's rotated values;
            // quantize them in place with the literal reference sequence
            if (!ok) literal_sym_h16(out + off, out + off, lig, LPG, 4, 4, s, SymFmt<FMT>::GT);
        }
    }
    if constexpr (CODES) zero_codes_padding(co, n_rows, cpr);
}

// ------------------------------------------------------------------------------------------------------------
// Streaming kernel (everything from a few thousand chunks on; rows of 4 .. 36 chunks).
//   work split      a CTA has one warp per group of 4 chunk columns (rows of 15 chunks, VAR-d30: 4 warps; 18 chunks,
//                   VAR-d36: 5 warps) and owns a contiguous range of rows (ranges differ by at most one row over the
//                   grid: no partial wave at the end); several CTAs per SM (about 20 warps, the register budget).  A warp
//                   walks down its rows two at a time, always on the same 4 columns, so that the multipliers (and, with
//                   MOD, the adaLN operands of the current batch) live in registers.
//   staging         every warp has a PRIVATE double buffer of 2 x 4 KB in shared memory and is its own producer: lane 0
//                   fetches the warp's next 2 rows x 4 chunks with 1-D bulk async copies (cp.async.bulk -> UBLKCP, the TMA
//                   engine; 2 KB of contiguous bytes per row) that complete on the buffer's mbarrier.  The bytes in flight
//                   cost shared memory, not registers, no warp ever waits for another one (no CTA barrier after the
//                   prologue), and the copy for step k+2 is issued as soon as step k has left its buffer.
//   transform       two passes over the 8 chunks in shared memory, so that no butterfly crosses lanes (no SHFL at all):
//       pass 1   8 lanes x 16 values per chunk: lane l holds the 16-byte units u = 8a + l (a = 0..3) of its chunk,
//                i.e. index bits 0,1 (inside a unit) and 5,6 (a) -- multiply, butterflies 0,1,5,6, write back IN PLACE;
//                done twice per step (row r, then row r + 1, same columns);
//       pass 2   4 lanes x 32 values per chunk: lane l' holds the units 8l' + i (i = 0..7), index bits 0..4 --
//                butterflies 2,3,4, round to fp16, per-group quantizer on the register tile, 128-bit stores of 32
//                CONTIGUOUS elements per lane.
//   bank conflicts  a chunk is 512 B = 4 x 128 B bank windows, and an LDS.128 / STS.128 is served 8 lanes at a time.
//                Pass 1 reads 8 consecutive units per chunk: conflict-free as it is.  Pass 2 reads units 128 B apart
//                in 4 lanes x 2 chunks per phase; the units are therefore stored XOR-swizzled inside their 128-byte
//                window by pass 1: unit (a, c) sits at slot c ^ (2a + s), s = parity of the chunk among the warp's 8.
//                Both the swizzled pass-1 stores and the pass-2 loads then touch 8 distinct 16-byte slots per phase
//                (tests/rotate_layout_model.py replays the choreography on the host).
// ------------------------------------------------------------------------------------------------------------
// The streaming kernel's quantizer runs on the FP4 / FP6 conversion hardware (sym_pair_h16_hw, exhaustively checked by
// fpq_selftest_f16_flow(32 + format)).  Measured against the magic-number path in the same kernel (same box, same run):
// VAR-d30 step 24.89 vs 25.29 ms, VAR-d36 step 24.19 vs 24.82 ms; the largest launch alone is 2 % slower (5.66 vs 5.79 TB/s).
constexpr bool ROT_HW_QUANT = true;
constexpr int ROT_MIN_CPR = 4, ROT_MAX_CPR = 36;       // rows the streaming kernel takes, in chunks
constexpr int ROT_WARP_STAGE_BYTES = 4096;             // 2 rows x 4 chunks x 512 B
constexpr int ROT_WARP_SMEM = 2 * ROT_WARP_STAGE_BYTES + 16;      // + the two mbarriers

// Loop bookkeeping is kept to a minimum (ncu r2: the first version of this body spent 10 of its 27 instructions per
// element on 64-bit row arithmetic, re-derived shared-memory addresses and branches): rows are 32-bit counters relative to
// the CTA's first row, global pointers are advanced instead of recomputed, every shared-memory address is a lane constant
// plus an immediate, and the two buffers are two copies of the step body with compile-time offsets.
// CODES: pass 2's 32 contiguous elements of a lane are two 16-byte K pieces of codes of one row, 128 B apart (an 8-row line is
// completed over four steps of the same warp and merged in L2); the padding rows are written at the end of the launch.
template <int FMT, bool QUANT, bool MOD, bool CODES>
struct RotStream {
    // lane constants
    uint32_t p1;            // pass 1: this lane's first unit of its chunk (row 0, buffer 0)
    uint32_t q1[4];         // pass 1: swizzled store addresses of its four units
    uint32_t a2[8];         // pass 2: swizzled load addresses of its eight units (buffer 0)
    bool colok1, colok2;
    int row2;
    int lq;
    uint64_t ms[8];
    uint64_t A[MOD ? 8 : 1], SH[MOD ? 8 : 1];
    float delta;
    // MOD: adaLN operands of the batch the next row belongs to
    const float* pa;
    const float* psh;
    uint32_t left, rpb, row_elems;
    bool reload;
    // output
    __half* op;             // this lane's 32 output elements of row `row2` of the current step
    __half* rp;             // same in `rotated` (or nullptr)
    // CODES output: two 32-bit counters only (the addresses are rebuilt from the kernel parameters every step; 64-bit pointers
    // here pushed the plain kernel past its 96 registers)
    uint32_t cslab;         // this lane's chunk column (slab)
    uint32_t crow;          // row `row2` of the current step (the launcher keeps rows_pad below 2^32)

    // this lane's (scale + 1) and shift of the batch `pa` / `psh` point at
    __device__ __forceinline__ void load_operands() {
        reload = false;
        if (colok1) {
            Modulate m{pa, psh, 0, mod_one};
#pragma unroll
            for (int a = 0; a < 4; ++a) load_mod4(m, size_t(32 * a), A[2 * a], A[2 * a + 1], SH[2 * a], SH[2 * a + 1]);
        }
    }
    __device__ __forceinline__ void pass1(uint32_t buf_off, int nr) {
#pragma unroll
        for (int sub = 0; sub < 2; ++sub) {
            if (sub < nr) {
                if constexpr (MOD) {
                    if (reload) load_operands();                  // first row of a batch
                    if (--left == 0) { left = rpb; pa += row_elems; psh += row_elems; reload = true; }
                }
                {
                    // every lane runs (no branch, no partial-warp barrier): a lane whose column does not exist (the last warp
                    // may own fewer than four) has zero multipliers and works on its own, unused slice of the buffer
                    const uint32_t off = buf_off + uint32_t(sub) * 2048u;
                    uint64_t P[8];
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        uint4 u;
                        asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(p1 + off + uint32_t(a * 128)));
                        P[2 * a] = (uint64_t(u.y) << 32) | u.x;
                        P[2 * a + 1] = (uint64_t(u.w) << 32) | u.z;
                    }
                    if constexpr (MOD) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) P[i] = modulate2(P[i], A[i], SH[i]);
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) P[i] = fmul2(P[i], ms[i]);
                    pair_stage(P);          // index bit 0
                    reg_stage(P, 1);        // index bit 1
                    reg_stage(P, 2);        // index bit 5
                    reg_stage(P, 4);        // index bit 6
                    // in place: the 8 lanes of the chunk have all read their units before any of them overwrites one
                    __syncwarp();
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        const F2 p0 = unpk(P[2 * a]), p1v = unpk(P[2 * a + 1]);
                        asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(q1[a] + off), "f"(p0.lo), "f"(p0.hi), "f"(p1v.lo), "f"(p1v.hi) : "memory");
                    }
                }
            }
        }
    }
    float mod_one;
    uint32_t lanes8;

    // returns after the loads of pass 2 (the caller then hands the buffer back to the producer) -- Q holds the values
    __device__ __forceinline__ void pass2_load(uint32_t buf_off, bool valid, uint64_t (&Q)[16]) {
        // unconditional: a lane set without a chunk (missing column, or the odd last row) reads its own stale slice of the
        // buffer and its results are never stored
        (void)valid;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            uint4 u;
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(a2[i] + buf_off));
            Q[2 * i] = (uint64_t(u.y) << 32) | u.x;
            Q[2 * i + 1] = (uint64_t(u.w) << 32) | u.z;
        }
    }
    __device__ __forceinline__ void pass2_finish(bool valid, uint64_t (&Q)[16], const CodesOut& co) {
        reg_stage(Q, 2);                // index bit 2
        reg_stage(Q, 4);                // index bit 3
        reg_stage(Q, 8);                // index bit 4
        // rounded to fp16: the fp16 GEMM output of the reference.  Lane l' holds elements 32*l' .. 32*l' + 31 in order.
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) w[i] = pack_h2_u64(Q[i]);
        if constexpr (CODES) {
            float sc;
            const bool ok = sym_quant_tile_h16<FMT, 4, 16, ROT_HW_QUANT, true>(w, sc, delta);
            if (valid) {
                uint8_t* p = co.codes + (size_t(cslab) * (co.rows_pad / 8) + (crow >> 3)) * CODES_BLOCK_BYTES + uint32_t(lq) * 256u + (crow & 7u) * 16u;
                if (ok) {
                    stg_stream(p, make_uint4(e4m3x4_h2(w[0], w[1]), e4m3x4_h2(w[2], w[3]), e4m3x4_h2(w[4], w[5]), e4m3x4_h2(w[6], w[7])));
                    stg_stream(p + 128, make_uint4(e4m3x4_h2(w[8], w[9]), e4m3x4_h2(w[10], w[11]), e4m3x4_h2(w[12], w[13]), e4m3x4_h2(w[14], w[15])));
                } else {
                    irregular_codes32<typename SymFmt<FMT>::HG>(w, sc, delta, p);
                }
                if (lq == 0) co.scales[size_t(cslab) * co.rows_pad + crow] = sc;
            }
            crow += 2;
            return;
        }
        if (rp != nullptr) {
            if (valid) {
#pragma unroll
                for (int q = 0; q < 4; ++q) stg_stream(rp + q * 8, make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]));
            }
            rp += 2 * size_t(row_elems);
        }
        bool ok = true;
        float sc = 0.0f;
        if constexpr (QUANT) ok = sym_quant_tile_h16<FMT, 4, 16, ROT_HW_QUANT>(w, sc, delta);
        if (valid) {
#pragma unroll
            for (int q = 0; q < 4; ++q) stg_stream(op + q * 8, make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]));
            // irregular scale (zero / subnormal / inf / NaN): `out` now holds this lane's rotated values;
            // quantize them in place with the literal reference sequence
            if (!ok) literal_sym_h16(op - lq * 32, op - lq * 32, lq, 4, 32, 1, sc, SymFmt<FMT>::GT);
        }
        op += 2 * size_t(row_elems);
    }
};

template <int FMT, bool QUANT, bool MOD, bool CODES>
__device__ __forceinline__ void rotate_stream_body(const float* __restrict__ x, const float* __restrict__ smooth,
                                                   SignMask sm, __half* __restrict__ out, __half* __restrict__ rotated,
                                                   size_t n_rows, int cpr, Modulate mod, const CodesOut& co) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_warps = blockDim.x >> 5;
    unsigned char* stage0 = smem + size_t(warp) * (2 * ROT_WARP_STAGE_BYTES);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + size_t(n_warps) * (2 * ROT_WARP_STAGE_BYTES)) + 2 * warp;
    if (lane == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        mbar_fence_init();
    }
    pdl_launch_dependents();
    __syncwarp();

    // this CTA's rows: [r_begin, r_begin + n_mine), sizes differ by at most one row over the grid (the launcher keeps
    // n_mine below 2^31)
    const size_t per = n_rows / gridDim.x, rem = n_rows % gridDim.x;
    const size_t r_begin = size_t(blockIdx.x) * per + (blockIdx.x < rem ? blockIdx.x : rem);
    const uint32_t n_mine = uint32_t(per) + (blockIdx.x < rem ? 1u : 0u);
    const uint32_t row_elems = uint32_t(cpr) * 128u;
    const int col0 = 4 * warp;                                          // first chunk column of this warp
    const int ncols = cpr - col0 < 4 ? cpr - col0 : 4;                  // its columns that exist (the last warp may own fewer)

    RotStream<FMT, QUANT, MOD, CODES> st;
    const uint32_t smem_base = smem_u32(stage0);
    // pass 1: 8 lanes per chunk; sub-iteration = row, g4 = column within the warp
    const int g4 = lane >> 3, l8 = lane & 7;
    st.colok1 = g4 < ncols;
    st.lanes8 = 0xFFu << (8 * g4);
    st.p1 = smem_base + uint32_t(g4) * 512u + uint32_t(l8) * 16u;
#pragma unroll
    for (int a = 0; a < 4; ++a)                                         // unit (a, c = l8) at slot c ^ (2a + s), s = column parity
        st.q1[a] = smem_base + uint32_t(g4) * 512u + uint32_t(a) * 128u + ((uint32_t(l8 ^ (g4 & 1)) ^ uint32_t(2 * a)) << 4);
    // pass 2: 4 lanes per chunk, lane set g8 = 4 * row + column
    const int g8 = lane >> 2, c2 = g8 & 3;
    st.lq = lane & 3;
    st.row2 = g8 >> 2;
    st.colok2 = c2 < ncols;
    {
        const uint32_t chunk2 = smem_base + uint32_t(st.row2) * 2048u + uint32_t(c2) * 512u + uint32_t(st.lq) * 128u;
        const uint32_t key2 = uint32_t(2 * st.lq + (g8 & 1));
#pragma unroll
        for (int i = 0; i < 8; ++i) st.a2[i] = chunk2 + ((uint32_t(i) ^ key2) << 4);
    }
    st.delta = tie_delta_kernel(uint32_t((r_begin + size_t(lane)) >> 44));       // 0, but not provably uniform (fpq_h16.cuh)
    st.row_elems = row_elems;
    st.mod_one = mod.one;
    st.op = out + (r_begin + size_t(st.row2)) * row_elems + size_t(col0 + c2) * 128 + st.lq * 32;
    st.rp = rotated != nullptr ? rotated + (r_begin + size_t(st.row2)) * row_elems + size_t(col0 + c2) * 128 + st.lq * 32 : nullptr;
    if constexpr (CODES) {
        st.cslab = uint32_t(col0 + c2);
        st.crow = uint32_t(r_begin) + uint32_t(st.row2);
    }
    st.pa = st.psh = nullptr;
    st.left = st.rpb = 1;
    st.reload = false;
    if constexpr (MOD) {
#pragma unroll
        for (int i = 0; i < 8; ++i) st.A[i] = st.SH[i] = 0ull;
    }
    if constexpr (MOD) {
        const size_t batch = r_begin / mod.rows_per_batch;
        st.rpb = uint32_t(mod.rows_per_batch);
        st.left = st.rpb - uint32_t(r_begin - batch * mod.rows_per_batch);
        const size_t lane_off = batch * row_elems + size_t(col0 + (st.colok1 ? g4 : 0)) * 128 + 4 * l8;
        st.pa = mod.scale + lane_off;
        st.psh = mod.shift + lane_off;
        st.reload = true;
    }
    // Nothing is read from global memory before pdl_wait(): x comes from the previous kernel, and `smooth` may too.
    pdl_wait();

    // ---- producer side (lane 0): the copy of step k + 2 is issued when step k has left its buffer ----
    const unsigned char* gsrc = reinterpret_cast<const unsigned char*>(x + r_begin * row_elems + size_t(col0) * 128);
    const uint32_t row_bytes = uint32_t(ncols) * 512u, row_stride_b = row_elems * 4u;
    uint32_t issued = 0;
    auto issue = [&](uint32_t s) {
        if (issued < n_mine) {
            if (lane == 0) {
                const bool two = n_mine - issued >= 2u;
                mbar_arrive_expect_tx(&full[s], two ? 2u * row_bytes : row_bytes);
                bulk_load(stage0 + s * ROT_WARP_STAGE_BYTES, gsrc, row_bytes, &full[s]);
                if (two) bulk_load(stage0 + s * ROT_WARP_STAGE_BYTES + 2048, gsrc + row_stride_b, row_bytes, &full[s]);
            }
            gsrc += 2 * size_t(row_stride_b);
            issued += 2u;
        }
    };
    issue(0);
    issue(1);
    if constexpr (MOD) st.load_operands();          // the first batch's adaLN operands travel while the first copy does

    // multipliers of this lane's 16 columns (pass 1): units u = 8a + l8, elements 32a + 4*l8 + k
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int e0 = 32 * a + 4 * l8;
        if (st.colok1) load_mult4(smooth, sm, size_t(col0 + g4) * 128 + e0, e0, st.ms[2 * a], st.ms[2 * a + 1]);
        else st.ms[2 * a] = st.ms[2 * a + 1] = 0ull;
    }

    auto step = [&](uint32_t s, uint32_t done, uint32_t phase) {
        const int nr = n_mine - done >= 2u ? 2 : 1;
        const uint32_t buf_off = s * ROT_WARP_STAGE_BYTES;
        mbar_wait(&full[s], phase);
        st.pass1(buf_off, nr);
        __syncwarp();
        const bool valid = st.colok2 && st.row2 < nr;
        uint64_t Q[16];
        st.pass2_load(buf_off, valid, Q);
        // the buffer is refilled by the async proxy: order this warp's generic-proxy accesses (reads and the in-place
        // writes of pass 1) before the copy that lane 0 issues next
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        issue(s);                       // step k + 2 into the buffer step k just left
        st.pass2_finish(valid, Q, co);
    };
    uint32_t phase = 0;
    for (uint32_t done = 0; done < n_mine; done += 4u) {
        step(0, done, phase);
        if (done + 2u < n_mine) step(1, done + 2u, phase);
        phase ^= 1u;
    }
    if constexpr (CODES) zero_codes_padding(co, n_rows, cpr);
}

// Registers: about 20 resident warps per SM at 96 registers; the adaLN variant keeps 32 more operands live and gets 128
// (16 warps).
template <int FMT, bool QUANT, bool CODES>
__global__ void __maxnreg__(96) transform_rotate_quant_stream_kernel(const float* __restrict__ x, const float* __restrict__ smooth,
                                                                    SignMask sm, __half* __restrict__ out, __half* __restrict__ rotated,
                                                                    size_t n_rows, int cpr, Modulate mod, CodesOut co) {
    rotate_stream_body<FMT, QUANT, false, CODES>(x, smooth, sm, out, rotated, n_rows, cpr, mod, co);
}
template <int FMT, bool QUANT, bool CODES>
__global__ void __maxnreg__(128) modulate_transform_rotate_quant_stream_kernel(const float* __restrict__ x, const float* __restrict__ smooth,
                                                                              SignMask sm, __half* __restrict__ out, __half* __restrict__ rotated,
                                                                              size_t n_rows, int cpr, Modulate mod, CodesOut co) {
    rotate_stream_body<FMT, QUANT, true, CODES>(x, smooth, sm, out, rotated, n_rows, cpr, mod, co);
}

// Weight side: one warp per (row, chunk); lane l holds elements 4l..4l+3 in fp64.  w_out may alias w (in place): every
// element is read and written by the same thread, and neither pointer is declared __restrict__.
__global__ void __launch_bounds__(256) transform_rotate_weight_kernel(const float* w, const float* __restrict__ smooth,
                                                                      SignMask sm, float* w_out, size_t n_chunks,
                                                                      int chunks_per_row) {
    const int lane = threadIdx.x & 31;
    const size_t warp_global = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = (size_t(gridDim.x) * blockDim.x) >> 5;
    for (size_t c = warp_global; c < n_chunks; c += n_warps) {
        const float4 w4 = *reinterpret_cast<const float4*>(w + c * 128 + 4 * lane);
        float f[4] = {w4.x, w4.y, w4.z, w4.w};
        if (smooth != nullptr) {
            const float4 s4 = __ldg(reinterpret_cast<const float4*>(smooth + size_t(c % chunks_per_row) * 128 + 4 * lane));
            f[0] = __fdiv_rn(f[0], s4.x); f[1] = __fdiv_rn(f[1], s4.y);          // transform_model_utils.py:12 (fp32)
            f[2] = __fdiv_rn(f[2], s4.z); f[3] = __fdiv_rn(f[3], s4.w);
        }
        double d[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int e = 4 * lane + k;
            const bool plus = (sm.w[e >> 5] >> (e & 31)) & 1u;
            d[k] = plus ? double(f[k]) : -double(f[k]);
        }
        // strides 1, 2 in registers
        { const double a = d[0] + d[1], b = d[0] - d[1], c2 = d[2] + d[3], e2 = d[2] - d[3];
          d[0] = a + c2; d[2] = a - c2; d[1] = b + e2; d[3] = b - e2; }
        // strides 4..64 across the 32 lanes
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const bool upper = lane & o;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const double p = __shfl_xor_sync(0xffffffffu, d[k], o);
                d[k] = upper ? p - d[k] : d[k] + p;
            }
        }
        const double c64 = double(11.313708305358887f);       // fl32(sqrt(128)) widened, hadamard_utils.py:85
        float4 o4;
        o4.x = float(d[0] / c64); o4.y = float(d[1] / c64); o4.z = float(d[2] / c64); o4.w = float(d[3] / c64);
        *reinterpret_cast<float4*>(w_out + c * 128 + 4 * lane) = o4;
    }
}

}  // namespace fpq

using namespace fpq;

// Launch geometry of the streaming kernel: warps per CTA (one per 4 chunk columns) and CTAs per SM (register budget:
// about 20 warps, 16 with the adaLN operands).
struct RotPlan { int warps; int ctas_per_sm; };
static bool rot_plan(int cpr, bool mod, RotPlan& p) {
    if (cpr < ROT_MIN_CPR || cpr > ROT_MAX_CPR) return false;
    p.warps = (cpr + 3) / 4;
    p.ctas_per_sm = (mod ? 16 : 20) / p.warps;
    // shared-memory budget: the carveout every activation kernel asks for (1 KB per CTA is reserved by the system)
    const int kb = g_tun.smem_kb > 0 ? g_tun.smem_kb : 228;
    const int by_smem = kb * 1024 / (p.warps * ROT_WARP_SMEM + 1024);
    if (p.ctas_per_sm > by_smem) p.ctas_per_sm = by_smem;
    if (p.ctas_per_sm < 1) p.ctas_per_sm = 1;
    return true;
}

template <int FMT, bool QUANT, bool MOD, bool CODES>
static int launch_stream(const float* x, const float* smooth, const SignMask& sm, __half* o, __half* rot, const CodesOut& co, size_t n_rows,
                         int cpr, const RotPlan& plan, const Modulate& m, cudaStream_t st) {
    void (*kernel)(const float*, const float*, SignMask, __half*, __half*, size_t, int, Modulate, CodesOut);
    if constexpr (MOD) kernel = modulate_transform_rotate_quant_stream_kernel<FMT, QUANT, CODES>;
    else kernel = transform_rotate_quant_stream_kernel<FMT, QUANT, CODES>;
    const size_t smem = size_t(plan.warps) * ROT_WARP_SMEM;
    static bool attr_done[64] = {};                    // per instantiation and device
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_done[dev & 63]) {
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (ROT_MAX_CPR + 3) / 4 * ROT_WARP_SMEM) != cudaSuccess) return FPQ_ERR_CUDA;
        attr_done[dev & 63] = true;
    }
    const size_t steps = (n_rows + 1) / 2;
    const size_t cap = size_t(sm_count()) * plan.ctas_per_sm;
    const unsigned grid = unsigned(steps < cap ? steps : cap);
    launch_pdl(kernel, grid, unsigned(32 * plan.warps), smem, st, x, smooth, sm, o, rot, n_rows, cpr, m, co);
    return finish_launch();
}

template <int FMT, bool QUANT, bool MOD, bool CODES>
static int launch_small(const float* x, const float* smooth, const SignMask& sm, __half* o, __half* rot, const CodesOut& co, size_t n_rows,
                        int cpr, const Modulate& m, cudaStream_t st) {
    // lane sets, one per (chunk column, row phase); enough to fill every SM's thread slots (the modulate variant holds
    // three operand tables in registers: 2 resident CTAs instead of 4)
    const size_t max_sets = size_t(sm_count()) * (MOD ? 1024 : 2048) / 8;
    size_t sets_per_col = max_sets / size_t(cpr);
    if (sets_per_col < 1) sets_per_col = 1;
    if (sets_per_col > n_rows) sets_per_col = n_rows;
    // equal work per set: with `trips` passes over the rows, use just enough sets that every pass is full
    const size_t trips = (n_rows + sets_per_col - 1) / sets_per_col;
    sets_per_col = (n_rows + trips - 1) / trips;
    const size_t n_sets = sets_per_col * size_t(cpr);
    const unsigned grid = unsigned((n_sets + 31) / 32);            // 32 lane sets per 256-thread block
    launch_pdl(transform_rotate_quant_small_kernel<FMT, QUANT, MOD, CODES>, grid, 256, 0, st, x, smooth, sm, o, rot, n_rows, cpr, sets_per_col, m, co);
    return finish_launch();
}

template <int FMT, bool QUANT, bool CODES>
static int launch_fmt(const float* x, const Modulate* mod, const float* smooth, const SignMask& sm, __half* o, __half* rot, const CodesOut& co,
                      size_t n_rows, int cpr, cudaStream_t st) {
    const Modulate m = mod ? *mod : Modulate{nullptr, nullptr, 1, 1.0f};
    RotPlan plan;
    const bool big = n_rows * size_t(cpr) > size_t(g_tun.rot_small_max_chunks) && rot_plan(cpr, mod != nullptr, plan) &&
                     (mod == nullptr || mod->rows_per_batch >= 2) &&
                     ((reinterpret_cast<uintptr_t>(o) | reinterpret_cast<uintptr_t>(rot)) & 15) == 0;      // 128-bit stores
    if (big) return mod ? launch_stream<FMT, QUANT, true, CODES>(x, smooth, sm, o, rot, co, n_rows, cpr, plan, m, st)
                        : launch_stream<FMT, QUANT, false, CODES>(x, smooth, sm, o, rot, co, n_rows, cpr, plan, m, st);
    return mod ? launch_small<FMT, QUANT, true, CODES>(x, smooth, sm, o, rot, co, n_rows, cpr, m, st)
               : launch_small<FMT, QUANT, false, CODES>(x, smooth, sm, o, rot, co, n_rows, cpr, m, st);
}

// Checks shared by both outputs
static int check_rotate_args(const float* x, const Modulate* mod, const float* smooth, const uint32_t* sign_bits_host, size_t n_rows, size_t n_cols) {
    if (n_cols == 0 || n_cols % 128 != 0 || n_cols / 128 > 0x7fffffff / 512 || !sign_bits_host || (n_rows && !x)) return FPQ_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(smooth)) & 15) return FPQ_ERR_ARG;
    if (mod != nullptr) {
        if (!mod->scale || !mod->shift || mod->rows_per_batch == 0 || n_rows % mod->rows_per_batch != 0) return FPQ_ERR_ARG;
        if ((reinterpret_cast<uintptr_t>(mod->scale) | reinterpret_cast<uintptr_t>(mod->shift)) & 15) return FPQ_ERR_ARG;
    }
    return FPQ_OK;
}

// format: FPQ_FMT_*, or -1 (rotation only) for the fp16 output
template <bool CODES>
static int launch_rotate(const float* x, const Modulate* mod, const float* smooth, const uint32_t* sign_bits_host, __half* o, __half* rot,
                         const CodesOut& co, size_t n_rows, size_t n_cols, int format, void* stream) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    SignMask sm;
    for (int i = 0; i < 4; ++i) sm.w[i] = sign_bits_host[i];
    const int cpr = int(n_cols / 128);
    if constexpr (!CODES) {
        if (format == -1) return launch_fmt<0, false, false>(x, mod, smooth, sm, o, rot, co, n_rows, cpr, st);
    }
    return with_sym_format(format, [&](auto fmt) { return launch_fmt<fmt.value, true, CODES>(x, mod, smooth, sm, o, rot, co, n_rows, cpr, st); });
}

static int launch_rotate_quant(const float* x, const Modulate* mod, const float* smooth, const uint32_t* sign_bits_host, void* out, void* rotated,
                               size_t n_rows, size_t n_cols, int format, void* stream) {
    if (int rc = check_rotate_args(x, mod, smooth, sign_bits_host, n_rows, n_cols)) return rc;
    if ((n_rows && !out) || format < -1 || format >= FPQ_NUM_SYM_FORMATS) return FPQ_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(rotated)) & 7) return FPQ_ERR_ARG;
    if (n_rows == 0) return FPQ_OK;
    return launch_rotate<false>(x, mod, smooth, sign_bits_host, static_cast<__half*>(out), static_cast<__half*>(rotated), CodesOut{nullptr, nullptr, 0},
                                n_rows, n_cols, format, stream);
}

static int launch_rotate_codes(const float* x, const Modulate* mod, const float* smooth, const uint32_t* sign_bits_host, uint8_t* codes, float* scales,
                               size_t n_rows, size_t n_cols, int format, void* stream) {
    if (int rc = check_rotate_args(x, mod, smooth, sign_bits_host, n_rows, n_cols)) return rc;
    if ((n_rows && (!codes || !scales)) || format < 0 || format >= FPQ_NUM_SYM_FORMATS) return FPQ_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(codes) & 15) || (reinterpret_cast<uintptr_t>(scales) & 3)) return FPQ_ERR_ARG;
    if (n_rows == 0) return FPQ_OK;
    if (fpq_codes_rows_padded(n_rows) > 0xFFFFFFFFull) return FPQ_ERR_UNSUPPORTED;      // the streaming kernel counts rows in 32 bits
    return launch_rotate<true>(x, mod, smooth, sign_bits_host, nullptr, nullptr, CodesOut{codes, scales, fpq_codes_rows_padded(n_rows)}, n_rows,
                               n_cols, format, stream);
}

// Introspection for the CPU tests (tests/rotate_layout_model.py mirrors the launcher): plan[2] = {warps per CTA, CTAs per SM}.
extern "C" int fpq_rotate_plan(int chunks_per_row, int with_modulate, int* plan_host) {
    RotPlan p;
    if (plan_host == nullptr || chunks_per_row < 1) return FPQ_ERR_ARG;
    if (!rot_plan(chunks_per_row, with_modulate != 0, p)) return FPQ_ERR_UNSUPPORTED;
    plan_host[0] = p.warps;
    plan_host[1] = p.ctas_per_sm;
    return FPQ_OK;
}

extern "C" int fpq_transform_rotate_quant(const float* x, const float* smooth, const uint32_t* sign_bits_host, void* out, void* rotated,
                                          size_t n_rows, size_t n_cols, int format, void* stream) {
    return launch_rotate_quant(x, nullptr, smooth, sign_bits_host, out, rotated, n_rows, n_cols, format, stream);
}

extern "C" int fpq_modulate_transform_rotate_quant(const float* x, const float* scale, const float* shift, size_t rows_per_batch,
                                                   const float* smooth, const uint32_t* sign_bits_host, void* out, void* rotated,
                                                   size_t n_rows, size_t n_cols, int format, int flags, void* stream) {
    if (flags & ~FPQ_MOD_GAIN) return FPQ_ERR_ARG;
    const Modulate m{scale, shift, rows_per_batch, (flags & FPQ_MOD_GAIN) ? -0.0f : 1.0f};
    return launch_rotate_quant(x, &m, smooth, sign_bits_host, out, rotated, n_rows, n_cols, format, stream);
}

extern "C" int fpq_transform_rotate_pack_codes(const float* x, const float* smooth, const uint32_t* sign_bits_host, uint8_t* codes, float* scales,
                                               size_t n_rows, size_t n_cols, int format, void* stream) {
    return launch_rotate_codes(x, nullptr, smooth, sign_bits_host, codes, scales, n_rows, n_cols, format, stream);
}

extern "C" int fpq_modulate_transform_rotate_pack_codes(const float* x, const float* scale, const float* shift, size_t rows_per_batch,
                                                        const float* smooth, const uint32_t* sign_bits_host, uint8_t* codes, float* scales,
                                                        size_t n_rows, size_t n_cols, int format, int flags, void* stream) {
    if (flags & ~FPQ_MOD_GAIN) return FPQ_ERR_ARG;
    const Modulate m{scale, shift, rows_per_batch, (flags & FPQ_MOD_GAIN) ? -0.0f : 1.0f};
    return launch_rotate_codes(x, &m, smooth, sign_bits_host, codes, scales, n_rows, n_cols, format, stream);
}

extern "C" int fpq_transform_rotate_weight(const float* w, const float* smooth, const uint32_t* sign_bits_host, float* w_out, size_t n_rows,
                                           size_t n_cols, void* stream) {
    if (n_cols == 0 || n_cols % 128 != 0 || !sign_bits_host || (n_rows && (!w || !w_out))) return FPQ_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(smooth) | reinterpret_cast<uintptr_t>(w_out)) & 15) return FPQ_ERR_ARG;
    if (n_rows == 0) return FPQ_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    SignMask sm;
    for (int i = 0; i < 4; ++i) sm.w[i] = sign_bits_host[i];
    const int cpr = int(n_cols / 128);
    const size_t n_chunks = n_rows * size_t(cpr);
    transform_rotate_weight_kernel<<<grid_for(n_chunks, 8, 64), 256, 0, st>>>(w, smooth, sm, w_out, n_chunks, cpr);
    return finish_launch();
}
