/*
 * fpq_b200.h -- C ABI of libfpq_b200.so: the B200 (sm_100a) implementation of FPQVAR's
 * floating-point fake-quantization hot path.
 *
 * Conventions (every entry point):
 *   - plain C types only; pointers are DEVICE pointers unless a name ends in `_host`;
 *   - nothing allocates, nothing synchronises; work is enqueued on `stream`
 *     (a cudaStream_t passed as void*; NULL = the legacy default stream);
 *   - the return value is 0 on success or a negative FPQ_ERR_* code; launch errors are
 *     reported as FPQ_ERR_CUDA and the CUDA error is retrievable with fpq_last_cuda_error();
 *   - inputs are never modified (the reference's in-place `x.div_(scale)`,
 *     models_fp_quant_transform_rotate/quant_utils.py:306, is a host-side concern).
 *
 * Reference interfaces replaced (paths relative to the reference repository root;
 * "qu.py" = models_fp_quant_transform_rotate/quant_utils.py, "qu0.py" =
 * models_fp_quant/quant_utils.py):
 *   fpq_quant_grid            quant_cuda.quant            quant/quant.cpp:17-29, quant/quant_kernel.cu:11-62
 *   fpq_fake_quant            fp_quant_e{1,2,3}_per_group_cuda qu.py:265-378, fp6_quant_*_per_{group,token}_cuda
 *                             qu.py:503-574, argmin variants qu.py:237-358, quantize_to_nearest_grid qu.py:209-230
 *   fpq_fake_quant_signsplit  fp_quant_e1m2_neg_e2m1_pos_per_group[_cuda] qu.py:381-452,
 *                             fp6_quant_int_neg_e2m3_pos_per_{group,token}_cuda qu.py:577-646,
 *                             fp4_afpq_per_group_cuda qu0.py:498-535
 *   fpq_transform_rotate_quant   basic_var.py:263,266 (`.mul(s)` + `matmul(., Q)`) fused with the
 *                             following QuantizedLinear.forward act_quant qu.py:764-769
 *   fpq_transform_rotate_weight  learnable_transformation/transform_model_utils.py:8-28 +
 *                             rotate_utils/rotation_utils.py:129-154
 *   fpq_score_formats         search/search_fp4_format.py:340-374,472-476,840-893 and
 *                             search/search_fp6_format.py:547-554 (tensor-level quantize + MSE)
 *   fpq_pack_codes / fpq_gemm_codes   QuantizedLinear.forward qu.py:764-769 (act_quant + F.linear) as a real low-bit GEMM
 *   fpq_[modulate_]transform_rotate_pack_codes   basic_var.py:263,266 fused with the act_quant of that GEMM, emitting codes
 */
#ifndef FPQ_B200_H
#define FPQ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define FPQ_API __attribute__((visibility("default")))
#else
#define FPQ_API
#endif

/* ---- error codes ---------------------------------------------------------------- */
#define FPQ_OK               0
#define FPQ_ERR_ARG         -1   /* bad enum / size / alignment                         */
#define FPQ_ERR_UNSUPPORTED -2   /* valid request this build has no kernel for          */
#define FPQ_ERR_CUDA        -3   /* CUDA runtime reported an error at launch            */

/* ---- element types -------------------------------------------------------------- */
#define FPQ_F32 0
#define FPQ_F16 1

/* ---- symmetric formats (qu.py:233-235, 458-486) ---------------------------------- */
#define FPQ_FMT_E2M1 0   /* "fp_e2"    +-{0,.5,1,1.5,2,3,4,6}             max 6    */
#define FPQ_FMT_E1M2 1   /* "fp_e1"    +-{0,.25,...,1.75}                 max 1.75 */
#define FPQ_FMT_E3M0 2   /* "fp_e3"    +-{0,.25,.5,1,2,4,8,16}            max 16   */
#define FPQ_FMT_E2M3 3   /* "fp6_e2m3" 6-bit, 3 mantissa bits             max 7.5  */
#define FPQ_FMT_E3M2 4   /* "fp6_e3m2" 6-bit, 2 mantissa bits             max 28   */
#define FPQ_NUM_SYM_FORMATS 5

/* ---- sign-split formats: separate grid and scale for x<=0 and x>0 ----------------- */
#define FPQ_SPLIT_E1M2NEG_E2M1POS 0  /* "fp_e1m2_neg_e2m1_pos" qu.py:415-452         */
#define FPQ_SPLIT_INTNEG_E2M3POS  1  /* "fp6_int_neg_e2m3_pos" qu.py:577-646         */
#define FPQ_SPLIT_AFPQ_E2M1       2  /* "fp4_afpq"             qu0.py:498-535        */
#define FPQ_NUM_SPLIT_FORMATS 3

/* ---- tie rule -------------------------------------------------------------------- */
#define FPQ_TIE_KERNEL 0  /* quant_cuda.quant: exact ties -> the LARGER grid value, NaN/inf -> +0
                             (quant/quant_kernel.cu:25-37)                                     */
#define FPQ_TIE_ARGMIN 1  /* torch.argmin:     exact ties -> the SMALLER grid value, NaN/inf -> grid[0]
                             (qu.py:224-230)                                                   */

/* ---- flags ----------------------------------------------------------------------- */
#define FPQ_FLAG_CLAMP3      1u  /* torch.clamp(x,-3,3) first (qu.py:241,254,289,337,350)          */
#define FPQ_FLAG_GLOBAL_CLIP 2u  /* sign-split only: reproduce the whole-tensor clip of qu.py:421-422
                                    at clipping_strength 1.0, i.e. "a NaN anywhere poisons the whole
                                    tensor"; needs `workspace` (see fpq_fake_quant_signsplit)       */

FPQ_API const char *fpq_version(void);
/* cudaGetErrorString of the last CUDA error seen by this library on the calling thread. */
FPQ_API const char *fpq_last_cuda_error(void);
/* How many of this library's kernels the calling thread has launched (bench.py's gpu_launches). */
FPQ_API uint64_t fpq_launch_count(void);

/*
 * Measurement aid: launch-geometry choices that were made from measurements can be moved at run time (by tools/ and the
 * GPU tests; never through the environment).  Process-wide; not meant to be changed while other threads launch.
 *   "pdl"                  1 (default) | 0: programmatic dependent launch of the activation kernels on / off
 *   "row_v"                0 (default: chosen per row length) | 1 | 2 | 4: 16-byte vectors per thread of the per-token kernels
 *   "rot_small_max_chunks" rotate launches of up to this many 128-chunks take the small-launch kernel (default 40000)
 *   "smem_kb"              0 (default: the driver chooses per kernel) | 1..228: the shared-memory carveout (KB per SM) every
 *                          activation kernel asks for, and the streaming rotate kernel's shared-memory budget
 *   "gemm_tile_n", "gemm_epi_cols", "gemm_stages", "gemm_pair"   tile shape, epilogue split, ring depth and CTA pairing of
 *                          fpq_gemm_codes (see there)
 * Results never depend on a tunable (tests/test_gpu_shapes.py).  Returns FPQ_ERR_ARG for an unknown name or value.
 */
FPQ_API int fpq_set_tunable(const char *name, long long value);

/*
 * z[i] = nearest entry of grid[0..k) to x[i] (fp32, n elements), reference scan semantics;
 * k <= 256.  tie_mode FPQ_TIE_KERNEL reproduces quant_cuda.quant exactly, including grids it
 * has never seen (unsorted, duplicated entries); the reference's own grids take a closed-form
 * path that is proven equal to the scan over all 2^32 inputs (fpq_selftest_rounding).
 * The reference's second output (`idx`, never written, quant/quant_kernel.cu:49,58) is the
 * binding's business, not this library's.
 */
FPQ_API int fpq_quant_grid(const float *x, const float *grid, int k, size_t n, float *z,
                   int tie_mode, void *stream);

/*
 * Symmetric fake-quant: absmax scale -> divide -> grid rounding -> multiply back, in one pass.
 *   x, out      : n_rows * row_len elements, contiguous; may NOT alias
 *   row_len     : elements that share one scale: the group size for per_group (128 in the
 *                 reference; 32..512 powers of two take the group kernel) or the last-dim
 *                 length for per_token / per_channel (any length >= 1)
 *   in_dtype    : FPQ_F32 | FPQ_F16;  out_dtype: FPQ_F32 | FPQ_F16
 *                 (fp16 input reproduces the reference's fp16 scale and fp16 normalised
 *                 value roundings bit for bit)
 *   format      : FPQ_FMT_*;  tie_mode: FPQ_TIE_*;  flags: FPQ_FLAG_CLAMP3 or 0
 */
FPQ_API int fpq_fake_quant(const void *x, void *out, size_t n_rows, size_t row_len,
                   int in_dtype, int out_dtype, int format, int tie_mode,
                   unsigned flags, void *stream);

/*
 * Symmetric fake-quant of `n_segments` equally long pieces of a larger fp16 tensor, optionally IN PLACE: segment i starts at
 * x + i * pitch_x (elements) and holds rows_per_segment rows of row_len (64 | 128) contiguous halves; kernel tie rule,
 * fp16 in and out.  out may equal x (with pitch_out == pitch_x); no other overlap.  This is the KV-cache call: the
 * reference re-quantizes `self.cached_k` / `self.cached_v` before every append (models_fp_quant_transform_rotate/
 * basic_var.py:192-197, fp6_quant_e2m3_per_token_cuda rows of head_dim = 64 / fp_quant_e2_per_group_cuda groups of 128);
 * with a preallocated cache [B, L_max, H, head_dim] the rows appended at one scale are B segments of pitch
 * L_max * H * head_dim, quantized where they lie (fpqvar_b200/kv_cache.py).
 */
FPQ_API int fpq_fake_quant_segments(const void *x, void *out, size_t n_segments, size_t rows_per_segment,
                   size_t row_len, size_t pitch_x, size_t pitch_out, int format, void *stream);

/*
 * Sign-split fake-quant (fc2 inputs): x<=0 and x>0 get their own grid and their own absmax
 * scale per row; out = q_neg*s_neg + q_pos*s_pos.  Arguments as fpq_fake_quant;
 * `split_format` is FPQ_SPLIT_*.  With FPQ_FLAG_GLOBAL_CLIP, `workspace` must point to 8 bytes
 * of device memory that were zero when first used ({flag, ticket}); the kernel raises the flag
 * when the tensor holds a NaN, the last CTA to finish then rewrites `out` as the reference would
 * (all +0) and zeroes the workspace again, so one workspace serves any number of calls on one
 * stream without a memset in between.  Without the flag a NaN element is treated as 0 locally
 * (qu.py:428-429) and `workspace` is unused.
 */
FPQ_API int fpq_fake_quant_signsplit(const void *x, void *out, size_t n_rows, size_t row_len,
                             int in_dtype, int out_dtype, int split_format, int tie_mode,
                             unsigned flags, void *workspace, void *stream);

/*
 * Fused activation path of the rotated/transformed model (basic_var.py:263,266 followed by
 * QuantizedLinear.forward qu.py:764-769):
 *     y   = half( FWHT_128( x[., c] * m[c] ) ),   m[c] = fl32(smooth[c] * fl32(1/sqrt(128))) * sign[c % 128]
 *     out = fake_quant_group128(y, format)         (fp16 in, fp16 out, FPQ_TIE_KERNEL)
 *   x        : fp32 [n_rows, n_cols], n_cols % 128 == 0 (adaLN-modulated LayerNorm output)
 *   smooth   : fp32 [n_cols] GALT factor s, or NULL for 1
 *   sign_bits: 128-bit mask, bit i of word i/32 set = +1 (the seed-42 vector of
 *              rotate_utils/hadamard_utils.py:95-97); host memory, read at call time
 *   out      : fp16 [n_rows, n_cols] fake-quantized; 8-byte aligned (16-byte aligned outputs let large launches take the
 *              streaming kernel; the values do not depend on which kernel runs)
 *   rotated  : optional fp16 [n_rows, n_cols]: the pre-quantization rotated values (NULL to skip)
 *   format   : FPQ_FMT_* or -1 to skip quantization (then `out` receives the rotated values)
 */
FPQ_API int fpq_transform_rotate_quant(const float *x, const float *smooth, const uint32_t *sign_bits_host,
                               void *out, void *rotated, size_t n_rows, size_t n_cols,
                               int format, void *stream);

/*
 * Same, with the adaLN modulate that precedes it in the reference fused in as well (SURVEY.md section 8f,
 * rank 1; basic_var.py:263,266 `self.ln_wo_grad(x).mul(scale1.add(1)).add_(shift1).mul(best_s)`):
 *     t[r, c] = ( x[r, c] * (scale[b, c] + 1) + shift[b, c] ) * smooth[c],   b = r / rows_per_batch
 * computed as the reference's four separately rounded fp32 operations, then rotated and quantized as above.
 *   x            : fp32 [n_rows, n_cols], the LayerNorm output; n_rows % rows_per_batch == 0
 *   scale, shift : fp32 [n_rows / rows_per_batch, n_cols] (the [B, 1, C] adaLN tensors), 16-byte aligned
 *   flags        : 0, or FPQ_MOD_GAIN: `scale` already holds the gain (scale + 1).  The reference's evaluation runs
 *                  under fp16 autocast (evaluate_fp_quant_transform_rotate.py:195), where scale1/shift1 are fp16 and
 *                  `scale1.add(1)` is rounded to fp16 before the fp32 multiply; such a caller passes
 *                  float(half(scale + 1)) and float(shift), both exact, and the kernel skips its own fp32 `+ 1`.
 */
#define FPQ_MOD_GAIN 1
FPQ_API int fpq_modulate_transform_rotate_quant(const float *x, const float *scale, const float *shift, size_t rows_per_batch,
                                        const float *smooth, const uint32_t *sign_bits_host, void *out, void *rotated,
                                        size_t n_rows, size_t n_cols, int format, int flags, void *stream);

/*
 * Launch plan of the streaming rotate kernel for rows of `chunks_per_row` 128-element chunks, without / with the adaLN
 * modulate (host-only query, no CUDA call; the CPU tests use it to keep tests/rotate_layout_model.py in step with the
 * launcher): plan_host[2] = {warps per CTA (one per 4 chunk columns), CTAs per SM}.  FPQ_ERR_UNSUPPORTED when such
 * rows only take the small-launch kernel.
 */
FPQ_API int fpq_rotate_plan(int chunks_per_row, int with_modulate, int *plan_host);

/*
 * Weight side of the same transform (transform_model_utils.py:8-28, rotation_utils.py:129-154):
 *     w_out[r, :] = float( FWHT_128_f64( (w[r, c] / smooth[c]) * sign[c % 128] ) / fl32(sqrt(128)) )
 * fp32 in/out, fp64 butterflies; in-place allowed (w_out == w).  smooth may be NULL.
 */
FPQ_API int fpq_transform_rotate_weight(const float *w, const float *smooth, const uint32_t *sign_bits_host,
                                float *w_out, size_t n_rows, size_t n_cols, void *stream);

/*
 * Batched format scoring: for every candidate c in formats[0..n_formats) accumulate
 *     sse[c] += sum_i (x[i] - fake_quant(x, format c)[i])^2          (fp64 accumulators)
 * reading x ONCE.  formats[] entries: FPQ_FMT_* (0..4) or 16+FPQ_SPLIT_* for sign-split
 * candidates; host array.  sse: n_formats doubles on the device, accumulated into (the caller
 * zeroes them and divides by the element count for the reference's mean).
 */
FPQ_API int fpq_score_formats(const void *x, size_t n_rows, size_t row_len, int in_dtype,
                      const int *formats_host, int n_formats, int tie_mode,
                      double *sse, void *stream);

/*
 * GELU(tanh) + sign-split fake-quant of an fp16 tensor in one pass, groups of 128, kernel tie rule:
 *     out = fp_quant_*_neg_*_pos_per_group_cuda( gelu(x, approximate="tanh") )
 * i.e. `fc2.act_quant(self.act(self.fc1(x)))` of the reference (models_fp_quant_transform_rotate/basic_var.py:108,120 ->
 * quant_utils.py:991-996) with x = the fp16 output of fc1.  The GELU reproduces ATen's CUDA kernel for Half tensors bit for bit
 * (fpq_selftest_gelu: all 65 536 inputs).  flags / workspace as fpq_fake_quant_signsplit.  SURVEY.md section 8 f1.
 */
FPQ_API int fpq_gelu_fake_quant_signsplit(const void *x, void *out, size_t n_groups, int split_format,
                   unsigned flags, void *workspace, void *stream);
/* table[i] = fp16( gelu_tanh( fp16 bit pattern i ) ) for i in [0, 65536): the device function of the kernel above */
FPQ_API int fpq_selftest_gelu(void *table_65536_halves, void *stream);

/*
 * Output-level loss of the format search: *out += sum_r w[r] * sum_c (a[r,c] - b[r,c])^2 over two row-major
 * [n_rows, n_cols] matrices of the same dtype (FPQ_F32 | FPQ_F16), read once each; row_weight (float64, n_rows entries) may
 * be NULL (= 1); out is one float64 accumulator the caller zeroes.  n_cols must fill whole 16-byte vectors.  Replaces
 * compute_quant_error(y_fp, y_q) = mean((y_fp - y_q)^2) inside the reference's search loop
 * (search/search_fp4_format.py:472-476, :798-816; search_fp6_format.py:807-868).
 */
FPQ_API int fpq_sse_rows(const void *a, const void *b, size_t n_rows, size_t n_cols, int dtype,
                   const double *row_weight, double *out, void *stream);

/*
 * Exhaustive self-check used by the GPU test-suite: for ALL 2^32 fp32 bit patterns compare the
 * closed-form rounding of `format` (FPQ_FMT_* or 16+half-grid id, 16 = int_neg, 17 = e2m3_pos, 18 = e1m2_neg, 19 = e2m1_pos, 20 = e2m1_neg; fpq_grid.cu) under
 * `tie_mode` with the literal reference scan over the same grid.  result[0] = mismatch count,
 * result[1] = bit pattern of the first mismatch found (device memory, 2 x uint64).
 */
FPQ_API int fpq_selftest_rounding(int format, int tie_mode, unsigned long long *result, void *stream);

/*
 * Exhaustive self-check of the packed fp16 activation path (fp16 in, fp16 out, FPQ_TIE_KERNEL):
 * for EVERY pair (x, scale) of fp16 values that can meet in a group with a normal scale, compare
 * the division-free element function of the fast kernels with the literal reference sequence
 * divide -> half -> scan -> multiply -> half (qu.py:320-329 / :432-451).  `format`: FPQ_FMT_*,
 * 16+FPQ_SPLIT_*, or 32+FPQ_FMT_{E2M1,E1M2,E2M3,E3M2} for the element function on the FP4/FP6 conversion
 * hardware (the format scorer's).  result as in fpq_selftest_rounding.
 */
FPQ_API int fpq_selftest_f16_flow(int format, unsigned long long *result, void *stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Packed low-bit operands and the real low-bit GEMM (SURVEY.md section 8 f4).  NOT in the reference: QuantizedLinear.forward
 * (qu.py:764-769, :991-996) fake-quantizes the activation and calls F.linear on fp16 tensors whose values happen to lie on
 * scale * grid.  Here the same quantizer emits what those tensors ARE -- one grid value per element and one scale per
 * (row, 128-group) -- and the product runs on the tensor cores in 8-bit containers (tcgen05.mma kind::f8f6f4), the scales
 * applied per 128-deep K slab.  Numerics contract: fpq_unpack_codes(fpq_pack_codes(x)) is bit-identical to
 * fp_quant_*_per_group_cuda(x) (qu.py:265-378, :537-574; the reference's dtype rules: an fp16 input has an fp16-rounded scale);
 * fpq_gemm_codes is bit-identical to oracle/gemm_codes.c (fixed fp32 operation order) inside the exact-accumulation envelope
 *   k_acc * max|q_a| * max|q_w| / (u_a * u_w) <= 2^24        (u: the grid's resolution; k_acc = 128 with groups of 128, k with
 *                                                              row scales; oracle/lowbit.py exact_accumulation)
 * where every partial sum of a scale group is an fp32 number: every 128-group pair but e3m2 x e3m2 (24.6 bits); with row scales
 * e3m0 x e3m0 up to k = 4096, e2m1 x e2m1 up to k = 116480, FP6 pairs far less (e3m2 x e3m2 not even at k = 2304).  Outside
 * it a slab sum may differ from the exact one by (k_acc - 1) * 2^-24 * sum |qa * qw|.  It differs from the reference's fp16
 * GEMM of the fake-quantized tensors only by that GEMM's own roundings (each product term fp16-rounded once in the reference,
 * never here; tolerance stated in tests/test_gpu_gemm_codes.py).
 *
 * Layout of an operand of `rows` x k (k % 128 == 0), rows_pad = fpq_codes_rows_padded(rows) = rows rounded up to 128:
 *   codes  : rows_pad * k bytes, [k/128 slabs][rows_pad/8][8 chunks of 16 K][8 rows][16 bytes]; byte = e4m3 encoding of the grid
 *            value (every FP4 / FP6 grid of the reference is a subset of e4m3); padding rows hold 0
 *   scales : fp32 [k/128][rows_pad] (one per row and 128-group) or [1][rows_pad] (one per row); 0 for the padding rows
 * so that a 128-row x 128-K tile is 16 KB of contiguous memory in the tensor core's K-major core-matrix order.
 * ------------------------------------------------------------------------------------------------------------------ */
FPQ_API size_t fpq_codes_rows_padded(size_t rows);
/*
 * x: [rows, k] contiguous, FPQ_F16 | FPQ_F32, 16-byte aligned; format: FPQ_FMT_*; kernel tie rule.
 * scale_group: 128 = one scale per (row, 128-group), fp_quant_*_per_group_cuda (qu.py:265-378, 537-574); scales [k/128][rows_pad]
 *              k   = one scale per row, the per_token / per_channel functions (qu.py:503-534);          scales [1][rows_pad]
 */
FPQ_API int fpq_pack_codes(const void *x, size_t rows, size_t k, size_t scale_group, int in_dtype, int format, uint8_t *codes,
                   float *scales, void *stream);
/* out[r, c] = out_dtype( fl32(q) * scale ): the fake-quantized tensor the codes stand for, [rows, k] contiguous. */
FPQ_API int fpq_unpack_codes(const uint8_t *codes, const float *scales, size_t rows, size_t k, size_t scale_group,
                   int out_dtype, void *out, void *stream);
/* 4-bit storage of the FP4 formats (FPQ_FMT_E2M1 | E1M2 | E3M0): nibble = sign << 3 | index of |q| in the ascending
 * non-negative half grid; byte i of `nibbles` holds codes 2i (low nibble) and 2i+1.  n_codes % 8 == 0.  Lossless both ways. */
FPQ_API int fpq_codes_to_nibbles(const uint8_t *codes, size_t n_codes, int format, uint8_t *nibbles, void *stream);
FPQ_API int fpq_nibbles_to_codes(const uint8_t *nibbles, size_t n_codes, int format, uint8_t *codes, void *stream);
/*
 * The fused activation path straight to codes: fpq_transform_rotate_quant / fpq_modulate_transform_rotate_quant with the
 * quantized tensor emitted as an operand of fpq_gemm_codes (scale_group = 128) instead of as fp16, in ONE launch (padding rows
 * included): 4 bytes read and 1 + 4/128 written per element, instead of the fp16 rotation (4 + 2) followed by fpq_pack_codes
 * (2 + 1 + 1/32).  Arguments, alignment rules, FPQ_MOD_GAIN, the kernel tie rule and the choice between the small-launch and
 * the streaming kernel are those of the fp16 siblings, except:
 *   codes  : rows_pad * n_cols bytes in the layout above, 16-byte aligned (rows_pad = fpq_codes_rows_padded(n_rows))
 *   scales : fp32 [n_cols/128][rows_pad], 4-byte aligned; each an fp16-rounded value, as fpq_pack_codes stores for fp16 input
 *   format : FPQ_FMT_* (no -1: there is nothing to pack without a quantizer)
 * Numerics contract: codes and scales are bit-identical to fpq_pack_codes(rotated, n_rows, n_cols, 128, FPQ_F16, format), where
 * `rotated` is the fp16 output of the sibling call with format = -1; equivalently, fpq_unpack_codes of them to fp16 is
 * bit-identical to the sibling's fake-quantized output.
 */
FPQ_API int fpq_transform_rotate_pack_codes(const float *x, const float *smooth, const uint32_t *sign_bits_host,
                   uint8_t *codes, float *scales, size_t n_rows, size_t n_cols, int format, void *stream);
FPQ_API int fpq_modulate_transform_rotate_pack_codes(const float *x, const float *scale, const float *shift, size_t rows_per_batch,
                   const float *smooth, const uint32_t *sign_bits_host, uint8_t *codes, float *scales,
                   size_t n_rows, size_t n_cols, int format, int flags, void *stream);
/*
 * F.linear(A, W, bias) for A = [m, k] and W = [n, k] given as codes that share `scale_group` (128 or k):
 *   C[i, j] = bias[j] + fma-chain over the scale groups t (ascending) of  (P_t[i, j] * sa[t, i]) * sw[t, j],
 *             P_t[i, j] = sum over the group's k of qa[i, k] * qw[j, k]        (fp32 accumulate in tensor memory; exact inside
 *                                                                              the envelope above, within (k_acc - 1) * 2^-24 *
 *                                                                              sum |qa * qw| outside it)
 * c: [m, ldc] row-major, FPQ_F16 | FPQ_F32, 16-byte aligned, n % 8 == 0, ldc % 8 == 0; bias: fp32 [n] or NULL.
 * Persistent kernel, one CTA per SM, 128 x 256 (or 128 x 128) tiles of C, ~205 KB of shared memory.  With groups of 128 every
 * accumulator is handed to the epilogue warps once per 128 K (1.0-1.45 PFLOP/s on a B200); with row scales once per tile
 * (2.1-2.6 PFLOP/s; the fp16 library GEMM on the fake-quantized tensors runs at 1.4-1.5).
 * Tunables: "gemm_tile_n" (128 | 256, default 256), "gemm_epi_cols" (columns per epilogue warp: 32 | 64 | 128, default 128),
 * "gemm_stages" (2..6, default 6; as many as fit: 3 with 256-column tiles and the fp16 staging buffer), "gemm_pair" (1: clusters
 * of two CTAs with cta_group::2 MMAs, each holding half of the B tile; 0: single CTAs; -1 = default: pairs for row scales and >= 4
 * row tiles, where they measured 3-4 % faster).  Results never depend on them.
 */
FPQ_API int fpq_gemm_codes(const uint8_t *a_codes, const float *a_scales, size_t m, const uint8_t *b_codes,
                   const float *b_scales, size_t n, size_t k, size_t scale_group, const float *bias, int out_dtype,
                   void *c, size_t ldc, void *stream);
/*
 * Output-level loss of the format search without materialising the quantized layer's output (SURVEY.md section 8 f3;
 * search/search_fp4_format.py:472-476, :798-816: compute_quant_error(y_fp, F.linear(x_q, W_q))):
 *   *sse += sum_{i<m} row_weight[i] * sum_{j<n} (ref[i, j] - C[i, j])^2,   C as fpq_gemm_codes computes it in fp32 (never stored)
 * ref: [m, ldr] row-major, FPQ_F16 | FPQ_F32, the full-precision layer output; row_weight: float64 [m] or NULL (= 1): with the
 * calibration tensors stacked into one matrix, 1 / (rows_of_its_tensor * n * tensors) turns the sum into the reference's mean of
 * per-tensor means; sse: one float64 accumulator the caller zeroes.
 */
FPQ_API int fpq_gemm_codes_sse(const uint8_t *a_codes, const float *a_scales, size_t m, const uint8_t *b_codes,
                   const float *b_scales, size_t n, size_t k, size_t scale_group, const float *bias, int ref_dtype,
                   const void *ref, size_t ldr, const double *row_weight, double *sse, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FPQ_B200_H */
