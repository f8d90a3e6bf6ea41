/*
 * ORACLE (test infrastructure only; nothing in fpqvar_b200/ may load this).
 *
 * CPU statement of fpq_gemm_codes (include/fpq_b200.h): the product F.linear(q_x, W_q) of the reference's
 * QuantizedLinear.forward (models_fp_quant_transform_rotate/quant_utils.py:764-769) for operands given as
 * (grid value, scale per row and 128-group) pairs instead of the fp16 tensors q * scale the reference materialises
 * (qu.py:313-330).  Operation order of the fp32 arithmetic, which the CUDA kernel follows to the letter:
 *     for group t = 0 .. K/group - 1: P = sum_{k in group} qa[i,k] * qw[j,k]    (exact here, in double; the tensor core
 *                                    accumulates in fp32, which is exact too while every partial sum fits 24 bits:
 *                                    group * max|qa| * max|qw| / (u_a * u_w) <= 2^24, u the grid's resolution
 *                                    (oracle/lowbit.py exact_accumulation: every 128-group pair but e3m2 x e3m2; one scale
 *                                    per row: e3m0 x e3m0 up to K = 4096).  Outside it the kernel's P may differ from this
 *                                    one by (group - 1) * 2^-24 * sum |qa * qw|)
 *                                    acc = fmaf( P * sa[t,i]  (rounded to fp32),  sw[t,j],  acc )
 *     c[i,j] = acc + bias[j]
 * "parity unpinned" by the reference (it has no such operator); pinned instead against a float64 evaluation of the
 * reference's own expression in tests/test_oracle_gemm_codes.py.
 */
#include <math.h>
#include <stddef.h>

void gemm_codes_ref(const float *qa, const float *sa, size_t m, const float *qw, const float *sw, size_t n, size_t k,
                    size_t group, const float *bias, float *c) {
    const size_t slabs = k / group;          /* group = 128 (per_group) or k (per_token x per_channel: one scale pair) */
    for (size_t i = 0; i < m; ++i) {
        for (size_t j = 0; j < n; ++j) {
            float acc = 0.0f;
            for (size_t t = 0; t < slabs; ++t) {
                const float *a = qa + i * k + t * group, *w = qw + j * k + t * group;
                double p = 0.0;                      /* exact: |terms| <= 28*28, multiples of 2^-8 */
                for (size_t e = 0; e < group; ++e) p += (double)a[e] * (double)w[e];
                const float ps = (float)p * sa[t * m + i];
                acc = fmaf(ps, sw[t * n + j], acc);
            }
            c[i * n + j] = bias ? acc + bias[j] : acc;
        }
    }
}
