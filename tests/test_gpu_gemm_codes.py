"""GPU parity of the packed low-bit operands and the low-bit GEMM (csrc/fpq_gemm.cu) through the C ABI, against
oracle/lowbit.py + oracle/gemm_codes.c.  Bars: codes, scales and dequantized tensors bit-exact; GEMM bit-exact against the
fixed-order oracle (the slab sums are exact, the fp32 scale chain has a defined order); against the reference's own expression
-- F.linear on the fake-quantized fp16 tensors, QuantizedLinear.forward qu.py:764-769 -- within the tolerance written below."""
import numpy as np
import pytest
import torch

from fpqvar_b200 import _lib as L, lowbit, ops
from oracle import lowbit as LB, oracle as O          # checker only

pytestmark = pytest.mark.gpu
FMTS = ["e2m1", "e1m2", "e3m0", "e2m3", "e3m2"]


def bits(a):
    return a.view({1: np.uint8, 2: np.uint16, 4: np.uint32}[a.dtype.itemsize])


def dev():
    return torch.device("cuda:0")


def same_bits(a, b):
    """bit-identical, NaN payloads aside (signed zeros and NaN positions count)"""
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(bits(a)[~na], bits(b)[~nb])


def adversarial(rng, rows, k, dtype):
    x = rng.standard_normal((rows, k)).astype(dtype)
    x[0, :128] = 0
    x[1, 5] = np.inf
    x[2, 130] = np.nan
    x[3, :128] = (x[3, :128].astype(np.float32) * 2.0 ** -20).astype(dtype)
    x[4, :8] = np.asarray([0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0, 6.0], dtype=dtype)
    return x


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("dtype", [np.float16, np.float32])
@pytest.mark.parametrize("rows", [1, 300])
def test_pack_codes_bit_exact(fmt, dtype, rows):
    rng = np.random.default_rng(rows)
    x = adversarial(rng, max(rows, 5), 384, dtype)[:rows] if rows >= 5 else rng.standard_normal((rows, 384)).astype(dtype)
    p = lowbit.pack_codes(torch.from_numpy(x).to(dev()), fmt)
    wc, ws = LB.pack_codes(x, fmt)
    assert np.array_equal(p.codes.cpu().numpy(), wc)
    assert same_bits(p.scales.cpu().numpy(), ws)
    # and the codes stand for exactly the tensor the fake-quant kernels (and the reference) produce
    out_dt = torch.float16 if dtype == np.float16 else torch.float32
    got = p.dequantize(out_dt)
    want = ops.fake_quant(torch.from_numpy(x).to(dev()), fmt, 128, "kernel")
    if want.dtype != out_dt:                        # the FP6 functions force fp16 (qu.py:553,573)
        got = p.dequantize(want.dtype)
    assert same_bits(got.cpu().numpy(), want.cpu().numpy())
    assert same_bits(got.cpu().numpy(), O.fake_quant(x, fmt, 128, "kernel", out_dtype=got.cpu().numpy().dtype))


@pytest.mark.parametrize("fmt", ["e2m1", "e1m2", "e3m0"])
def test_nibble_storage_round_trip(fmt):
    rng = np.random.default_rng(7)
    x = rng.standard_normal((200, 256)).astype(np.float16)
    p = lowbit.pack_codes(torch.from_numpy(x).to(dev()), fmt)
    nib = p.to_nibbles()
    assert nib.numel() * 2 == p.codes.numel()
    assert np.array_equal(nib.cpu().numpy(), LB.codes_to_nibbles(p.codes.cpu().numpy(), fmt))
    back = lowbit.PackedCodes.from_nibbles(nib, p.scales, p.rows, p.k, fmt)
    assert torch.equal(back.codes, p.codes)


def test_nibble_storage_rejects_fp6():
    p = lowbit.pack_codes(torch.randn(8, 128, device=dev(), dtype=torch.float16), "e2m3")
    with pytest.raises(L.FpqError):
        p.to_nibbles()


def _operands(rng, m, n, k, fmt_a, fmt_w, dtype_a=np.float16):
    x = rng.standard_normal((m, k)).astype(dtype_a)
    w = (rng.standard_normal((n, k)) * 0.05).astype(np.float32)
    return x, w, LB.quantize_codes(x, fmt_a), LB.quantize_codes(w, fmt_w)


@pytest.mark.parametrize("m,n,k", [(128, 128, 128), (128, 128, 256), (1, 8, 128), (100, 136, 384), (300, 384, 1920), (257, 128, 7680),
                                   (700, 640, 640)])
@pytest.mark.parametrize("tile_n,epi_cols,stages,pair", [(256, 128, 3, 1), (256, 64, 4, 0), (256, 128, 2, 0), (256, 128, 2, 1), (128, 32, 6, 0),
                                                         (128, 64, 2, 0), (128, 128, 3, 0)])
def test_gemm_codes_bit_exact_against_the_fixed_order_oracle(m, n, k, tile_n, epi_cols, stages, pair):
    rng = np.random.default_rng(m + n + k)
    x, w, (qa, sa), (qw, sw) = _operands(rng, m, n, k, "e2m1", "e2m1")
    bias = rng.standard_normal(n).astype(np.float32)
    a = lowbit.pack_codes(torch.from_numpy(x).to(dev()), "e2m1")
    ww = lowbit.pack_codes(torch.from_numpy(w).to(dev()), "e2m1")
    L.set_tunable("gemm_stages", stages)
    L.set_tunable("gemm_tile_n", tile_n)
    L.set_tunable("gemm_epi_cols", epi_cols)
    L.set_tunable("gemm_pair", pair)
    try:
        c32 = lowbit.linear_codes(a, ww, torch.from_numpy(bias).to(dev()), torch.float32).cpu().numpy()
        c16 = lowbit.linear_codes(a, ww, None, torch.float16).cpu().numpy()
    finally:
        L.set_tunable("gemm_stages", 6)
        L.set_tunable("gemm_tile_n", 256)
        L.set_tunable("gemm_epi_cols", 128)
        L.set_tunable("gemm_pair", -1)
    assert np.array_equal(bits(c32), bits(LB.gemm_codes(qa, sa, qw, sw, bias)))
    assert np.array_equal(bits(c16), bits(LB.gemm_codes(qa, sa, qw, sw).astype(np.float16)))


def test_gemm_codes_many_tiles_per_cta():
    """more tiles than SMs: the persistent loop, the scale ring and both accumulators wrap several times"""
    rng = np.random.default_rng(99)
    m, n, k = 128 * 21 - 5, 256 * 9 + 128, 384          # 21 row tiles: the last CTA pair has a phantom second tile
    x, w, (qa, sa), (qw, sw) = _operands(rng, m, n, k, "e2m1", "e1m2")
    a = lowbit.pack_codes(torch.from_numpy(x).to(dev()), "e2m1")
    ww = lowbit.pack_codes(torch.from_numpy(w).to(dev()), "e1m2")
    want = LB.gemm_codes(qa, sa, qw, sw)
    for tile_n, epi_cols, pair in ((256, 128, 1), (256, 64, 0), (256, 128, 0), (128, 32, 0), (128, 64, 0), (128, 128, 0)):
        L.set_tunable("gemm_tile_n", tile_n)
        L.set_tunable("gemm_epi_cols", epi_cols)
        L.set_tunable("gemm_pair", pair)
        try:
            c = lowbit.linear_codes(a, ww, None, torch.float32).cpu().numpy()
            c16 = lowbit.linear_codes(a, ww, None, torch.float16).cpu().numpy()
        finally:
            L.set_tunable("gemm_tile_n", 256)
            L.set_tunable("gemm_epi_cols", 128)
            L.set_tunable("gemm_pair", -1)
        assert np.array_equal(bits(c), bits(want))
        assert np.array_equal(bits(c16), bits(want.astype(np.float16)))


@pytest.mark.parametrize("fmt_a,fmt_w,dtype", [("e2m1", "e2m1", np.float16), ("e1m2", "e3m0", np.float32), ("e2m3", "e2m3", np.float16),
                                               ("e3m2", "e3m2", np.float16)])
def test_row_scaled_codes_and_gemm(fmt_a, fmt_w, dtype):
    """per_token activations x per_channel weights (the README's W6A6 commands; fp6_quant_*_per_token_cuda qu.py:503-534):
    one scale per row, the whole K accumulates in tensor memory.  Inside the exact-accumulation envelope (LB.exact_accumulation:
    every partial sum is an fp32 number) bit-exact; outside it the fp32 sums may round: tolerance 2^-20 of sum |terms| (the
    contract's bound is (K - 1) * 2^-24; on these normal-distributed operands the rounding errors stay far below it)."""
    rng = np.random.default_rng(13)
    m, n, k = 300, 384, 2304
    x = rng.standard_normal((m, k)).astype(dtype)
    w = (rng.standard_normal((n, k)) * 0.05).astype(np.float32)
    a = lowbit.pack_codes(torch.from_numpy(x).to(dev()), fmt_a, per_row=True)
    ww = lowbit.pack_codes(torch.from_numpy(w).to(dev()), fmt_w, per_row=True)
    wc, ws = LB.pack_codes(x, fmt_a, None)
    assert np.array_equal(a.codes.cpu().numpy(), wc) and same_bits(a.scales.cpu().numpy(), ws)
    out_dt = np.float16 if (dtype == np.float16 or fmt_a in ("e2m3", "e3m2")) else np.float32
    got = a.dequantize(torch.float16 if out_dt == np.float16 else torch.float32).cpu().numpy()
    assert same_bits(got, O.fake_quant(x, fmt_a, None, "kernel", out_dtype=out_dt))
    (qa, sa), (qw, sw) = LB.quantize_codes(x, fmt_a, None), LB.quantize_codes(w, fmt_w, None)
    c = lowbit.linear_codes(a, ww, None, torch.float32).cpu().numpy()
    want = LB.gemm_codes(qa, sa, qw, sw)
    if LB.exact_accumulation(fmt_a, fmt_w, k):
        assert np.array_equal(bits(c), bits(want))
    else:
        mag = (np.abs(qa) * sa) @ (np.abs(qw) * sw).T
        assert np.all(np.abs(c.astype(np.float64) - want) <= 2.0 ** -20 * mag)


@pytest.mark.parametrize("pair", [-1, 0, 1])
def test_row_scaled_gemm_default_pairing(pair):
    """Row scales with enough row tiles for the default (gemm_pair = -1) to launch CTA pairs with cta_group::2 MMAs, an odd number of
    row tiles (phantom second tile in the last pair) and a half tile column: bit-exact (e2m1: the sums are exact), whatever the pairing."""
    rng = np.random.default_rng(17)
    m, n, k = 128 * 7 - 3, 256 * 2 + 128, 2304
    x = rng.standard_normal((m, k)).astype(np.float16)
    w = (rng.standard_normal((n, k)) * 0.05).astype(np.float32)
    bias = rng.standard_normal(n).astype(np.float32)
    a = lowbit.pack_codes(torch.from_numpy(x).to(dev()), "e2m1", per_row=True)
    ww = lowbit.pack_codes(torch.from_numpy(w).to(dev()), "e2m1", per_row=True)
    (qa, sa), (qw, sw) = LB.quantize_codes(x, "e2m1", None), LB.quantize_codes(w, "e2m1", None)
    L.set_tunable("gemm_pair", pair)
    try:
        c32 = lowbit.linear_codes(a, ww, torch.from_numpy(bias).to(dev()), torch.float32).cpu().numpy()
        c16 = lowbit.linear_codes(a, ww, None, torch.float16).cpu().numpy()
    finally:
        L.set_tunable("gemm_pair", -1)
    assert np.array_equal(bits(c32), bits(LB.gemm_codes(qa, sa, qw, sw, bias)))
    assert np.array_equal(bits(c16), bits(LB.gemm_codes(qa, sa, qw, sw).astype(np.float16)))


@pytest.mark.parametrize("ref_dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("per_row", [False, True])
def test_fused_output_level_loss(ref_dtype, per_row):
    """fpq_gemm_codes_sse == sum((ref - linear_codes)^2) in float64, without the product ever being stored
    (compute_quant_error of search/search_fp4_format.py:472-476 at the layer output)."""
    torch.manual_seed(3)
    m, n, k = 1000, 640, 1920
    x = torch.randn(m, k, device=dev(), dtype=torch.float16)
    w = torch.randn(n, k, device=dev()) * 0.03
    bias = torch.randn(n, device=dev())
    ref = torch.nn.functional.linear(x.float(), w, bias).to(ref_dtype)
    a, ww = lowbit.pack_codes(x, "e2m1", per_row), lowbit.pack_codes(w, "e2m1", per_row)
    y = lowbit.linear_codes(a, ww, bias, torch.float32)
    want = ((ref.double() - y.double()) ** 2).sum().item()
    for tile_n, pair in ((256, 1), (256, 0), (128, 0)):
        L.set_tunable("gemm_tile_n", tile_n)
        L.set_tunable("gemm_pair", pair)
        try:
            got = lowbit.linear_codes_sse(a, ww, ref, bias).item()
            rw = torch.rand(m, device=dev(), dtype=torch.float64)
            got_w = lowbit.linear_codes_sse(a, ww, ref, bias, None, rw).item()
        finally:
            L.set_tunable("gemm_tile_n", 256)
            L.set_tunable("gemm_pair", -1)
        assert abs(got - want) <= 2e-6 * want          # fp32 squares along a row piece, then float64
        want_w = (((ref.double() - y.double()) ** 2).sum(1) * rw).sum().item()
        assert abs(got_w - want_w) <= 2e-6 * want_w


@pytest.mark.parametrize("fmt_a,fmt_w", [("e1m2", "e3m0"), ("e2m3", "e2m3"), ("e3m2", "e2m1"), ("e3m2", "e3m2")])
def test_gemm_codes_other_formats(fmt_a, fmt_w):
    rng = np.random.default_rng(11)
    x, w, (qa, sa), (qw, sw) = _operands(rng, 130, 256, 640, fmt_a, fmt_w, np.float32)
    a = lowbit.pack_codes(torch.from_numpy(x).to(dev()), fmt_a)
    ww = lowbit.pack_codes(torch.from_numpy(w).to(dev()), fmt_w)
    c = lowbit.linear_codes(a, ww, None, torch.float32).cpu().numpy()
    assert np.array_equal(bits(c), bits(LB.gemm_codes(qa, sa, qw, sw)))


def test_gemm_codes_against_the_reference_expression_fp16_linear():
    """QuantizedLinear.forward (qu.py:764-769): F.linear(act_quant(x), W_q, b) under fp16 autocast.  The fp16 GEMM rounds every
    activation value q*s to fp16 (done by the quantizer, qu.py:329), the weight to fp16 (autocast), accumulates in fp32 and rounds
    the output to fp16.  Stated tolerance: |diff| <= 2^-10 * sum_k |x_q w_q| (operand roundings) + 1 fp16 ulp of the result."""
    torch.manual_seed(0)
    m, n, k = 1000, 384, 1920
    x = torch.randn(m, k, device=dev(), dtype=torch.float16)
    lin = torch.nn.Linear(k, n, bias=True, device=dev())
    mod = lowbit.QuantizedLinearLowBit.from_float(lin, "e2m1", "e2m1")
    y = mod(x)
    xq = ops.fake_quant(x, "e2m1", 128, "kernel")
    wq = ops.fake_quant(lin.weight.detach(), "e2m1", 128, "kernel")
    ref = torch.nn.functional.linear(xq, wq.half(), lin.bias.detach().half())
    mag = xq.abs().double() @ wq.abs().double().T + lin.bias.detach().abs().double()
    tol = 2.0 ** -10 * mag + 2.0 ** -10 * ref.abs().double() + 1e-7
    assert y.shape == ref.shape and y.dtype == torch.float16
    assert bool(((y.double() - ref.double()).abs() <= tol).all())
    # and against float64 on the exact operand values the codes stand for: fp32-chain accuracy
    exact = xq.double() @ wq.double().T + lin.bias.detach().double()
    y32 = lowbit.linear_codes(lowbit.pack_codes(x, "e2m1"), mod.weight_packed(), lin.bias.detach(), torch.float32)
    assert bool(((y32.double() - exact).abs() <= 2.0 ** -11 * mag + 1e-7).all())        # q*s fp16-rounded in xq, exact in the codes


def test_gemm_codes_full_size_properties():
    """BASELINE configs[2] largest mat_qkv call (25 600 token rows of stage 9, C = 1920 -> 5760): exact power-of-two scale
    equivariance, row-block independence, and agreement with the fp16 library GEMM on the fake-quantized tensors."""
    torch.manual_seed(1)
    m, n, k = 25600, 5760, 1920
    x = torch.randn(m, k, device=dev(), dtype=torch.float16)
    w = torch.randn(n, k, device=dev()) * 0.02
    a, ww = lowbit.pack_codes(x, "e2m1"), lowbit.pack_codes(w, "e2m1")
    y = lowbit.linear_codes(a, ww, None, torch.float32)
    a4 = lowbit.PackedCodes(a.codes, a.scales * 4.0, a.rows, a.k, a.fmt)
    assert torch.equal(lowbit.linear_codes(a4, ww, None, torch.float32), y * 4.0)
    sub = lowbit.linear_codes(lowbit.pack_codes(x[5000:5300], "e2m1"), ww, None, torch.float32)
    assert torch.equal(sub, y[5000:5300])
    ref = torch.nn.functional.linear(ops.fake_quant(x, "e2m1", 128, "kernel"), ops.fake_quant(w, "e2m1", 128, "kernel").half())
    err = (y - ref.float()).abs().max().item()
    assert err <= 2.0 ** -8 * ref.float().abs().max().item()


@pytest.mark.parametrize("per", ["group", "row"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_search_loss_table_from_codes(per, dtype):
    """search.search_layer_lowbit (low-bit GEMM + fused loss) against search.search_layer_batched (fake-quant + library GEMMs +
    fpq_sse_rows), the path pinned to the reference's loop by tests/test_reference_search.py.  Calibration tensors of unequal
    row counts, as the reference's [2, pn^2, C] stages.  Stated tolerance: 2e-3 relative per entry (fp16 library GEMM output
    rounding on one side, none on the other), same winner."""
    from fpqvar_b200 import search
    torch.manual_seed(5)
    torch.backends.cuda.matmul.allow_tf32 = False
    c_in, c_out = 640, 384
    w = (torch.randn(c_out, c_in, device=dev()) * 0.04).to(dtype)
    acts = [torch.randn(2, pn * pn, c_in, device=dev()).to(dtype) for pn in (1, 2, 3, 4, 5, 6, 8, 10, 13)]
    fmts = ["e2m1", "e1m2", "e3m0"]
    want = search.search_layer_batched(w, acts, fmts, fmts, per if per == "group" else "token")
    got = search.search_layer_lowbit(w, acts, fmts, fmts, per if per == "group" else "token")
    assert torch.allclose(got, want, rtol=2e-3, atol=0)
    assert search.best_formats(got, fmts, fmts)["weight_format"] == search.best_formats(want, fmts, fmts)["weight_format"]
    assert search.best_formats(got, fmts, fmts)["activation_format"] == search.best_formats(want, fmts, fmts)["activation_format"]


def test_gemm_codes_argument_errors():
    a = lowbit.pack_codes(torch.randn(8, 256, device=dev(), dtype=torch.float16), "e2m1")
    w = lowbit.pack_codes(torch.randn(16, 128, device=dev()), "e2m1")
    with pytest.raises(L.FpqError):
        lowbit.linear_codes(a, w)
    with pytest.raises(L.FpqError):
        lowbit.pack_codes(torch.randn(8, 100, device=dev()), "e2m1")
    with pytest.raises(L.FpqError):
        lowbit.pack_codes(torch.randn(8, 128), "e2m1")
    with pytest.raises(ValueError):
        lowbit.pack_codes(torch.randn(8, 128, device=dev()), "fp_e9")
    # hand-made PackedCodes whose buffers do not match their shape never reach the kernel
    bad = lowbit.PackedCodes(a.codes[:-128], a.scales, a.rows, a.k, a.fmt)
    with pytest.raises(L.FpqError):
        lowbit.linear_codes(bad, a)
    bad = lowbit.PackedCodes(a.codes, a.scales.double(), a.rows, a.k, a.fmt)
    with pytest.raises(L.FpqError):
        bad.dequantize()
    bad = lowbit.PackedCodes(a.codes.cpu(), a.scales, a.rows, a.k, a.fmt)
    with pytest.raises(L.FpqError):
        lowbit.linear_codes(a, bad)
