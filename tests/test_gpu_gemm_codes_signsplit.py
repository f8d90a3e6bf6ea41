"""GPU parity of the sign-split codes operand (the fc2 input) and of the split low-bit GEMM (csrc/fpq_gemm.cu) against
oracle/lowbit_split.py, whose GEMM is oracle/gemm_codes.c on the expanded operands A' (depth 2k) and W' (every 128-slab twice).
Bars: codes, scales and dequantized tensors bit-exact; GEMM bit-exact (every split half x weight format pair is inside the
exact-accumulation envelope); against the reference's fc2 expression within the tolerance of tests/test_gpu_gemm_codes.py."""
import numpy as np
import pytest
import torch

from fpqvar_b200 import _lib as L, lowbit, ops
from oracle import lowbit as LB, lowbit_split as LS, oracle as O          # checker only

pytestmark = pytest.mark.gpu
SPLITS = list(LS.FORMATS)
WEIGHT_FMTS = ["e2m1", "e1m2", "e3m0", "e2m3", "e3m2"]
TUNABLES = [(256, 128, 3, 1), (256, 64, 4, 0), (256, 128, 2, 0), (256, 128, 2, 1), (128, 32, 6, 0), (128, 64, 2, 0), (128, 128, 3, 0)]


def bits(a):
    return a.view({1: np.uint8, 2: np.uint16, 4: np.uint32}[a.dtype.itemsize])


def same_bits(a, b):
    """bit-identical, NaN payloads aside (signed zeros and NaN positions count)"""
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(bits(a)[~na], bits(b)[~nb])


def dev():
    return torch.device("cuda:0")


def cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev())


def adversarial(rng, rows, k, dtype, nan=False):
    """zero, all-negative and all-positive groups, -0.0, subnormals, +-inf, GELU-like rows, grid points; a NaN if asked"""
    x = rng.standard_normal((rows, k)).astype(dtype)
    if rows == 1:
        x[0, :64] = -np.abs(x[0, :64])
        x[0, 200:260] = dtype(-0.0)
        x[0, 300] = np.inf
        if nan:
            x[0, 17] = np.nan
        return x
    x[0, :128] = 0
    x[1, :128] = -np.abs(x[1, :128])
    x[2, 128:256] = np.abs(x[2, 128:256])
    x[3, ::3] = dtype(-0.0)
    x[4, :128] = (x[4, :128].astype(np.float32) * np.float32(2.0 ** -20 if dtype == np.float16 else 2.0 ** -140)).astype(dtype)
    x[5, 7] = np.inf
    x[6, 300] = -np.inf
    x[7, :128] = -0.0
    x[8:100] = np.where(x[8:100] > 0, x[8:100], x[8:100] * dtype(0.05))
    x[100, :8] = np.asarray([0.25, -0.125, 0.375, -1.75, 3.0, -0.5, 5.0, 6.0], dtype=dtype)
    if nan:
        x[150, 130] = np.nan
    return x


def tunables(tile_n, epi_cols, stages, pair):
    L.set_tunable("gemm_stages", stages)
    L.set_tunable("gemm_tile_n", tile_n)
    L.set_tunable("gemm_epi_cols", epi_cols)
    L.set_tunable("gemm_pair", pair)


def reset_tunables():
    tunables(256, 128, 6, -1)


@pytest.mark.parametrize("fmt", SPLITS)
@pytest.mark.parametrize("dtype", [np.float16, np.float32])
@pytest.mark.parametrize("rows", [1, 300])
def test_pack_codes_signsplit_bit_exact(fmt, dtype, rows):
    rng = np.random.default_rng(rows)
    out_dt = torch.float16 if dtype == np.float16 else torch.float32
    for clip, nan in ((True, False), (False, True)):
        x = adversarial(rng, rows, 384, dtype, nan)
        p = lowbit.pack_codes(cuda(x), fmt, global_clip=clip)
        assert p.split and p.codes.numel() == 2 * p.rows_pad * 384
        wc, ws = LS.pack_codes_signsplit(x, fmt, clip)
        assert np.array_equal(p.codes.cpu().numpy(), wc)
        assert same_bits(p.scales.cpu().numpy().reshape(ws.shape), ws)
        got = p.dequantize(out_dt).cpu().numpy()
        want = ops.fake_quant_signsplit(cuda(x), fmt, 128, "kernel", global_clip=clip).cpu().numpy()
        assert same_bits(got, want)
        assert same_bits(got, O.fake_quant_signsplit(x, fmt, 128, "kernel", clipping_strength=1.0 if clip else None))


@pytest.mark.parametrize("fmt", SPLITS)
@pytest.mark.parametrize("dtype", [np.float16, np.float32])
def test_global_clip_nan_gives_the_all_zero_operand_and_the_next_call_is_normal(fmt, dtype):
    rng = np.random.default_rng(2)
    x = adversarial(rng, 300, 512, dtype, nan=True)
    p = lowbit.pack_codes(cuda(x), fmt)
    assert not p.codes.any().item() and not p.scales.view(torch.int32).any().item()
    assert not bits(p.dequantize(torch.float32).cpu().numpy()).any()
    ws = ops._clip_workspace(dev())
    y = adversarial(rng, 300, 512, dtype, nan=False)
    q = lowbit.pack_codes(cuda(y), fmt)
    torch.cuda.synchronize()
    assert not ws.any().item()                                   # the last CTA re-zeroed {flag, ticket}
    wc, wsc = LS.pack_codes_signsplit(y, fmt)
    assert np.array_equal(q.codes.cpu().numpy(), wc) and same_bits(q.scales.cpu().numpy(), wsc)


@pytest.mark.parametrize("fmt", SPLITS)
@pytest.mark.parametrize("clip", [False, True])
def test_gelu_pack_codes_every_fp16_pattern(fmt, clip):
    """all 65 536 fp16 bit patterns as 512 groups of 128 (NaN patterns included: with the clip the result is all zero)"""
    x = cuda(np.arange(65536, dtype=np.uint16).view(np.float16).reshape(64, 1024))
    g = ops.gelu_table().reshape(64, 1024)                        # the library's GELU of the same patterns, in the same order
    p = lowbit.gelu_pack_codes(x, fmt, clip)
    q = lowbit.pack_codes(g, fmt, global_clip=clip)
    assert torch.equal(p.codes, q.codes)
    assert same_bits(p.scales.cpu().numpy(), q.scales.cpu().numpy())
    assert same_bits(p.dequantize(torch.float16).cpu().numpy(), ops.gelu_fake_quant_signsplit(x, fmt, clip).cpu().numpy())
    wc, ws = LS.pack_codes_signsplit(g.cpu().numpy(), fmt, clip)
    assert np.array_equal(p.codes.cpu().numpy(), wc) and same_bits(p.scales.cpu().numpy(), ws)


def _split_operands(rng, m, n, k, fmt, wfmt, dtype=np.float16):
    x = rng.standard_normal((m, k)).astype(dtype)
    x = np.where(x > 0, x, x * dtype(0.1)).astype(dtype)
    w = (rng.standard_normal((n, k)) * 0.05).astype(np.float32)
    return x, w, LS.quantize_codes_signsplit(x, fmt), LB.quantize_codes(w, wfmt)


@pytest.mark.parametrize("m,n,k", [(1, 8, 128), (100, 136, 384), (300, 384, 1920), (257, 128, 7680)])
@pytest.mark.parametrize("tile_n,epi_cols,stages,pair", TUNABLES)
def test_split_gemm_bit_exact_against_the_expanded_oracle(m, n, k, tile_n, epi_cols, stages, pair):
    rng = np.random.default_rng(m + n + k)
    fmt = "e1m2_neg_e2m1_pos"
    x, w, qa, (qw, sw) = _split_operands(rng, m, n, k, fmt, "e2m1")
    bias = rng.standard_normal(n).astype(np.float32)
    a = lowbit.pack_codes(cuda(x), fmt)
    ww = lowbit.pack_codes(cuda(w), "e2m1")
    tunables(tile_n, epi_cols, stages, pair)
    try:
        c32 = lowbit.linear_codes(a, ww, cuda(bias), torch.float32).cpu().numpy()
        c16 = lowbit.linear_codes(a, ww, None, torch.float16).cpu().numpy()
    finally:
        reset_tunables()
    assert np.array_equal(bits(c32), bits(LS.gemm_codes_signsplit(*qa, qw, sw, bias)))
    assert np.array_equal(bits(c16), bits(LS.gemm_codes_signsplit(*qa, qw, sw).astype(np.float16)))


def test_split_gemm_many_tiles_per_cta():
    """more tiles than SMs: the persistent loop, the scale ring and the accumulators wrap several times"""
    rng = np.random.default_rng(99)
    m, n, k = 128 * 21 - 5, 256 * 9 + 128, 384
    x, w, qa, (qw, sw) = _split_operands(rng, m, n, k, "afpq_e2m1", "e1m2")
    a = lowbit.pack_codes(cuda(x), "afpq_e2m1")
    ww = lowbit.pack_codes(cuda(w), "e1m2")
    want = LS.gemm_codes_signsplit(*qa, qw, sw)
    for tile_n, epi_cols, stages, pair in TUNABLES:
        tunables(tile_n, epi_cols, stages, pair)
        try:
            c = lowbit.linear_codes(a, ww, None, torch.float32).cpu().numpy()
            c16 = lowbit.linear_codes(a, ww, None, torch.float16).cpu().numpy()
        finally:
            reset_tunables()
        assert np.array_equal(bits(c), bits(want))
        assert np.array_equal(bits(c16), bits(want.astype(np.float16)))


@pytest.mark.parametrize("fmt", SPLITS)
@pytest.mark.parametrize("wfmt", WEIGHT_FMTS)
def test_split_gemm_every_weight_format(fmt, wfmt):
    rng = np.random.default_rng(11)
    x, w, qa, (qw, sw) = _split_operands(rng, 130, 264, 640, fmt, wfmt, np.float32)
    a = lowbit.pack_codes(cuda(x), fmt)
    ww = lowbit.pack_codes(cuda(w), wfmt)
    c = lowbit.linear_codes(a, ww, None, torch.float32).cpu().numpy()
    assert np.array_equal(bits(c), bits(LS.gemm_codes_signsplit(*qa, qw, sw)))


def test_split_gemm_with_an_infinite_scale():
    """a -inf element makes sn = inf in its group: 0 * inf = NaN through the scale chain of that row, as in the oracle"""
    rng = np.random.default_rng(5)
    x, w, _, (qw, sw) = _split_operands(rng, 200, 256, 512, "e1m2_neg_e2m1_pos", "e2m1")
    x[7, 300] = -np.inf
    x[9, 3] = np.inf
    qa = LS.quantize_codes_signsplit(x, "e1m2_neg_e2m1_pos")
    assert np.isinf(qa[2][7]).any() and np.isinf(qa[3][9]).any()
    a = lowbit.pack_codes(cuda(x), "e1m2_neg_e2m1_pos")
    ww = lowbit.pack_codes(cuda(w), "e2m1")
    c = lowbit.linear_codes(a, ww, None, torch.float32).cpu().numpy()
    want = LS.gemm_codes_signsplit(*qa, qw, sw)
    assert np.isnan(want[7]).all() and np.isnan(want[9]).all()
    assert same_bits(c, want)


@pytest.mark.parametrize("ref_dtype", [torch.float32, torch.float16])
def test_split_fused_output_level_loss(ref_dtype):
    torch.manual_seed(3)
    m, n, k = 1000, 640, 1920
    h = torch.nn.functional.gelu(torch.randn(m, k, device=dev()), approximate="tanh").half()
    w = torch.randn(n, k, device=dev()) * 0.03
    bias = torch.randn(n, device=dev())
    ref = torch.nn.functional.linear(h.float(), w, bias).to(ref_dtype)
    a, ww = lowbit.pack_codes(h, "e1m2_neg_e2m1_pos"), lowbit.pack_codes(w, "e2m1")
    y = lowbit.linear_codes(a, ww, bias, torch.float32)
    want = ((ref.double() - y.double()) ** 2).sum().item()
    rw = torch.rand(m, device=dev(), dtype=torch.float64)
    want_w = (((ref.double() - y.double()) ** 2).sum(1) * rw).sum().item()
    for tile_n, pair in ((256, 1), (256, 0), (128, 0)):
        tunables(tile_n, 128, 6, pair)
        try:
            got = lowbit.linear_codes_sse(a, ww, ref, bias).item()
            got_w = lowbit.linear_codes_sse(a, ww, ref, bias, None, rw).item()
        finally:
            reset_tunables()
        assert abs(got - want) <= 2e-6 * want
        assert abs(got_w - want_w) <= 2e-6 * want_w


def test_fc2_layer_against_the_reference_expression():
    """QuantizedLinear_fc2 (qu.py:870-1093: sign-split act_quant + F.linear under fp16 autocast) with the W4A4 README formats.
    Tolerance as test_gemm_codes_against_the_reference_expression_fp16_linear; forward_gelu(h) == forward(gelu(h)) bit for bit."""
    from fpqvar_b200 import quant_utils as qu
    torch.manual_seed(0)
    m, k, n = 1000, 1920, 384
    h = torch.randn(m, k, device=dev(), dtype=torch.float16)
    x = torch.nn.functional.gelu(h, approximate="tanh")
    lin = torch.nn.Linear(k, n, bias=True, device=dev())
    mod = lowbit.QuantizedLinearLowBit.from_float(lin, "e2m1", "e1m2_neg_e2m1_pos")
    assert "sign-split" in mod.extra_repr()
    y = mod(x)
    ref_mod = qu.QuantizedLinear_fc2.from_float(lin, weight_quant="per_group", act_quant="per_group", w_bit=4, a_bit=4,
                                                activation_fp_quant=True, weight_fp_quant=True, act_fp_type="fp_e1m2_neg_e2m1_pos",
                                                weight_fp_type="fp_e2")
    with torch.autocast("cuda", dtype=torch.float16):
        ref = ref_mod(x)
    xq = ops.fake_quant_signsplit(x, "e1m2_neg_e2m1_pos", 128, "kernel", global_clip=True)
    wq = ops.fake_quant(lin.weight.detach(), "e2m1", 128, "kernel")
    mag = xq.abs().double() @ wq.abs().double().T + lin.bias.detach().abs().double()
    tol = 2.0 ** -10 * mag + 2.0 ** -10 * ref.abs().double() + 1e-7
    assert y.shape == ref.shape and y.dtype == torch.float16 == ref.dtype
    assert bool(((y.double() - ref.double()).abs() <= tol).all())
    assert torch.equal(mod.forward_gelu(h).view(torch.int16), y.view(torch.int16))


def test_fc2_search_from_codes():
    """search_layer_lowbit with sign-split activation candidates against search_layer_batched: 2e-3 relative, same winner"""
    from fpqvar_b200 import search
    torch.manual_seed(5)
    torch.backends.cuda.matmul.allow_tf32 = False
    c_in, c_out = 768, 256
    w = (torch.randn(c_out, c_in, device=dev()) * 0.04).half()
    acts = [torch.nn.functional.gelu(torch.randn(2, pn * pn, c_in, device=dev()), approximate="tanh").half()
            for pn in (1, 2, 3, 4, 5, 6, 8, 10, 13)]
    wf, af = ["e2m1", "e1m2", "e3m0"], ["e1m2_neg_e2m1_pos", "afpq_e2m1", "e2m1"]
    want = search.search_layer_batched(w, acts, wf, af, "group")
    got = search.search_layer_lowbit(w, acts, wf, af, "group")
    assert torch.allclose(got, want, rtol=2e-3, atol=0)
    assert search.best_formats(got, wf, af) | {"loss": 0} == search.best_formats(want, wf, af) | {"loss": 0}


def test_side_stream_and_graph_capture_match_eager():
    torch.manual_seed(7)
    h = torch.randn(300, 1920, device=dev(), dtype=torch.float16)
    w = lowbit.pack_codes(torch.randn(384, 1920, device=dev()) * 0.03, "e2m1")
    bias = torch.randn(384, device=dev())

    def run():
        return lowbit.linear_codes(lowbit.gelu_pack_codes(h, "e1m2_neg_e2m1_pos"), w, bias, torch.float16)

    eager = run()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        side = run()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            captured = run()
    torch.cuda.current_stream().wait_stream(s)
    captured.fill_(float("nan"))
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(side.view(torch.int16), eager.view(torch.int16))
    assert torch.equal(captured.view(torch.int16), eager.view(torch.int16))


def test_argument_errors_launch_nothing():
    x = torch.randn(8, 256, device=dev(), dtype=torch.float16)
    a = lowbit.pack_codes(x, "e1m2_neg_e2m1_pos")
    w = lowbit.pack_codes(torch.randn(16, 256, device=dev()), "e2m1")
    w_row = lowbit.pack_codes(torch.randn(16, 256, device=dev()), "e2m1", per_row=True)
    w_k = lowbit.pack_codes(torch.randn(16, 128, device=dev()), "e2m1")
    ref = torch.zeros(8, 16, device=dev())
    torch.cuda.synchronize()
    before = L.lib().fpq_launch_count()
    bad_calls = [
        lambda: lowbit.pack_codes(x, "int_neg_e2m3_pos"),
        lambda: lowbit.gelu_pack_codes(x, "int_neg_e2m3_pos"),
        lambda: lowbit.pack_codes(x, "afpq_e2m1", per_row=True),
        lambda: lowbit.gelu_pack_codes(x, "e2m1"),
        lambda: lowbit.gelu_pack_codes(x.float(), "afpq_e2m1"),
        lambda: lowbit.linear_codes(w, a),                                           # sign-split weight
        lambda: lowbit.linear_codes(a, w_row),                                       # row-scaled weight
        lambda: lowbit.linear_codes(a, w_k),                                         # k differs
        lambda: lowbit.linear_codes_sse(a, w_k, ref),
        lambda: lowbit.linear_codes(lowbit.PackedCodes(a.codes[: a.codes.numel() // 2], a.scales, a.rows, a.k, a.fmt), w),
        lambda: lowbit.linear_codes(lowbit.PackedCodes(a.codes, a.scales[:2], a.rows, a.k, a.fmt), w),
        lambda: lowbit.PackedCodes(w.codes, w.scales, w.rows, w.k, "afpq_e2m1").dequantize(),     # symmetric-sized buffers
        lambda: lowbit.PackedCodes(a.codes, a.scales, a.rows, a.k, a.fmt, a.k).dequantize(),      # split with row scales
        lambda: a.to_nibbles(),
        lambda: lowbit.QuantizedLinearLowBit(w_row, None, "e1m2_neg_e2m1_pos"),
    ]
    for call in bad_calls:
        with pytest.raises(L.FpqError):
            call()
    with pytest.raises(ValueError):
        lowbit.pack_codes(x, "fp_e9")
    codes = torch.empty(2 * 128 * 256, dtype=torch.uint8, device=dev())
    scales = torch.empty(4 * 128, dtype=torch.float32, device=dev())
    ws = torch.zeros(2, dtype=torch.int32, device=dev())
    lib = L.lib()
    assert lib.fpq_pack_codes_signsplit(x.data_ptr(), 8, 256, L.FPQ_F16, L.SPLIT["int_neg_e2m3_pos"], 0, None, codes.data_ptr(),
                                        scales.data_ptr(), None) == L.FPQ_ERR_UNSUPPORTED
    assert lib.fpq_pack_codes_signsplit(x.data_ptr(), 8, 192, L.FPQ_F16, 0, 0, None, codes.data_ptr(), scales.data_ptr(), None) == L.FPQ_ERR_ARG
    assert lib.fpq_pack_codes_signsplit(x.data_ptr(), 8, 256, L.FPQ_F16, 0, L.FLAG_GLOBAL_CLIP, None, codes.data_ptr(),
                                        scales.data_ptr(), None) == L.FPQ_ERR_ARG
    assert lib.fpq_pack_codes_signsplit(x.data_ptr(), 8, 256, L.FPQ_F16, 0, 4, ws.data_ptr(), codes.data_ptr(), scales.data_ptr(),
                                        None) == L.FPQ_ERR_ARG
    assert lib.fpq_gelu_pack_codes_signsplit(x.data_ptr(), 8, 256, 3, 0, None, codes.data_ptr(), scales.data_ptr(), None) == L.FPQ_ERR_ARG
    assert lib.fpq_unpack_codes_signsplit(codes.data_ptr(), scales.data_ptr(), 8, 256, 7, ref.data_ptr(), None) == L.FPQ_ERR_ARG
    assert lib.fpq_gemm_codes_signsplit(a.codes.data_ptr(), a.scales.data_ptr(), 8, w.codes.data_ptr(), w.scales.data_ptr(), 16, 192,
                                        None, L.FPQ_F32, ref.data_ptr(), 16, None) == L.FPQ_ERR_ARG
    assert lib.fpq_gemm_codes_signsplit_sse(a.codes.data_ptr(), a.scales.data_ptr(), 8, w.codes.data_ptr(), w.scales.data_ptr(), 16,
                                            256, None, L.FPQ_F32, ref.data_ptr(), 16, None, None, None) == L.FPQ_ERR_ARG
    torch.cuda.synchronize()
    assert L.lib().fpq_launch_count() == before
