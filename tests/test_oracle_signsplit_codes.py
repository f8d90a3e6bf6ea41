"""CPU: the sign-split codes operand (oracle/lowbit_split.py) against the reference's sign-split quantizer (oracle.fake_quant_signsplit,
qu.py:415-452) and the split GEMM as oracle/gemm_codes.c on the expanded operands.  No GPU."""
import numpy as np
import pytest

from oracle import lowbit as LB, lowbit_split as LS, oracle as O

WEIGHT_FMTS = ["e2m1", "e1m2", "e3m0", "e2m3", "e3m2"]


def bits(a):
    return a.view({1: np.uint8, 2: np.uint16, 4: np.uint32}[a.dtype.itemsize])


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(bits(a)[~na], bits(b)[~nb])


def adversarial(dtype, with_nan):
    """groups: zero, all-negative, all-positive, -0.0 mixed in, subnormals, +-inf, a NaN element (with_nan), GELU-like."""
    rng = np.random.default_rng(1)
    x = rng.standard_normal((12, 512)).astype(dtype)
    x[0, :128] = 0
    x[1, :128] = -np.abs(x[1, :128])
    x[2, 128:256] = np.abs(x[2, 128:256])
    x[3, ::3] = dtype(-0.0)
    x[4, :128] = (x[4, :128].astype(np.float32) * np.float32(2.0 ** -20 if dtype == np.float16 else 2.0 ** -140)).astype(dtype)
    x[5, 7] = np.inf
    x[6, 300] = -np.inf
    x[7, :128] = -0.0
    x[8] = np.where(x[8] > 0, x[8], x[8] * dtype(0.05))
    x[9, 256:] = np.asarray(np.tile([0.25, -0.125, 0.375, -1.75, 3.0, -0.5, 5.0, 6.0], 32), dtype=dtype)
    if with_nan:
        x[10, 200] = np.nan
    return x


@pytest.mark.parametrize("fmt", LS.FORMATS)
@pytest.mark.parametrize("dtype", [np.float16, np.float32])
def test_dequantized_codes_are_the_reference_sign_split_quantizer(fmt, dtype):
    x = adversarial(dtype, with_nan=False)
    got = LS.dequantize_signsplit(*LS.quantize_codes_signsplit(x, fmt), dtype)
    assert same_bits(got, O.fake_quant_signsplit(x, fmt, 128, "kernel"))
    # NaN elements without the whole-tensor clip count as 0 locally (qu.py:428-429)
    x = adversarial(dtype, with_nan=True)
    got = LS.dequantize_signsplit(*LS.quantize_codes_signsplit(x, fmt, global_clip=False), dtype)
    assert same_bits(got, O.fake_quant_signsplit(x, fmt, 128, "kernel", clipping_strength=None))


@pytest.mark.parametrize("fmt", LS.FORMATS)
@pytest.mark.parametrize("dtype", [np.float16, np.float32])
def test_global_clip_of_a_nan_tensor_is_the_all_zero_operand(fmt, dtype):
    x = adversarial(dtype, with_nan=True)
    qn, qp, sn, sp = LS.quantize_codes_signsplit(x, fmt)
    for t in (qn, qp, sn, sp):
        assert np.array_equal(bits(t), np.zeros_like(bits(t)))          # +0 everywhere
    codes, scales = LS.pack_codes_signsplit(x, fmt)
    assert not codes.any() and not bits(scales).any()
    got = LS.dequantize_signsplit(qn, qp, sn, sp, dtype)
    assert same_bits(got, O.fake_quant_signsplit(x, fmt, 128, "kernel"))


def test_half_grids_are_e4m3_numbers_and_int_neg_is_not():
    for fmt in LS.FORMATS:
        for half in O.SPLIT[fmt]:
            assert LS.e4m3_representable(O.GRIDS[half]).all(), half
    neg, pos = O.SPLIT["int_neg_e2m3_pos"]
    assert LS.e4m3_representable(O.GRIDS[pos]).all()
    bad = O.GRIDS[neg][~LS.e4m3_representable(O.GRIDS[neg])]
    assert sorted(-bad.astype(int)) == list(range(17, 32, 2))


@pytest.mark.parametrize("fmt", LS.FORMATS)
def test_layout_round_trip(fmt):
    x = adversarial(np.float16, with_nan=False)[:11]
    qn, qp, sn, sp = LS.quantize_codes_signsplit(x, fmt)
    codes, scales = LS.pack_codes_signsplit(x, fmt)
    rows, k = x.shape
    assert codes.size == 2 * LB.rows_padded(rows) * k and scales.shape == (2 * k // 128, LB.rows_padded(rows))
    a2 = LB.e4m3_decode(LB.from_blocked(codes, rows, 2 * k))
    back = LS.split_halves(a2, scales[:, :rows].T)
    for want, got in zip((qn, qp, sn, sp), back):
        assert same_bits(np.ascontiguousarray(got), want)
    assert not scales[:, rows:].any()
    # slab 2t is group t's negative half, slab 2t + 1 its positive half
    for t in range(k // 128):
        assert np.array_equal(a2[:, 256 * t:256 * t + 128], qn[:, 128 * t:128 * (t + 1)])
        assert np.array_equal(a2[:, 256 * t + 128:256 * (t + 1)], qp[:, 128 * t:128 * (t + 1)])
        assert (qn[:, 128 * t:128 * (t + 1)] <= 0).all() and (qp[:, 128 * t:128 * (t + 1)] >= 0).all()
    assert not ((qn != 0) & (qp != 0)).any()


@pytest.mark.parametrize("half", sorted({h for f in LS.FORMATS for h in O.SPLIT[f]}))
@pytest.mark.parametrize("wfmt", WEIGHT_FMTS)
def test_every_split_half_and_weight_pair_accumulates_exactly(half, wfmt):
    assert LB.exact_accumulation(half, wfmt, 128)
    assert LB.accumulation_bits(half, wfmt, 128) <= LB.accumulation_bits("e2m1_pos", "e3m2", 128) < 19.5


@pytest.mark.parametrize("fmt", LS.FORMATS)
@pytest.mark.parametrize("wfmt", ["e2m1", "e3m2"])
def test_expanded_gemm_is_the_scale_chain_of_exact_slab_sums(fmt, wfmt):
    rng = np.random.default_rng(3)
    m, n, k = 37, 24, 384
    x = rng.standard_normal((m, k)).astype(np.float16)
    w = (rng.standard_normal((n, k)) * 0.05).astype(np.float32)
    bias = rng.standard_normal(n).astype(np.float32)
    qn, qp, sn, sp = LS.quantize_codes_signsplit(x, fmt)
    qw, sw = LB.quantize_codes(w, wfmt)
    c = LS.gemm_codes_signsplit(qn, qp, sn, sp, qw, sw, bias)
    a2, s2 = LS.expand_signsplit(qn, qp, sn, sp)
    w2, sw2 = LS.repeat_weight_slabs(qw, sw)
    p = np.stack([a2[:, 128 * u:128 * (u + 1)].astype(np.float64) @ w2[:, 128 * u:128 * (u + 1)].T.astype(np.float64)
                  for u in range(2 * k // 128)])            # exact: small multiples of the grid units
    assert np.array_equal(bits(c), bits(LB.scale_chain(p, s2, sw2, bias)))
    # against float64 on the values the codes stand for: one rounding per scale-chain step
    av = (qn.reshape(m, -1, 128) * sn[:, :, None].astype(np.float64) + qp.reshape(m, -1, 128) * sp[:, :, None]).reshape(m, k)
    wv = (qw.reshape(n, -1, 128) * sw[:, :, None].astype(np.float64)).reshape(n, k)
    exact = av @ wv.T + bias
    mag = np.abs(av) @ np.abs(wv).T + np.abs(bias)
    assert np.all(np.abs(c - exact) <= (2 * (2 * k // 128) + 2) * 2.0 ** -24 * mag)


def test_c_abi_exports_the_sign_split_entry_points():
    import ctypes
    import os
    so = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fpqvar_b200", "libfpq_b200.so")
    if not os.path.exists(so):
        pytest.skip("libfpq_b200.so is not built")
    lib = ctypes.CDLL(so)
    for name in ("fpq_pack_codes_signsplit", "fpq_gelu_pack_codes_signsplit", "fpq_unpack_codes_signsplit", "fpq_gemm_codes_signsplit",
                 "fpq_gemm_codes_signsplit_sse"):
        assert hasattr(lib, name)


def test_sign_split_host_layer_has_no_cpu_path():
    import torch
    from fpqvar_b200 import _lib as L, lowbit
    assert lowbit.SPLIT_FORMATS == LS.FORMATS
    for fmt in ("e1m2_neg_e2m1_pos", "int_neg_e2m3_pos"):
        with pytest.raises(L.FpqError):
            lowbit.pack_codes(torch.randn(8, 128), fmt)
        with pytest.raises(L.FpqError):
            lowbit.gelu_pack_codes(torch.randn(8, 128).half(), fmt)
    p = lowbit.PackedCodes(torch.zeros(2 * 128 * 128, dtype=torch.uint8), torch.zeros(2, 128), 8, 128, "afpq_e2m1")
    assert p.split
    for call in (p.dequantize, p.to_nibbles, lambda: lowbit.linear_codes(p, p)):
        with pytest.raises(L.FpqError):
            call()
