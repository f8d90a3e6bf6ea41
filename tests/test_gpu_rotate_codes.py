"""The fused rotate kernels' codes output (fpq_transform_rotate_pack_codes, fpq_modulate_transform_rotate_pack_codes,
lowbit.rotate_pack_codes): codes and scales bit-identical to fpq_pack_codes of the fp16 rotation the sibling call writes with
format -1 (and to oracle/lowbit.py's pack_codes of those values), whichever kernel runs; one launch per call, padding rows
included; and the product of those codes through QuantizedLinearLowBit equal to the unfused two-step path."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import bits_equal
from oracle import lowbit as LB

FORMATS = ["e2m1", "e1m2", "e3m0", "e2m3", "e3m2"]
# (chunks per row, rows, rows per batch for the modulated entry): widths the small kernel alone takes (1, 3, 40) and the
# streaming kernel's (4 .. 36); row counts around the 8-row blocks and 128-row tiles of the codes layout; 25 600 x 1920 is the
# largest VAR-d30 stage (rows_per_batch 256)
SHAPES = [(1, 1, 1), (3, 7, 7), (4, 8, 4), (5, 127, 127), (15, 128, 64), (15, 129, 43), (18, 4097, 241), (36, 129, 3), (40, 4097, 17),
          (15, 25600, 256)]
ENTRIES = ["plain", "plain_smooth", "mod_f32", "mod_f16"]


@pytest.fixture(scope="module")
def mods():
    from fpqvar_b200 import _lib, lowbit, ops
    assert torch.cuda.is_available()
    return ops, lowbit, _lib


@pytest.fixture(scope="module")
def sign_bits():
    from fpqvar_b200.hotpath import seed42_sign_bits
    return seed42_sign_bits()


def make_inputs(cpr, rows, rpb, entry, seed):
    """x with the irregular chunks of the quantizer (all-zero, NaN, inf, fp16 overflow after the rotation, subnormal fp16
    scale) in its first rows; smooth with a non-positive entry; fp32 or fp16 adaLN operands with the special gains."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    C = 128 * cpr
    x = torch.randn(rows, C, device="cuda", generator=g) * torch.exp(torch.randn(rows, 1, device="cuda", generator=g))
    # "overflow": a constant 1e8 chunk rotates to values far past the fp16 range (checked in the bit-identity test)
    specials = [("zero", 0.0), ("nan", None), ("inf", None), ("overflow", 1.0e8), ("subnormal", 1.0e-6)]
    for i, (kind, v) in enumerate(specials):
        r, c = i % rows, (i * 7) % cpr
        if kind == "nan":
            x[r, 128 * c + 5] = float("nan")
        elif kind == "inf":
            x[r, 128 * c + 17] = float("inf")
        else:
            x[r, 128 * c:128 * (c + 1)] = v
    smooth = None
    if entry != "plain":
        smooth = torch.exp(torch.rand(C, device="cuda", generator=g) * 2 - 1)
        smooth[3 % C] = -0.0883
        smooth[(C - 1) // 2] = 0.0
    scale = shift = None
    if entry.startswith("mod"):
        B = rows // rpb
        scale = torch.randn(B, 1, C, device="cuda", generator=g) * 0.3
        shift = torch.randn(B, 1, C, device="cuda", generator=g) * 0.5
        if entry == "mod_f16":
            scale, shift = scale.half(), shift.half()
        n = min(8, C)
        scale[0, 0, :n] = torch.tensor([-1.0, 2.0 ** -12, -(2.0 ** -12), 6e-8, -6e-8, 0.0, -0.0, -1.0005][:n], device="cuda").to(scale.dtype)
        shift[0, 0, :n] = torch.tensor([0.0, -0.0, 0.0, -0.0, 1.0, 0.0, -0.0, 0.0][:n], device="cuda").to(shift.dtype)
        x = x.view(B, rpb, C)
    return x, smooth, scale, shift


def sibling(ops, x, smooth, scale, shift, bits, fmt):
    if scale is None:
        return ops.transform_rotate_quant(x, smooth, bits, fmt)
    return ops.modulate_transform_rotate_quant(x, scale, shift, smooth, bits, fmt)


def same_bytes(a, b):
    return torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("cpr,rows,rpb", SHAPES)
def test_codes_bit_identical_to_pack_codes_of_the_rotation(mods, sign_bits, cpr, rows, rpb, entry):
    ops, lowbit, _ = mods
    x, smooth, scale, shift = make_inputs(cpr, rows, rpb, entry, cpr * 100003 + rows)
    C = 128 * cpr
    rot = sibling(ops, x, smooth, scale, shift, sign_bits, None).reshape(rows, C)
    rot_host = rot.cpu().numpy()
    if rows >= 5:                          # each special in a row of its own: the overflow chunk is inf in fp16
        c_ovf = 21 % cpr
        assert bool(torch.isinf(rot[3, 128 * c_ovf:128 * (c_ovf + 1)]).any())
    n_or = min(rows, 256)                 # the oracle restates the first rows (the irregular chunks are among them)
    for fmt in FORMATS:
        got = lowbit.rotate_pack_codes(x, smooth, sign_bits, fmt, scale, shift)
        assert (got.rows, got.k, got.scale_group, got.fmt) == (rows, C, 128, fmt)
        want = lowbit.pack_codes(rot, fmt)
        assert same_bytes(got.codes, want.codes), f"{fmt}: codes differ from pack_codes of the rotation"
        assert same_bytes(got.scales, want.scales), f"{fmt}: scales differ from pack_codes of the rotation"
        fq = sibling(ops, x, smooth, scale, shift, sign_bits, fmt).reshape(rows, C)
        assert same_bytes(got.dequantize(torch.float16), fq), f"{fmt}: dequantized codes differ from the fused fake quant"
        q, s = LB.quantize_codes(rot_host[:n_or], fmt)
        codes_rows = LB.from_blocked(got.codes.cpu().numpy(), rows, C)[:n_or]
        assert np.array_equal(codes_rows, LB.e4m3_encode(q)), f"{fmt}: codes differ from the oracle"
        assert bits_equal(np.ascontiguousarray(got.scales.cpu().numpy()[:, :n_or].T), s), f"{fmt}: scales differ from the oracle"


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["plain_smooth", "mod_f16"])
@pytest.mark.parametrize("cpr,rows,rpb", [(4, 1000, 8), (15, 4097, 241), (36, 300, 2)])
def test_kernel_choice_does_not_change_the_bytes(mods, sign_bits, cpr, rows, rpb, entry):
    """Both kernels (and both PDL settings and shared-memory budgets) on one input give the same codes and scales."""
    ops, lowbit, L = mods
    x, smooth, scale, shift = make_inputs(cpr, rows, rpb, entry, 7 * cpr + rows)
    runs = []
    try:
        for small_max, smem_kb, pdl in ((1 << 40, 0, 1), (0, 0, 1), (0, 100, 0), (1 << 40, 0, 0)):
            L.set_tunable("rot_small_max_chunks", small_max)
            L.set_tunable("smem_kb", smem_kb)
            L.set_tunable("pdl", pdl)
            runs.append(lowbit.rotate_pack_codes(x, smooth, sign_bits, "e2m1", scale, shift))
    finally:
        L.set_tunable("rot_small_max_chunks", 40000)
        L.set_tunable("smem_kb", 0)
        L.set_tunable("pdl", 1)
    for r in runs[1:]:
        assert same_bytes(r.codes, runs[0].codes) and same_bytes(r.scales, runs[0].scales)


def _raw_call(L, x, smooth, bits, codes_ptr, scales_ptr, rows, C, fmt, mod=None, rpb=1):
    sb = (ctypes.c_uint32 * 4)(*[int(b) & 0xFFFFFFFF for b in bits])
    sp = smooth.data_ptr() if smooth is not None else None
    stream = torch.cuda.current_stream().cuda_stream
    if mod is None:
        return L.lib().fpq_transform_rotate_pack_codes(x.data_ptr(), sp, sb, codes_ptr, scales_ptr, rows, C, fmt, stream)
    return L.lib().fpq_modulate_transform_rotate_pack_codes(x.data_ptr(), mod[0].data_ptr(), mod[1].data_ptr(), rpb, sp, sb, codes_ptr,
                                                            scales_ptr, rows, C, fmt, 0, stream)


@pytest.mark.gpu
@pytest.mark.parametrize("cpr,rows", [(3, 5), (15, 129), (15, 25000), (36, 1001)])
@pytest.mark.parametrize("modulate", [False, True])
def test_padding_rows_and_one_launch(mods, sign_bits, cpr, rows, modulate):
    """Outputs pre-filled with 0xFF: the padding rows read back as code 0 / scale 0, written by the call's single launch."""
    ops, lowbit, L = mods
    C = 128 * cpr
    x = torch.randn(rows, C, device="cuda")
    mod = (torch.randn(1, C, device="cuda"), torch.randn(1, C, device="cuda")) if modulate else None
    rp = LB.rows_padded(rows)
    codes = torch.full((rp * C,), 0xFF, dtype=torch.uint8, device="cuda")
    scales = torch.full((cpr, rp), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    n0 = L.lib().fpq_launch_count()
    assert _raw_call(L, x, None, sign_bits, codes.data_ptr(), scales.data_ptr(), rows, C, L.FMT["e2m3"], mod, rows) == 0
    assert L.lib().fpq_launch_count() - n0 == 1
    want = lowbit.rotate_pack_codes(x.view(1, rows, C) if modulate else x, None, sign_bits, "e2m3",
                                    *((mod[0].view(1, 1, C), mod[1].view(1, 1, C)) if modulate else (None, None)))
    assert same_bytes(codes, want.codes) and same_bytes(scales, want.scales)
    blocked = codes.view(cpr, rp // 8, 8, 8, 16).permute(1, 3, 0, 2, 4).reshape(rp, C)
    assert int(blocked[rows:].count_nonzero()) == 0
    assert int(scales[:, rows:].count_nonzero()) == 0
    n0 = L.lib().fpq_launch_count()
    lowbit.rotate_pack_codes(x, None, sign_bits, "e2m1")
    assert L.lib().fpq_launch_count() - n0 == 1


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["e2m1", "e3m2"])
def test_forward_packed_equals_forward_of_the_rotation(mods, sign_bits, fmt):
    ops, lowbit, L = mods
    B, Lr, C, N = 4, 160, 1920, 640
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn(B, Lr, C, device="cuda", generator=g)
    scale = torch.randn(B, 1, C, device="cuda", generator=g) * 0.3
    shift = torch.randn(B, 1, C, device="cuda", generator=g) * 0.5
    smooth = torch.exp(torch.rand(C, device="cuda", generator=g) * 2 - 1)
    lin = torch.nn.Linear(C, N).cuda()
    with torch.no_grad():
        lin.weight.copy_(ops.transform_rotate_weight(lin.weight.detach().float().contiguous(), smooth, sign_bits))
    layer = lowbit.QuantizedLinearLowBit.from_float(lin, "e2m1", fmt)
    rot = ops.modulate_transform_rotate_quant(x, scale, shift, smooth, sign_bits, None)
    want = layer(rot)
    got = layer.forward_packed(lowbit.rotate_pack_codes(x, smooth, sign_bits, fmt, scale, shift))
    assert got.shape == (B * Lr, N)
    assert same_bytes(got, want.reshape(B * Lr, N))
    with pytest.raises(L.FpqError):
        layer.forward_packed(lowbit.rotate_pack_codes(x, smooth, sign_bits, "e1m2" if fmt != "e1m2" else "e2m1", scale, shift))
    with pytest.raises(L.FpqError):
        layer.forward_packed(lowbit.pack_codes(rot, fmt, per_row=True))


@pytest.mark.gpu
def test_argument_errors(mods, sign_bits):
    ops, lowbit, L = mods
    x = torch.randn(6, 256, device="cuda")
    with pytest.raises(L.FpqError):
        lowbit.rotate_pack_codes(x.cpu(), None, sign_bits, "e2m1")
    with pytest.raises(L.FpqError):
        lowbit.rotate_pack_codes(torch.randn(6, 200, device="cuda"), None, sign_bits, "e2m1")
    with pytest.raises(L.FpqError):
        lowbit.rotate_pack_codes(x, None, sign_bits, None)
    xm = x.view(2, 3, 256)
    ok = torch.zeros(2, 1, 256, device="cuda")
    with pytest.raises(L.FpqError):
        lowbit.rotate_pack_codes(xm, None, sign_bits, "e2m1", torch.zeros(3, 1, 256, device="cuda"), ok)
    with pytest.raises(L.FpqError):
        lowbit.rotate_pack_codes(xm, None, sign_bits, "e2m1", ok, ok.cpu())
    # scale 0 / shift 0 is no modulate at all
    a = lowbit.rotate_pack_codes(xm, None, sign_bits, "e2m1", ok, ok)
    b = lowbit.rotate_pack_codes(x, None, sign_bits, "e2m1")
    assert same_bytes(a.codes, b.codes) and same_bytes(a.scales, b.scales)
    # through the C ABI: rows not a multiple of rows_per_batch, format -1, misaligned outputs
    rp = LB.rows_padded(6)
    codes = torch.empty(rp * 256 + 64, dtype=torch.uint8, device="cuda")
    scales = torch.empty(2 * rp + 4, dtype=torch.float32, device="cuda")
    mod = (torch.zeros(2, 256, device="cuda"), torch.zeros(2, 256, device="cuda"))
    assert _raw_call(L, x, None, sign_bits, codes.data_ptr(), scales.data_ptr(), 6, 256, 0, mod, 4) == L.FPQ_ERR_ARG
    assert _raw_call(L, x, None, sign_bits, codes.data_ptr(), scales.data_ptr(), 6, 256, -1) == L.FPQ_ERR_ARG
    assert _raw_call(L, x, None, sign_bits, codes.data_ptr() + 8, scales.data_ptr(), 6, 256, 0) == L.FPQ_ERR_ARG
    assert _raw_call(L, x, None, sign_bits, codes.data_ptr(), scales.data_ptr() + 2, 6, 256, 0) == L.FPQ_ERR_ARG
    assert _raw_call(L, x, None, sign_bits, codes.data_ptr(), scales.data_ptr(), 6, 200, 0) == L.FPQ_ERR_ARG
    assert _raw_call(L, x, None, sign_bits, codes.data_ptr(), scales.data_ptr() + 4, 6, 256, 0) == 0     # 4-byte aligned scales


@pytest.mark.gpu
def test_more_than_2pow31_elements(mods, sign_bits):
    """Windows of one launch over > 2^31 elements equal separate launches of the same rows (64-bit indexing of the codes)."""
    ops, lowbit, L = mods
    free, _ = torch.cuda.mem_get_info()
    C = 1920
    rows = (1 << 31) // C + 500
    if free < rows * C * 6 + (6 << 30):
        pytest.skip("not enough free HBM")
    x = torch.empty(rows, C, device="cuda")
    step = 1 << 16
    for i in range(0, rows, step):
        m = min(step, rows - i)
        idx = torch.arange(i * C, (i + m) * C, device="cuda", dtype=torch.int64).view(m, C)
        x[i:i + m] = (((idx * 2654435761) % 2001 - 1000).float() * ((idx // 128) % 8191 + 1).float() * 1e-3)
    s = torch.exp(torch.linspace(-1, 1, C, device="cuda"))
    cpr = C // 128

    def window(p, r0, n):
        rb = p.rows_pad // 8
        return p.codes.view(cpr, rb, 1024)[:, r0 // 8:(r0 + n) // 8], p.scales[:, r0:r0 + n]

    big = lowbit.rotate_pack_codes(x, s, sign_bits, "e2m1")
    rp = big.rows_pad
    for r0 in (0, ((1 << 31) // C) // 128 * 128 - 128, rp - 256):
        part = lowbit.rotate_pack_codes(x[r0:min(r0 + 256, rows)].clone(), s, sign_bits, "e2m1")
        (bc, bs), (pc, ps) = window(big, r0, 256), window(part, 0, 256)
        assert torch.equal(bc, pc) and same_bytes(bs, ps), f"rows [{r0}, {r0 + 256})"
        assert bool((pc != 0).any())
    del big
    # adaLN entry past 2^31 elements as well: 971 batches of 1152 rows = 2 147 696 640 elements
    B, rpb = 971, 1152
    assert B * rpb * C > (1 << 31) and B * rpb <= rows
    xm = x[:B * rpb].view(B, rpb, C)
    sc = torch.randn(B, 1, C, device="cuda") * 0.3
    sh = torch.randn(B, 1, C, device="cuda") * 0.5
    bigm = lowbit.rotate_pack_codes(xm, s, sign_bits, "e2m1", sc, sh)
    for b in (0, B // 2, B - 1):
        part = lowbit.rotate_pack_codes(xm[b:b + 1].clone(), s, sign_bits, "e2m1", sc[b:b + 1].clone(), sh[b:b + 1].clone())
        (bc, bs), (pc, ps) = window(bigm, b * rpb, rpb), window(part, 0, rpb)
        assert torch.equal(bc, pc) and same_bytes(bs, ps), f"modulate batch {b}"


def test_cpu_tensors_are_rejected_before_any_kernel_is_loaded(monkeypatch):
    from fpqvar_b200 import _lib as L, lowbit, ops

    def no_load(*_a, **_k):
        raise AssertionError("a kernel library was loaded")

    monkeypatch.setattr(L, "lib", no_load)
    monkeypatch.setattr(ops, "_ext", no_load)
    monkeypatch.setattr(lowbit, "_ext", no_load)
    from fpqvar_b200.hotpath import seed42_sign_bits
    with pytest.raises(L.FpqError):
        lowbit.rotate_pack_codes(torch.randn(4, 256), None, seed42_sign_bits(), "e2m1")
    with pytest.raises(L.FpqError):
        lowbit.rotate_pack_codes(torch.randn(2, 2, 256), None, seed42_sign_bits(), "e2m1", torch.zeros(2, 1, 256), torch.zeros(2, 1, 256))
