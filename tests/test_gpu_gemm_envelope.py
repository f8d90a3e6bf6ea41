"""The low-bit GEMM (csrc/fpq_gemm.cu) at the edges of its numerics contract, against oracle/gemm_codes.c:
  - F1-F3 accumulation probes (oracle/lowbit.py envelope_probe) for all 25 format pairs, 128-groups and row scales: bit-exact
    inside the exact-accumulation envelope (oracle/lowbit.py exact_accumulation), within the stated bound outside it;
  - the fp32 scale epilogue on scales that overflow, underflow, vanish or are not finite, and on +-0 / +-inf biases;
  - degenerate activations and weights through the quantizer end to end, against the oracle and against the reference's
    expression F.linear(fake_quant(x), fake_quant(W));
  - the fused loss (fpq_gemm_codes_sse) on the same probes;
  - the host checks of linear_codes_sse, with a library stub that records every launch.
The operands of the probes are built from exact grid values, so the quantizer stays out of the way."""
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from fpqvar_b200 import _lib as L, lowbit, ops
from oracle import lowbit as LB, oracle as O          # checker only

pytestmark = pytest.mark.gpu
FMTS = ["e2m1", "e1m2", "e3m0", "e2m3", "e3m2"]
PAIRS = [(a, w) for a in FMTS for w in FMTS]
SHAPES = [(128, 128), (640, 128), (1920, 1920), (2304, 2304), (7680, 7680)]       # (k, scale group)
VARIANTS = [(256, 1), (256, 0), (128, 0)]                                           # (gemm_tile_n, gemm_pair)


def dev():
    return torch.device("cuda:0")


def bits(a):
    return a.view({2: np.uint16, 4: np.uint32, 8: np.uint64}[a.dtype.itemsize])


def same_bits(a, b):
    """bit-identical, NaN payloads aside (signed zeros and NaN positions count)"""
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(bits(a)[~na], bits(b)[~nb])


@contextmanager
def variant(tile_n, pair):
    L.set_tunable("gemm_tile_n", tile_n)
    L.set_tunable("gemm_pair", pair)
    try:
        yield
    finally:
        L.set_tunable("gemm_tile_n", 256)
        L.set_tunable("gemm_pair", -1)


def packed(q, s, fmt, group):
    """PackedCodes straight from grid values and scales [rows, k / group]."""
    codes = torch.from_numpy(LB.to_blocked(LB.e4m3_encode(q))).to(dev())
    scales = torch.from_numpy(LB.scales_layout(np.ascontiguousarray(s, dtype=np.float32))).to(dev())
    return lowbit.PackedCodes(codes, scales, q.shape[0], q.shape[1], fmt, group).check("probe")


def ulps(got, want):
    """|got - want| in fp32 ulps of want (finite entries)."""
    f = np.isfinite(want)
    d = np.abs(got[f].astype(np.float64) - want[f].astype(np.float64))
    return float(np.max(d / np.spacing(np.abs(want[f])).astype(np.float64)))


@pytest.mark.parametrize("k,group", SHAPES)
@pytest.mark.parametrize("fmt_a,fmt_w", PAIRS)
def test_accumulation_probes(fmt_a, fmt_w, k, group):
    """Inside the envelope every slab sum is exact in fp32 whatever the order of the additions: bit-exact.  Outside it the slab
    sums may round: |C - oracle| <= (k_acc - 1) * 2^-24 * sum_t |sa sw| sum |qa qw| plus one fp32 rounding of the scale chain
    per group; the fp16 output is the fp32 one rounded.  The fused loss against the oracle's own C is exactly 0 inside the
    envelope, and sum d^2 for ref = C + d."""
    qa, sa, qw, sw = LB.envelope_probe(fmt_a, fmt_w, k, group)
    want = LB.gemm_codes(qa, sa, qw, sw)
    a, w = packed(qa, sa, fmt_a, group), packed(qw, sw, fmt_w, group)
    exact = LB.exact_accumulation(fmt_a, fmt_w, group)
    unit = LB.grid_unit(fmt_a) * LB.grid_unit(fmt_w)
    mag = np.einsum("tij,it,jt->ij", LB.slab_sums_units(np.abs(qa), fmt_a, np.abs(qw), fmt_w, group) * unit,
                    sa.astype(np.float64), sw.astype(np.float64))
    tol = (group - 1) * 2.0 ** -24 * mag + (k // group) * 2.0 ** -24 * mag
    rng = np.random.default_rng(k + group)
    d = (rng.integers(-2, 3, size=want.shape) * np.spacing(np.abs(want))).astype(np.float32)
    ref_d = (want + d).astype(np.float32)
    assert np.array_equal(ref_d.astype(np.float64) - want, d.astype(np.float64))        # C + d is exact, so is the difference
    worst = 0.0
    for tile_n, pair in VARIANTS:
        with variant(tile_n, pair):
            c32 = lowbit.linear_codes(a, w, None, torch.float32).cpu().numpy()
            c16 = lowbit.linear_codes(a, w, None, torch.float16).cpu().numpy()
            if exact:
                sse0 = lowbit.linear_codes_sse(a, w, torch.from_numpy(want).to(dev())).item()
                sse_d = lowbit.linear_codes_sse(a, w, torch.from_numpy(ref_d).to(dev())).item()
        if exact:
            assert same_bits(c32, want), f"{fmt_a} x {fmt_w} k {k} group {group} tile {tile_n} pair {pair}"
            assert same_bits(c16, want.astype(np.float16))
            assert sse0 == 0.0
            want_d = float((d.astype(np.float64) ** 2).sum())
            assert abs(sse_d - want_d) <= 2e-6 * want_d
        else:
            assert np.all(np.abs(c32.astype(np.float64) - want) <= tol)
            assert same_bits(c16, c32.astype(np.float16))         # the same slab sums, rounded to fp16 at the end
            worst = max(worst, ulps(c32, want))
    print(f"ENVELOPE {fmt_a} x {fmt_w} k={k} k_acc={group} bits={LB.accumulation_bits(fmt_a, fmt_w, group):.2f} "
          f"{'exact' if exact else 'outside'}: {'bit-exact' if exact else f'max deviation {worst:g} ulp'}")


SCALE_CASES = [("e2m1", "e2m1", 640, 128), ("e3m2", "e2m3", 640, 128), ("e1m2", "e3m0", 640, 128),
               ("e2m1", "e2m1", 256, 256), ("e3m2", "e2m3", 256, 256)]


@pytest.mark.parametrize("fmt_a,fmt_w,k,group", SCALE_CASES)
def test_scale_chain_probes(fmt_a, fmt_w, k, group):
    """Generic non-power-of-two scales (whose other operation orders give other bits, tests/test_oracle_gemm_envelope.py),
    scales near 2^+-60, fp32-subnormal scales, overflowing scale products, zero scales with P != 0, NaN and inf scales with
    P = 0 and P != 0, bias +-0 and +-inf: bit-exact, NaN positions included.  The fused loss of a product with NaN entries is
    NaN, also with every row weight 0 (0 * NaN = NaN: a NaN never vanishes from the loss)."""
    assert LB.exact_accumulation(fmt_a, fmt_w, group)
    qa, sa, qw, sw, bias = LB.scale_chain_probe(fmt_a, fmt_w, 160, 136, k, group)
    a, w = packed(qa, sa, fmt_a, group), packed(qw, sw, fmt_w, group)
    want_b, want = LB.gemm_codes(qa, sa, qw, sw, bias), LB.gemm_codes(qa, sa, qw, sw)
    assert np.isnan(want).any() and np.isinf(want).any()
    tb = torch.from_numpy(bias).to(dev())
    for tile_n, pair in VARIANTS:
        with variant(tile_n, pair):
            c32b = lowbit.linear_codes(a, w, tb, torch.float32).cpu().numpy()
            c16b = lowbit.linear_codes(a, w, tb, torch.float16).cpu().numpy()
            c32 = lowbit.linear_codes(a, w, None, torch.float32).cpu().numpy()
            ref = torch.from_numpy(want).to(dev())
            sse = lowbit.linear_codes_sse(a, w, ref).item()
            sse_rw0 = lowbit.linear_codes_sse(a, w, ref, None, None, torch.zeros(160, dtype=torch.float64, device=dev())).item()
        assert same_bits(c32b, want_b), (tile_n, pair)
        assert same_bits(c16b, want_b.astype(np.float16)), (tile_n, pair)
        assert same_bits(c32, want), (tile_n, pair)
        assert np.isnan(sse) and np.isnan(sse_rw0)


def degenerate(rng, rows, k, dtype):
    """standard normal rows with: a zero group, a single +inf and a single -inf element, a single NaN, a group whose fp16 scale
    is subnormal, and a group at the top of the dtype's range (fp16: 65504 and 65000, where q * s of e3m2 overflows fp16 in the
    fake-quantized tensor but not in the codes; fp32: 1e38)."""
    x = rng.standard_normal((rows, k)).astype(dtype)
    x[0, :128] = 0
    x[1, 5] = np.inf
    x[2, 130] = np.nan
    x[3, :128] = (x[3, :128].astype(np.float32) * 2.0 ** -20).astype(dtype)
    x[4, 128:256] = (np.sign(x[4, 128:256]) * (65504.0 if dtype == np.float16 else 1e38)).astype(dtype)
    x[4, 128] = 65000.0 if dtype == np.float16 else 3e37
    x[5, 7] = -np.inf
    return x


@pytest.mark.parametrize("per_row", [False, True])
@pytest.mark.parametrize("dtype", [np.float16, np.float32])
@pytest.mark.parametrize("fmt_a,fmt_w", [("e2m1", "e2m1"), ("e3m2", "e3m2"), ("e3m2", "e2m1"), ("e1m2", "e3m0")])
def test_degenerate_inputs_end_to_end(fmt_a, fmt_w, dtype, per_row):
    """Bit-exact against the oracle, and against the reference's expression F.linear(fake_quant(x), fake_quant(W)) (evaluated in
    float64 on the ops.fake_quant tensors) on the NaN / inf pattern.  An inf or NaN element makes its group's scale inf or NaN
    and every code of the group 0 (x / inf = 0, inf / inf = NaN -> 0), so the group's slab sum is 0 and 0 * inf = NaN: the
    product is NaN exactly where the reference's is -- a non-finite group never yields inf.  The documented differences:
    (1) where q * s overflows fp16 in the reference's fake-quantized tensor (e3m2 near 65504), the reference is NaN and the
    codes, which never form q * s, give a finite number; (2) the fp32 product overflows to +-inf where the float64 value is
    beyond (or, for a partial sum of the fp32 chain, near) the fp32 range, with the sign of the float64 value."""
    rng = np.random.default_rng(11)
    m, n, k = 200, 136, 384
    x = degenerate(rng, m, k, dtype)
    wt = degenerate(rng, n, k, np.float32)
    group = None if per_row else 128
    tx, tw = torch.from_numpy(x).to(dev()), torch.from_numpy(wt).to(dev())
    a, w = lowbit.pack_codes(tx, fmt_a, per_row), lowbit.pack_codes(tw, fmt_w, per_row)
    (qa, sa), (qw, sw) = LB.quantize_codes(x, fmt_a, group), LB.quantize_codes(wt, fmt_w, group)
    want = LB.gemm_codes(qa, sa, qw, sw)
    c32 = lowbit.linear_codes(a, w, None, torch.float32).cpu().numpy()
    c16 = lowbit.linear_codes(a, w, None, torch.float16).cpu().numpy()
    assert same_bits(c32, want) and same_bits(c16, want.astype(np.float16))
    xq = ops.fake_quant(tx, fmt_a, group, "kernel").cpu().double().numpy()
    wq = ops.fake_quant(tw, fmt_w, group, "kernel").cpu().double().numpy()
    with np.errstate(invalid="ignore", over="ignore"):
        ref = xq @ wq.T
    nan_c, nan_r = np.isnan(c32), np.isnan(ref)
    assert nan_c.any() and not (nan_c & ~nan_r).any()              # every NaN of the product is a NaN of the reference
    overflowed = np.isinf(xq).any(1)[:, None] | np.isinf(wq).any(1)[None, :]
    assert np.array_equal(nan_r & ~nan_c, nan_r & ~nan_c & overflowed)           # (1)
    if dtype == np.float32:
        assert not overflowed.any() and np.array_equal(nan_c, nan_r)
    inf_c = np.isinf(c32)
    assert np.all(nan_r[inf_c] | (np.abs(ref[inf_c]) >= 2.0 ** 120))             # (2)
    fin = inf_c & ~nan_r
    assert np.array_equal(np.sign(c32[fin]), np.sign(ref[fin]))


class _StubLib:
    """Stands in for the CUDA library: records every entry point called and returns success without launching anything."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def call(*args):
            self.calls.append(name)
            return 0
        return call


def test_linear_codes_sse_checks_its_arguments_on_the_host(monkeypatch):
    a = lowbit.pack_codes(torch.randn(8, 256, device=dev(), dtype=torch.float16), "e2m1")
    w = lowbit.pack_codes(torch.randn(16, 256, device=dev()), "e2m1")
    ref = torch.zeros(8, 16, device=dev())
    stub = _StubLib()
    monkeypatch.setattr(L, "lib", lambda: stub)
    bad = [dict(bias=torch.zeros(16)),                                     # on the CPU
           dict(bias=torch.zeros(15, device=dev())),                       # one entry short: the epilogue would read past it
           dict(bias=torch.zeros(17, device=dev()))]
    if torch.cuda.device_count() > 1:
        other = torch.device("cuda:1")
        bad += [dict(ref=ref.to(other)), dict(sse=torch.zeros(1, dtype=torch.float64, device=other)),
                dict(row_weight=torch.ones(8, dtype=torch.float64, device=other))]
    for kw in bad:
        args = dict(ref=ref, bias=None, sse=None, row_weight=None)
        args.update(kw)
        with pytest.raises(L.FpqError):
            lowbit.linear_codes_sse(a, w, args["ref"], args["bias"], args["sse"], args["row_weight"])
    assert stub.calls == []
    lowbit.linear_codes_sse(a, w, ref, torch.zeros(16, device=dev()))
    assert stub.calls == ["fpq_gemm_codes_sse"]                                   # the stub does stand in for the library
