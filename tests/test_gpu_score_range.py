"""GPU: the format scorers and the search losses across the whole fp16 / fp32 scale range, group by group.

fpq_score_formats returns one float64 total per candidate, and the search picks a layer's format from those totals.  A test
on one total hides every group that is small next to the largest ones, so every call here holds groups of one class only
(tests/score_range_cases.py): one binade of the group absmax with one content kind, or one boundary case of the scorers'
branch switches, or one probe group among all-zero groups.  Then the bar on the call's total is a bar on each group.

The bar, 2e-6 relative, against the float64 sum of the oracle port's per-element errors (which are exact: x and x_q are
fp16 / fp32 values and their difference and square are exact in float64):
  * generic kernel (fp32 input, fp16 input under the argmin rule): 16 terms per lane in an fp32 fmaf chain (<= 16 roundings
    of 2^-24 relative each), then float64;
  * fp16 kernel-rule kernel: 2 x 16 FHFMA (fp16 * fp16 + fp32), acc0 + acc1, then 8 groups' lane sums over 5 fp32 shuffle
    levels: about 16 + 1 + 5 = 22 roundings, 22 * 2^-24 = 1.3e-6;
  2e-6 covers both.  All terms are >= 0, so no cancellation widens it.

fp32 squares: the kernels square and sum in fp32 (see include/fpq_b200.h at fpq_score_formats), so a group whose exact
error is beyond the fp32 range scores +inf where a float64 statement is finite (test_fp32_square_overflow pins that
contract on both sides of its band), and squares below the fp32 range count as 0: the bar has an absolute part of
n * 2^-149 for n elements, so fp32 groups with an absmax below about 2^-60 score 0.

Also here: the strided-output and strided-reference forms of the low-bit GEMM (ldc / ldr > n) and the edges of
fpq_sse_rows."""
import ctypes

import numpy as np
import pytest
import torch

import score_range_cases as C
from oracle import lowbit as LB
from test_gpu_persistent_loops import assert_same, grid_caps, ref_split, sym, split

pytestmark = pytest.mark.gpu
F16, F32 = torch.float16, torch.float32
TORCH = {np.float16: F16, np.float32: F32}
BAR = 2e-6
FORMATS = C.FORMATS
GPW = {("f16", "kernel"): 8, ("f16", "argmin"): 4, ("f32", "kernel"): 4, ("f32", "argmin"): 4}     # groups per warp trip
VARIANTS = [(np.float32, "kernel"), (np.float32, "argmin"), (np.float16, "kernel"), (np.float16, "argmin")]
VIDS = [f"{np.dtype(d).name}-{t}" for d, t in VARIANTS]


@pytest.fixture(scope="module")
def L():
    from fpqvar_b200 import _lib
    _lib.lib()
    return _lib


def _stream():
    return torch.cuda.current_stream().cuda_stream


def fmt_code(L, f):
    return L.FMT[f] if f in L.FMT else 16 + L.SPLIT[f]


def score_into(L, ptr, n_groups, dt, fmts, tie, sse_ptr):
    codes = (ctypes.c_int * len(fmts))(*[fmt_code(L, f) for f in fmts])
    return L.lib().fpq_score_formats(ptr, n_groups, 128, L.FPQ_F16 if dt == np.float16 else L.FPQ_F32, codes, len(fmts), L.TIE[tie],
                                     sse_ptr, _stream())


def score_calls(L, xs, tie, fmts=FORMATS):
    """One fpq_score_formats call per array of xs ([G, 128] each, one dtype); returns [len(xs), len(fmts)] float64."""
    dt = xs[0].dtype.type
    dev = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in xs]
    sse = torch.zeros(len(xs), len(fmts), dtype=torch.float64, device="cuda")
    for i, x in enumerate(dev):
        L.check(score_into(L, x.data_ptr(), x.shape[0], dt, fmts, tie, sse[i].data_ptr()), "fpq_score_formats")
    return sse.cpu().numpy()


def lane_pieces(d):
    """float64 SSE of every 16-element lane piece of the generic scorer, [.., G, 8]: element i of a group is in piece
    (i / 4) % 8.  (The fp16 kernel's pieces are of fp16 errors, whose squares never leave the fp32 range.)"""
    with np.errstate(over="ignore", invalid="ignore"):
        d2 = d * d
    return d2.reshape(d.shape[:-1] + (4, 8, 4)).sum(axis=(-3, -1))


def oracle(xs, tie, fmts=FORMATS):
    """float64 totals [len(xs), len(fmts)] of the oracle port's errors and the largest lane piece of each call; xs of one
    shape are stacked into one port call."""
    big = np.stack(xs) if len({x.shape for x in xs}) == 1 else None
    tot, top = np.empty((len(xs), len(fmts))), np.empty((len(xs), len(fmts)))
    for j, f in enumerate(fmts):
        for i, d in ([(None, C.errors(big, f, tie))] if big is not None else [(i, C.errors(x, f, tie)) for i, x in enumerate(xs)]):
            sl = slice(None) if i is None else i
            with np.errstate(over="ignore", invalid="ignore"):
                tot[sl, j] = (d * d).sum(axis=(-2, -1))
            p = lane_pieces(d)
            top[sl, j] = np.where(np.isnan(p), 0.0, p).max(axis=(-2, -1))
    return tot, top


def floor(n_elements):
    """The absolute part of the bar: each fp32 rounding of a square or partial sum can be off by up to 2^-150, so squares
    below the fp32 range count as 0 (include/fpq_b200.h at fpq_score_formats)."""
    return n_elements * 2.0 ** -149


def mismatches(got, want, top, n_elements, labels, fmts=FORMATS, bar=BAR):
    """(label, fmt, got, want) of every entry that breaks the contract of include/fpq_b200.h: the class (NaN, +-inf,
    finite) of a non-finite float64 sum; +inf once a lane piece's float64 SSE exceeds 2 FLT_MAX; below FLT_MAX / 2 in every
    piece, finite and within bar * want + floor(n_elements).  Entries in the band between are left out."""
    bad = []
    for i in range(want.shape[0]):
        for j, f in enumerate(fmts):
            g, w, t = float(got[i, j]), float(want[i, j]), float(top[i, j])
            if np.isnan(w) or np.isinf(w):
                ok = (np.isnan(g) and np.isnan(w)) or g == w
            elif t > 2 * C.FLT_MAX:
                ok = g == np.inf
            elif t >= C.FLT_MAX / 2:
                continue
            else:
                ok = np.isfinite(g) and abs(g - w) <= bar * w + floor(n_elements[i])
            if not ok:
                bad.append((labels[i], f, g, w))
    return bad


def report(bad, what):
    assert not bad, f"{what}: {len(bad)} (class, candidate) entries off the bar, first:\n" + "\n".join(
        f"  {lab}  {f}: got {g!r} want {w!r}" for lab, f, g, w in bad[:12])


# ------------------------------------------------------------------------------------------------------------------------
# per-class calls: binade sweep and boundary cases, all eight candidates in one call, and the ranking the search takes
# ------------------------------------------------------------------------------------------------------------------------
_CASES = {}


def cases(dt):
    if dt not in _CASES:
        _CASES[dt] = C.binade_cases(dt) + C.boundary_cases(dt)
    return _CASES[dt]


@pytest.mark.parametrize("dt,tie", VARIANTS, ids=VIDS)
def test_score_formats_per_class(L, dt, tie):
    cs = cases(dt)
    xs = [c.x for c in cs]
    got = score_calls(L, xs, tie)
    want, top = oracle(xs, tie)
    n = [x.size for x in xs]
    report(mismatches(got, want, top, n, [c.label for c in cs]), f"score_formats {np.dtype(dt).name} {tie}")
    # ranking: wherever the oracle's best two candidates are further apart than the bar, the scorer picks the same one
    wrong = []
    for i, c in enumerate(cs):
        w = np.sort(want[i])
        if (np.all(np.isfinite(got[i])) and np.all(top[i] < C.FLT_MAX / 2) and w[1] - w[0] > 2 * (BAR * w[1] + floor(n[i]))
                and int(np.argmin(got[i])) != int(np.argmin(want[i]))):
            wrong.append(f"{c.label}: picks {FORMATS[int(np.argmin(got[i]))]}, oracle {FORMATS[int(np.argmin(want[i]))]}")
    assert not wrong, f"{len(wrong)} classes ranked differently:\n" + "\n".join(wrong[:12])


# ------------------------------------------------------------------------------------------------------------------------
# isolation: one probe group among all-zero groups, at every slot of a warp trip, as the last group before dead lane
# sets, and on a later trip of the grid-stride loop
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt,tie", VARIANTS, ids=VIDS)
def test_zero_group_scores_exactly_zero(L, dt, tie):
    z = np.zeros((37, 128), dtype=dt)
    z[::2, 5] = dt(-0.0)
    got = score_calls(L, [z], tie)
    assert np.all(got == 0.0), got


@pytest.mark.parametrize("dt,tie", VARIANTS, ids=VIDS)
def test_probe_group_isolated(L, dt, tie):
    gpw = GPW[(np.dtype(dt).name[0] + np.dtype(dt).name[-2:], tie)]
    probes = [c.x[:1] for c in C.boundary_cases(dt)]
    labels = [c.label for c in C.boundary_cases(dt)]
    want, top = oracle(probes, tie)
    cap = grid_caps()["score"]
    late = 3 * cap + 5 * gpw + 3                       # > 3 x the grid: every warp makes at least three trips
    layouts = [(2 * gpw, gpw + j) for j in range(gpw)]                     # every slot of a warp trip
    layouts += [(3 * gpw + r, 3 * gpw + r - 1) for r in (1, gpw - 1)]      # the last group, dead lane sets behind it
    layouts += [(late, late - 1), (late, 3 * cap + 2)]                     # a later trip of the grid-stride loop
    buf = torch.zeros(late, 128, dtype=TORCH[dt], device="cuda")
    sse = torch.zeros(len(layouts), len(probes), len(FORMATS), dtype=torch.float64, device="cuda")
    dev = torch.from_numpy(np.concatenate(probes)).cuda()
    for li, (n, at) in enumerate(layouts):
        for pi in range(len(probes)):
            buf[at] = dev[pi]
            L.check(score_into(L, buf.data_ptr(), n, dt, FORMATS, tie, sse[li, pi].data_ptr()), "fpq_score_formats")
            buf[at] = 0
    got = sse.cpu().numpy()
    bad = []
    for li, (n, at) in enumerate(layouts):
        bad += mismatches(got[li], want, top, [128] * len(probes), [f"{lab} at group {at} of {n}" for lab in labels])
    report(bad, f"probe {np.dtype(dt).name} {tie}")


@pytest.mark.parametrize("fmt", ["e2m1", "e3m0"])
def test_literal_fallback_lanes_score_their_own_elements(L, fmt):
    """fp16, kernel rule: a group on the literal path (fp16-subnormal scale) in the same warp trip as a fast-path group.
    The per-lane sums are exact here, and each lane of the literal group scores its own 32 elements, so lane 0 adds the fast
    group's 2^-24 to the literal group's 0 and the total is 2^-24 + 2 * 2^-48 exactly.  A lane that scored its neighbour's
    elements would add 2^-48 to 2^-24 first, which rounds away in fp32."""
    v = C.vmax(fmt)
    u = 2.0 ** -24
    lit = np.zeros(128, dtype=np.float64)
    lit[8 * 4] = 4 * u * v             # chunk 4 (lane 0): the absmax, scale 4u (fp16-subnormal), on the grid
    lit[8 * 1] = 5 * u                 # lane 1: x / s = 1.25, one u from the grid
    lit[8 * 3] = 5 * u                 # lane 3
    fast = np.zeros(128, dtype=np.float64)
    fast[8 * 1] = 2.0 ** -10 * v       # lane 1: the absmax, scale 2^-10 (normal), on the grid
    fast[8 * 0] = 1.25 * 2.0 ** -10    # lane 0: error 2^-12
    for a, b in ((lit, fast), (fast, lit)):
        x = np.zeros((8, 128), dtype=np.float16)
        x[0], x[1] = a, b
        want = float(C.group_sse(x, fmt, "kernel").sum())
        assert want == 2.0 ** -24 + 2.0 ** -47
        got = score_calls(L, [x], "kernel", [fmt])[0, 0]
        assert got == want, (fmt, got, want)


# ------------------------------------------------------------------------------------------------------------------------
# candidate independence: alone, among all eight, reversed, duplicated
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt,tie", VARIANTS, ids=VIDS)
def test_candidates_score_independently(L, dt, tie):
    cs = C.boundary_cases(dt) + [c for c in cases(dt) if c.binade is not None and c.binade % 7 == 0]
    x = np.concatenate([c.x for c in cs])
    base = score_calls(L, [x], tie)[0]
    rev = score_calls(L, [x], tie, FORMATS[::-1])[0][::-1]
    for j, f in enumerate(FORMATS):
        alone = score_calls(L, [x], tie, [f])[0, 0]
        dup = score_calls(L, [x], tie, [f, FORMATS[(j + 3) % 8], f])[0]
        for tag, g in (("alone", alone), ("reversed", rev[j]), ("duplicated", dup[0]), ("duplicated twice", dup[2])):
            assert g == base[j] or abs(g - base[j]) <= 1e-12 * abs(base[j]), (f, tag, g, base[j])


# ------------------------------------------------------------------------------------------------------------------------
# non-finite groups
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt,tie", VARIANTS, ids=VIDS)
def test_nonfinite_groups(L, dt, tie):
    rng = np.random.default_rng(11)
    base = rng.standard_normal((16, 128)).astype(dt)
    xs, labels = [], []
    specials = [("nan", np.nan), ("+inf", np.inf), ("-inf", -np.inf)]
    if dt == np.float16:
        specials += [("65504", 65504.0), ("-65504", -65504.0)]
    for name, val in specials:
        for col in (0, 77, 127):
            x = base.copy()
            x[:, col] = dt(val)
            xs.append(x)
            labels.append(f"{name} at {col}")
    got = score_calls(L, xs, tie)
    want, top = oracle(xs, tie)
    if dt == np.float16 and tie == "kernel":      # fp16 output: 65504 quantizes to inf on every candidate but e3m0
        i = labels.index("65504 at 0")
        assert [bool(np.isinf(want[i, j])) for j in range(8)] == [f != "e3m0" for f in FORMATS], want[i]
    report(mismatches(got, want, top, [x.size for x in xs], labels), f"non-finite {np.dtype(dt).name} {tie}")


# ------------------------------------------------------------------------------------------------------------------------
# fp32 overflow of the squares
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tie", ["kernel", "argmin"])
def test_fp32_square_overflow(L, tie):
    """+inf (never NaN, never finite) once some lane piece's float64 SSE exceeds 2 FLT_MAX; finite and within the bar while
    every piece's stays below FLT_MAX / 2; the band between is left to fp32 rounding."""
    rng = np.random.default_rng(5)
    mags = [10.0 ** p for p in np.arange(16.0, 22.01, 0.25)] + [1e30, 1e37]
    xs = [(rng.standard_normal((8, 128)) * m).astype(np.float32) for m in mags]
    got = score_calls(L, xs, tie)
    n_inf = n_fin = 0
    for j, f in enumerate(FORMATS):
        for i, x in enumerate(xs):
            pieces = lane_pieces(C.errors(x, f, tie))
            if np.max(pieces) > 2 * C.FLT_MAX:
                assert got[i, j] == np.inf, (f, mags[i], got[i, j])
                n_inf += 1
            elif np.max(pieces) < C.FLT_MAX / 2:
                w = float(pieces.sum())
                assert np.isfinite(got[i, j]) and abs(got[i, j] - w) <= BAR * w, (f, mags[i], got[i, j], w)
                n_fin += 1
    assert n_inf >= 16 and n_fin >= 16, (n_inf, n_fin)


# ------------------------------------------------------------------------------------------------------------------------
# argument checks: no launch
# ------------------------------------------------------------------------------------------------------------------------
def test_score_formats_argument_checks(L):
    x = torch.zeros(4 * 128 + 16, dtype=F32, device="cuda")
    sse = torch.full((9,), 7.0, dtype=torch.float64, device="cuda")
    lib = L.lib()

    def call(fmts, n_rows=4, row_len=128, ptr=None, tie="kernel"):
        codes = (ctypes.c_int * max(1, len(fmts)))(*fmts)
        return lib.fpq_score_formats(ptr or x.data_ptr(), n_rows, row_len, L.FPQ_F32, codes, len(fmts), L.TIE[tie], sse.data_ptr(), _stream())

    before = lib.fpq_launch_count()
    assert call([]) == L.FPQ_ERR_ARG
    assert call([0] * 9) == L.FPQ_ERR_ARG
    for bad in (-1, 5, 15, 19):
        assert call([0, bad]) == L.FPQ_ERR_ARG, bad
    for rl in (64, 256):
        assert call([0], row_len=rl) == L.FPQ_ERR_UNSUPPORTED, rl
    for off in (2, 8):
        assert call([0], ptr=x.data_ptr() + off) == L.FPQ_ERR_ARG, off
    assert call([0, 16, 18], n_rows=0) == L.FPQ_OK
    torch.cuda.synchronize()
    assert lib.fpq_launch_count() == before
    assert bool((sse == 7.0).all())


# ------------------------------------------------------------------------------------------------------------------------
# the quantizers on the same cases, bit for bit
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("row_len", [128, 1920])
@pytest.mark.parametrize("dt,tie", VARIANTS, ids=VIDS)
def test_quantizers_bit_exact_on_the_range_cases(L, dt, tie, row_len):
    cs = cases(dt)
    xh = np.concatenate([c.x[:8] for c in cs])
    xh = xh[: xh.shape[0] // 15 * 15].reshape(-1, row_len)
    x = torch.from_numpy(xh).cuda()
    dout = TORCH[dt] if tie == "kernel" else F32
    npo = np.float16 if dout == F16 else np.float32
    for f in C.SYM:
        want = C.P.fake_quant(xh, f, None, tie, clamp3=False, out_dtype=npo)
        assert_same(sym(L, x, f, tie, False, dout), want, f"fake_quant {f} {np.dtype(dt).name} {tie} rows of {row_len}")
    for f in C.SPLIT:
        want = ref_split(xh, f, tie, npo)
        assert_same(split(L, x, f, tie, dout), want, f"signsplit {f} {np.dtype(dt).name} {tie} rows of {row_len}")


# ------------------------------------------------------------------------------------------------------------------------
# the low-bit GEMM with a row stride: C as the middle third of an [m, 3n] matrix, ref as a slice of a NaN-filled buffer
# ------------------------------------------------------------------------------------------------------------------------
GEMM_CFGS = [(256, 128, 0), (256, 128, 1), (256, 64, 0), (128, 32, 0), (128, 64, 0), (128, 128, 0)]
SENTINEL = -1234.0


def with_gemm_cfg(L, cfg, fn):
    tile_n, ec, pair = cfg
    L.set_tunable("gemm_tile_n", tile_n)
    L.set_tunable("gemm_epi_cols", ec)
    L.set_tunable("gemm_pair", pair)
    try:
        return fn()
    finally:
        L.set_tunable("gemm_tile_n", 256)
        L.set_tunable("gemm_epi_cols", 128)
        L.set_tunable("gemm_pair", -1)


def gemm_operands(m, n, k, seed):
    from fpqvar_b200 import lowbit
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((m, k)).astype(np.float16)
    w = (rng.standard_normal((n, k)) * 0.05).astype(np.float32)
    a = lowbit.pack_codes(torch.from_numpy(x).cuda(), "e2m1")
    ww = lowbit.pack_codes(torch.from_numpy(w).cuda(), "e2m1")
    return a, ww, LB.quantize_codes(x, "e2m1"), LB.quantize_codes(w, "e2m1"), rng.standard_normal(n).astype(np.float32)


@pytest.mark.parametrize("n", [136, 384])
def test_gemm_codes_strided_output(L, n):
    from fpqvar_b200 import lowbit
    m, k = 300, 256
    a, w, (qa, sa), (qw, sw), bias = gemm_operands(m, n, k, n)
    bias_d = torch.from_numpy(bias).cuda()
    for out in (F16, F32):
        for b in (None, bias_d):
            want = LB.gemm_codes(qa, sa, qw, sw, None if b is None else bias)
            want = torch.from_numpy(want.astype(np.float16) if out == F16 else want).cuda()
            for cfg in GEMM_CFGS:
                def run():
                    dense = lowbit.linear_codes(a, w, b, out)
                    buf = torch.full((m + 8, 3 * n), SENTINEL, dtype=out, device="cuda")
                    L.check(L.lib().fpq_gemm_codes(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), n, k,
                                                   128, None if b is None else b.data_ptr(), L.FPQ_F16 if out == F16 else L.FPQ_F32,
                                                   buf.data_ptr() + n * buf.element_size(), 3 * n, _stream()), "fpq_gemm_codes")
                    return dense, buf
                dense, buf = with_gemm_cfg(L, cfg, run)
                tag = f"gemm ldc=3n m={m} n={n} {out} bias={b is not None} cfg={cfg}"
                assert_same(dense, want, tag + " (dense)")
                assert_same(buf[:m, n:2 * n], want, tag)
                rest = buf.clone()
                rest[:m, n:2 * n] = SENTINEL
                assert bool((rest == SENTINEL).all()), f"{tag}: wrote outside the slice"


@pytest.mark.parametrize("n", [136, 384])
def test_gemm_codes_sse_strided_reference(L, n):
    from fpqvar_b200 import lowbit
    m, k = 300, 256
    a, w, _, _, bias = gemm_operands(m, n, k, 10 + n)
    g = torch.Generator(device="cuda").manual_seed(n)
    y = torch.randn(m, n, device="cuda", generator=g)
    rw = torch.rand(m, device="cuda", generator=g, dtype=torch.float64)
    bias_d = torch.from_numpy(bias).cuda()
    for rdt in (F16, F32):
        ref = y.to(rdt)
        wide = torch.full((m + 8, 3 * n), float("nan"), dtype=rdt, device="cuda")
        wide[:m, n:2 * n] = ref
        for weights in (None, rw):
            for cfg in [None] + GEMM_CFGS:
                def run():
                    dense = lowbit.linear_codes_sse(a, w, ref, bias_d, row_weight=weights)
                    sse = torch.zeros(1, dtype=torch.float64, device="cuda")
                    L.check(L.lib().fpq_gemm_codes_sse(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), n,
                                                       k, 128, bias_d.data_ptr(), L.FPQ_F16 if rdt == F16 else L.FPQ_F32,
                                                       wide.data_ptr() + n * wide.element_size(), 3 * n,
                                                       None if weights is None else weights.data_ptr(), sse.data_ptr(), _stream()),
                            "fpq_gemm_codes_sse")
                    return float(dense), float(sse)
                d, s = run() if cfg is None else with_gemm_cfg(L, cfg, run)
                assert np.isfinite(s) and np.isfinite(d) and abs(s - d) <= 1e-12 * d, (rdt, weights is not None, cfg, s, d)


def test_gemm_codes_stride_argument_checks(L):
    from fpqvar_b200 import lowbit
    m, n, k = 16, 64, 128
    a, w, *_ = gemm_operands(m, n, k, 3)
    c = torch.full((m, 2 * n + 16), SENTINEL, dtype=F32, device="cuda")
    lib = L.lib()
    before = lib.fpq_launch_count()
    for ldc, off in ((n - 8, 0), (n + 4, 0), (2 * n, 4), (2 * n, 8)):
        rc = lib.fpq_gemm_codes(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), n, k, 128, None,
                                L.FPQ_F32, c.data_ptr() + off, ldc, _stream())
        assert rc == L.FPQ_ERR_ARG, (ldc, off, rc)
        sse = torch.zeros(1, dtype=torch.float64, device="cuda")
        rc = lib.fpq_gemm_codes_sse(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), n, k, 128, None,
                                    L.FPQ_F32, c.data_ptr() + off, ldc, None, sse.data_ptr(), _stream())
        assert rc == L.FPQ_ERR_ARG, (ldc, off, rc)
    torch.cuda.synchronize()
    assert lib.fpq_launch_count() == before
    assert bool((c == SENTINEL).all())


# ------------------------------------------------------------------------------------------------------------------------
# fpq_sse_rows edges
# ------------------------------------------------------------------------------------------------------------------------
def _cls(v):
    return "nan" if np.isnan(v) else ("+inf" if v == np.inf else ("-inf" if v == -np.inf else "finite"))


@pytest.mark.parametrize("din", [F32, F16], ids=["f32", "f16"])
def test_sse_rows_nonfinite_and_empty(L, din):
    from fpqvar_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(4)
    a0 = torch.randn(16, 64, device="cuda", generator=g).to(din)
    b0 = (a0.float() + 0.01 * torch.randn(16, 64, device="cuda", generator=g)).to(din)
    w = torch.rand(16, device="cuda", generator=g, dtype=torch.float64)
    w[5] = 0.0
    for which in ("a", "b"):
        for val in (float("nan"), float("inf"), float("-inf")):
            for row in (3, 5):
                a, b = a0.clone(), b0.clone()
                (a if which == "a" else b)[row, 17] = val
                d2 = (a.double() - b.double()).square().sum(dim=1)
                for ww in (None, w):
                    want = float(d2.sum() if ww is None else (d2 * ww).sum())
                    got = float(ops.sse_rows(a, b, ww))
                    assert _cls(got) == _cls(want), (which, val, row, ww is not None, got, want)
                    if _cls(want) == "finite":
                        assert abs(got - want) <= BAR * want
    # a row weight of 0 does not hide a NaN in its row
    a = a0.clone()
    a[5, 0] = float("nan")
    assert np.isnan(float(ops.sse_rows(a, b0, w)))
    out = torch.full((1,), 7.0, dtype=torch.float64, device="cuda")
    L.check(L.lib().fpq_sse_rows(a0.data_ptr(), b0.data_ptr(), 0, 64, L.FPQ_F16 if din == F16 else L.FPQ_F32, None, out.data_ptr(), _stream()),
            "fpq_sse_rows")
    torch.cuda.synchronize()
    assert float(out) == 7.0
