"""GPU: the persistent activation kernels against the oracle once every CTA loops over many rows.

The launchers cap their grids at a few CTAs per SM and every CTA strides over rows or groups, carrying state from one trip
to the next (the prefetched next row of the row-in-registers kernels, shared row scalars, the whole-tensor clip flag).  Each
case here sizes its tensor past three times an upper bound of its launcher's grid, so every CTA makes at least three trips
and the last trip's prefetch runs past the end, and puts irregular rows (zero, NaN, +-inf, one-sided, fp16-subnormal
scales, GELU skew, fp16 overflow) among regular ones, the last row included.  References: the multi-threaded C port of
the oracle (oracle/port.py, pinned to oracle/oracle.py by test_oracle_port.py) on whole tensors, oracle/lowbit.py on a row
sample (per-row and per-group quantization is row-local), float64 sums for the scorers."""
import numpy as np
import pytest
import torch

from conftest import mismatch_report
from oracle import lowbit as LB, oracle as O, port as P

pytestmark = pytest.mark.gpu
NP = {torch.float32: np.float32, torch.float16: np.float16}
F16, F32 = torch.float16, torch.float32
SYM_FMTS = ["e2m3", "e2m1", "e3m2", "e1m2", "e3m0"]
SPLIT_FMTS = ["int_neg_e2m3_pos", "e1m2_neg_e2m1_pos", "afpq_e2m1"]
SENTINEL = -1234.0                      # what an output element holds until a kernel writes it (exact in fp16 and fp32)


@pytest.fixture(scope="module")
def L():
    from fpqvar_b200 import _lib
    _lib.lib()
    return _lib


# ------------------------------------------------------------------------------------------------------------------------
# sizing
# ------------------------------------------------------------------------------------------------------------------------
def grid_caps():
    """Upper bounds of each launcher's grid, in the launcher's work items, from the device's SM count."""
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count

    def row_reg(row_len, elem_size):
        # rows: resident_row_grid (csrc/fpq_common.cuh:113-121) launches at most the resident CTAs per SM; bound them by the
        # hardware (32 CTAs and 2048 threads per SM) at the smallest CTA any values-per-thread choice gives (fpq_common.cuh:93-111)
        row_vecs = row_len * elem_size // 16
        best = 0
        for v in (1, 2, 4):
            while -(-row_vecs // v) > 1024:
                v *= 2
            threads = (-(-row_vecs // v) + 31) // 32 * 32
            best = max(best, sms * min(32, 2048 // threads))
        return best

    return {
        "row_reg": row_reg,
        "row_two_pass": 16 * sms,                       # rows: grid_for(n_rows, 1, 16), fpq_sym.inc.cuh:248, fpq_split.inc.cuh:343
        "group": lambda gs: 64 * sms * 8 * (32 // (gs // 16)),   # groups: grid_for(n, 8 * 32/LPG, 64), fpq_sym.inc.cuh:242, fpq_split.inc.cuh:337
        "score": 256 * sms,                             # groups of 128: grid_for(n, 32, 8) / grid_for(n, 64, 4), fpq_score.cu:423-428
        "sse_rows": 64 * sms,                           # rows: grid_for(n_rows, 8, 8), one row per warp, fpq_score.cu:401
        "quant_grid": 64 * sms * 256 * 4,               # elements: grid_for(n, 1024, 64), 4 per thread and trip, fpq_grid.cu:186
        "pack_tasks": 64 * sms,                         # (128-slab, 8-row block) tasks: grid_for(tasks, 8, 8), fpq_gemm.cu:678
        "pack_row_blocks": 64 * sms,                    # 8-row blocks: grid_for(rows_pad / 8, 8, 8), fpq_gemm.cu:669
        "unpack_chunks": 8 * sms * 256,                 # 16-code chunks: grid_for(chunks, 256, 8), fpq_gemm.cu:720
        "segment_groups": lambda n_seg: 64 * (-(-8 * sms // n_seg)),   # groups per segment and trip: per_seg CTAs of 64, fpq_h16.cu:472
    }


def past_three_caps(cap, which):
    """n = 3 cap + r, r in {1, cap - 1, a prime}: every CTA makes at least three trips."""
    n = 3 * cap + (1, cap - 1, 97)[which % 3]
    assert n > 2 * cap
    return n


def sample_rows(n, cap, irregular):
    """Rows [0, 64), +-32 around cap and 2 cap, the last 64 rows and every irregular row."""
    parts = [np.arange(64), np.arange(cap - 32, cap + 32), np.arange(2 * cap - 32, 2 * cap + 32), np.arange(n - 64, n), irregular]
    idx = np.unique(np.concatenate(parts))
    return idx[(idx >= 0) & (idx < n)]


# ------------------------------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------------------------------
IRREGULAR = ["zero", "nan", "+inf", "-inf", "no_neg", "no_pos", "tiny", "gelu", "big"]


def make_rows(n_rows, row_len, dtype, seed, nonfinite=True):
    """[n_rows, row_len] on the GPU with per-row magnitudes spread over e^+-6; about 15 % of the rows (seeded, scattered),
    one contiguous block of 24 and the last row are irregular, their kinds cycling so that regular and irregular rows
    alternate inside any CTA's sequence of rows.  nonfinite=False leaves out NaN and +-inf.  Returns (x, irregular rows)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(n_rows, row_len, device="cuda", generator=g)
    x *= torch.exp(torch.rand(n_rows, 1, device="cuda", generator=g) * 12 - 6)
    rng = np.random.default_rng(seed)
    start = int(rng.integers(0, max(1, n_rows - 24)))
    irr = np.unique(np.concatenate([rng.choice(n_rows, size=max(1, int(0.15 * n_rows)), replace=False),
                                    np.arange(start, min(n_rows, start + 24)), [n_rows - 1]]))
    kinds = [k for k in IRREGULAR if nonfinite or k not in ("nan", "+inf", "-inf")]
    col = torch.from_numpy((irr * 7919) % row_len).cuda()
    for i, kind in enumerate(kinds):
        sel = torch.from_numpy(irr[i::len(kinds)]).cuda()
        if sel.numel() == 0:
            continue
        if kind == "zero":
            x[sel] = 0.0
        elif kind in ("nan", "+inf", "-inf"):
            x[sel, col[i::len(kinds)]] = {"nan": float("nan"), "+inf": float("inf"), "-inf": float("-inf")}[kind]
        elif kind == "no_neg":                           # sign-split: zero negative scale
            x[sel] = x[sel].abs()
        elif kind == "no_pos":                           # sign-split: zero positive scale
            x[sel] = -x[sel].abs()
        elif kind == "tiny":                             # scales in the fp16-subnormal range
            x[sel] = torch.randn(sel.numel(), row_len, device="cuda", generator=g) * 1e-6
        elif kind == "gelu":
            x[sel] = torch.where(x[sel] > 0, x[sel], x[sel] * 0.02)
        else:                                            # fp32 values whose quantized outputs overflow fp16 (finite in fp16 input)
            big = torch.randn(sel.numel(), row_len, device="cuda", generator=g)
            x[sel] = (big * 4e4) if dtype == F32 else (big * 1e4).clamp(-6e4, 6e4)
    return x.to(dtype), irr


# ------------------------------------------------------------------------------------------------------------------------
# launches (the C ABI, into outputs pre-filled with SENTINEL so that a row no CTA reaches cannot pass)
# ------------------------------------------------------------------------------------------------------------------------
def _dt(L, t):
    return {F32: L.FPQ_F32, F16: L.FPQ_F16}[t]


def _stream():
    return torch.cuda.current_stream().cuda_stream


def sym(L, x, fmt, tie, clamp3, dout, row_len=None, n_rows=None, ptr=None, din=None):
    row_len = row_len or x.shape[-1]
    n_rows = n_rows or x.numel() // row_len
    out = torch.full((n_rows, row_len), SENTINEL, dtype=dout, device="cuda")
    L.check(L.lib().fpq_fake_quant(ptr or x.data_ptr(), out.data_ptr(), n_rows, row_len, _dt(L, din or x.dtype), _dt(L, dout), L.FMT[fmt],
                                   L.TIE[tie], L.FLAG_CLAMP3 if clamp3 else 0, _stream()), "fpq_fake_quant")
    return out


def split(L, x, fmt, tie, dout, row_len=None, n_rows=None, ptr=None, din=None, ws=None):
    row_len = row_len or x.shape[-1]
    n_rows = n_rows or x.numel() // row_len
    out = torch.full((n_rows, row_len), SENTINEL, dtype=dout, device="cuda")
    L.check(L.lib().fpq_fake_quant_signsplit(ptr or x.data_ptr(), out.data_ptr(), n_rows, row_len, _dt(L, din or x.dtype), _dt(L, dout),
                                             L.SPLIT[fmt], L.TIE[tie], L.FLAG_GLOBAL_CLIP if ws is not None else 0,
                                             ws.data_ptr() if ws is not None else None, _stream()), "fpq_fake_quant_signsplit")
    return out


def ref_sym(xh, fmt, tie, clamp3, dout, row_len=None):
    return P.fake_quant(xh.reshape(-1, row_len or xh.shape[-1]), fmt, None, tie, clamp3=clamp3, out_dtype=dout)


def ref_split(xh, fmt, tie, dout, row_len=None):
    """The port's sign-split for any (in, out) pair: its C entry points take (f32, f32), (f16, f16) and (f16, f32); an fp32
    tensor with an fp16 output is the fp32 result rounded once, as the kernels store it."""
    xh = np.ascontiguousarray(xh.reshape(-1, row_len or xh.shape[-1]))
    if xh.dtype == np.float32 and dout == np.float16:
        with np.errstate(over="ignore"):
            return ref_split(xh, fmt, tie, np.float32).astype(np.float16)
    out = np.empty(xh.shape, dtype=dout)
    gneg, gpos = (O.GRIDS[n] for n in O.SPLIT[fmt])
    fn = getattr(P._lib(), f"port_signsplit_{P._TAG[xh.dtype]}_{P._TAG[np.dtype(dout)]}")
    fn(xh.ctypes.data, out.ctypes.data, xh.shape[0], xh.shape[1], gneg.ctypes.data, gneg.size, float(np.max(np.abs(gneg))),
       gpos.ctypes.data, gpos.size, float(np.max(np.abs(gpos))), P._TIE[tie])
    return out


def assert_same(got, want, tag):
    """Bit-identical on the device (every NaN equals every NaN; signed zeros differ); a host report of the first mismatches
    and the rows they are in otherwise."""
    w = want if isinstance(want, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(want)).to(got.device)
    assert got.dtype == w.dtype and got.shape == w.shape, (tag, got.dtype, w.dtype, tuple(got.shape), w.shape)
    it = {2: torch.int16, 4: torch.int32}[got.element_size()]
    gn, wn = torch.isnan(got), torch.isnan(w)
    bad = (gn != wn) | (~gn & (got.view(it) != w.view(it)))
    if bool(bad.any()):
        rows = torch.nonzero(bad.reshape(got.shape[0], -1).any(dim=1)).flatten()
        raise AssertionError(f"{tag}: {rows.numel()} rows differ, first {rows[:8].tolist()}\n"
                             + mismatch_report(got.cpu().numpy(), w.cpu().numpy()))


def with_row_v(L, v, fn):
    L.set_tunable("row_v", v)
    try:
        return fn()
    finally:
        L.set_tunable("row_v", 0)


# ------------------------------------------------------------------------------------------------------------------------
# 1, 2: per-row symmetric and sign-split through the row-in-registers kernels
# ------------------------------------------------------------------------------------------------------------------------
ROW_REG = [(256, F16), (1920, F16), (7680, F16), (9216, F16), (16384, F16), (1920, F32), (4096, F32)]


@pytest.mark.parametrize("case", range(len(ROW_REG)), ids=[f"{r}-{str(d)[6:]}" for r, d in ROW_REG])
def test_sym_row_reg_kernel_many_rows_per_cta(L, case):
    row_len, din = ROW_REG[case]
    cap = grid_caps()["row_reg"](row_len, din.itemsize)
    n = past_three_caps(cap, case)
    fmt = SYM_FMTS[case % len(SYM_FMTS)]
    x, _ = make_rows(n, row_len, din, seed=100 + case)
    xh = x.cpu().numpy()
    for dout in (F16, F32):
        for tie, clamp3 in (("kernel", False), ("argmin", True)):
            want = torch.from_numpy(ref_sym(xh, fmt, tie, clamp3, NP[dout])).cuda()
            for v in (1, 2, 4, 0):
                got = with_row_v(L, v, lambda: sym(L, x, fmt, tie, clamp3, dout))
                assert_same(got, want, f"sym rows {n}x{row_len} {din}->{dout} {fmt} {tie} clamp3={clamp3} V={v or 'default'} cap={cap}")


@pytest.mark.parametrize("case", range(len(ROW_REG)), ids=[f"{r}-{str(d)[6:]}" for r, d in ROW_REG])
def test_signsplit_row_reg_kernel_many_rows_per_cta(L, case):
    row_len, din = ROW_REG[case]
    cap = grid_caps()["row_reg"](row_len, din.itemsize)
    n = past_three_caps(cap, case + 1)
    fmt = SPLIT_FMTS[case % len(SPLIT_FMTS)]
    x, _ = make_rows(n, row_len, din, seed=200 + case)
    xh = x.cpu().numpy()
    for dout in (F16, F32):
        for tie in ("kernel", "argmin"):
            want = torch.from_numpy(ref_split(xh, fmt, tie, NP[dout])).cuda()
            for v in (1, 2, 4, 0):
                got = with_row_v(L, v, lambda: split(L, x, fmt, tie, dout))
                assert_same(got, want, f"split rows {n}x{row_len} {din}->{dout} {fmt} {tie} V={v or 'default'} cap={cap}")


# ------------------------------------------------------------------------------------------------------------------------
# 3: the two-pass row kernels (rows shorter than 256, rows not 16-byte aligned, fp16 rows over 4096 vectors)
# ------------------------------------------------------------------------------------------------------------------------
TWO_PASS = [("short", 200, F16), ("short", 200, F32), ("odd_offset", 1000, F16), ("odd_offset", 1000, F32), ("long", 40000, F16)]


@pytest.mark.parametrize("case", range(len(TWO_PASS)), ids=[f"{k}-{r}-{str(d)[6:]}" for k, r, d in TWO_PASS])
def test_two_pass_row_kernels_many_rows_per_cta(L, case):
    kind, row_len, din = TWO_PASS[case]
    cap = grid_caps()["row_two_pass"]
    n = past_three_caps(cap, case if kind != "long" else 0)
    x, _ = make_rows(n, row_len, din, seed=300 + case)
    xh = x.cpu().numpy()
    ptr = None
    if kind == "odd_offset":                 # the same rows one element into a buffer: no 16-byte vector path
        buf = torch.empty(n * row_len + 1, dtype=din, device="cuda")
        buf[1:] = x.reshape(-1)
        ptr = buf.data_ptr() + din.itemsize
    for tie, clamp3 in (("kernel", False), ("argmin", True)):
        dout = din if tie == "kernel" else F32
        fmt = SYM_FMTS[case % len(SYM_FMTS)]
        got = sym(L, x, fmt, tie, clamp3, dout, n_rows=n, row_len=row_len, ptr=ptr)
        assert_same(got, ref_sym(xh, fmt, tie, clamp3, NP[dout]), f"sym two-pass {kind} {n}x{row_len} {din} {fmt} {tie} cap={cap}")
        sfmt = SPLIT_FMTS[case % len(SPLIT_FMTS)]
        got = split(L, x, sfmt, tie, dout, n_rows=n, row_len=row_len, ptr=ptr)
        assert_same(got, ref_split(xh, sfmt, tie, NP[dout]), f"split two-pass {kind} {n}x{row_len} {din} {sfmt} {tie} cap={cap}")


# ------------------------------------------------------------------------------------------------------------------------
# 4: the whole-tensor clip on the paths that finish with poison_fill_kernel
# ------------------------------------------------------------------------------------------------------------------------
CLIP = [(1920, F16, "kernel", "row_reg"), (1920, F32, "argmin", "row_reg"), (200, F16, "argmin", "row_two_pass"),
        (64, F32, "kernel", "group"), (64, F16, "argmin", "group"), (128, F32, "argmin", "group")]


@pytest.mark.parametrize("case", range(len(CLIP)), ids=[f"{r}-{str(d)[6:]}-{t}-{f}" for r, d, t, f in CLIP])
def test_whole_tensor_clip_found_on_a_later_trip(L, case):
    """A NaN in a row past the grid (found on a later trip) or in the last row only zeroes the whole output: +0 under the
    kernel rule, -0 under the argmin rule (fpq_split.inc.cuh:349-351).  The workspace is zero afterwards and a clean call
    right behind on the same stream matches the oracle."""
    from fpqvar_b200 import ops
    row_len, din, tie, fam = CLIP[case]
    caps = grid_caps()
    cap = caps["row_reg"](row_len, din.itemsize) if fam == "row_reg" else caps["group"](row_len) if fam == "group" else caps[fam]
    n = past_three_caps(cap, case)
    fmt = SPLIT_FMTS[case % len(SPLIT_FMTS)]
    dout = din if tie == "kernel" else F32
    clean, _ = make_rows(n, row_len, din, seed=400 + case, nonfinite=False)
    late, last = clean.clone(), clean.clone()
    late[2 * cap + 5, 3] = float("nan")
    last[n - 1, row_len - 1] = float("nan")
    ws = ops._clip_workspace(clean.device)
    outs = [split(L, t, fmt, tie, dout, ws=ws) for t in (clean, late, clean, last, clean)]
    torch.cuda.synchronize()
    assert ws.tolist() == [0, 0], "workspace not left zeroed"
    want = ref_split(clean.cpu().numpy(), fmt, tie, NP[dout])
    fill = torch.zeros((), dtype=dout) if tie == "kernel" else -torch.zeros((), dtype=dout)
    it = {2: torch.int16, 4: torch.int32}[dout.itemsize]
    fill_bits = int(fill.view(it))
    for i, o in enumerate(outs):
        if i in (1, 3):
            assert bool((o.view(it) == fill_bits).all()), f"poisoned call {i}: output is not all {float(fill)!r} ({fam} {n}x{row_len})"
        else:
            assert_same(o, want, f"clean call {i} ({fam} {n}x{row_len} {din} {fmt} {tie} cap={cap})")


# ------------------------------------------------------------------------------------------------------------------------
# 5: the generic group kernels (fp32 in, argmin, clamp3, fp16 -> fp32)
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gs", [64, 128])
@pytest.mark.parametrize("din", [F32, F16], ids=["f32", "f16"])
def test_generic_group_kernels_many_groups_per_warp(L, gs, din):
    cap = grid_caps()["group"](gs)
    n = past_three_caps(cap, gs // 64 + (din == F16))
    x, _ = make_rows(n, gs, din, seed=500 + gs + (din == F16))
    xh = x.cpu().numpy()
    if din == F32:
        sym_cases = [("e2m1", "kernel", False, F32), ("e3m2", "argmin", True, F32), ("e1m2", "argmin", False, F32)]
        split_cases = [("e1m2_neg_e2m1_pos", "kernel", F32), ("int_neg_e2m3_pos", "argmin", F32)]
    else:                                    # the fp16 -> fp16 kernel-rule calls without clamp3 take the packed kernels instead
        sym_cases = [("e2m3", "argmin", True, F32), ("e3m0", "kernel", False, F32), ("e2m1", "kernel", True, F16)]
        split_cases = [("afpq_e2m1", "argmin", F32)] + ([("e1m2_neg_e2m1_pos", "kernel", F16)] if gs == 64 else [])
    for fmt, tie, clamp3, dout in sym_cases:
        assert_same(sym(L, x, fmt, tie, clamp3, dout), ref_sym(xh, fmt, tie, clamp3, NP[dout]),
                    f"sym groups {n}x{gs} {din}->{dout} {fmt} {tie} clamp3={clamp3} cap={cap}")
    for fmt, tie, dout in split_cases:
        assert_same(split(L, x, fmt, tie, dout), ref_split(xh, fmt, tie, NP[dout]), f"split groups {n}x{gs} {din}->{dout} {fmt} {tie} cap={cap}")


# ------------------------------------------------------------------------------------------------------------------------
# 6: format scoring, the row-weighted SSE and the grid rounding
# ------------------------------------------------------------------------------------------------------------------------
ALL_FORMATS = SYM_FMTS + SPLIT_FMTS


@pytest.mark.parametrize("tie", ["kernel", "argmin"])
@pytest.mark.parametrize("din", [F32, F16], ids=["f32", "f16"])
def test_score_formats_many_groups_per_warp(tie, din):
    from fpqvar_b200 import ops
    cap = grid_caps()["score"]
    n = past_three_caps(cap, (tie == "argmin") + 2 * (din == F16))
    x, _ = make_rows(n, 128, din, seed=600 + (tie == "argmin") + 2 * (din == F16), nonfinite=False)
    xh = x.cpu().numpy()
    sse = ops.score_formats(x, ALL_FORMATS, tie).cpu().numpy()
    for got, fmt in zip(sse, ALL_FORMATS):
        xq = ref_split(xh, fmt, tie, np.float32 if tie == "argmin" else xh.dtype) if fmt in O.SPLIT else ref_sym(xh, fmt, tie, False, None)
        d = xh.astype(np.float64) - xq.astype(np.float64)
        want = float((d * d).sum())
        # per-element errors are exact; only the summation order differs (fp32 partial sums of 16, then fp64)
        assert abs(got - want) <= 2e-6 * want, (fmt, n, cap, got, want)


@pytest.mark.parametrize("din", [F32, F16], ids=["f32", "f16"])
def test_sse_rows_many_rows_per_warp(din):
    from fpqvar_b200 import ops
    cap = grid_caps()["sse_rows"]
    n = past_three_caps(cap, 1 + (din == F16))
    a, _ = make_rows(n, 1024, din, seed=700 + (din == F16), nonfinite=False)
    g = torch.Generator(device="cuda").manual_seed(7)
    b = (a.float() * (1 + 0.01 * torch.randn(a.shape, device="cuda", generator=g))).to(din)
    w = torch.rand(n, device="cuda", generator=g, dtype=torch.float64)
    d2 = (a.double() - b.double()).square().sum(dim=1)
    got, want = float(ops.sse_rows(a, b)), float(d2.sum())
    assert abs(got - want) <= 2e-6 * want, (n, cap, got, want)
    got, want = float(ops.sse_rows(a, b, w)), float((d2 * w).sum())
    assert abs(got - want) <= 2e-6 * want, (n, cap, got, want)


@pytest.mark.parametrize("tie", ["kernel", "argmin"])
def test_quant_grid_many_elements_per_thread(tie):
    """An unsorted grid with duplicates (the scan path) and a grid the library knows (the closed-form path)."""
    from fpqvar_b200 import ops
    cap = grid_caps()["quant_grid"]
    n = past_three_caps(cap, tie == "argmin")
    g = torch.Generator(device="cuda").manual_seed(8)
    x = torch.randn(n, device="cuda", generator=g) * torch.exp(torch.rand(n, device="cuda", generator=g) * 6 - 3)
    specials = torch.tensor([float("nan"), float("inf"), float("-inf"), 0.0, -0.0, 0.25, -1.5, 2.375, 6.0, -7.0], device="cuda")
    pos = torch.randint(0, n, (4096,), device="cuda", generator=g)
    x[pos] = specials[torch.arange(4096, device="cuda") % specials.numel()]
    x[-1] = float("nan")
    xh = x.cpu().numpy()
    for grid in (np.array([0.5, -1.0, 3.0, 0.5, -2.5, 0.0, 1.75, -1.0, 6.0, 0.0, -6.0], dtype=np.float32), O.GRIDS["e3m2"]):
        got = ops.quant_grid(x, torch.from_numpy(grid).cuda(), tie)
        want = (O.scan_quant if tie == "kernel" else O.argmin_quant)(xh, grid)
        assert_same(got.view(-1, 1), want.reshape(-1, 1), f"quant_grid {n} elements {tie} grid of {grid.size} cap={cap}")


# ------------------------------------------------------------------------------------------------------------------------
# 7: packed low-bit codes and their dequantization
# ------------------------------------------------------------------------------------------------------------------------
PACK = [("group", F16, "e2m1", 384), ("group", F32, "e3m2", 384), ("per_row", F16, "e2m3", 256), ("per_row", F32, "e1m2", 256)]


@pytest.mark.parametrize("case", range(len(PACK)), ids=[f"{m}-{str(d)[6:]}-{f}" for m, d, f, _ in PACK])
def test_pack_and_unpack_codes_many_tasks_per_warp(case):
    from fpqvar_b200 import lowbit
    mode, din, fmt, k = PACK[case]
    caps = grid_caps()
    per_row = mode == "per_row"
    slabs = k // 128
    cap = caps["pack_row_blocks"] * 8 if per_row else caps["pack_tasks"] * 8 // slabs        # in rows
    rows = past_three_caps(cap, case)
    assert LB.rows_padded(rows) * k // 16 > 3 * caps["unpack_chunks"]
    x, irr = make_rows(rows, k, din, seed=800 + case)
    p = lowbit.pack_codes(x, fmt, per_row=per_row)
    idx = sample_rows(rows, cap, irr)
    xs = x[torch.from_numpy(idx).cuda()].cpu().numpy()
    q, s = LB.quantize_codes(xs, fmt, None if per_row else 128)
    rp = LB.rows_padded(rows)
    codes = p.codes.cpu().numpy().reshape(slabs, rp // 8, 8, 8, 16).transpose(1, 3, 0, 2, 4).reshape(rp, k)
    tag = f"pack {mode} {rows}x{k} {din} {fmt} cap={cap}"
    got_codes = codes[idx]
    want_codes = LB.e4m3_encode(q)
    bad = np.nonzero((got_codes != want_codes).any(axis=1))[0]
    assert bad.size == 0, f"{tag}: codes of rows {idx[bad[:8]].tolist()} differ"
    assert not codes[rows:].any(), f"{tag}: padding rows hold codes"
    scales = p.scales.cpu().numpy()
    assert not scales[:, rows:].any(), f"{tag}: padding rows hold scales"
    assert_same(torch.from_numpy(np.ascontiguousarray(scales[:, idx].T)), s, f"{tag}: scales")
    for dout in (F16, F32):
        got = p.dequantize(dout)[torch.from_numpy(idx).cuda()]
        assert_same(got, LB.dequantize(q, s, NP[dout]), f"unpack {tag} -> {dout}")


# ------------------------------------------------------------------------------------------------------------------------
# 8: segmented fp16 fake quant (KV cache) with per_seg capped
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("smem_kb", [0, 100])
@pytest.mark.parametrize("pitched", [False, True], ids=["in_place", "pitched"])
@pytest.mark.parametrize("gs", [64, 128])
def test_fake_quant_segments_many_groups_per_cta(L, gs, pitched, smem_kb):
    n_seg = 37
    cap = grid_caps()["segment_groups"](n_seg)
    groups = past_three_caps(cap, gs // 64 + pitched)
    lo, pad = 4, 9                                       # one group per token: segments of tokens [lo, lo + groups) of [B, Lmax, gs]
    lmax = lo + groups + pad
    fmt = SYM_FMTS[(gs // 64 + 2 * pitched + smem_kb) % len(SYM_FMTS)]
    x, _ = make_rows(n_seg * lmax, gs, F16, seed=900 + gs + pitched)
    buf = x.view(n_seg, lmax, gs)
    orig = buf.clone()
    want = ref_sym(orig[:, lo:lo + groups].cpu().numpy(), fmt, "kernel", False, np.float16, row_len=gs)
    seg = groups * gs
    pitch_out = seg + 64 if pitched else lmax * gs
    out = torch.full((n_seg, pitch_out), SENTINEL, dtype=F16, device="cuda") if pitched else buf
    L.set_tunable("smem_kb", smem_kb)
    try:
        L.check(L.lib().fpq_fake_quant_segments(buf.data_ptr() + lo * gs * 2, out.data_ptr() + (0 if pitched else lo * gs * 2), n_seg, groups,
                                                gs, lmax * gs, pitch_out, L.FMT[fmt], _stream()), "fpq_fake_quant_segments")
        torch.cuda.synchronize()
    finally:
        L.set_tunable("smem_kb", 0)
    tag = f"segments {n_seg} x {groups} groups of {gs} {'pitched' if pitched else 'in place'} smem_kb={smem_kb} {fmt} cap={cap}"
    if pitched:
        assert_same(out[:, :seg].reshape(-1, gs), want, tag)
        assert bool((out[:, seg:] == SENTINEL).all()), f"{tag}: wrote past the segment"
        assert torch.equal(buf.view(torch.int16), orig.view(torch.int16)), f"{tag}: input changed"
    else:
        assert_same(buf[:, lo:lo + groups].reshape(-1, gs), want, tag)
        assert torch.equal(buf[:, :lo].view(torch.int16), orig[:, :lo].view(torch.int16)), f"{tag}: tokens before the range changed"
        assert torch.equal(buf[:, lo + groups:].view(torch.int16), orig[:, lo + groups:].view(torch.int16)), f"{tag}: tokens after the range changed"
