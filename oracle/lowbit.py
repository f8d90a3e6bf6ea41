"""ORACLE (test infrastructure only; nothing under fpqvar_b200/ may import this).

CPU statement of the packed low-bit operand format and of the low-bit GEMM of include/fpq_b200.h (fpq_pack_codes,
fpq_unpack_codes, fpq_codes_to_nibbles, fpq_gemm_codes).  The reference has no such operator -- QuantizedLinear.forward
(models_fp_quant_transform_rotate/quant_utils.py:764-769) multiplies fp16 tensors whose values are scale * grid value -- so
the statement is anchored on the reference's quantizer: `quantize_codes` returns exactly the (grid value, scale) pair that
oracle.fake_quant (fp_quant_*_per_group_cuda, qu.py:265-378, 537-574) multiplies in its last step, and
`dequantize(quantize_codes(x)) == fake_quant(x)` bit for bit is the first test (tests/test_oracle_gemm_codes.py).
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

from . import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
GROUP = 128
TILE_ROWS = 128


def _lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "liboracle_gemm.so")
        if not os.path.exists(so):
            subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle_gemm.so"])
        lib = ctypes.CDLL(so)
        lib.gemm_codes_ref.restype = None
        lib.gemm_codes_ref.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_size_t, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]
        _LIB = lib
    return _LIB


def rows_padded(rows: int) -> int:
    return (rows + TILE_ROWS - 1) // TILE_ROWS * TILE_ROWS


def quantize_codes(x: np.ndarray, fmt: str, scale_group=GROUP):
    """(q, s): q fp32 [rows, k] grid values, s fp32 [rows, k/scale_group] scales, as fp_quant_*_per_group_cuda computes them
    (qu.py:320-326: scale = absmax / max|grid| in the input dtype, x / scale in the input dtype, quant_cuda.quant);
    scale_group=None: one scale per row, the per_token / per_channel functions (qu.py:503-534)."""
    x = np.asarray(x)
    assert x.ndim == 2 and x.shape[1] % GROUP == 0 and x.dtype in (np.float16, np.float32)
    dt = x.dtype
    grid = O.GRIDS[fmt]
    scale_group = x.shape[1] if scale_group is None else scale_group
    g = O._as_groups(x, scale_group)
    a = O._absmax_lastdim(g)
    s = O._div(a, np.full_like(a, O.grid_absmax(fmt), dtype=np.float32), dt)
    v = O._div(g, s, dt)
    q = O.scan_quant(v.astype(np.float32), grid).reshape(x.shape)
    return q.astype(np.float32), s.astype(np.float32).reshape(x.shape[0], x.shape[1] // scale_group)


def dequantize(q: np.ndarray, s: np.ndarray, dtype) -> np.ndarray:
    """qu.py:328-329: quantized * scale in fp32, cast to the output dtype."""
    with np.errstate(invalid="ignore", over="ignore", under="ignore"):
        out = q.reshape(q.shape[0], s.shape[1], -1) * s[:, :, None]
        return out.reshape(q.shape).astype(dtype)


def e4m3_encode(q: np.ndarray) -> np.ndarray:
    """e4m3 (bias 7, 3 mantissa bits, no infinities) byte of every value; asserts that the value is representable --
    true for every grid of the reference (qu.py:233-235, 458-486)."""
    q = np.asarray(q, dtype=np.float32)
    sign = (np.signbit(q)).astype(np.uint8) << 7
    a = np.abs(q).astype(np.float64)
    out = np.zeros(q.shape, dtype=np.uint8)
    nz = a > 0
    m, e = np.frexp(a[nz])                      # a = m * 2^e, m in [0.5, 1)
    e = e - 1                                   # a = (2m) * 2^e, 2m in [1, 2)
    normal = e >= -6
    mant = np.where(normal, (2 * m - 1) * 8, a[nz] * 512)        # subnormals: multiples of 2^-9
    assert np.all(mant == np.round(mant)) and np.all(e <= 8), "value is not an e4m3 number"
    byte = np.where(normal, ((e + 7).astype(np.int64) << 3) | mant.astype(np.int64), mant.astype(np.int64))
    out[nz] = byte.astype(np.uint8)
    return out | sign


def e4m3_decode(b: np.ndarray) -> np.ndarray:
    b = np.asarray(b, dtype=np.uint8)
    e = ((b >> 3) & 0xF).astype(np.int32)
    m = (b & 7).astype(np.float32)
    mag = np.where(e == 0, m * np.float32(2.0 ** -9), (1 + m / 8) * np.exp2((e - 7).astype(np.float32))).astype(np.float32)
    return np.where(b >> 7 == 1, -mag, mag).astype(np.float32)


def to_blocked(codes2d: np.ndarray) -> np.ndarray:
    """[rows, k] bytes -> the flat array of include/fpq_b200.h:
    [k/128 slabs][rows_pad/8][8 chunks of 16 K][8 rows][16 bytes], padding rows = 0."""
    rows, k = codes2d.shape
    rp = rows_padded(rows)
    full = np.zeros((rp, k), dtype=np.uint8)
    full[:rows] = codes2d
    t = full.reshape(rp // 8, 8, k // GROUP, 8, 16)            # [rb, r, slab, chunk, byte]
    return np.ascontiguousarray(t.transpose(2, 0, 3, 1, 4)).reshape(-1)


def from_blocked(flat: np.ndarray, rows: int, k: int) -> np.ndarray:
    rp = rows_padded(rows)
    t = np.asarray(flat, dtype=np.uint8).reshape(k // GROUP, rp // 8, 8, 8, 16)       # [slab, rb, chunk, r, byte]
    return np.ascontiguousarray(t.transpose(1, 3, 0, 2, 4)).reshape(rp, k)[:rows]


def scales_layout(s: np.ndarray) -> np.ndarray:
    """[rows, k/128] -> [k/128, rows_pad] with zeros for the padding rows."""
    rows, slabs = s.shape
    out = np.zeros((slabs, rows_padded(rows)), dtype=np.float32)
    out[:, :rows] = s.T
    return out


def pack_codes(x: np.ndarray, fmt: str, scale_group=GROUP):
    """What fpq_pack_codes writes: (flat code bytes, scales [k/scale_group, rows_pad])."""
    q, s = quantize_codes(x, fmt, scale_group)
    return to_blocked(e4m3_encode(q)), scales_layout(s)


_HALF = {"e2m1": [0, .5, 1, 1.5, 2, 3, 4, 6], "e1m2": [0, .25, .5, .75, 1, 1.25, 1.5, 1.75], "e3m0": [0, .25, .5, 1, 2, 4, 8, 16]}


def codes_to_nibbles(codes: np.ndarray, fmt: str) -> np.ndarray:
    """nibble = sign << 3 | index of |q| in the ascending half grid; byte i = codes 2i (low nibble), 2i+1."""
    v = e4m3_decode(codes)
    half = np.asarray(_HALF[fmt], dtype=np.float32)
    idx = np.searchsorted(half, np.abs(v))
    assert np.all(half[idx] == np.abs(v))
    nib = (idx | ((np.asarray(codes) >> 7).astype(np.int64) << 3)).astype(np.uint8)
    return (nib[0::2] | (nib[1::2] << 4)).astype(np.uint8)


def nibbles_to_codes(nib: np.ndarray, fmt: str) -> np.ndarray:
    half = np.asarray(_HALF[fmt], dtype=np.float32)
    n = np.empty(nib.size * 2, dtype=np.uint8)
    n[0::2] = nib & 0xF
    n[1::2] = nib >> 4
    v = half[n & 7] * np.where((n >> 3) == 1, np.float32(-1), np.float32(1))
    return e4m3_encode(np.where(v == 0, np.float32(0), v))


def gemm_codes(qa: np.ndarray, sa: np.ndarray, qw: np.ndarray, sw: np.ndarray, bias=None) -> np.ndarray:
    """fp32 [m, n] in the fixed operation order of oracle/gemm_codes.c.  qa [m, k], sa [m, groups], qw [n, k], sw [n, groups]."""
    m, k = qa.shape
    assert sa.shape[1] == sw.shape[1] and k % sa.shape[1] == 0
    n = qw.shape[0]
    qa = np.ascontiguousarray(qa, dtype=np.float32)
    qw = np.ascontiguousarray(qw, dtype=np.float32)
    sat = np.ascontiguousarray(sa.T, dtype=np.float32)          # [slabs, m]
    swt = np.ascontiguousarray(sw.T, dtype=np.float32)
    b = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32)
    c = np.empty((m, n), dtype=np.float32)
    _lib().gemm_codes_ref(qa.ctypes.data, sat.ctypes.data, m, qw.ctypes.data, swt.ctypes.data, n, k, k // sa.shape[1],
                          None if b is None else b.ctypes.data, c.ctypes.data)
    return c


def grid_unit(fmt: str) -> float:
    """The grid's resolution u: the largest power of two that divides every value of O.GRIDS[fmt]."""
    v = np.abs(O.GRIDS[fmt].astype(np.float64))
    v = v[v > 0]
    u = 2.0 ** 16
    while np.any(v / u != np.round(v / u)):
        u /= 2
    return u


def grid_min(fmt: str) -> float:
    """The smallest non-zero magnitude of the grid."""
    v = np.abs(O.GRIDS[fmt].astype(np.float64))
    return float(v[v > 0].min())


def accumulation_bits(fmt_a: str, fmt_w: str, k_acc: int) -> float:
    """log2 of the largest partial sum of k_acc products qa*qw, counted in units of u_a*u_w: the fp32 significand bits an
    accumulator needs to hold every partial sum of such a product exactly."""
    return float(np.log2(k_acc * (O.grid_absmax(fmt_a) / grid_unit(fmt_a)) * (O.grid_absmax(fmt_w) / grid_unit(fmt_w))))


def exact_accumulation(fmt_a: str, fmt_w: str, k_acc: int) -> bool:
    """True when every partial sum of k_acc products of grid values of fmt_a and fmt_w is an fp32 number, so that an fp32
    accumulator (IEEE addition, 24 significand bits) sums them exactly in any order:
        k_acc * max|q_a| * max|q_w| / (u_a * u_w) <= 2^24
    k_acc is 128 for one scale per 128-group and k for one scale per row.  Outside this envelope a partial sum P_t of the
    low-bit GEMM may differ from the exact one by (k_acc - 1) * 2^-24 * sum |qa * qw| (one rounding per addition)."""
    units = k_acc * (O.grid_absmax(fmt_a) / grid_unit(fmt_a)) * (O.grid_absmax(fmt_w) / grid_unit(fmt_w))
    return bool(units <= 2.0 ** 24)


def fma32(a, b, c) -> np.ndarray:
    """fmaf(a, b, c) element-wise for float32 arrays: a*b is exact in float64, the sum a*b + c is rounded once to float32
    (the float64 sum plus its TwoSum error decide the one case where rounding through float64 first would differ: a
    float64 sum that falls exactly half-way between two float32 numbers)."""
    a, b, c = (np.asarray(t, dtype=np.float32) for t in (a, b, c))
    with np.errstate(invalid="ignore", over="ignore"):
        p = a.astype(np.float64) * b.astype(np.float64)
        s = p + c.astype(np.float64)
        bb = s - p
        err = (p - (s - bb)) + (c.astype(np.float64) - bb)            # TwoSum: exact value = s + err
        r = s.astype(np.float32)
        up = np.nextafter(r, np.float32(np.inf))
        dn = np.nextafter(r, np.float32(-np.inf))
        mid_up = (r.astype(np.float64) + up.astype(np.float64)) / 2 == s
        mid_dn = (r.astype(np.float64) + dn.astype(np.float64)) / 2 == s
        fin = np.isfinite(s) & np.isfinite(err)
        r = np.where(fin & mid_up & (err > 0), up, r)
        r = np.where(fin & mid_dn & (err < 0), dn, r)
    return r.astype(np.float32)


def slab_sums_units(qa: np.ndarray, fmt_a: str, qw: np.ndarray, fmt_w: str, group: int) -> np.ndarray:
    """P[t, i, j] / (u_a * u_w): the exact sum over scale group t of qa[i, k] * qw[j, k] as an integer (held in float64, where
    every partial sum below 2^53 is exact, so the order of the matrix product does not matter)."""
    ua, uw = grid_unit(fmt_a), grid_unit(fmt_w)
    ia = np.asarray(qa, np.float64) / ua
    iw = np.asarray(qw, np.float64) / uw
    assert np.array_equal(ia, np.round(ia)) and np.array_equal(iw, np.round(iw)), "values are not on the grids"
    slabs = qa.shape[1] // group
    return np.stack([ia[:, t * group:(t + 1) * group] @ iw[:, t * group:(t + 1) * group].T for t in range(slabs)])


def scale_chain(p: np.ndarray, sa: np.ndarray, sw: np.ndarray, bias=None) -> np.ndarray:
    """The fp32 epilogue of oracle/gemm_codes.c on given slab sums p [slabs, m, n] (float64, rounded to fp32 first):
    acc = fmaf(fl32(P_t) * sa[:, t], sw[:, t], acc) for t ascending, then acc + bias."""
    acc = np.zeros(p.shape[1:], dtype=np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        for t in range(p.shape[0]):
            ps = p[t].astype(np.float32) * sa[:, t].astype(np.float32)[:, None]
            acc = fma32(ps, sw[:, t].astype(np.float32)[None, :], acc)
        return acc if bias is None else acc + np.asarray(bias, dtype=np.float32)[None, :]


def _signs(pattern: int, k: int, group: int) -> np.ndarray:
    """+-1 over k: 0 all +, 1 alternating 32-blocks (one MMA each), 2 first half of every accumulation span + and second half -,
    3 alternating 128-slabs."""
    i = np.arange(k)
    s = {0: np.zeros(k, bool), 1: (i // 32) % 2 == 1, 2: (i % group) >= group // 2, 3: (i // GROUP) % 2 == 1}[pattern]
    return np.where(s, -1.0, 1.0)


def probe_saturate(fmt: str, rows: int, k: int, group: int) -> np.ndarray:
    """F1: every value at +max|grid| except one at the smallest non-zero magnitude, at offset r % 128 of every 128-slab
    (group 128) or of the last slab (one scale per row, where the partial sums are largest there).  The rows sweep the 128
    offsets of a slab, i.e. every position inside each of its four 32-deep MMAs; A row r against W row r holds one product at
    u_a * u_w and all others at the pair's maximum.  Odd rows also hold a 0 at offset (r + 64) % 128, so that their sum is an
    odd number of units even where the maximal product is odd and k_acc - 1 of them make an even number (e1m2 x e1m2)."""
    q = np.full((rows, k), O.grid_absmax(fmt), dtype=np.float32)
    slabs = range(k // GROUP) if group == GROUP else [k // GROUP - 1]
    for r in range(rows):
        for t in slabs:
            q[r, t * GROUP + r % GROUP] = grid_min(fmt)
            if r % 2 == 1:
                q[r, t * GROUP + (r + 64) % GROUP] = 0
    return q


def probe_cancel(fmt: str, rows: int, k: int, group: int, side: str) -> np.ndarray:
    """F2: +-max|grid| plus, in row r, one element at the smallest magnitude at a position that sweeps the span with r.  A rows
    (side "a") are all +; W rows (side "w") carry sign pattern 1 + r % 3 of _signs, so that A row r against W row r cancels in
    32-blocks, in halves of the accumulation span (whole slabs with one scale per row) or slab by slab: the result is small
    while partial sums are large, and it holds one product of u_a * u_w that an accumulator dropping low bits of a large
    partial sum loses."""
    q = np.empty((rows, k), dtype=np.float32)
    for r in range(rows):
        q[r] = O.grid_absmax(fmt) * _signs(0 if side == "a" else 1 + r % 3, k, group)
        p = ((r * k) // rows + (5 * r) % 32) % k
        q[r, p] = np.sign(q[r, p]) * grid_min(fmt)
    return q


def probe_random(fmt: str, rows: int, k: int, rng) -> np.ndarray:
    """F3: seeded random signs on the two largest magnitudes of the grid, one element in 16 on one of the three smallest."""
    v = np.unique(np.abs(O.GRIDS[fmt]))
    v = v[v > 0]
    q = rng.choice(v[-2:], size=(rows, k)) * rng.choice([-1.0, 1.0], size=(rows, k))
    small = rng.random((rows, k)) < 1 / 16
    q[small] = rng.choice(v[:3], size=int(small.sum())) * rng.choice([-1.0, 1.0], size=int(small.sum()))
    return q.astype(np.float32)


ENVELOPE_ROWS = (128, 64, 101)          # A rows of F1, F2, F3: 293 = two 128-row tiles and a remainder
ENVELOPE_COLS = (128, 64, 72)           # W rows: 264, not a multiple of 256


def envelope_probe(fmt_a: str, fmt_w: str, k: int, group: int, seed: int = 0, rows=ENVELOPE_ROWS, cols=ENVELOPE_COLS):
    """(qa [m, k], sa [m, k/group], qw [n, k], sw [n, k/group]): F1, F2, F3 stacked along the rows of A and of W (the cross
    blocks, F1 x F3 and so on, are adversarial too), exact grid values and power-of-two scales, so that every output is the
    slab sums times exact scale factors and differs from the exact product only through the accumulation."""
    rng = np.random.default_rng(seed)
    qa = np.concatenate([probe_saturate(fmt_a, rows[0], k, group), probe_cancel(fmt_a, rows[1], k, group, "a"),
                         probe_random(fmt_a, rows[2], k, rng)])
    qw = np.concatenate([probe_saturate(fmt_w, cols[0], k, group), probe_cancel(fmt_w, cols[1], k, group, "w"),
                         probe_random(fmt_w, cols[2], k, rng)])
    slabs = k // group
    t = np.arange(slabs)
    sa = np.exp2((np.arange(qa.shape[0])[:, None] + 3 * t[None, :]) % 5 - 2.0).astype(np.float32)
    sw = np.exp2((2 * np.arange(qw.shape[0])[:, None] + t[None, :]) % 7 - 3.0).astype(np.float32)
    return qa, sa, qw, sw


def scale_chain_probe(fmt_a: str, fmt_w: str, m: int, n: int, k: int, group: int, seed: int = 0):
    """(qa, sa, qw, sw, bias) whose scales stress the fp32 epilogue: generic non-power-of-two scales (rounding at every step, so
    that another operation order gives other bits), scales near 2^+-60 (products that overflow or fall to subnormals), fp32
    subnormal scales, scale products that overflow to +-inf, zero scales with P != 0, NaN and inf scales with P = 0 and P != 0
    (some (row, group) blocks of A are all zero), and a bias of +-0 and +-inf in some columns."""
    rng = np.random.default_rng(seed)
    grid_a, grid_w = O.GRIDS[fmt_a], O.GRIDS[fmt_w]
    qa = rng.choice(grid_a, size=(m, k)).astype(np.float32)
    qw = rng.choice(grid_w, size=(n, k)).astype(np.float32)
    slabs = k // group
    for i in range(m):
        for t in range(slabs):
            if (i + t) % 7 == 3:
                qa[i, t * group:(t + 1) * group] = 0
    r = lambda *shape: np.exp(rng.uniform(-3, 3, size=shape))                     # noqa: E731
    kinds_a = [lambda s: r(*s), lambda s: np.exp2(60.0) * r(*s), lambda s: np.exp2(-60.0) * r(*s),
               lambda s: np.exp2(-140.0) * r(*s), lambda s: np.exp2(100.0) * r(*s), lambda s: np.zeros(s),
               lambda s: np.full(s, np.nan), lambda s: np.full(s, np.inf)]
    kinds_w = [lambda s: r(*s), lambda s: np.exp2(-60.0) * r(*s), lambda s: np.exp2(60.0) * r(*s),
               lambda s: np.exp2(40.0) * r(*s), lambda s: np.exp2(-135.0) * r(*s), lambda s: np.zeros(s),
               lambda s: np.full(s, np.inf), lambda s: np.full(s, np.nan)]
    sa = np.empty((m, slabs))
    sw = np.empty((n, slabs))
    for i in range(m):                       # even rows generic; an odd row has one special scale, in group (i // 2) % slabs
        for t in range(slabs):
            kind = (i // 2) % len(kinds_a) if i % 2 == 1 and t == (i // 2) % slabs else 0
            sa[i, t] = kinds_a[kind]((1,))[0]
    for j in range(n):
        for t in range(slabs):
            kind = (j // 2) % len(kinds_w) if j % 2 == 1 and t == (j // 2 + 1) % slabs else 0
            sw[j, t] = kinds_w[kind]((1,))[0]
    bias = rng.standard_normal(n).astype(np.float32)
    bias[1::16], bias[3::16], bias[5::16], bias[7::16] = 0.0, -0.0, np.inf, -np.inf
    return qa, sa.astype(np.float32), qw, sw.astype(np.float32), bias


def linear_f64(qa, sa, qw, sw, bias=None) -> np.ndarray:
    """The reference's expression F.linear(q_x * s_x, W_q * s_w, b) evaluated in float64 on the exact operand values."""
    a = qa.astype(np.float64).reshape(qa.shape[0], sa.shape[1], -1) * sa.astype(np.float64)[:, :, None]
    w = qw.astype(np.float64).reshape(qw.shape[0], sw.shape[1], -1) * sw.astype(np.float64)[:, :, None]
    c = a.reshape(qa.shape) @ w.reshape(qw.shape).T
    return c if bias is None else c + np.asarray(bias, dtype=np.float64)
