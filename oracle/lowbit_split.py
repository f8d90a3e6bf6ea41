"""ORACLE (test infrastructure only; nothing under fpqvar_b200/ may import this).

CPU statement of the sign-split codes operand of include/fpq_b200.h (fpq_pack_codes_signsplit, fpq_unpack_codes_signsplit,
fpq_gemm_codes_signsplit).  The reference's fc2 quantizer (fp_quant_e1m2_neg_e2m1_pos_per_group_cuda, qu.py:415-452) gives
every 128-group two scales and returns qn*sn + qp*sp, one of qn, qp being 0 in every element.  `quantize_codes_signsplit`
returns exactly those four arrays, stated line by line as oracle.fake_quant_signsplit (kernel tie rule), and the operand is the
symmetric operand of depth 2k whose slab 2t holds qn of group t (scale sn) and slab 2t+1 qp (scale sp).  With the weight's
128-slabs repeated twice, the split GEMM is oracle/gemm_codes.c on those two operands (`gemm_codes_signsplit`): no new C.
"""
from __future__ import annotations

import numpy as np

from . import lowbit as LB
from . import oracle as O

GROUP = LB.GROUP
FORMATS = ("e1m2_neg_e2m1_pos", "afpq_e2m1")        # the sign-split formats with a codes form


def quantize_codes_signsplit(x: np.ndarray, fmt: str, global_clip: bool = True):
    """(qn, qp, sn, sp): qn / qp fp32 [rows, k] grid values of the two halves, sn / sp fp32 [rows, k/128] scales, as
    oracle.fake_quant_signsplit computes them (qu.py:421-444) before its last line.  global_clip: the whole-tensor clip of
    qu.py:421-422; a tensor holding a NaN then becomes all NaN, both halves 0, every scale 0 and every grid value 0 -- the
    all-zero operand."""
    x = np.asarray(x)
    assert x.ndim == 2 and x.shape[1] % GROUP == 0 and x.dtype in (np.float16, np.float32)
    dt = x.dtype
    gneg, gpos = (O.GRIDS[n] for n in O.SPLIT[fmt])
    if global_clip:
        x = O._global_clip(x, 1.0)                                                  # :421-422
    g = O._as_groups(x, GROUP)
    zero = np.zeros_like(g)
    with np.errstate(invalid="ignore"):
        xn = np.where(g <= 0, g, zero)                                              # :428 (NaN -> 0)
        xp = np.where(g > 0, g, zero)                                               # :429
    sn = O._div(O._absmax_lastdim(xn), np.full((1, 1), np.max(np.abs(gneg)), np.float32), dt)     # :432
    sp = O._div(O._absmax_lastdim(xp), np.full((1, 1), np.max(np.abs(gpos)), np.float32), dt)     # :433
    vn = O._div(xn, sn, dt)                                                         # :436
    vp = O._div(xp, sp, dt)                                                         # :437
    qn = O.scan_quant(vn.astype(np.float32), gneg)                                  # :443
    qp = O.scan_quant(vp.astype(np.float32), gpos)                                  # :444
    rows, k = x.shape
    return (qn.reshape(rows, k), qp.reshape(rows, k), sn.astype(np.float32).reshape(rows, k // GROUP),
            sp.astype(np.float32).reshape(rows, k // GROUP))


def dequantize_signsplit(qn, qp, sn, sp, dtype) -> np.ndarray:
    """qu.py:450-451: qn*sn + qp*sp in fp32 (two products and one sum, each rounded), cast to the output dtype."""
    rows, k = qn.shape
    with np.errstate(invalid="ignore", over="ignore", under="ignore"):
        a = qn.reshape(rows, -1, GROUP) * sn[:, :, None]
        b = qp.reshape(rows, -1, GROUP) * sp[:, :, None]
        return (a + b).reshape(rows, k).astype(dtype)


def expand_signsplit(qn, qp, sn, sp):
    """(A' [rows, 2k], S' [rows, 2k/128]): slab 2t = qn of group t with scale sn, slab 2t+1 = qp of group t with scale sp."""
    rows, k = qn.shape
    a = np.stack([qn.reshape(rows, -1, GROUP), qp.reshape(rows, -1, GROUP)], axis=2).reshape(rows, 2 * k)
    s = np.stack([sn, sp], axis=2).reshape(rows, 2 * (k // GROUP))
    return a.astype(np.float32), s.astype(np.float32)


def split_halves(a2, s2):
    """Inverse of expand_signsplit."""
    rows, k2 = a2.shape
    t = a2.reshape(rows, -1, 2, GROUP)
    return (t[:, :, 0].reshape(rows, k2 // 2), t[:, :, 1].reshape(rows, k2 // 2), s2[:, 0::2], s2[:, 1::2])


def repeat_weight_slabs(qw, sw):
    """(W' [n, 2k], SW' [n, 2k/128]): every 128-slab of the weight and its scale, twice in a row."""
    n, k = qw.shape
    w = np.repeat(qw.reshape(n, -1, 1, GROUP), 2, axis=2).reshape(n, 2 * k)
    return w.astype(np.float32), np.repeat(sw, 2, axis=1).astype(np.float32)


def pack_codes_signsplit(x: np.ndarray, fmt: str, global_clip: bool = True):
    """What fpq_pack_codes_signsplit writes: (flat code bytes of the depth-2k operand, scales [2k/128, rows_pad])."""
    a, s = expand_signsplit(*quantize_codes_signsplit(x, fmt, global_clip))
    return LB.to_blocked(LB.e4m3_encode(a)), LB.scales_layout(s)


def gemm_codes_signsplit(qn, qp, sn, sp, qw, sw, bias=None) -> np.ndarray:
    """fpq_gemm_codes_signsplit: oracle/gemm_codes.c on A' and W' (fp32 [m, n])."""
    a, s = expand_signsplit(qn, qp, sn, sp)
    w, s_w = repeat_weight_slabs(qw, sw)
    return LB.gemm_codes(a, s, w, s_w, bias)


def e4m3_representable(values) -> np.ndarray:
    """True where the value is an e4m3 number (bias 7, 3 mantissa bits, finite)."""
    table = LB.e4m3_decode(np.arange(256, dtype=np.uint8))
    table = table[np.isfinite(table)]
    return np.isin(np.asarray(values, dtype=np.float32), table)
