"""Host-only cases for the format scorers' range tests (tests/test_gpu_score_range.py): calls of 128-element groups that
all share one class, so that every group's squared error is of the same order and a relative bar on a call's total is a bar
on every group.

A class is either one binade of the group absmax (fp16: 2^-24 .. 2^15, fp32: 2^-149 .. 2^127) filled with one content
kind, or one boundary case: groups whose rounded scale fl(a / VMAX) sits on a chosen side of a switch of the scorers -- the
fp16 normal range (scale bits 0x03FE / 0x03FF / 0x0400 / 0x0401), the e1m2 conversion-hardware limit (0x77FE .. 0x7801) and
the fp32 2^+-100 range of `scale_regular<float>`.  A sign-split boundary case puts one side on the boundary and the other
side exactly on a power-of-two scale times its half grid, so that the other side's error is exactly 0 and the call's total
is the boundary side's error alone.  `self_check` (run by tests/test_score_range_cases.py without a GPU) recomputes every
claim on the host; without it the GPU tests could pass vacuously.

Nothing here touches a GPU; references are the multi-threaded C port of the oracle (oracle/port.py) with float64 sums."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from oracle import oracle as O, port as P

GS = 128
SYM = ["e2m1", "e1m2", "e3m0", "e2m3", "e3m2"]
SPLIT = ["e1m2_neg_e2m1_pos", "int_neg_e2m3_pos", "afpq_e2m1"]
FORMATS = SYM + SPLIT
KINDS = ["normal", "gelu", "pos", "pos0", "neg", "neg0", "ties", "far"]
BINADES = {np.float16: range(-24, 16), np.float32: range(-149, 128)}
F16_BOUNDARY = [0x03FE, 0x03FF, 0x0400, 0x0401]
E1M2_HW_BOUNDARY = [0x77FE, 0x77FF, 0x7800, 0x7801]
TIES_FROM = {np.float16: -6, np.float32: -118}    # every midpoint times the scale is a normal number from here on
FLT_MAX = float(np.finfo(np.float32).max)


def vmax(fmt, side=None):
    """VMAX of a symmetric format, or of the negative (side 0) / positive (side 1) half grid of a sign-split one."""
    name = fmt if side is None else O.SPLIT[fmt][side]
    return float(np.max(np.abs(O.GRIDS[name])))


def rounded_scale(a, v, dt):
    """The reference's scale: fl_dt(fl32(a) / fl32(VMAX)) (qu.py:320, :432-433)."""
    with np.errstate(divide="ignore", invalid="ignore", over="ignore", under="ignore"):
        return (np.asarray(a, dtype=np.float32) / np.float32(v)).astype(dt)


def regular(s, dt):
    """`scale_regular<InT>` (csrc/fpq_common.cuh): the range in which the scorers take the reciprocal fast path."""
    s = np.asarray(s, dtype=np.float64)
    if dt == np.float16:
        return (s >= 2.0 ** -14) & (s <= 65504.0)
    return (s >= 2.0 ** -100) & (s <= 2.0 ** 100)


@dataclass
class Case:
    """One call: x [G, 128] of dtype dt.  boundary cases carry the side (None: symmetric, 0: negative, 1: positive), the
    target scale (fp16 bit pattern or fp32 value) and whether that scale is regular."""
    dt: type
    label: str
    x: np.ndarray
    fmt: str | None = None
    side: int | None = None
    target: float | None = None
    claim_regular: bool | None = None
    binade: int | None = None
    meta: dict = field(default_factory=dict)


# ------------------------------------------------------------------------------------------------------------------------
# binade sweep
# ------------------------------------------------------------------------------------------------------------------------
def _tiny(dt):
    return float(np.finfo(dt).smallest_subnormal)


def binade_absmax(dt, e):
    a = dt(2.0 ** e * 1.6875)
    return a if 2.0 ** e <= float(a) < 2.0 ** (e + 1) else dt(2.0 ** e)


def _unit_rows(rng, g):
    y = rng.standard_normal((g, GS))
    return y / np.max(np.abs(y), axis=1, keepdims=True)


def _place_absmax(x, rng, a, sign=None):
    g = x.shape[0]
    pos = rng.integers(0, GS, g)
    sg = rng.choice([-1.0, 1.0], g) if sign is None else np.full(g, sign)
    x[np.arange(g), pos] = (sg * float(a)).astype(x.dtype)
    return x


def _ties(dt, e, g, rng):
    """Power-of-two scales and elements on grid midpoints: group i is built for candidate FORMATS[i % 8]."""
    x = np.zeros((g, GS), dtype=np.float64)
    for i in range(g):
        fmt = FORMATS[i % len(FORMATS)]
        halves = [(None, O.GRIDS[fmt])] if fmt in SYM else [(s, O.GRIDS[O.SPLIT[fmt][s]]) for s in (0, 1)]
        for side, grid in halves:
            mags = np.unique(np.abs(grid.astype(np.float64)))
            mids = (mags[1:] + mags[:-1]) / 2
            s = 2.0 ** (e - int(np.floor(np.log2(mags[-1]))))
            cols = np.arange(GS) if side is None else np.arange(side, GS, 2)
            sg = rng.choice([-1.0, 1.0], cols.size) if side is None else np.full(cols.size, 1.0 if side else -1.0)
            x[i, cols] = sg * rng.choice(mids, cols.size) * s
            x[i, cols[0]] = (1.0 if side != 0 else -1.0) * mags[-1] * s
    return x.astype(dt)


def binade_case(dt, e, kind, g, seed):
    rng = np.random.default_rng(seed)
    a = binade_absmax(dt, e)
    y = _unit_rows(rng, g) * float(a) * 0.98
    with np.errstate(under="ignore", over="ignore"):
        if kind == "normal":
            x = _place_absmax(y.astype(dt), rng, a)
        elif kind == "gelu":                              # the negative side six binades below the positive
            x = _place_absmax(np.where(y > 0, y, y * 2.0 ** -6).astype(dt), rng, a, 1.0)
        elif kind in ("pos", "pos0", "neg", "neg0"):
            sign = 1.0 if kind.startswith("pos") else -1.0
            x = (sign * np.abs(y)).astype(dt)
            x[x == 0] = dt(sign * float(a))
            if kind.endswith("0"):                        # exact +0 and -0 elements
                z = rng.random((g, GS))
                x[z < 0.125] = dt(0.0)
                x[z > 0.875] = dt(-0.0)
                x[:, :2] = [dt(0.0), dt(-0.0)]
                x[:, 2] = dt(sign * float(a))
            else:
                x = _place_absmax(x, rng, a, sign)
        elif kind == "ties":
            x = _ties(dt, e, g, rng)
        elif kind == "far":                               # x / s rounds to 0: far below the scale, subnormals included
            x = (y * 2.0 ** -12).astype(dt)
            small = np.array([_tiny(dt), 3 * _tiny(dt), 2.0 ** -20, 2.0 ** -130], dtype=np.float64)
            small = small[(small <= float(a) * 2.0 ** -10) & (small >= _tiny(dt))].astype(dt)
            if small.size:
                cols = rng.integers(0, GS, (g, 8))
                x[np.arange(g)[:, None], cols] = rng.choice([-1, 1], (g, 8)).astype(dt) * rng.choice(small, (g, 8))
            x = _place_absmax(x, rng, a)
        else:
            raise ValueError(kind)
    return Case(dt, f"{np.dtype(dt).name} 2^{e} {kind}", np.ascontiguousarray(x), binade=e, meta={"kind": kind})


def binade_cases(dt, g=64, kinds=KINDS):
    return [binade_case(dt, e, k, g, seed=(e + 200) * 16 + KINDS.index(k) + (dt == np.float16) * 100000)
            for e in BINADES[dt] for k in kinds if k != "ties" or e >= TIES_FROM[dt]]


# ------------------------------------------------------------------------------------------------------------------------
# boundary cases
# ------------------------------------------------------------------------------------------------------------------------
def _absmax_for_scale(target, v, dt):
    """An absmax a (a dt value) whose rounded scale is the target, or, if no a reaches it, the nearest one on the
    target's side of its neighbours (the self-check reports where each case landed)."""
    if dt == np.float16:
        a = np.arange(1, 0x7C00, dtype=np.uint16).view(np.float16)
        s = rounded_scale(a, v, np.float16).view(np.uint16).astype(np.int64)
        hit = np.nonzero(s == int(target))[0]
        if hit.size:
            return a[hit[hit.size // 2]]
        return a[np.argmin(np.abs(s - int(target)))]
    t = np.float32(target)
    a0 = np.float32(np.float64(t) * v)
    cand = (np.int64(a0.view(np.uint32)) + np.arange(-16, 17)).astype(np.uint32).view(np.float32)
    s = rounded_scale(cand, v, np.float32)
    hit = np.nonzero(s == t)[0]
    if hit.size:
        return cand[hit[hit.size // 2]]
    return cand[np.argmin(np.abs(s.astype(np.float64) - float(t)))]


def fp32_targets():
    out = []
    for b in (np.float32(2.0 ** -100), np.float32(2.0 ** 100)):
        lo = np.nextafter(b, np.float32(0))
        hi = np.nextafter(b, np.float32(np.inf))
        out += [np.nextafter(lo, np.float32(0)), lo, b, hi, np.nextafter(hi, np.float32(np.inf))]
    return out


def targets(dt, fmt, side):
    if dt == np.float32:
        return [float(t) for t in fp32_targets()]
    t = list(F16_BOUNDARY)
    if fmt == "e1m2" and side is None:
        t += E1M2_HW_BOUNDARY
    return t


def target_value(dt, t):
    return float(np.uint16(t).view(np.float16)) if dt == np.float16 else float(t)


def companion_scale(dt, a):
    """A regular power-of-two scale near a's binade for the other side of a sign-split boundary case."""
    lo, hi = (-13, 9) if dt == np.float16 else (-99, 99)
    return 2.0 ** int(np.clip(np.floor(np.log2(float(a))) - 3, lo, hi))


def boundary_case(dt, fmt, side, t, g, seed):
    rng = np.random.default_rng(seed)
    v = vmax(fmt, side)
    a = _absmax_for_scale(t, v, dt)
    y = np.abs(_unit_rows(rng, g)) * float(a) * 0.98
    with np.errstate(under="ignore", over="ignore"):
        if side is None:
            x = _place_absmax((y * rng.choice([-1.0, 1.0], y.shape)).astype(dt), rng, a)
        else:
            sign = 1.0 if side else -1.0
            x = np.empty((g, GS), dtype=dt)
            cols_b, cols_c = np.arange(0, GS, 2), np.arange(1, GS, 2)       # boundary side / companion side
            xb = (sign * y[:, : cols_b.size]).astype(dt)
            xb[xb == 0] = dt(sign * float(a))
            xb[:, 0] = dt(sign * float(a))
            x[:, cols_b] = xb
            cgrid = O.GRIDS[O.SPLIT[fmt][1 - side]].astype(np.float64)
            cvals = cgrid[cgrid * -sign > 0]
            sc = companion_scale(dt, a)
            xc = rng.choice(cvals, (g, cols_c.size)) * sc
            xc[:, 0] = cvals[np.argmax(np.abs(cvals))] * sc
            x[:, cols_c] = xc.astype(dt)
    claim = bool(regular(target_value(dt, t), dt))
    if dt == np.float32:                                  # not every fp32 scale is fl(a / VMAX) of some a: keep the one reached
        t = float(rounded_scale(a, v, dt))
    tv = target_value(dt, t)
    if dt == np.float16 and fmt == "e1m2" and side is None:
        claim = 0x0400 <= t <= 0x77FF                      # HwCvt<HG_E1M2>::S_MAX_BITS: 2 s stays finite
    where = "sym" if side is None else ("neg" if side == 0 else "pos")
    lab = f"0x{t:04X}" if dt == np.float16 else f"{tv!r}"
    return Case(dt, f"{np.dtype(dt).name} {fmt} {where} scale {lab}", np.ascontiguousarray(x), fmt=fmt, side=side, target=t,
                claim_regular=claim)


def every_value_case(fmt, t):
    """fp16, symmetric: every fp16 value below the absmax a whose rounded scale has bits t, 127 per group after a itself."""
    a = _absmax_for_scale(t, vmax(fmt), np.float16)
    mags = np.arange(1, int(np.float16(a).view(np.uint16)), dtype=np.uint16).view(np.float16)
    vals = np.concatenate([mags, -mags, np.float16([0.0, -0.0])])
    g = -(-vals.size // (GS - 1))
    x = np.zeros((g, GS), dtype=np.float16)
    x[:, 1:] = np.concatenate([vals, np.zeros(g * (GS - 1) - vals.size, dtype=np.float16)]).reshape(g, GS - 1)
    x[:, 0] = np.where(np.arange(g) % 2, -a, a)
    return Case(np.float16, f"float16 {fmt} sym scale 0x{t:04X} every x", np.ascontiguousarray(x), fmt=fmt, side=None, target=t,
                claim_regular=bool(0x0400 <= t <= (0x77FF if fmt == "e1m2" else 0x7BFF)))


def boundary_cases(dt, g=64, fmts=FORMATS):
    out = []
    for fi, fmt in enumerate(fmts):
        for side in ([None] if fmt in SYM else [0, 1]):
            for ti, t in enumerate(targets(dt, fmt, side)):
                out.append(boundary_case(dt, fmt, side, t, g, seed=7000 + 100 * fi + 10 * (side or 0) + ti + 50000 * (dt == np.float16)))
                if dt == np.float16 and side is None:
                    out.append(every_value_case(fmt, t))
    return out


# ------------------------------------------------------------------------------------------------------------------------
# the oracle
# ------------------------------------------------------------------------------------------------------------------------
def quantize(x, fmt, tie):
    """The port's fake quantization of [.., 128] groups in the scorers' output dtype: the input dtype under the kernel rule
    (the *_cuda functions), fp32 under the argmin rule."""
    xh = np.ascontiguousarray(x.reshape(-1, GS))
    dout = xh.dtype if tie == "kernel" else np.dtype(np.float32)
    if fmt in SYM:
        return P.fake_quant(xh, fmt, None, tie, clamp3=False, out_dtype=dout).reshape(x.shape)
    out = np.empty(xh.shape, dtype=dout)
    gneg, gpos = (O.GRIDS[n] for n in O.SPLIT[fmt])
    fn = getattr(P._lib(), f"port_signsplit_{P._TAG[xh.dtype]}_{P._TAG[np.dtype(dout)]}")
    fn(xh.ctypes.data, out.ctypes.data, xh.shape[0], GS, gneg.ctypes.data, gneg.size, float(np.max(np.abs(gneg))),
       gpos.ctypes.data, gpos.size, float(np.max(np.abs(gpos))), P._TIE[tie])
    return out.reshape(x.shape)


def errors(x, fmt, tie):
    """float64 x - x_q, element by element."""
    with np.errstate(invalid="ignore", over="ignore"):
        return x.astype(np.float64) - quantize(x, fmt, tie).astype(np.float64)


def group_sse(x, fmt, tie):
    """float64 squared error of every group, [..] over the leading dims of x [.., 128]."""
    d = errors(x, fmt, tie)
    with np.errstate(invalid="ignore", over="ignore"):
        return (d * d).sum(axis=-1)


# ------------------------------------------------------------------------------------------------------------------------
# the self-check
# ------------------------------------------------------------------------------------------------------------------------
def self_check(case: Case):
    """Every claim of a case, recomputed on the host; returns a list of violations (empty = fine)."""
    bad = []
    x = case.x
    if x.dtype != case.dt or x.shape[1] != GS or not np.all(np.isfinite(x)):
        bad.append("dtype, shape or finiteness")
        return bad
    if case.binade is not None:
        am = np.max(np.abs(x.astype(np.float64)), axis=1)
        if not np.all((am >= 2.0 ** case.binade) & (am < 2.0 ** (case.binade + 1))):
            bad.append(f"absmax outside the binade: {np.unique(am)[:4]}")
        kind = case.meta["kind"]
        if kind in ("pos", "neg") and np.any(x == 0):
            bad.append("one-sided group holds zeros")
        if kind in ("pos0", "neg0") and not (np.any(np.signbit(x) & (x == 0)) and np.any(~np.signbit(x) & (x == 0))):
            bad.append("one-sided group without both zeros")
        if kind.startswith("pos") and np.any(x < 0) or kind.startswith("neg") and np.any(x > 0):
            bad.append("one-sided group has the other sign")
        return bad
    side = case.side
    xs = x.astype(np.float64)
    if side is None:
        a = np.max(np.abs(xs), axis=1)
    else:
        sel = xs > 0 if side else xs <= 0
        a = np.max(np.where(sel, np.abs(xs), 0.0), axis=1)
    s = rounded_scale(a.astype(case.dt), vmax(case.fmt, side), case.dt)
    if case.dt == np.float16:
        got = set(int(b) for b in s.view(np.uint16))
        if got != {int(case.target)}:
            bad.append(f"rounded scale bits {sorted(got)} != 0x{case.target:04X}")
    elif set(float(v) for v in s) != {float(case.target)}:
        bad.append(f"rounded scale {sorted(set(float(v) for v in s))} != {case.target!r}")
    reg = regular(s, case.dt)
    if case.dt == np.float16 and case.fmt == "e1m2" and side is None:
        reg = (s.view(np.uint16) >= 0x0400) & (s.view(np.uint16) <= 0x77FF)
    if not np.all(reg == case.claim_regular):
        bad.append(f"regularity {reg[:4]} != claim {case.claim_regular}")
    if side is not None:
        other = xs > 0 if side == 0 else xs <= 0
        sc = rounded_scale(np.max(np.where(other, np.abs(xs), 0.0), axis=1).astype(case.dt), vmax(case.fmt, 1 - side), case.dt)
        if not np.all(regular(sc, case.dt)):
            bad.append("companion scale not regular")
        if not np.all(np.log2(sc.astype(np.float64)) == np.round(np.log2(sc.astype(np.float64)))):
            bad.append("companion scale not a power of two")
        for tie in ("kernel", "argmin"):
            d = errors(x, case.fmt, tie)
            if np.any(d[other] != 0):
                bad.append(f"companion side error not 0 under the {tie} rule")
    return bad
