"""The exact-accumulation envelope of the low-bit GEMM (oracle/lowbit.py exact_accumulation) and the probes that test it on
the GPU (tests/test_gpu_gemm_envelope.py), checked on the CPU:
  - the envelope k_acc * max|q_a| * max|q_w| / (u_a * u_w) <= 2^24 at the boundaries the contract text names;
  - the oracle (oracle/gemm_codes.c) equals the probe summed in integer units, and fp32 holds every in-envelope slab sum;
  - sensitivity: each probe set tells the oracle apart from an accumulator narrower than fp32 (truncating or rounding, 32-deep
    MMA chunks) wherever the envelope needs more bits than that accumulator keeps, and from the other fp32 orders of the
    scale epilogue.  Without this a green GPU run could not tell an exact accumulator from a narrower one."""
import numpy as np
import pytest

from oracle import lowbit as LB

FMTS = ["e2m1", "e1m2", "e3m0", "e2m3", "e3m2"]
PAIRS = [(a, w) for a in FMTS for w in FMTS]
# (k, scale group): 128-groups, then one scale per row; the GPU test runs the same shapes
SHAPES = [(128, 128), (640, 128), (1920, 1920), (2304, 2304), (7680, 7680)]
MODEL_BITS = (23, 22, 20, 16, 14)


def bits(a):
    return a.view({2: np.uint16, 4: np.uint32}[a.dtype.itemsize])


def same_bits(a, b):
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(bits(a)[~na], bits(b)[~nb])


def test_exact_accumulation_table():
    for a, w in PAIRS:
        assert LB.exact_accumulation(a, w, 128) == ((a, w) != ("e3m2", "e3m2")), (a, w)
    assert LB.exact_accumulation("e3m0", "e3m0", 4096) and not LB.exact_accumulation("e3m0", "e3m0", 4224)
    assert LB.exact_accumulation("e2m1", "e2m1", 9216)
    # the row-scaled boundaries the contract text quotes
    assert not LB.exact_accumulation("e3m2", "e3m2", 2304) and not LB.exact_accumulation("e3m2", "e3m0", 2304)
    assert not LB.exact_accumulation("e3m2", "e2m3", 2304) and not LB.exact_accumulation("e2m1", "e3m2", 7680)
    assert LB.exact_accumulation("e2m3", "e2m3", 2304) and not LB.exact_accumulation("e2m3", "e2m3", 7680)
    assert round(LB.accumulation_bits("e3m2", "e3m2", 128), 1) == 24.6
    assert round(LB.accumulation_bits("e3m0", "e3m2", 128), 1) == 21.8
    # the resolutions and maxima come from the grids
    assert [LB.grid_unit(f) for f in FMTS] == [0.5, 0.25, 0.25, 0.125, 0.0625]
    assert [LB.grid_min(f) for f in FMTS] == [0.5, 0.25, 0.25, 0.125, 0.0625]


def test_fma32_rounds_once():
    a, b, c = np.float32(1 + 2.0 ** -12), np.float32(1 + 2.0 ** -12), np.float32(2.0 ** -80)
    # a * b = 1 + 2^-11 + 2^-24, a float32 half-way point; + 2^-80 lifts the exact sum above it, but the float64 sum rounds back
    # onto it: rounded once, the result goes up, not to even
    assert LB.fma32(a, b, c) == np.nextafter(np.float32(1 + 2.0 ** -11), np.float32(2))
    assert LB.fma32(a, b, np.float32(0)) == np.float32(1 + 2.0 ** -11)
    assert LB.fma32(a, b, -c) == np.float32(1 + 2.0 ** -11)


@pytest.mark.parametrize("k,group", SHAPES)
@pytest.mark.parametrize("fmt_a,fmt_w", PAIRS)
def test_oracle_is_exact_on_envelope_probes(fmt_a, fmt_w, k, group):
    qa, sa, qw, sw = LB.envelope_probe(fmt_a, fmt_w, k, group)
    units = LB.slab_sums_units(qa, fmt_a, qw, fmt_w, group)
    p = units * (LB.grid_unit(fmt_a) * LB.grid_unit(fmt_w))
    want = LB.gemm_codes(qa, sa, qw, sw)
    assert same_bits(LB.scale_chain(p, sa, sw), want)
    if LB.exact_accumulation(fmt_a, fmt_w, group):
        assert np.array_equal(p.astype(np.float32).astype(np.float64), p)       # every slab sum is an fp32 number
        # and the probes reach into the top of the envelope: F1 row r x F1 column r is k_acc-1 maximal products + 1 unit
        top = (group - 1) * (LB.O.grid_absmax(fmt_a) / LB.grid_unit(fmt_a)) * (LB.O.grid_absmax(fmt_w) / LB.grid_unit(fmt_w))
        assert units[-1, 0, 0] == top + 1


def _round_bits(x, b, mode):
    """x (integers in float64) kept to b significant bits, by truncation or round-to-nearest-even."""
    ax = np.abs(x)
    e = np.floor(np.log2(np.where(ax > 0, ax, 1)))
    ulp = np.maximum(np.exp2(e - b + 1), 1.0)
    r = np.floor(ax / ulp) if mode == "trunc" else np.round(ax / ulp)
    return np.sign(x) * r * ulp


def _narrow_accumulators(qa, fmt_a, qw, fmt_w, group, models):
    """Slab sums of accumulators that keep b bits, for every (b, mode) of `models`: each 32-deep MMA's sum is exact, its
    addition to the accumulator rounds."""
    ia, iw = qa.astype(np.float64) / LB.grid_unit(fmt_a), qw.astype(np.float64) / LB.grid_unit(fmt_w)
    slabs = qa.shape[1] // group
    out = {bm: np.empty((slabs, qa.shape[0], qw.shape[0])) for bm in models}
    for t in range(slabs):
        acc = {bm: 0.0 for bm in models}
        for c in range(t * group, (t + 1) * group, 32):
            chunk = ia[:, c:c + 32] @ iw[:, c:c + 32].T
            acc = {(b, mode): _round_bits(acc[b, mode] + chunk, b, mode) for b, mode in models}
        for bm in models:
            out[bm][t] = acc[bm]
    return {bm: p * (LB.grid_unit(fmt_a) * LB.grid_unit(fmt_w)) for bm, p in out.items()}


@pytest.mark.parametrize("k,group", [(128, 128), (1920, 1920), (2304, 2304), (7680, 7680)])
@pytest.mark.parametrize("fmt_a,fmt_w", PAIRS)
def test_probes_detect_a_narrower_accumulator(fmt_a, fmt_w, k, group):
    need = LB.accumulation_bits(fmt_a, fmt_w, group)
    narrower = [b for b in MODEL_BITS if need > b]
    if not narrower:
        pytest.skip(f"{fmt_a} x {fmt_w} at {group} needs {need:.1f} bits, no model is narrower")
    qa, sa, qw, sw = LB.envelope_probe(fmt_a, fmt_w, k, group)
    want = LB.gemm_codes(qa, sa, qw, sw)
    models = [(b, mode) for b in narrower for mode in ("trunc", "rn")] + [(60, "trunc")]
    p = _narrow_accumulators(qa, fmt_a, qw, fmt_w, group, models)
    for b, mode in models[:-1]:
        assert not same_bits(LB.scale_chain(p[b, mode], sa, sw), want), \
            f"{fmt_a} x {fmt_w}, k_acc {group}: a {b}-bit {mode} accumulator is not detected"
    # and a model wide enough to be exact is the oracle: the models differ from it by their width alone
    assert same_bits(LB.scale_chain(p[60, "trunc"], sa, sw), want)


def _chain(p, sa, sw, order):
    acc = np.zeros(p.shape[1:], dtype=np.float32)
    slabs = range(p.shape[0]) if order != "descending" else range(p.shape[0] - 1, -1, -1)
    with np.errstate(invalid="ignore", over="ignore"):
        for t in slabs:
            p32, a, w = p[t].astype(np.float32), sa[:, t][:, None], sw[:, t][None, :]
            if order == "scale_product":                    # fma(P, sa * sw, acc)
                acc = LB.fma32(p32, a * w, acc)
            elif order == "no_fma":                         # (P * sa) * sw + acc, two roundings
                acc = (p32 * a) * w + acc
            else:                                           # fma(P * sa, sw, acc): the contract
                acc = LB.fma32(p32 * a, w, acc)
    return acc


@pytest.mark.parametrize("fmt_a,fmt_w", [("e2m1", "e2m1"), ("e3m2", "e2m3"), ("e1m2", "e3m0")])
def test_scale_probes_detect_another_epilogue_order(fmt_a, fmt_w):
    qa, sa, qw, sw, _ = LB.scale_chain_probe(fmt_a, fmt_w, 160, 136, 640, 128)
    p = LB.slab_sums_units(qa, fmt_a, qw, fmt_w, 128) * (LB.grid_unit(fmt_a) * LB.grid_unit(fmt_w))
    want = LB.gemm_codes(qa, sa, qw, sw)
    assert same_bits(_chain(p, sa, sw, "ascending"), want)
    for order in ("scale_product", "no_fma", "descending"):
        assert not same_bits(_chain(p, sa, sw, order), want), order
