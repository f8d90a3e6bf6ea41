"""CPU self-check of the scorer range cases (tests/score_range_cases.py): every case lands where it claims -- the binade of
its absmax, the side of each scale boundary, an exactly-zero error on the companion side of a sign-split boundary case --
so that the GPU tests in tests/test_gpu_score_range.py cannot pass vacuously."""
import numpy as np
import pytest

import score_range_cases as C


@pytest.mark.parametrize("dt", [np.float16, np.float32], ids=["f16", "f32"])
def test_every_case_lands_where_it_claims(dt):
    cs = C.binade_cases(dt) + C.boundary_cases(dt)
    bad = [(c.label, b) for c in cs for b in [C.self_check(c)] if b]
    assert not bad, bad[:10]
    # every binade of the range, every content kind, both sides of every boundary of every candidate
    seen = {(c.binade, c.meta["kind"]) for c in cs if c.binade is not None}
    assert {e for e, _ in seen} == set(C.BINADES[dt])
    assert {k for _, k in seen} == set(C.KINDS)
    for fmt in C.FORMATS:
        for side in ([None] if fmt in C.SYM else [0, 1]):
            claims = {c.claim_regular for c in cs if c.fmt == fmt and c.side == side}
            assert claims == {True, False}, (fmt, side, claims)


@pytest.mark.parametrize("dt", [np.float16, np.float32], ids=["f16", "f32"])
def test_boundary_cases_have_nonzero_error(dt):
    """The per-class bar only bites where the oracle's error is not zero."""
    cs = C.boundary_cases(dt)
    for tie in ("kernel", "argmin"):
        want = np.array([[C.group_sse(c.x, f, tie).sum() for f in C.FORMATS] for c in cs])
        bites = (want > 0) | np.isnan(want)              # a NaN total is checked too: by its class
        assert np.mean(bites) > 0.9, (tie, np.mean(bites))
        own = [want[i, C.FORMATS.index(c.fmt)] for i, c in enumerate(cs)]
        assert all(np.isfinite(v) and v > 0 for v in own), [(c.label, v) for c, v in zip(cs, own) if not v > 0][:5]


def test_e1m2_hardware_boundary_and_fp32_targets():
    t = C.targets(np.float16, "e1m2", None)
    assert t == C.F16_BOUNDARY + C.E1M2_HW_BOUNDARY
    f32 = C.fp32_targets()
    assert len(f32) == 10 and sum(bool(C.regular(v, np.float32)) for v in f32) == 6
