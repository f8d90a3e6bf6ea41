"""GPU: the UNMODIFIED reference CUDA extension (compiled from a checkout of the reference's quant/ sources into
oracle/_ref by oracle/build_ref.sh) against (1) the oracle's restatement of its scan -- which
closes the chain reference -> golden fixtures -- and (2) this repo's kernels, on the real device
with real torch-CUDA glue arithmetic (fp16 division, type promotion)."""
import numpy as np
import pytest
import torch

from conftest import bits_equal, mismatch_report
from oracle import oracle as O
import ref_glue

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    mod = ref_glue.load_ref_ext()
    if mod is None:
        # no stored stand-in: these tests compare with the reference's own kernel, and without a build of it there is
        # nothing of it to compare with (its outputs were never recorded)
        pytest.skip("oracle/_ref/ref_quant_cuda*.so not built: oracle/build_ref.sh builds it from a checkout of the reference")
    return mod


@pytest.fixture(scope="module")
def ops():
    from fpqvar_b200 import ops as _ops
    return _ops


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


def _probe(golden):
    rng = np.random.default_rng(9)
    return np.concatenate([golden["in/probe"], (rng.standard_normal(1 << 20) * 4).astype(np.float32),
                           rng.uniform(-40, 40, 1 << 18).astype(np.float32)])


@pytest.mark.parametrize("gname", list(O.GRIDS))
def test_reference_kernel_equals_oracle_scan_and_ours(ref, ops, golden, gname):
    x = _probe(golden)
    grid = O.GRIDS[gname]
    z_ref, idx = ref.quant(dev(x), dev(grid))
    torch.cuda.synchronize()
    z_ref = host(z_ref)
    assert float(idx.abs().sum()) == 0.0                                  # never written (quant_kernel.cu:49,58)
    want = O.scan_quant(x, grid)
    assert bits_equal(z_ref, want), "oracle scan != real reference kernel\n" + mismatch_report(want, z_ref)
    ours = host(ops.quant_grid(dev(x), dev(grid), "kernel"))
    assert bits_equal(ours, z_ref), mismatch_report(ours, z_ref)


@pytest.mark.parametrize("dt", [torch.float32, torch.float16])
@pytest.mark.parametrize("fmt", ["e2m1", "e1m2", "e3m0", "e2m3", "e3m2"])
def test_fused_group_equals_reference_glue_plus_reference_kernel(ref, ops, fmt, dt):
    torch.manual_seed(5)
    x = (torch.randn(8192, 1920, device="cuda") * torch.exp(torch.randn(8192, 1, device="cuda"))).to(dt)
    x[17] = 0
    x[33, :128] = 1e-7                                                     # fp16: scale underflows to 0
    want = ref_glue.sym_group_cuda(ref.quant, x, dev(O.GRIDS[fmt]))
    torch.cuda.synchronize()
    got = ops.fake_quant(x, fmt, 128, "kernel")
    assert got.dtype == want.dtype
    assert bits_equal(host(got), host(want)), mismatch_report(host(got), host(want))


@pytest.mark.parametrize("dt", [torch.float32, torch.float16])
@pytest.mark.parametrize("split", ["e1m2_neg_e2m1_pos", "int_neg_e2m3_pos"])
def test_fused_signsplit_equals_reference_glue_plus_reference_kernel(ref, ops, split, dt):
    torch.manual_seed(6)
    x = torch.nn.functional.gelu(torch.randn(4096, 7680, device="cuda") * 1.5, approximate="tanh").to(dt)
    x[3] = x[3].abs()
    x[4] = -x[4].abs()
    gn, gp = (dev(O.GRIDS[n]) for n in O.SPLIT[split])
    clip = 1.0 if split == "e1m2_neg_e2m1_pos" else None
    want = ref_glue.signsplit_group_cuda(ref.quant, x, gn, gp, 128, clip)
    torch.cuda.synchronize()
    got = ops.fake_quant_signsplit(x, split, 128, "kernel", global_clip=clip is not None)
    assert bits_equal(host(got), host(want)), mismatch_report(host(got), host(want))


def test_config1_full_size_against_reference_kernel(ref, ops):
    """BASELINE configs[0] tensor at full size, GPU reference path vs ours."""
    torch.manual_seed(0)
    x = torch.randn(4096, 4096).cuda()
    want = ref_glue.sym_group_cuda(ref.quant, x, dev(O.GRIDS["e2m1"]))
    torch.cuda.synchronize()
    got = ops.fake_quant(x, "e2m1", 128, "kernel")
    assert bits_equal(host(got), host(want))
