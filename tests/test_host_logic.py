"""CPU: host-side logic -- C-ABI surface, workload model, sharding (incl. a 2-rank gloo run), the
drop-in API surface and its error behaviour.  No kernel is launched here."""
import ctypes
import inspect
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------
# C ABI: the library loads and exports every symbol include/fpq_b200.h declares
# ---------------------------------------------------------------------------------------------
def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "fpq_b200.h")).read()
    return sorted(set(re.findall(r"FPQ_API[^;(]*?\b(fpq_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from fpqvar_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        pytest.fail(f"{_lib.LIB_PATH} missing: run __graft_entry__.build()")
    handle = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 11
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in include/fpq_b200.h but not exported"
    # the ctypes signature table covers exactly the declared entry points
    assert sorted(_lib.SIGNATURES) == declared
    assert handle.fpq_version is not None
    _lib.lib().fpq_version.restype = ctypes.c_char_p
    assert b"sm_100a" in _lib.lib().fpq_version()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "fpqvar_b200")
    for dirpath, _d, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{f} imports the oracle"
                assert "liboracle" not in src, f"{f} links the oracle"


def test_cpu_tensors_are_rejected_loudly():
    from fpqvar_b200 import ops, quant_utils as Q
    from fpqvar_b200._lib import FpqError
    x = torch.zeros(4, 128)
    for fn in (lambda: ops.fake_quant(x, "e2m1"), lambda: Q.fp_quant_e2_per_group_cuda(x, 4, 128),
               lambda: Q.fp6_quant_e2m3_per_token_cuda(x, 6), lambda: ops.score_formats(x, ["e2m1"]),
               lambda: Q.fp_quant_e1m2_neg_e2m1_pos_per_group_cuda(x, 4)):
        with pytest.raises(FpqError, match="no CPU fallback"):
            fn()


# ---------------------------------------------------------------------------------------------
# workload model (SURVEY.md appendix C)
# ---------------------------------------------------------------------------------------------
def test_var_workload_shapes_and_bytes():
    from fpqvar_b200.var_workload import WORKLOADS
    d30 = WORKLOADS["var_d30_w4a4_rot"]
    assert d30.width == 1920 and d30.stage_rows() == [100, 400, 900, 1600, 2500, 3600, 6400, 10000, 16900, 25600]
    calls = d30.calls()
    assert len(calls) == 10 * 30 * 4
    assert {c.site for c in calls} == {"mat_qkv", "proj", "fc1", "fc2"}
    # 548 M activation elements per image (SURVEY.md section 8d): 68000 rows x 7C x 30 blocks / 50 images
    assert d30.elems_per_pass() == 68000 * 7 * 1920 * 30
    # 6C + 4C + 6C + 16C bytes per token and block, plus the adaLN rows the fused mat_qkv / fc1 kernel reads:
    # 2 sites x (scale, shift) x 100 batch rows x C x 4 bytes per block and stage
    assert d30.modulate and all(c.op == "mod_rotate_quant" and c.rows_per_batch * 100 == c.rows for c in calls if c.site in ("mat_qkv", "fc1"))
    assert d30.bytes_per_pass() == 68000 * 30 * 32 * 1920 + 10 * 30 * 2 * 2 * 100 * 1920 * 4
    nomod = WORKLOADS["var_d30_w4a4_rot_nomod"]
    assert nomod.bytes_per_pass() == 68000 * 30 * 32 * 1920 and all(c.op != "mod_rotate_quant" for c in nomod.calls())
    d16 = WORKLOADS["var_d16_w4a4"]
    assert d16.stage_rows()[-1] == 32768 and d16.width == 1024
    assert all(c.op == "group" for c in d16.calls())
    d36 = WORKLOADS["var_d36_w6a6_rot"]
    assert d36.stage_rows() == [20, 80, 180, 320, 720, 1620, 3380, 6480, 11520, 20480] and d36.width == 2304
    assert all(c.elems % 128 == 0 for w in WORKLOADS.values() for c in w.calls())


# ---------------------------------------------------------------------------------------------
# streaming rotate kernel: launch plan and shared-memory choreography (tests/rotate_layout_model.py)
# ---------------------------------------------------------------------------------------------
def test_rotate_plan_model_matches_the_launcher():
    """The Python mirror of rot_plan() plans exactly like the C++ launcher (fpq_rotate_plan is a host-only query)."""
    import ctypes
    import rotate_layout_model as M
    from fpqvar_b200 import _lib as L
    lib = L.lib()
    for cpr in list(range(1, 80)) + [128, 1000]:
        for mod in (False, True):
            out = (ctypes.c_int * 2)()
            rc = lib.fpq_rotate_plan(cpr, int(mod), out)
            want = M.rot_plan(cpr, mod)
            if want is None:
                assert rc == L.FPQ_ERR_UNSUPPORTED, cpr
                continue
            assert rc == 0 and tuple(out) == want, (cpr, mod)
            assert want[0] * want[1] <= 20 or want[1] == 1
    assert M.rot_plan(15) == (4, 5) and M.rot_plan(18) == (5, 4) and M.rot_plan(8) == (2, 10)     # VAR-d30 / d36 / d16


@pytest.mark.parametrize("ncols,nr", [(4, 2), (3, 2), (1, 2), (4, 1), (2, 1)])
def test_rotate_streaming_layout_covers_every_unit_without_bank_conflicts(ncols, nr):
    import rotate_layout_model as M
    seen1, seen2 = {}, {}
    for sub in range(2):
        for ph in range(4):                                   # a phase of pass 1 = the 8 lanes of one chunk
            accs = [M.pass1_accesses(lane, sub, ncols, nr) for lane in range(8 * ph, 8 * ph + 8)]
            for a in range(4):
                assert M.conflict_free([x[a][0] if x else None for x in accs]), ("pass-1 load", sub, ph, a)
                assert M.conflict_free([x[a][1] if x else None for x in accs]), ("pass-1 store", sub, ph, a)
            lds = {ld for x in accs if x for ld, _ in x}
            sts = {st for x in accs if x for _, st in x}
            assert lds == sts                                 # in place: stores stay inside the chunk's own units
            for ld in lds:
                seen1[ld] = seen1.get(ld, 0) + 1
    for ph in range(4):
        accs = [M.pass2_accesses(lane, ncols, nr) for lane in range(8 * ph, 8 * ph + 8)]
        for i in range(8):
            assert M.conflict_free([x[i] if x else None for x in accs]), ("pass-2 load", ph, i)
        for x in accs:
            for a in (x or []):
                seen2[a] = seen2.get(a, 0) + 1
    want = {row * 2048 + col * 512 + u * 16 for row in range(nr) for col in range(ncols) for u in range(32)}
    assert set(seen1) == want and set(seen1.values()) == {1}
    assert set(seen2) == want and set(seen2.values()) == {1}


@pytest.mark.parametrize("ncols,nr", [(4, 2), (3, 2), (4, 1), (1, 1)])
def test_rotate_streaming_two_pass_butterflies_are_the_hadamard_transform(ncols, nr):
    """Pass 1 (bits 0,1,5,6, written back swizzled in place) + pass 2 (bits 2,3,4) == x * m @ H_128 on every chunk."""
    import rotate_layout_model as M
    rng = np.random.default_rng(10 * ncols + nr)
    tile = rng.standard_normal((nr, ncols * 128))
    mult = rng.standard_normal(ncols * 128)
    h = np.array([[1.0]])
    for _ in range(7):
        h = np.block([[h, h], [h, -h]])
    want = ((tile * mult).reshape(nr, ncols, 128) @ h).reshape(nr, -1)
    got = M.simulate_step(tile, mult, ncols)
    assert not np.isnan(got).any()
    assert np.abs(got - want).max() <= 1e-11 * np.abs(want).max()


def test_shard_units_partition():
    from fpqvar_b200.var_workload import shard_units
    for world in (1, 2, 3, 8):
        seen = sorted(u for r in range(world) for u in shard_units(37, r, world))
        assert seen == list(range(37))
    with pytest.raises(ValueError):
        shard_units(4, 2, 2)


# ---------------------------------------------------------------------------------------------
# rotation host utilities
# ---------------------------------------------------------------------------------------------
def test_block_hadamard_matrix_matches_reference_fixture(golden):
    from fpqvar_b200 import rotation_utils as R
    from fpqvar_b200.hotpath import SIGN_BITS_SEED42_128
    q = R.block_random_hadamard_matrix(256, 128, "cpu", 42)
    assert q.dtype == torch.float64
    assert np.array_equal(q.numpy().view(np.uint64), golden["rot/q256"].view(np.uint64))
    s = R.sign_vector(128, 42)
    assert "".join("1" if v > 0 else "0" for v in s.tolist()) == SIGN_BITS_SEED42_128
    bits = R.block_sign_bits(128, 42)
    for i, c in enumerate(SIGN_BITS_SEED42_128):
        assert ((bits[i >> 5] >> (i & 31)) & 1) == int(c)
    # like the reference, building the matrix leaves the global RNG seeded with `seed`
    R.block_random_hadamard_matrix(128, 128, "cpu", 7)
    a = torch.rand(3)
    torch.manual_seed(7)
    torch.randint(low=0, high=2, size=(128,))
    assert torch.equal(a, torch.rand(3))
    assert torch.equal(R.block_random_hadamard_matrix(256, 128, "cpu", 42, force_identity=True), torch.eye(256, dtype=torch.float64))
    # hadamard_utils mirror: the reference's butterfly builds the same matrix; non power-of-two sizes are out of scope
    from fpqvar_b200 import hadamard_utils as H, block_rotation_utils as BR
    signs = R.sign_vector(128, 42)
    q128 = H.matmul_hadU(torch.diag(signs))
    assert np.array_equal(q128.numpy().view(np.uint64), golden["rot/q256"][:128, :128].view(np.uint64))
    assert H.get_hadK(128) == (None, 1) and BR.rotate_model is R.rotate_model
    with pytest.raises(NotImplementedError):
        H.matmul_hadU(torch.zeros(2, 1920, dtype=torch.float64))


# ---------------------------------------------------------------------------------------------
# drop-in API surface
# ---------------------------------------------------------------------------------------------
REFERENCE_SIGNATURES = {     # models_fp_quant_transform_rotate/quant_utils.py (+ models_fp_quant for the last two)
    "quantize_to_nearest_grid": ["x", "quant_grid"],
    "fp_quant_e1_per_token": ["x", "n_bits"], "fp_quant_e2_per_token": ["x", "n_bits"], "fp_quant_e3_per_token": ["x", "n_bits"],
    "fp_quant_e1_per_group": ["x", "n_bits", "group_size"], "fp_quant_e2_per_group": ["x", "n_bits", "group_size"],
    "fp_quant_e3_per_group": ["x", "n_bits", "group_size"],
    "fp_quant_e1_per_group_cuda": ["x", "n_bits", "group_size"], "fp_quant_e2_per_group_cuda": ["x", "n_bits", "group_size"],
    "fp_quant_e3_per_group_cuda": ["x", "n_bits", "group_size"],
    "fp_quant_e1m2_neg_e2m1_pos_per_group": ["x", "n_bits", "group_size", "clipping_strength"],
    "fp_quant_e1m2_neg_e2m1_pos_per_group_cuda": ["x", "n_bits", "group_size", "clipping_strength"],
    "fp6_quant_e2m3_per_token_cuda": ["x", "n_bits"], "fp6_quant_e3m2_per_token_cuda": ["x", "n_bits"],
    "fp6_quant_e2m3_per_group_cuda": ["x", "n_bits", "group_size"], "fp6_quant_e3m2_per_group_cuda": ["x", "n_bits", "group_size"],
    "fp6_quant_int_neg_e2m3_pos_per_group_cuda": ["x", "n_bits", "group_size"],
    "fp6_quant_int_neg_e2m3_pos_per_token_cuda": ["x", "n_bits"],
    "fp4_afpq_per_group_cuda": ["x", "n_bits", "group_size", "clipping_strength"],
    "fp_neg_reverse_quant_per_group_cuda": ["x", "n_bits", "group_size"],
}
CTOR = ["in_features", "out_features", "bias", "act_quant", "quantize_output", "w_bit", "a_bit", "act_quant_sym",
        "fc2_act_log2_quant", "activation_fp_quant", "weight_fp_quant", "act_fp_type", "weight_fp_type"]
FROM_FLOAT = ["module", "weight_quant", "act_quant", "quantize_output", "w_bit", "a_bit", "act_quant_sym", "fc2_act_log2_quant",
              "activation_fp_quant", "weight_fp_quant", "act_fp_type", "weight_fp_type"]
QUANTIZE_VAR = ["model", "weight_quant", "act_quant", "quantize_bmm_input", "w_bit", "a_bit", "kv_bit", "act_quant_sym",
                "fc2_act_log2_quant", "quant_kv", "activation_fp_quant", "weight_fp_quant", "act_fp_type", "weight_fp_type", "fc2_fp_type"]


def test_quant_utils_signatures_match_the_reference():
    from fpqvar_b200 import quant_utils as Q
    for name, params in REFERENCE_SIGNATURES.items():
        assert list(inspect.signature(getattr(Q, name)).parameters) == params, name
    for cls in (Q.QuantizedLinear, Q.QuantizedLinear_fc2):
        assert list(inspect.signature(cls.__init__).parameters)[1:] == CTOR
        assert list(inspect.signature(cls.from_float).parameters) == FROM_FLOAT
    assert list(inspect.signature(Q.quantize_VAR).parameters) == QUANTIZE_VAR
    assert inspect.signature(Q.fp_quant_e2_per_group_cuda).parameters["group_size"].default == 128


def test_quantized_linear_dispatch_and_errors():
    from fpqvar_b200 import quant_utils as Q
    m = Q.QuantizedLinear(256, 128, True, act_quant="per_group", a_bit=4, activation_fp_quant=True, act_fp_type="fp_e2")
    assert m.act_quant.func is Q.fp_quant_e2_per_group_cuda and m.act_quant.keywords == {"n_bits": 4, "group_size": 128}
    assert m.act_quant_name == "per_group" and m.output_quant_name == "None"
    assert m.weight.dtype == torch.float16 and tuple(m.weight.shape) == (128, 256) and tuple(m.bias.shape) == (1, 128)
    assert "weight" in dict(m.named_buffers()) and not list(m.parameters())
    m2 = Q.QuantizedLinear_fc2(256, 128, False, act_quant="per_group", a_bit=4, activation_fp_quant=True, act_fp_type="fp_e1m2_neg_e2m1_pos")
    assert m2.act_quant.func is Q.fp_quant_e1m2_neg_e2m1_pos_per_group_cuda and m2.bias is None
    m3 = Q.QuantizedLinear(64, 64, act_quant="per_token", a_bit=6, activation_fp_quant=True, act_fp_type="fp6_e3m2", quantize_output=True)
    assert m3.act_quant.func is Q.fp6_quant_e3m2_per_token_cuda and m3.output_quant is m3.act_quant
    with pytest.raises(ValueError, match="Unsupported fp_type"):
        Q.QuantizedLinear(8, 8, act_quant="per_group", activation_fp_quant=True, act_fp_type="fp_e1m2_neg_e2m1_pos")   # fc2-only type
    with pytest.raises(ValueError, match="Unsupported fp_type"):
        Q.QuantizedLinear_fc2(8, 8, act_quant="per_token", activation_fp_quant=True, act_fp_type="nope")
    with pytest.raises(ValueError, match="Invalid act_quant"):
        Q.QuantizedLinear(8, 8, act_quant="per_row")
    with pytest.raises(AssertionError):
        Q.fp_quant_e2_per_group_cuda(torch.zeros(128), 6)
    with pytest.raises(AssertionError):
        Q.fp6_quant_e2m3_per_token_cuda(torch.zeros(128), 4)
    # integer baselines are out of scope and say so
    with pytest.raises(NotImplementedError, match="outside the FP"):
        Q.QuantizedLinear(8, 8, act_quant="per_token", a_bit=8)(torch.zeros(1, 8))


def test_quant_cuda_is_an_importable_extension_module_on_sys_path():
    """`import quant_cuda` with fpqvar_b200/dropin on sys.path loads the torch extension over the C ABI (a real module file,
    not a sys.modules entry): what replaces the reference's quant/ build directory."""
    code = ("import sys; sys.path.insert(0, %r); import torch, quant_cuda; "
            "assert quant_cuda.__file__.endswith('.so') and 'dropin' in quant_cuda.__file__; "
            "print(quant_cuda.version())") % os.path.join(ROOT, "fpqvar_b200", "dropin")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "fpq_b200" in r.stdout


def test_dropin_install_registers_reference_module_names():
    import sys
    import fpqvar_b200.dropin as dropin
    saved = {k: sys.modules.get(k) for k in ("quant_cuda", "quant_utils", "rotation_utils", "transform_model_utils",
                                             "block_rotation_utils", "hadamard_utils")}
    try:
        dropin.install()
        import quant_cuda
        assert callable(quant_cuda.quant) and "quant(x: torch.Tensor, y: torch.Tensor)" in quant_cuda.quant.__doc__     # quant/quant.cpp:27-29
        import quant_utils
        assert quant_utils.QuantizedLinear.__name__ == "QuantizedLinear"
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


# ---------------------------------------------------------------------------------------------
# multi-rank search sharding over gloo (world_size 2), CPU stand-in scorer
# ---------------------------------------------------------------------------------------------
def _fake_layer_fn(weight, activations, weight_formats, act_formats):
    # deterministic stand-in for search_layer: depends on the layer, the weight format and the act format
    base = float(weight.sum())
    row = [base + 10.0 * len(wf) + sum(ord(c) for c in wf) * 0.01 + ai + float(activations[0].sum()) for wf in weight_formats
           for ai, _ in enumerate(act_formats)]
    return torch.tensor(row, dtype=torch.float64).view(len(weight_formats), len(act_formats))


def _make_layers():
    g = torch.Generator().manual_seed(0)
    return [{"name": f"blk{i}", "weight": torch.randn(4, 4, generator=g), "activations": [torch.randn(2, 4, generator=g)]} for i in range(5)]


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fpqvar_b200 import search
    res = search.search_layers(_make_layers(), rank=rank, world=world, layer_fn=_fake_layer_fn)
    if rank == 0:
        torch.save(res, out)
    dist.destroy_process_group()


def test_search_sharding_two_ranks_gloo(tmp_path):
    import socket
    import torch.multiprocessing as mp
    from fpqvar_b200 import search
    want = search.search_layers(_make_layers(), layer_fn=_fake_layer_fn)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "res.pt")
    mp.spawn(_gloo_worker, args=(2, port, out), nprocs=2, join=True)
    got = torch.load(out)
    assert got == want
    assert all(r["weight_format"] in search.FP4_FORMATS for r in got)


# ---------------------------------------------------------------------------------------------
# bench.py reference arm (CPU port) prints the contract's JSON line
# ---------------------------------------------------------------------------------------------
def test_bench_reference_arm_json_contract():
    import json
    import subprocess
    import sys
    env = dict(os.environ, ORACLE_THREADS=str(min(8, os.cpu_count() or 1)))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--workload", "var_d16_w4a4", "--sample-stages", "6"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "GB/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["config"]["workload"] == "var_d16_w4a4"


def test_var_generation_harness_runs_on_cpu_in_fp16_mode():
    """tools/var_generate.py (the images/sec harness, SURVEY.md section 8d): the caller-side model steps through all
    ten scales with a KV cache and produces a finite f_hat of the right shape.  The quantized modes need the GPU
    (tests/test_gpu_dropin.py); here only the unquantized plumbing runs."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("var_generate", os.path.join(ROOT, "tools", "var_generate.py"))
    vg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(vg)
    import torch
    model = vg.Var(2, (1, 2, 3, 4), False).eval()
    model.init_weights(0)
    for b in model.blocks:
        for lin in (b.attn.mat_qkv, b.attn.proj, b.ffn.fc1, b.ffn.fc2, b.ada_lin):
            lin.half()
    f_hat = model.generate(2, torch.tensor([1, 2]), torch.Generator().manual_seed(0))
    assert f_hat.shape == (2, 32, 4, 4) and bool(torch.isfinite(f_hat).all())
    assert model.blocks[0].attn.cur == 1 + 4 + 9 + 16


def test_kv_cache_host_checks_without_a_gpu():
    """fpqvar_b200.kv_cache: argument errors surface before anything touches the device; a CPU tensor reaches the
    quantizer's own 'no CPU fallback' error only when there is history to quantize."""
    import torch
    from fpqvar_b200.kv_cache import IncrementalKVQuant
    from fpqvar_b200._lib import FpqError
    with pytest.raises(NotImplementedError):
        IncrementalKVQuant(8, 16)                                         # basic_var.py:199: only kv_bit 4 and 6 exist
    c = IncrementalKVQuant(6, 16)
    with pytest.raises(ValueError):
        c.append(torch.zeros(1, 2, 2, 64), torch.zeros(1, 2, 2, 64))      # fp32: the cache is fp16 (autocast attention)
    k = torch.zeros(1, 2, 2, 64, dtype=torch.float16)
    kk, vv = c.append(k, k)                                               # first scale: nothing to quantize yet
    assert kk.shape == (1, 2, 2, 64) and c.cur == 2 and c.done == 0 and c.exact
    with pytest.raises(FpqError):
        c.append(k, k)                                                    # history on the CPU: the quantizer refuses
    c4 = IncrementalKVQuant(4, 16)
    with pytest.raises(ValueError):
        c4.append(torch.zeros(1, 2, 3, 64, dtype=torch.float16), torch.zeros(1, 2, 3, 64, dtype=torch.float16))


def test_mixed_datatype_variants_issue_the_reference_call_sequence(monkeypatch):
    """quantize_VAR_mixed_fp4_datatype / _mixed_fp6_datatype (imported by evaluate_fp_quant.py:18) and
    quantize_VAR_use_different_datatype: the same (module, class, keyword arguments) sequence as the reference's own
    functions on a 30-block model (tests/golden/make_golden_mixed.py recorded them with `from_float` patched out)."""
    import json
    import torch
    from torch import nn
    from fpqvar_b200 import quant_utils as Q
    plans = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_mixed_plans.json")))

    class SelfAttention(nn.Module):
        def __init__(self):
            super().__init__()
            self.mat_qkv, self.proj = nn.Linear(128, 384, bias=False), nn.Linear(128, 128)

    class FFN(nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1, self.fc2 = nn.Linear(128, 128), nn.Linear(128, 128)

    class AdaLNSelfAttn(nn.Module):
        def __init__(self):
            super().__init__()
            self.attn, self.ffn = SelfAttention(), FFN()
            self.ada_lin = nn.Sequential(nn.SiLU(), nn.Linear(128, 768))

    class Model(nn.Module):
        def __init__(self):
            super().__init__()
            self.blocks = nn.ModuleList(AdaLNSelfAttn() for _ in range(30))

    fixture_key = {"quantize_VAR_with_ada_lin": "models_fp_quant_rotate.quantize_VAR", "quantize_VAR": "models_fp_quant_transform_rotate.quantize_VAR"}
    for fn_name in ("quantize_VAR_mixed_fp4_datatype", "quantize_VAR_mixed_fp6_datatype", "quantize_VAR_use_different_datatype",
                    "quantize_VAR_with_ada_lin", "quantize_VAR"):
        model = Model()
        paths = {id(m): n for n, m in model.named_modules()}
        calls = []

        def recorder(cls_name):
            def from_float(module, **kwargs):
                calls.append({"module": paths[id(module)], "class": cls_name, "kwargs": {k: kwargs[k] for k in sorted(kwargs)}})
                return module
            return staticmethod(from_float)

        monkeypatch.setattr(Q.QuantizedLinear, "from_float", recorder("QuantizedLinear"))
        monkeypatch.setattr(Q.QuantizedLinear_fc2, "from_float", recorder("QuantizedLinear_fc2"))
        kw = dict(plans["kwargs"])
        if "fp6" in fn_name:
            kw.update(w_bit=6, a_bit=6, act_fp_type="fp6_e2m3", weight_fp_type="fp6_e2m3", fc2_fp_type="fp6_int_neg_e2m3_pos")
        out = getattr(Q, fn_name)(model, **kw)
        assert out is model
        want = plans[fixture_key.get(fn_name, fn_name)]
        assert len(calls) == len(want) == (120 if fn_name == "quantize_VAR" else 150)
        if fn_name == "quantize_VAR":                          # same calls; this repo's walk visits ffn / attn in registration order too
            key = lambda c: (c["module"],)  # noqa: E731
            assert sorted(calls, key=key) == sorted(want, key=key)
        for got, ref in zip(calls, want):
            assert got == ref, (fn_name, got, ref)


def test_rotation_module_exports_what_the_reference_scripts_use():
    """evaluate_fp_quant_transform_rotate.py calls rotation_utils.cleanup_memory() / get_orthogonal_matrix(...), and
    rotation_utils.py:7 imports apply_exact_had_to_linear / is_pow2 from hadamard_utils: a drop-in must carry the names."""
    import torch
    from fpqvar_b200 import hadamard_utils as H, rotation_utils as R
    from fpqvar_b200._lib import FpqError
    R.cleanup_memory()                                                    # no GPU here: gc only
    q = R.get_orthogonal_matrix(128, "hadamard", "cpu")
    assert torch.equal(q, R.random_hadamard_matrix(128, "cpu", 42))
    assert torch.allclose(q @ q.T, torch.eye(128, dtype=torch.float64), atol=1e-12)
    torch.manual_seed(0)
    r = R.get_orthogonal_matrix(64, "random", "cpu")
    assert r.dtype == torch.float64 and torch.allclose(r @ r.T, torch.eye(64, dtype=torch.float64), atol=1e-10)
    with pytest.raises(ValueError):
        R.get_orthogonal_matrix(64, "givens", "cpu")
    with pytest.raises(FpqError):
        R.get_orthogonal_matrix(1920, "hadamard", "cpu")                  # the K = 60 tables of the full-width rotation: out of scope
    lin = torch.nn.Linear(64, 32, bias=False)
    w0 = lin.weight.data.clone()
    H.apply_exact_had_to_linear(lin)                                       # W @ H_64 / 8
    assert torch.allclose(lin.weight.data.double(), w0.double() @ (R._sylvester(64) / 8.0), atol=1e-6)
    H.apply_exact_had_to_linear(lin)                                       # H is an involution up to the scale: back to W
    assert torch.allclose(lin.weight.data, w0, atol=1e-5)
    lin2 = torch.nn.Linear(16, 64, bias=False)
    w1 = lin2.weight.data.clone()
    H.apply_exact_had_to_linear(lin2, output=True)
    assert torch.allclose(lin2.weight.data.double(), (R._sylvester(64) / 8.0) @ w1.double(), atol=1e-6)
    with pytest.raises(NotImplementedError):
        H.apply_exact_had_to_linear(lin, had_dim=16)


def test_rotate_fc2_and_ada_lin_match_their_regression_snapshot():
    """rotation_utils.rotate_fc2 / rotate_ada_lin / block_diag (defined by the reference, unused by its rotate_model):
    bit-identical to a REGRESSION SNAPSHOT of this project's own output (tests/golden/make_snapshot_rotate.py).  The
    reference's functions are not available to compare with, so this pins the current behaviour, not the reference's."""
    from fpqvar_b200 import rotation_utils as R
    G = np.load(os.path.join(ROOT, "tests", "golden", "snapshot_rotate.npz"))
    layer = torch.nn.Module()
    layer.ffn = torch.nn.Module()
    layer.ffn.fc2 = torch.nn.Linear(64, 16)
    layer.ada_lin = torch.nn.Sequential(torch.nn.SiLU(), torch.nn.Linear(16, 96))
    names = list(layer.state_dict())
    layer.load_state_dict({k: torch.from_numpy(G[f"in/{k}"]) for k in names})
    q64, q16 = torch.from_numpy(G["Q64"]), torch.from_numpy(G["Q16"])
    R.rotate_fc2(layer, q64)
    R.rotate_ada_lin(layer, q16)
    for k, v in layer.state_dict().items():
        assert torch.equal(v, torch.from_numpy(G[f"out/{k}"])), k
    assert torch.equal(R.block_diag([q16, q16]), torch.from_numpy(G["block_diag"]))


def test_bench_b200_arm_refuses_to_run_without_a_gpu():
    """The product arm of bench.py has no CPU path: without a CUDA device it exits with an explicit message instead of
    timing anything (the CPU numbers come only from `--impl reference`)."""
    import subprocess
    import sys
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode != 0
    assert "no CUDA device" in (out.stderr + out.stdout) and "no CPU fallback" in (out.stderr + out.stdout)
    assert not any(line.startswith("{") for line in out.stdout.splitlines())
