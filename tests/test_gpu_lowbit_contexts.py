"""The low-bit path (fpq_pack_codes, the nibble converters, the fused rotate-to-codes entries, fpq_gemm_codes and
fpq_gemm_codes_sse) in every way a layer loop runs it, not only eagerly on the current stream: captured on a side stream in a
CUDA graph and replayed, with the process's first call of each launcher inside the capture, back to back through buffers the
previous call still owns, from several host threads at once, and on a second device.

Every output is compared with a reference that does not share the code under test: codes, scales, nibbles and dequantized
tensors bit for bit with oracle/lowbit.py; GEMM outputs bit for bit with the fixed-order oracle LB.gemm_codes (e2m1 x e2m1:
inside the exact-accumulation envelope, so the order of the tensor core's sums does not matter); the codes of the fused rotate
entries with their numerics contract (pack_codes of the fp16 rotation the sibling call writes with fmt=None, computed eagerly
beforehand, and LB.pack_codes of its host copy); the fused loss with the float64 sum of (ref - C_oracle)^2 within 2e-6 relative
(its float64 atomicAdds land in no fixed order).  Layers are those of a VAR-d16 block (C = 1024): mat_qkv C -> 3C from the
adaLN-modulated rotate-to-codes entry, proj C -> C from pack_codes (per 128-group and per row), fc1 C -> 4C from rotate-to-codes.
"""
import contextlib
import ctypes
import hashlib
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from oracle import lowbit as LB          # checker only

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C = 1024
FMT = "e2m1"
SSE_RTOL = 2e-6
# rows: one row; 513 = five 128-row tiles, the last one holding a single row (the default launches CTA pairs for row scales)
ROWS = (1, 513)
BATCHES = {1: 1, 513: 3}                 # adaLN batches of the modulated entry (rows per batch = rows / batches)
DEFAULTS = {"pdl": 1, "rot_small_max_chunks": 40000, "smem_kb": 0, "gemm_stages": 6, "gemm_pair": -1, "gemm_tile_n": 256,
            "gemm_epi_cols": 128}
CHILD_TIMEOUT = 300


@pytest.fixture(scope="module")
def mods():
    from fpqvar_b200 import _lib, lowbit, ops
    assert torch.cuda.is_available()
    return ops, lowbit, _lib


@pytest.fixture(scope="module")
def sign_bits():
    from fpqvar_b200.hotpath import seed42_sign_bits
    return seed42_sign_bits()


@contextlib.contextmanager
def tunables(L, **values):
    """Set launch-geometry tunables for the duration of a block; every one is back at its default afterwards."""
    try:
        for k, v in values.items():
            L.set_tunable(k, v)
        yield
    finally:
        for k in values:
            L.set_tunable(k, DEFAULTS[k])


def host(t):
    return t.detach().cpu().numpy()


def assert_bits(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype, f"{what}: {got.shape} {got.dtype} vs {want.shape} {want.dtype}"
    u = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[got.dtype.itemsize]
    bad = int(np.count_nonzero(got.view(u) != want.view(u)))
    assert bad == 0, f"{what}: {bad} of {got.size} elements differ from the oracle"


def assert_sse(got, want, what):
    assert abs(got - want) <= SSE_RTOL * want, f"{what}: {got!r} vs {want!r}"


_GEMM = {}


def gemm_oracle(qa, sa, q_w, bias=None):
    """LB.gemm_codes, memoized on the operands' bytes (the same products recur across launch forms and PDL settings)."""
    qw, sw = q_w
    h = hashlib.sha1()
    for a in (qa, sa, qw, sw) + (() if bias is None else (bias,)):
        h.update(np.ascontiguousarray(a).tobytes())
    key = h.hexdigest()
    if key not in _GEMM:
        _GEMM[key] = LB.gemm_codes(qa, sa, qw, sw, bias)
    return _GEMM[key]


def rotate_contract(ops, lowbit, x, smooth, bits, scale=None, shift=None):
    """The codes a rotate-to-codes call must write: pack_codes of the sibling call's fp16 rotation (fmt=None), which must equal
    LB.pack_codes of its host copy; returns (codes, scales, qa, sa) on the host."""
    if scale is None:
        rot = ops.transform_rotate_quant(x, smooth, bits, None)
    else:
        rot = ops.modulate_transform_rotate_quant(x, scale, shift, smooth, bits, None)
    rot = rot.reshape(-1, x.shape[-1])
    dev = lowbit.pack_codes(rot, FMT)
    r = host(rot)
    codes, scales = LB.pack_codes(r, FMT)
    assert_bits(host(dev.codes), codes, "contract: pack_codes of the rotation")
    assert_bits(host(dev.scales), scales, "contract: scales of the rotation")
    qa, sa = LB.quantize_codes(r, FMT)
    return codes, scales, qa, sa


@pytest.fixture(scope="module")
def weights(mods):
    """mat_qkv, proj and fc1 of a d16 block: fp32 weights packed per 128-group (proj also per row), biases, host codes."""
    _, lowbit, _ = mods
    rng = np.random.default_rng(1234)
    out = {}
    for name, n in (("qkv", 3 * C), ("proj", C), ("fc1", 4 * C)):
        w = (rng.standard_normal((n, C)) / np.sqrt(C)).astype(np.float32)
        b = rng.standard_normal(n).astype(np.float32)
        wd = torch.from_numpy(w).cuda()
        out[name] = dict(w=w, b=b, bd=torch.from_numpy(b).cuda(), p=lowbit.pack_codes(wd, FMT), q=LB.quantize_codes(w, FMT))
        if name == "proj":
            out["proj_row"] = dict(p=lowbit.pack_codes(wd, FMT, per_row=True), q=LB.quantize_codes(w, FMT, None))
    torch.cuda.synchronize()
    return out


def block(lowbit, w, inp, bits, sse_zeroed, sse_acc):
    """One d16 block's low-bit calls in layer order; `sse_zeroed` is cleared in the sequence, `sse_acc` is not."""
    o = {}
    a = lowbit.rotate_pack_codes(inp["x"], inp["smooth"], bits, FMT, inp["scale"], inp["shift"])
    o["qkv_codes"], o["qkv_scales"] = a.codes, a.scales
    o["qkv"] = lowbit.linear_codes(a, w["qkv"]["p"], w["qkv"]["bd"], torch.float16)          # fp16 out, bias
    h = o["qkv"][:, :C]                                                                       # a column slice: pack_codes copies it
    p = lowbit.pack_codes(h, FMT)
    o["proj_codes"], o["proj_scales"] = p.codes, p.scales
    o["nibbles"] = p.to_nibbles()
    back = lowbit.PackedCodes.from_nibbles(o["nibbles"], p.scales, p.rows, C, FMT)
    o["back_codes"] = back.codes
    o["dequant"] = back.dequantize(torch.float16)
    o["proj"] = lowbit.linear_codes(back, w["proj"]["p"], None, torch.float32)                # fp32 out, no bias
    r = lowbit.pack_codes(h, FMT, per_row=True)
    o["row_codes"], o["row_scales"] = r.codes, r.scales
    o["proj_row"] = lowbit.linear_codes(r, w["proj_row"]["p"], w["proj"]["bd"], torch.float32)  # row scales, fp32 out, bias
    sse_zeroed.zero_()
    lowbit.linear_codes_sse(back, w["proj"]["p"], inp["ref"], w["proj"]["bd"], sse_zeroed)
    lowbit.linear_codes_sse(back, w["proj"]["p"], inp["ref"], w["proj"]["bd"], sse_acc)
    f = lowbit.rotate_pack_codes(inp["x2"], inp["smooth2"], bits, FMT)
    o["fc1_codes"], o["fc1_scales"] = f.codes, f.scales
    o["fc1"] = lowbit.linear_codes(f, w["fc1"]["p"], None, torch.float16)                     # fp16 out, no bias
    return o


_BLOCKS = {}


def block_case(mods, weights, bits, rows):
    """Inputs of one block and the oracle of every output (computed once per row count)."""
    if rows in _BLOCKS:
        return _BLOCKS[rows]
    ops, lowbit, _ = mods
    g = torch.Generator(device="cuda").manual_seed(rows)
    nb = BATCHES[rows]
    inp = dict(x=torch.randn(nb, rows // nb, C, device="cuda", generator=g),
               scale=torch.randn(nb, 1, C, device="cuda", generator=g) * 0.3,
               shift=torch.randn(nb, 1, C, device="cuda", generator=g) * 0.5,
               smooth=torch.exp(torch.rand(C, device="cuda", generator=g) - 0.5),
               x2=torch.randn(rows, C, device="cuda", generator=g),
               smooth2=torch.exp(torch.rand(C, device="cuda", generator=g) - 0.5),
               ref=torch.randn(rows, C, device="cuda", generator=g))
    want = {}
    want["qkv_codes"], want["qkv_scales"], qa, sa = rotate_contract(ops, lowbit, inp["x"], inp["smooth"], bits, inp["scale"], inp["shift"])
    want["qkv"] = gemm_oracle(qa, sa, weights["qkv"]["q"], weights["qkv"]["b"]).astype(np.float16)
    h = np.ascontiguousarray(want["qkv"][:, :C])
    want["proj_codes"], want["proj_scales"] = LB.pack_codes(h, FMT)
    qh, sh = LB.quantize_codes(h, FMT)
    want["nibbles"] = LB.codes_to_nibbles(want["proj_codes"], FMT)
    want["back_codes"] = want["proj_codes"]
    want["dequant"] = LB.dequantize(qh, sh, np.float16)
    want["proj"] = gemm_oracle(qh, sh, weights["proj"]["q"])
    want["row_codes"], want["row_scales"] = LB.pack_codes(h, FMT, None)
    qr, sr = LB.quantize_codes(h, FMT, None)
    want["proj_row"] = gemm_oracle(qr, sr, weights["proj_row"]["q"], weights["proj"]["b"])
    c = gemm_oracle(qh, sh, weights["proj"]["q"], weights["proj"]["b"])
    want["sse"] = float(((host(inp["ref"]).astype(np.float64) - c.astype(np.float64)) ** 2).sum())
    want["fc1_codes"], want["fc1_scales"], qf, sf = rotate_contract(ops, lowbit, inp["x2"], inp["smooth2"], bits)
    want["fc1"] = gemm_oracle(qf, sf, weights["fc1"]["q"]).astype(np.float16)
    torch.cuda.synchronize()
    _BLOCKS[rows] = (inp, want)
    return inp, want


def check_block(o, want, what):
    for k, v in o.items():
        assert_bits(host(v), want[k], f"{what}: {k}")


FORMS = {"default": {}, "pair": {"gemm_pair": 1}, "single_cta": {"gemm_pair": 0}, "tile_n_128": {"gemm_tile_n": 128},
         "streaming_rotate": {"rot_small_max_chunks": 0}}


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("rows", ROWS)
def test_block_on_a_side_stream_and_in_graph_replay(mods, weights, sign_bits, rows, form):
    """The whole block captured on a side stream and replayed twice (outputs poisoned before each): every output equals the
    oracle after each replay.  The loss: with its zeroing captured, each replay gives the eager value; the accumulator zeroed
    once before the capture holds twice that after two replays.  Then the block eagerly on the side stream."""
    ops, lowbit, L = mods
    inp, want = block_case(mods, weights, sign_bits, rows)
    s = torch.cuda.Stream()
    with tunables(L, **FORMS[form]):
        sse_z = torch.zeros(1, dtype=torch.float64, device="cuda")
        sse_acc = torch.zeros(1, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            o = block(lowbit, weights, inp, sign_bits, sse_z, sse_acc)
        for replay in (1, 2):
            for v in o.values():                               # whatever the replay leaves unwritten differs from the oracle
                v.view(torch.uint8).fill_(0xFF)
            torch.cuda.synchronize()
            with torch.cuda.stream(s):
                g.replay()
            s.synchronize()
            check_block(o, want, f"{form}, replay {replay}")
            assert_sse(sse_z.item(), want["sse"], f"{form}: loss with its zeroing captured, replay {replay}")
            assert_sse(sse_acc.item(), replay * want["sse"], f"{form}: accumulated loss after {replay} replays")
        del g
        ez = torch.zeros(1, dtype=torch.float64, device="cuda")
        ea = torch.zeros(1, dtype=torch.float64, device="cuda")
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            e = block(lowbit, weights, inp, sign_bits, ez, ea)
        s.synchronize()
    check_block(e, want, f"{form}, eager on a side stream")
    assert_sse(ez.item(), want["sse"], f"{form}: eager loss")
    assert_sse(ea.item(), want["sse"], f"{form}: eager loss into a zeroed accumulator")


def run_child(code, *args):
    """Runs `code` in a fresh interpreter (nothing of it outlives the call: it is killed at the timeout)."""
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", textwrap.dedent(code), ROOT, *map(str, args)]
    try:
        r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=CHILD_TIMEOUT)
    except subprocess.TimeoutExpired:
        pytest.fail(f"child process did not finish within {CHILD_TIMEOUT} s")
    assert r.returncode == 0, f"child process failed ({r.returncode}):\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}"
    return r.stdout


# The child of the first-call test: no kernel of the library has run when the capture starts; inside it, the first call of the
# streaming rotate kernel (under a shared-memory carveout), of the pack kernels, of the single-CTA GEMM with 128- and 256-column
# tiles, of the pair GEMM and of the pair SSE GEMM.
CHILD_FIRST_CALLS = """
    import sys
    import numpy as np
    import torch
    root, src, dst = sys.argv[1:4]
    sys.path.insert(0, root)
    from fpqvar_b200 import _lib as L, lowbit, ops
    from fpqvar_b200.hotpath import seed42_sign_bits

    d = np.load(src)
    t = {k: torch.from_numpy(d[k]).cuda() for k in d.files}
    bits = seed42_sign_bits()
    ops._ext()
    lib = L.lib()
    assert lib.fpq_launch_count() == 0
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    try:
        L.set_tunable("smem_kb", 100)
        L.set_tunable("rot_small_max_chunks", 0)
        with torch.cuda.graph(g, stream=s):
            a = lowbit.rotate_pack_codes(t["x"], t["smooth"], bits, "e2m1")
            w = lowbit.pack_codes(t["w"], "e2m1")
            ar = lowbit.pack_codes(t["h"], "e2m1", per_row=True)
            wr = lowbit.pack_codes(t["w"], "e2m1", per_row=True)
            L.set_tunable("gemm_tile_n", 128)
            c128 = lowbit.linear_codes(a, w, t["b"], torch.float32)
            L.set_tunable("gemm_tile_n", 256)
            c256 = lowbit.linear_codes(a, w, None, torch.float16)
            cpair = lowbit.linear_codes(ar, wr, t["b"], torch.float16)
            sse = torch.zeros(1, dtype=torch.float64, device="cuda")
            lowbit.linear_codes_sse(ar, wr, t["ref"], t["b"], sse)
    finally:
        for k, v in (("smem_kb", 0), ("rot_small_max_chunks", 40000), ("gemm_tile_n", 256)):
            L.set_tunable(k, v)
    assert lib.fpq_launch_count() == 8, lib.fpq_launch_count()
    out = {}
    for replay in range(2):
        with torch.cuda.stream(s):
            g.replay()
        s.synchronize()
        out.update({f"{k}{replay}": v.cpu().numpy() for k, v in (("codes", a.codes), ("scales", a.scales), ("c128", c128),
                                                                  ("c256", c256), ("cpair", cpair), ("sse", sse))})
    np.savez(dst, **out)
"""


def test_first_call_of_every_launcher_inside_a_capture(mods, sign_bits, tmp_path):
    """The one-time setup of the launchers (dynamic shared-memory attributes, the cluster occupancy query, the SM count, the
    carveout) runs in a global-mode capture: the capture succeeds and both replays equal the oracle."""
    ops, lowbit, L = mods
    rng = np.random.default_rng(21)
    m = 520                                                   # five row tiles: the default launches CTA pairs for row scales
    d = dict(x=rng.standard_normal((m, C)).astype(np.float32), smooth=np.exp(rng.uniform(-0.5, 0.5, C)).astype(np.float32),
             w=(rng.standard_normal((C, C)) / np.sqrt(C)).astype(np.float32), h=rng.standard_normal((m, C)).astype(np.float16),
             b=rng.standard_normal(C).astype(np.float32), ref=rng.standard_normal((m, C)).astype(np.float32))
    np.savez(tmp_path / "in.npz", **d)
    run_child(CHILD_FIRST_CALLS, tmp_path / "in.npz", tmp_path / "out.npz")
    got = np.load(tmp_path / "out.npz")
    codes, scales, qa, sa = rotate_contract(ops, lowbit, torch.from_numpy(d["x"]).cuda(), torch.from_numpy(d["smooth"]).cuda(), sign_bits)
    qw = LB.quantize_codes(d["w"], FMT)
    qwr = LB.quantize_codes(d["w"], FMT, None)
    qr, sr = LB.quantize_codes(d["h"], FMT, None)
    cpair = gemm_oracle(qr, sr, qwr, d["b"])
    sse = float(((d["ref"].astype(np.float64) - cpair.astype(np.float64)) ** 2).sum())
    for r in range(2):
        assert_bits(got[f"codes{r}"], codes, f"replay {r}: rotate codes")
        assert_bits(got[f"scales{r}"], scales, f"replay {r}: rotate scales")
        assert_bits(got[f"c128{r}"], gemm_oracle(qa, sa, qw, d["b"]), f"replay {r}: 128-column tiles")
        assert_bits(got[f"c256{r}"], gemm_oracle(qa, sa, qw).astype(np.float16), f"replay {r}: 256-column tiles")
        assert_bits(got[f"cpair{r}"], cpair.astype(np.float16), f"replay {r}: CTA pairs")
        assert_sse(float(got[f"sse{r}"][0]), sse, f"replay {r}: fused loss")


CHAIN_ROWS, CHAIN_LAYERS, CHAIN_BATCHES = 264, 12, 2


def _sign_words(bits):
    return (ctypes.c_uint32 * 4)(*[int(b) & 0xFFFFFFFF for b in bits])


def _raw_rotate(L, x, smooth, sb, codes, scales, rows, stream, mod=None):
    if mod is None:
        return L.lib().fpq_transform_rotate_pack_codes(x.data_ptr(), smooth.data_ptr(), sb, codes.data_ptr(), scales.data_ptr(), rows, C,
                                                       L.FMT[FMT], stream)
    return L.lib().fpq_modulate_transform_rotate_pack_codes(x.data_ptr(), mod[0].data_ptr(), mod[1].data_ptr(), rows // CHAIN_BATCHES,
                                                            smooth.data_ptr(), sb, codes.data_ptr(), scales.data_ptr(), rows, C,
                                                            L.FMT[FMT], 0, stream)


def _raw_gemm(L, codes, scales, rows, wp, out, stream, bias=None):
    dt = L.FPQ_F16 if out.dtype == torch.float16 else L.FPQ_F32
    return L.lib().fpq_gemm_codes(codes.data_ptr(), scales.data_ptr(), rows, wp.codes.data_ptr(), wp.scales.data_ptr(), wp.rows, C, 128,
                                  None if bias is None else bias.data_ptr(), dt, out.data_ptr(), wp.rows, stream)


@pytest.mark.parametrize("pdl", [1, 0])
def test_layer_chain_writes_codes_the_previous_gemm_still_reads(mods, weights, sign_bits, pdl):
    """Twelve layers share ONE activation codes / scales pair: each layer's rotate-to-codes call (a PDL launch; plain and
    modulated alternate) overwrites the codes the previous layer's GEMM reads, with nothing in between on the stream."""
    ops, lowbit, L = mods
    rows, wp, bias = CHAIN_ROWS, weights["proj"]["p"], weights["proj"]["bd"]
    g = torch.Generator(device="cuda").manual_seed(77)
    xs = [torch.randn(rows, C, device="cuda", generator=g) for _ in range(CHAIN_LAYERS)]
    mod = (torch.randn(CHAIN_BATCHES, C, device="cuda", generator=g) * 0.3, torch.randn(CHAIN_BATCHES, C, device="cuda", generator=g) * 0.5)
    smooth = torch.exp(torch.rand(C, device="cuda", generator=g) - 0.5)
    want = []
    for i, x in enumerate(xs):                                 # the contract of each layer's codes, eagerly beforehand
        if i % 2:
            x3 = x.view(CHAIN_BATCHES, rows // CHAIN_BATCHES, C)
            _, _, qa, sa = rotate_contract(ops, lowbit, x3, smooth, sign_bits, mod[0].view(CHAIN_BATCHES, 1, C), mod[1].view(CHAIN_BATCHES, 1, C))
        else:
            _, _, qa, sa = rotate_contract(ops, lowbit, x, smooth, sign_bits)
        want.append(gemm_oracle(qa, sa, weights["proj"]["q"], weights["proj"]["b"] if i % 3 == 0 else None))
    rp = LB.rows_padded(rows)
    codes = torch.empty(rp * C, dtype=torch.uint8, device="cuda")
    scales = torch.empty(C // 128, rp, dtype=torch.float32, device="cuda")
    outs = [torch.empty(rows, C, dtype=torch.float16 if i % 2 else torch.float32, device="cuda") for i in range(CHAIN_LAYERS)]
    sb = _sign_words(sign_bits)
    stream = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    with tunables(L, pdl=pdl):
        for i in range(CHAIN_LAYERS):
            assert _raw_rotate(L, xs[i], smooth, sb, codes, scales, rows, stream, mod if i % 2 else None) == 0
            assert _raw_gemm(L, codes, scales, rows, wp, outs[i], stream, bias if i % 3 == 0 else None) == 0
        torch.cuda.synchronize()
    for i in range(CHAIN_LAYERS):
        w = want[i].astype(np.float16) if i % 2 else want[i]
        assert_bits(host(outs[i]), w, f"pdl {pdl}, layer {i}")


@pytest.mark.parametrize("pdl", [1, 0])
def test_layer_chain_packs_the_previous_gemm_output(mods, weights, sign_bits, pdl):
    """Each layer's output is the next layer's input: an fp32 output goes through rotate-to-codes (PDL), an fp16 output through
    pack_codes (plain launch), into one shared codes / scales pair; every layer's output equals the oracle of its own input."""
    ops, lowbit, L = mods
    rows, wp = CHAIN_ROWS, weights["proj"]["p"]
    g = torch.Generator(device="cuda").manual_seed(78)
    h0 = torch.randn(rows, C, device="cuda", generator=g).half()
    smooth = torch.exp(torch.rand(C, device="cuda", generator=g) - 0.5)
    rp = LB.rows_padded(rows)
    codes = torch.empty(rp * C, dtype=torch.uint8, device="cuda")
    scales = torch.empty(C // 128, rp, dtype=torch.float32, device="cuda")
    # layer i reads an fp16 input when i is even (pack_codes) and writes fp32; odd layers rotate that fp32 output and write fp16
    outs = [torch.empty(rows, C, dtype=torch.float32 if i % 2 == 0 else torch.float16, device="cuda") for i in range(CHAIN_LAYERS)]
    ins = [h0] + outs[:-1]
    sb = _sign_words(sign_bits)
    stream = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    with tunables(L, pdl=pdl):
        for i in range(CHAIN_LAYERS):
            if i % 2 == 0:
                rc = L.lib().fpq_pack_codes(ins[i].data_ptr(), rows, C, 128, L.FPQ_F16, L.FMT[FMT], codes.data_ptr(), scales.data_ptr(), stream)
            else:
                rc = _raw_rotate(L, ins[i], smooth, sb, codes, scales, rows, stream)
            assert rc == 0
            assert _raw_gemm(L, codes, scales, rows, wp, outs[i], stream) == 0
        torch.cuda.synchronize()
    for i in range(CHAIN_LAYERS):
        if i % 2 == 0:
            qa, sa = LB.quantize_codes(host(ins[i]), FMT)
        else:
            _, _, qa, sa = rotate_contract(ops, lowbit, ins[i], smooth, sign_bits)
        w = gemm_oracle(qa, sa, weights["proj"]["q"])
        assert_bits(host(outs[i]), w if i % 2 == 0 else w.astype(np.float16), f"pdl {pdl}, layer {i}")


# The child of the thread test: four threads make their first calls of the pair GEMM (row scales), the group GEMM, the SSE GEMM
# and the streaming rotate-to-codes kernel at once, each on its own stream, then 20 more rounds; every call returns FPQ_OK and
# adds exactly one to the thread's launch count; every result equals the serial one, which goes to the parent for the oracle.
CHILD_THREADS = """
    import ctypes
    import sys
    import threading
    import numpy as np
    import torch
    root, src, dst = sys.argv[1:4]
    sys.path.insert(0, root)
    from fpqvar_b200 import _lib as L, lowbit
    from fpqvar_b200.hotpath import seed42_sign_bits

    d = np.load(src)
    n_threads, rounds, C = 4, 21, d["w"].shape[1]
    lib = L.lib()
    w = lowbit.pack_codes(torch.from_numpy(d["w"]).cuda(), "e2m1")
    wr = lowbit.pack_codes(torch.from_numpy(d["w"]).cuda(), "e2m1", per_row=True)
    b = torch.from_numpy(d["b"]).cuda()
    smooth = torch.from_numpy(d["smooth"]).cuda()
    xs = [torch.from_numpy(d[f"x{t}"]).cuda() for t in range(n_threads)]
    refs = [torch.from_numpy(d[f"ref{t}"]).cuda() for t in range(n_threads)]
    a = [lowbit.pack_codes(torch.from_numpy(d[f"h{t}"]).cuda(), "e2m1") for t in range(n_threads)]
    ar = [lowbit.pack_codes(torch.from_numpy(d[f"h{t}"]).cuda(), "e2m1", per_row=True) for t in range(n_threads)]
    m = a[0].rows
    sb = (ctypes.c_uint32 * 4)(*[int(v) & 0xFFFFFFFF for v in seed42_sign_bits()])

    def buffers():
        return dict(pair=torch.empty(m, C, dtype=torch.float16, device="cuda"), group=torch.empty(m, C, dtype=torch.float32, device="cuda"),
                    sse=torch.zeros(1, dtype=torch.float64, device="cuda"), codes=torch.empty(a[0].codes.numel(), dtype=torch.uint8, device="cuda"),
                    scales=torch.empty_like(a[0].scales))

    def calls(t, o, st):
        p, q = ar[t], a[t]
        yield "pair", lambda: lib.fpq_gemm_codes(p.codes.data_ptr(), p.scales.data_ptr(), m, wr.codes.data_ptr(), wr.scales.data_ptr(), C, C,
                                                 C, b.data_ptr(), L.FPQ_F16, o["pair"].data_ptr(), C, st)
        yield "group", lambda: lib.fpq_gemm_codes(q.codes.data_ptr(), q.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), C, C,
                                                  128, None, L.FPQ_F32, o["group"].data_ptr(), C, st)
        yield "sse", lambda: lib.fpq_gemm_codes_sse(q.codes.data_ptr(), q.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), C, C,
                                                    128, b.data_ptr(), L.FPQ_F32, refs[t].data_ptr(), C, None, o["sse"].data_ptr(), st)
        yield "rotate", lambda: lib.fpq_transform_rotate_pack_codes(xs[t].data_ptr(), smooth.data_ptr(), sb, o["codes"].data_ptr(),
                                                                    o["scales"].data_ptr(), m, C, L.FMT["e2m1"], st)

    L.set_tunable("rot_small_max_chunks", 0)
    try:
        bufs = [[buffers() for _ in range(rounds)] for _ in range(n_threads)]
        torch.cuda.synchronize()
        barrier = threading.Barrier(n_threads)
        errors = []

        def worker(t):
            try:
                s = torch.cuda.Stream()
                barrier.wait()
                for r in range(rounds):
                    for name, call in calls(t, bufs[t][r], s.cuda_stream):
                        n0 = lib.fpq_launch_count()
                        rc = call()
                        n = lib.fpq_launch_count() - n0
                        if rc != 0 or n != 1:
                            errors.append(f"thread {t}, round {r}, {name}: rc {rc} ({lib.fpq_last_cuda_error().decode()}), {n} launches")
                s.synchronize()
            except Exception as e:
                errors.append(f"thread {t}: {type(e).__name__}: {e}")

        threads = [threading.Thread(target=worker, args=(t,)) for t in range(n_threads)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        assert not errors, errors
        serial = [buffers() for _ in range(n_threads)]
        st = torch.cuda.current_stream().cuda_stream
        for t in range(n_threads):
            for name, call in calls(t, serial[t], st):
                assert call() == 0, name
        torch.cuda.synchronize()
    finally:
        L.set_tunable("rot_small_max_chunks", 40000)
    for t in range(n_threads):
        for r in range(rounds):
            for k in ("pair", "group", "codes", "scales"):
                assert torch.equal(bufs[t][r][k].view(torch.uint8), serial[t][k].view(torch.uint8)), (t, r, k)
            got, want = bufs[t][r]["sse"].item(), serial[t]["sse"].item()
            assert abs(got - want) <= 4e-6 * want, (t, r, got, want)
    np.savez(dst, **{f"{k}{t}": v.cpu().numpy() for t in range(n_threads) for k, v in serial[t].items()})
"""


def test_first_calls_from_concurrent_host_threads(mods, sign_bits, tmp_path):
    """Guards the one-time setup of the GEMM and rotate launchers against concurrent first calls (the cluster count of the pair
    path is published in one atomic after its attribute is set): a race cannot be provoked at will, so this pins the behaviour
    rather than proving the absence of one."""
    ops, lowbit, L = mods
    rng = np.random.default_rng(31)
    m, n_threads = 520, 4
    d = dict(w=(rng.standard_normal((C, C)) / np.sqrt(C)).astype(np.float32), b=rng.standard_normal(C).astype(np.float32),
             smooth=np.exp(rng.uniform(-0.5, 0.5, C)).astype(np.float32))
    for t in range(n_threads):
        d[f"x{t}"] = rng.standard_normal((m, C)).astype(np.float32)
        d[f"h{t}"] = rng.standard_normal((m, C)).astype(np.float16)
        d[f"ref{t}"] = rng.standard_normal((m, C)).astype(np.float32)
    np.savez(tmp_path / "in.npz", **d)
    run_child(CHILD_THREADS, tmp_path / "in.npz", tmp_path / "out.npz")
    got = np.load(tmp_path / "out.npz")
    qw, qwr = LB.quantize_codes(d["w"], FMT), LB.quantize_codes(d["w"], FMT, None)
    for t in range(n_threads):
        qr, sr = LB.quantize_codes(d[f"h{t}"], FMT, None)
        qa, sa = LB.quantize_codes(d[f"h{t}"], FMT)
        assert_bits(got[f"pair{t}"], gemm_oracle(qr, sr, qwr, d["b"]).astype(np.float16), f"thread {t}: pair GEMM")
        assert_bits(got[f"group{t}"], gemm_oracle(qa, sa, qw), f"thread {t}: group GEMM")
        c = gemm_oracle(qa, sa, qw, d["b"])
        assert_sse(float(got[f"sse{t}"][0]), float(((d[f"ref{t}"].astype(np.float64) - c) ** 2).sum()), f"thread {t}: fused loss")
        codes, scales, _, _ = rotate_contract(ops, lowbit, torch.from_numpy(d[f"x{t}"]).cuda(), torch.from_numpy(d["smooth"]).cuda(), sign_bits)
        assert_bits(got[f"codes{t}"], codes, f"thread {t}: rotate codes")
        assert_bits(got[f"scales{t}"], scales, f"thread {t}: rotate scales")


# The child of the two-device test: with cuda:0 current, the process's first GEMM calls (group, pair, SSE) and a streaming
# rotate-to-codes call take operands on cuda:1, then the same on cuda:0.
CHILD_TWO_DEVICES = """
    import sys
    import numpy as np
    import torch
    root, src, dst = sys.argv[1:4]
    sys.path.insert(0, root)
    from fpqvar_b200 import _lib as L, lowbit
    from fpqvar_b200.hotpath import seed42_sign_bits

    d = np.load(src)
    torch.cuda.set_device(0)
    out = {}
    L.set_tunable("rot_small_max_chunks", 0)
    try:
        for dev in (1, 0):
            t = {k: torch.from_numpy(v).to(f"cuda:{dev}") for k, v in d.items()}
            a, w = lowbit.pack_codes(t["h"], "e2m1"), lowbit.pack_codes(t["w"], "e2m1")
            ar, wr = lowbit.pack_codes(t["h"], "e2m1", per_row=True), lowbit.pack_codes(t["w"], "e2m1", per_row=True)
            out[f"group{dev}"] = lowbit.linear_codes(a, w, None, torch.float32)
            out[f"pair{dev}"] = lowbit.linear_codes(ar, wr, t["b"], torch.float16)
            out[f"sse{dev}"] = lowbit.linear_codes_sse(a, w, t["ref"], t["b"])
            r = lowbit.rotate_pack_codes(t["x"], t["smooth"], seed42_sign_bits(), "e2m1")
            out[f"codes{dev}"], out[f"scales{dev}"] = r.codes, r.scales
            assert torch.cuda.current_device() == 0
            torch.cuda.synchronize(dev)
    finally:
        L.set_tunable("rot_small_max_chunks", 40000)
    assert torch.cuda.current_device() == 0
    np.savez(dst, **{k: v.cpu().numpy() for k, v in out.items()})
"""


def test_second_device_first(mods, sign_bits, tmp_path):
    """The launchers' per-device caches and the SM count follow the operands' device, not the current one."""
    ops, lowbit, L = mods
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    rng = np.random.default_rng(41)
    m = 520
    d = dict(w=(rng.standard_normal((C, C)) / np.sqrt(C)).astype(np.float32), b=rng.standard_normal(C).astype(np.float32),
             h=rng.standard_normal((m, C)).astype(np.float16), ref=rng.standard_normal((m, C)).astype(np.float32),
             x=rng.standard_normal((m, C)).astype(np.float32), smooth=np.exp(rng.uniform(-0.5, 0.5, C)).astype(np.float32))
    np.savez(tmp_path / "in.npz", **d)
    run_child(CHILD_TWO_DEVICES, tmp_path / "in.npz", tmp_path / "out.npz")
    got = np.load(tmp_path / "out.npz")
    qa, sa = LB.quantize_codes(d["h"], FMT)
    qr, sr = LB.quantize_codes(d["h"], FMT, None)
    qw, qwr = LB.quantize_codes(d["w"], FMT), LB.quantize_codes(d["w"], FMT, None)
    c = gemm_oracle(qa, sa, qw, d["b"])
    sse = float(((d["ref"].astype(np.float64) - c) ** 2).sum())
    codes, scales, _, _ = rotate_contract(ops, lowbit, torch.from_numpy(d["x"]).cuda(), torch.from_numpy(d["smooth"]).cuda(), sign_bits)
    for dev in (1, 0):
        assert_bits(got[f"group{dev}"], gemm_oracle(qa, sa, qw), f"cuda:{dev}: group GEMM")
        assert_bits(got[f"pair{dev}"], gemm_oracle(qr, sr, qwr, d["b"]).astype(np.float16), f"cuda:{dev}: pair GEMM")
        assert_sse(float(got[f"sse{dev}"][0]), sse, f"cuda:{dev}: fused loss")
        assert_bits(got[f"codes{dev}"], codes, f"cuda:{dev}: rotate codes")
        assert_bits(got[f"scales{dev}"], scales, f"cuda:{dev}: rotate scales")
