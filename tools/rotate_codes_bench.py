"""Fused rotate -> codes against the two ways it replaces, on the B200 (DESIGN.md sections 3.3 / 3.6).

Per VAR-d30 mat_qkv / fc1 call shape of every stage (var_workload: rows = 2 * B * pn^2, C = 1920, the adaLN modulate fused in,
rows_per_batch = pn^2) and per VAR-d36 stage (C = 2304):
  (a) fp16   ops.modulate_transform_rotate_quant(fmt)         the fused fake-quant sibling: 4 B read + 2 B written per element
  (b) codes  lowbit.rotate_pack_codes(fmt, scale, shift)      one launch: 4 + 1 + 4/128 B
  (c) 2-step rotate with fmt=None, then lowbit.pack_codes      (4 + 2) + (2 + 1 + 4/128) B
and the same three without the modulate (`*_plain`: ops.transform_rotate_quant / rotate_pack_codes without scale, shift; the
other streaming instantiation, 96 registers instead of 128),
and, at the largest d30 stage, the whole linear of mat_qkv (N = 5760) and fc1 (N = 7680), K = 1920:
  (b) + linear_codes,  (c) + linear_codes,  (a) + F.linear (the fp16 library GEMM on the fake-quantized tensors).
Kernel time: every variant is captured in a CUDA graph of back-to-back calls (no host time between kernels) and replayed between
CUDA events; the inputs rotate over copies totalling more than 256 MB (twice the 126 MB L2), so every call reads x from HBM.
The three variants are measured interleaved, `--repeats` rounds, median reported.  TB/s is algorithmic: the bytes above (from
the shapes) over kernel time.  Card name and power limit are read in the same run.  Needs a GPU; no fallback.

    python tools/rotate_codes_bench.py --out /tmp/rotate_codes_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from fpqvar_b200 import lowbit, ops  # noqa: E402
from fpqvar_b200.hotpath import seed42_sign_bits  # noqa: E402
from fpqvar_b200.var_workload import WORKLOADS  # noqa: E402

BYTES = {"a_fp16": 4 + 2, "b_codes": 4 + 1 + 4 / 128, "c_two_step": (4 + 2) + (2 + 1 + 4 / 128)}
BYTES.update({k + "_plain": v for k, v in list(BYTES.items())})
L2_BYTES = 126 << 20


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip()}


def graph_of(fn, n_calls):
    """CUDA graph of n_calls back-to-back calls fn(i)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(min(n_calls, 3)):          # warm up (module loads, attributes) outside the capture
            fn(i)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(n_calls):
            fn(i)
    return g


def time_graph(g, n_calls, replays):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    g.replay()
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(replays):
        g.replay()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / (replays * n_calls) * 1e3          # us per call


def bench_shape(rows, C, rpb, fmt, bits, repeats, layer_n=()):
    B = rows // rpb
    n_copies = max(2, -(-2 * L2_BYTES // (rows * C * 4)))
    n_calls = max(n_copies, 16)
    g = torch.Generator(device="cuda").manual_seed(rows + C)
    xs = [torch.randn(B, rpb, C, device="cuda", generator=g) for _ in range(n_copies)]
    scale = torch.randn(B, 1, C, device="cuda", generator=g) * 0.3
    shift = torch.randn(B, 1, C, device="cuda", generator=g) * 0.5
    smooth = torch.exp(torch.rand(C, device="cuda", generator=g) * 2 - 1)

    def a(i):
        return ops.modulate_transform_rotate_quant(xs[i % n_copies], scale, shift, smooth, bits, fmt)

    def b(i):
        return lowbit.rotate_pack_codes(xs[i % n_copies], smooth, bits, fmt, scale, shift)

    def c(i):
        return lowbit.pack_codes(ops.modulate_transform_rotate_quant(xs[i % n_copies], scale, shift, smooth, bits, None), fmt)

    def a_plain(i):
        return ops.transform_rotate_quant(xs[i % n_copies].view(rows, C), smooth, bits, fmt)

    def b_plain(i):
        return lowbit.rotate_pack_codes(xs[i % n_copies].view(rows, C), smooth, bits, fmt)

    def c_plain(i):
        return lowbit.pack_codes(ops.transform_rotate_quant(xs[i % n_copies].view(rows, C), smooth, bits, None), fmt)

    # the three outputs of each entry agree before anything is timed
    for fb, fc, fa in ((b, c, a), (b_plain, c_plain, a_plain)):
        pb, pc = fb(0), fc(0)
        assert torch.equal(pb.codes, pc.codes) and torch.equal(pb.scales, pc.scales)
        assert torch.equal(pb.dequantize().view(torch.int16), fa(0).reshape(rows, C).view(torch.int16))
    variants = {"a_fp16": a, "b_codes": b, "c_two_step": c, "a_fp16_plain": a_plain, "b_codes_plain": b_plain, "c_two_step_plain": c_plain}
    for n in layer_n:
        lin = torch.nn.Linear(C, n).cuda()
        w = lowbit.pack_codes(lin.weight.detach().float().contiguous(), "e2m1")
        w16 = w.dequantize(torch.float16)
        b16 = lin.bias.detach().half()
        variants[f"layer{n}_b_codes_gemm"] = lambda i, w=w, lin=lin: lowbit.linear_codes(b(i), w, lin.bias)
        variants[f"layer{n}_c_two_step_gemm"] = lambda i, w=w, lin=lin: lowbit.linear_codes(c(i), w, lin.bias)
        variants[f"layer{n}_a_fp16_flinear"] = lambda i, w16=w16, b16=b16: F.linear(a(i).view(rows, C), w16, b16)
    graphs = {k: graph_of(f, n_calls) for k, f in variants.items()}
    est_us = max(rows * C * 6 / 6e12 * 1e6, 4.0)                                        # a call: bytes at ~6 TB/s, or a small launch
    replays = max(3, int(2e4 // (est_us * n_calls)))                                    # ~20 ms of kernels per timed window
    samples = {k: [] for k in variants}
    for _ in range(repeats):
        for k, gr in graphs.items():
            samples[k].append(time_graph(gr, n_calls, replays))
    out = {}
    elems = rows * C
    for k, v in samples.items():
        us = statistics.median(v)
        rec = {"us": round(us, 3), "spread_us": [round(min(v), 3), round(max(v), 3)]}
        if k in BYTES:
            rec["tb_s"] = round(elems * BYTES[k] / (us * 1e-6) / 1e12, 3)
            rec["bytes_per_elem"] = round(BYTES[k], 5)
        out[k] = rec
    del graphs
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="JSON file to write (the table is printed either way)")
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "rotate_codes_bench needs a CUDA device"
    bits = seed42_sign_bits()
    res = {"card": card(), "method": "CUDA graph of back-to-back calls, CUDA events, inputs rotated over > 256 MB, "
                                     "median of interleaved repeats", "shapes": []}
    print(json.dumps(res["card"]))
    for wname in ("var_d30_w4a4_rot", "var_d36_w6a6_rot"):
        w = WORKLOADS[wname]
        rows_all = w.stage_rows()
        for si, rows in enumerate(rows_all):
            pn = w.patch_nums[si]
            largest = wname == "var_d30_w4a4_rot" and rows == max(rows_all)
            r = bench_shape(rows, w.width, pn * pn, w.act_fmt, bits, args.repeats, (5760, 7680) if largest else ())
            entry = {"workload": wname, "stage": si, "rows": rows, "C": w.width, "rows_per_batch": pn * pn, "fmt": w.act_fmt, **r}
            res["shapes"].append(entry)
            print(f"{wname} stage {si:2d} rows {rows:6d} C {w.width}: " + "  ".join(
                f"{k} {v['us']:.2f} us" + (f" ({v['tb_s']:.2f} TB/s)" if "tb_s" in v else "") for k, v in r.items()), flush=True)
    res["card_after"] = card()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
