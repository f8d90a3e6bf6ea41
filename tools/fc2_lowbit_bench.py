"""fc2 of VAR-d30 (k = 7680 -> n = 1920) at the token rows of every stage (2 x 50 images x pn^2, up to 25 600): today's path
against the sign-split codes path, and the fc2 format search from codes against the fake-quant search.

  (a) fake   ops.gelu_fake_quant_signsplit + F.linear fp16 (the library GEMM on the fake-quantized tensors)
  (b) codes  lowbit.gelu_pack_codes + lowbit.linear_codes (split GEMM, depth 2k), also split into its two launches
  (s) sym    lowbit.linear_codes of a symmetric per-group operand of the same shape (reference point, GEMM only)

CUDA events over many launches; the fc1 outputs are rotated over more than the 126 MB of L2, so every launch reads its input
from HBM.  Prints the card and its power limit.  Usage: python tools/fc2_lowbit_bench.py [--out FILE]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fpqvar_b200 import lowbit, ops, search  # noqa: E402

K, N = 7680, 1920
PATCH_NUMS = (1, 2, 3, 4, 5, 6, 8, 10, 13, 16)
BATCH2 = 100                       # 2 x 50 images (classifier-free guidance doubles the batch)
FMT = "e1m2_neg_e2m1_pos"
L2_BYTES = 126 << 20


def card() -> str:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:          # noqa: BLE001
        q = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {e})"
    return q


def timed(fn, n_inputs: int, min_ms: float = 150.0) -> float:
    """mean ms per call of fn(i) over rotating inputs i, after a warm-up, the window at least min_ms long"""
    for i in range(n_inputs):
        fn(i)
    torch.cuda.synchronize()
    reps = n_inputs
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            fn(i % n_inputs)
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= min_ms or reps >= 4096:
            return ms / reps
        reps = min(4096, max(reps * 2, int(reps * min_ms / max(ms, 1e-3)) + 1))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)

    torch.manual_seed(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    log(f"card: {card()}")
    log(f"fc2 of VAR-d30: [rows, {K}] fp16 fc1 output -> GELU(tanh) -> sign-split {FMT} act x e2m1 weight (groups of 128) -> [rows, {N}] fp16")
    log("times: ms per call, CUDA events, inputs rotated over > 126 MB (L2)")
    lin_w = torch.randn(N, K, device="cuda") * 0.02
    wq16 = ops.fake_quant(lin_w, "e2m1", 128, "kernel").half()
    w_codes = lowbit.pack_codes(lin_w, "e2m1")
    log()
    log(f"{'rows':>6} {'(a) fake':>9} {'(b) codes':>10} {'b: pack':>8} {'b: gemm':>8} {'(s) sym gemm':>12} {'b/a':>6} "
        f"{'gemm TFLOP/s b / s':>19} {'max|b-a|/max|a|':>16}")
    for pn in PATCH_NUMS:
        rows = BATCH2 * pn * pn
        n_in = max(2, min(64, -(-3 * L2_BYTES // (rows * K * 2))))
        hs = [torch.randn(rows, K, device="cuda", dtype=torch.float16) for _ in range(n_in)]
        packed = [lowbit.gelu_pack_codes(h, FMT) for h in hs]
        sym = [lowbit.pack_codes(torch.nn.functional.gelu(h, approximate="tanh"), "e2m1") for h in hs]
        out = torch.empty(rows, N, device="cuda", dtype=torch.float16)
        t_a = timed(lambda i: torch.nn.functional.linear(ops.gelu_fake_quant_signsplit(hs[i], FMT, global_clip=True), wq16), n_in)
        t_b = timed(lambda i: lowbit.linear_codes(lowbit.gelu_pack_codes(hs[i], FMT), w_codes, None, torch.float16, out), n_in)
        t_pack = timed(lambda i: lowbit.gelu_pack_codes(hs[i], FMT), n_in)
        t_gemm = timed(lambda i: lowbit.linear_codes(packed[i], w_codes, None, torch.float16, out), n_in)
        t_sym = timed(lambda i: lowbit.linear_codes(sym[i], w_codes, None, torch.float16, out), n_in)
        ya = torch.nn.functional.linear(ops.gelu_fake_quant_signsplit(hs[0], FMT, global_clip=True), wq16).float()
        yb = lowbit.linear_codes(packed[0], w_codes, None, torch.float16).float()
        err = ((yb - ya).abs().max() / ya.abs().max()).item()
        flop = 2.0 * rows * N * K
        log(f"{rows:>6} {t_a:>9.4f} {t_b:>10.4f} {t_pack:>8.4f} {t_gemm:>8.4f} {t_sym:>12.4f} {t_b / t_a:>6.2f} "
            f"{flop / t_gemm * 1e-9:>9.0f} / {flop / t_sym * 1e-9:<7.0f} {err:>16.2e}")
        del hs, packed, sym
        torch.cuda.empty_cache()

    # the fc2 format search: one calibration set of every stage ([2, pn^2, 7680] per stage), three weight formats,
    # the two sign-split activation candidates with a codes form
    log()
    acts = [torch.nn.functional.gelu(torch.randn(2, pn * pn, K, device="cuda"), approximate="tanh").half() for pn in PATCH_NUMS]
    w16 = lin_w.half()
    wf, af = ["e2m1", "e1m2", "e3m0"], ["e1m2_neg_e2m1_pos", "afpq_e2m1"]
    rows_total = sum(a.numel() // K for a in acts)
    for name, fn in (("search_layer_batched (fake-quant + fp16 library GEMMs)", search.search_layer_batched),
                     ("search_layer_lowbit  (codes + fused-loss split GEMM)  ", search.search_layer_lowbit)):
        fn(w16, acts, wf, af, "group")
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        a.record()
        for _ in range(reps):
            table = fn(w16, acts, wf, af, "group")
        b.record()
        b.synchronize()
        log(f"fc2 search, {len(wf)} weight x {len(af)} split act formats, {rows_total} calibration rows: {name} "
            f"{a.elapsed_time(b) / reps:8.3f} ms   winner {search.best_formats(table, wf, af)}")
    text = "\n".join(lines) + "\n"
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
