"""Format search (search/search_fp4_format.py, search/search_fp6_format.py) on the B200 kernels.

Two scoring levels, as in the reference:
  * tensor level  mean((x - x_q)^2) per candidate format (compute_quant_error, search_fp4_format.py:472-476,
    loops :840-893) -- `score_tensor_formats`: ONE kernel reads x once and scores every candidate.
  * output level  mean((x W^T - x_q W_q^T)^2) over the calibration activations per (weight format,
    activation format) pair (loop :781-836) -- `search_layer`: fused quantizers + library GEMMs; y_fp is
    computed once per activation instead of once per pair; `search_layer_batched`: the whole calibration
    set of a layer as one row-stacked matrix (large GEMMs, a handful of quantizer launches).
Candidates are independent, so `search_layers` shards (layer, weight-format) units over ranks and
gathers the small loss table at the end (SURVEY.md section 8e) -- the only collective.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch

from . import ops
from .var_workload import shard_units

FP4_FORMATS = ("e1m2", "e2m1", "e3m0")                       # search_fp4_format.py:797
FP6_FORMATS = ("e2m3", "e3m2")                               # search_fp6_format.py
_SPLIT = ("e1m2_neg_e2m1_pos", "int_neg_e2m3_pos", "afpq_e2m1")


def fp4_quant(x, format):
    """search_fp4_format.py:544-553."""
    if format not in FP4_FORMATS:
        raise NotImplementedError
    return ops.fake_quant(x, format, 128, "kernel")


def fp6_quant(x, format):
    """search_fp6_format.py:547-554 (per-token, always fp16)."""
    if format not in FP6_FORMATS:
        raise NotImplementedError
    return ops.fake_quant(x, format, None, "kernel", out_dtype=torch.float16)


def quantize(x, fmt: str, per: str = "group"):
    if fmt in _SPLIT:
        return ops.fake_quant_signsplit(x, fmt, 128 if per == "group" else None, "kernel")
    out_dtype = torch.float16 if fmt in FP6_FORMATS else None
    return ops.fake_quant(x, fmt, 128 if per == "group" else None, "kernel", out_dtype=out_dtype)


class FPQuant(torch.autograd.Function):
    """search_fp4_format.py:340-374 (also the GALT trainers): whole-tensor clip, per-group absmax scale, argmin
    rounding onto e1m2 / e2m1 / e3m0, straight-through gradient."""

    @staticmethod
    def forward(ctx, x, n_bits=4, group_size=128, format=None, clipping_strength=1.0):
        assert n_bits == 4
        if format not in FP4_FORMATS:
            raise ValueError("Unsupported format type")
        clip_value = clipping_strength * x.abs().max()                     # identity at 1.0 for finite data; NaN poisons, as in the reference
        x = torch.clamp(x, -clip_value, clip_value)
        return ops.fake_quant(x, format, group_size, "argmin")

    @staticmethod
    def backward(ctx, grad_output):
        return grad_output.clone(), None, None, None, None


class FPQuant_e1m2_neg_e2m1_pos(torch.autograd.Function):
    """search_fp4_format.py:378-422: the sign-split fc2 format with argmin rounding, straight-through gradient."""

    @staticmethod
    def forward(ctx, x, n_bits=4, group_size=128, clipping_strength=1.0):
        assert n_bits == 4
        if clipping_strength != 1.0:
            clip_value = clipping_strength * x.abs().max()
            x = torch.clamp(x, -clip_value, clip_value)
        return ops.fake_quant_signsplit(x, "e1m2_neg_e2m1_pos", group_size, "argmin", global_clip=True)

    @staticmethod
    def backward(ctx, grad_output):
        return grad_output.clone(), None, None, None


def compute_quant_error(x_fp, x_quant):
    """search_fp4_format.py:472-476."""
    return torch.mean((x_fp - x_quant) ** 2)


def score_tensor_formats(x: torch.Tensor, formats: Sequence[str], tie: str = "kernel") -> torch.Tensor:
    """mean((x - fake_quant(x, f))^2) for every f in `formats`, x read once; float64 [len(formats)]."""
    return ops.score_formats(x, list(formats), tie) / x.numel()


def search_layer(weight: torch.Tensor, activations: Sequence[torch.Tensor], weight_formats: Sequence[str] = FP4_FORMATS,
                 act_formats: Sequence[str] = FP4_FORMATS, per: str = "group") -> torch.Tensor:
    """Loss table [len(weight_formats), len(act_formats)] of search_fp4_format.py:798-816:
    loss[w, a] = mean_j mean((x_j W^T - q_a(x_j) q_w(W)^T)^2)."""
    wq = [quantize(weight, wf, per).to(weight.dtype) for wf in weight_formats]
    loss = torch.zeros(len(weight_formats), len(act_formats), dtype=torch.float64, device=weight.device)
    for x in activations:
        y_fp = torch.matmul(x, weight.T)
        for ai, af in enumerate(act_formats):
            xq = quantize(x, af, per).to(x.dtype)
            for wi in range(len(weight_formats)):
                loss[wi, ai] += compute_quant_error(y_fp, torch.matmul(xq, wq[wi].T)).double()
    return loss / max(1, len(activations))


def search_layer_batched(weight: torch.Tensor, activations: Sequence[torch.Tensor], weight_formats: Sequence[str] = FP4_FORMATS,
                         act_formats: Sequence[str] = FP4_FORMATS, per: str = "group", max_rows: int = 32768) -> torch.Tensor:
    """The same loss table as `search_layer`, computed on the calibration set as ONE row-stacked matrix.

    Scales are shared only along the last dim (groups of 128 or whole rows), so quantizing the stacked
    [sum_j rows_j, C_in] matrix gives every row exactly the values it gets inside its own tensor.  The
    reference's 1000 small tensors per layer ([2, pn^2, C_in], search_fp4_format.py:781-836) then cost
    len(act_formats) fused quantizer launches and (1 + W*A) large library GEMMs per `max_rows` slab instead
    of ~25 launch-bound kernels per tensor.  Per-tensor means are recovered with a segment sum of per-row
    squared errors, accumulated in float64:
        loss[w, a] = (1/J) sum_j  SSE_rows(j) / (rows_j * C_out).
    Differs from `search_layer` only in floating-point summation order."""
    if not activations:
        return torch.zeros(len(weight_formats), len(act_formats), dtype=torch.float64, device=weight.device)
    c_in = weight.shape[1]
    flat = [x.reshape(-1, c_in) for x in activations]
    rows = torch.tensor([f.shape[0] for f in flat], device=weight.device)
    X = torch.cat(flat)
    # weight of every row in the final mean: 1 / (rows_j * C_out * J)
    row_w = torch.repeat_interleave(1.0 / (rows.double() * weight.shape[0] * len(flat)), rows)
    wq = [quantize(weight, wf, per).to(weight.dtype) for wf in weight_formats]
    loss = torch.zeros(len(weight_formats), len(act_formats), dtype=torch.float64, device=weight.device)
    for r0 in range(0, X.shape[0], max_rows):
        xs = X[r0:r0 + max_rows]
        ws = row_w[r0:r0 + max_rows]
        y_fp = torch.matmul(xs, weight.T)
        for ai, af in enumerate(act_formats):
            xq = quantize(xs, af, per).to(xs.dtype)
            for wi in range(len(weight_formats)):
                ops.sse_rows(torch.matmul(xq, wq[wi].T), y_fp, ws, out=loss[wi, ai])      # one read of y_q and y_fp, nothing written
    return loss


def search_layer_lowbit(weight: torch.Tensor, activations: Sequence[torch.Tensor], weight_formats: Sequence[str] = FP4_FORMATS,
                        act_formats: Sequence[str] = FP4_FORMATS, per: str = "group", max_rows: int = 65536) -> torch.Tensor:
    """The loss table of `search_layer_batched` with the quantized layer evaluated from codes on the tensor cores and compared
    with y_fp inside the GEMM's epilogue (lowbit.linear_codes_sse: SURVEY.md section 8 f3): every candidate pair costs one
    low-bit GEMM that writes nothing, every activation format one quantizer pass, every weight format one; the only library
    GEMM left is y_fp.  Weight formats are symmetric; activation formats may also be the sign-split formats with a codes form
    (lowbit.SPLIT_FORMATS, per="group": the fc2 search), packed without the whole-tensor clip as `quantize` applies none.
    Rounding is the kernel tie rule of the evaluation path
    (fp_quant_*_per_group_cuda) where the search scripts' FPQuant uses torch.argmin (search_fp4_format.py:340-363): the two
    differ on exact midpoints only.  The products are exact where the reference's fp16 / fp32 GEMMs round; measured agreement
    of the loss tables: tests/test_gpu_gemm_codes.py."""
    from . import lowbit
    if not activations:
        return torch.zeros(len(weight_formats), len(act_formats), dtype=torch.float64, device=weight.device)
    per_row = per != "group"
    c_in = weight.shape[1]
    flat = [x.reshape(-1, c_in) for x in activations]
    rows = torch.tensor([f.shape[0] for f in flat], device=weight.device)
    X = torch.cat(flat)
    row_w = torch.repeat_interleave(1.0 / (rows.double() * weight.shape[0] * len(flat)), rows)
    wq = [lowbit.pack_codes(weight, wf, per_row) for wf in weight_formats]
    loss = torch.zeros(len(weight_formats), len(act_formats), dtype=torch.float64, device=weight.device)
    for r0 in range(0, X.shape[0], max_rows):
        xs = X[r0:r0 + max_rows].contiguous()
        ws = row_w[r0:r0 + max_rows].contiguous()
        y_fp = torch.matmul(xs, weight.T.to(xs.dtype)).contiguous()
        for ai, af in enumerate(act_formats):
            a = lowbit.pack_codes(xs, af, per_row, global_clip=False)
            for wi in range(len(weight_formats)):
                lowbit.linear_codes_sse(a, wq[wi], y_fp, None, loss[wi, ai:ai + 1], ws)
    return loss


def best_formats(loss: torch.Tensor, weight_formats: Sequence[str], act_formats: Sequence[str]) -> Dict[str, object]:
    """argmin in the reference's iteration order (weight format outer, activation format inner; the first
    strictly smaller loss wins, search_fp4_format.py:818-821)."""
    flat = loss.reshape(-1).cpu()
    best, best_i = float("inf"), 0
    for i, v in enumerate(flat.tolist()):
        if v < best:
            best, best_i = v, i
    wi, ai = divmod(best_i, len(act_formats))
    return {"weight_format": weight_formats[wi], "activation_format": act_formats[ai], "loss": best}


def search_layers(layers: Sequence[dict], weight_formats: Sequence[str] = FP4_FORMATS, act_formats: Sequence[str] = FP4_FORMATS,
                  rank: int = 0, world: int = 1, group=None, layer_fn=None) -> Optional[List[Dict[str, object]]]:
    """`layers`: [{"name": ..., "weight": W, "activations": [x_j]}].  Units (layer, weight format) are dealt
    round-robin to ranks; every rank fills its rows of the [layers, w, a] table and the tables are
    summed at the end (each entry is written by exactly one rank).  Returns the per-layer optimum on
    every rank.  `layer_fn` (default `search_layer`) scores one (layer, [weight format]) unit."""
    layer_fn = layer_fn or search_layer
    table = torch.zeros(len(layers), len(weight_formats), len(act_formats), dtype=torch.float64,
                        device=layers[0]["weight"].device if layers else "cpu")
    units = [(li, wi) for li in range(len(layers)) for wi in range(len(weight_formats))]
    for u in shard_units(len(units), rank, world):
        li, wi = units[u]
        table[li, wi] = layer_fn(layers[li]["weight"], layers[li]["activations"], [weight_formats[wi]], act_formats)[0]
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(table, group=group)
    return [dict(name=layers[li].get("name", li), **best_formats(table[li], weight_formats, act_formats)) for li in range(len(layers))]
