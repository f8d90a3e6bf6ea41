"""Packed low-bit operands and the real low-bit linear layer (SURVEY.md section 8 f4).

The reference's QuantizedLinear.forward is `act_quant(x)` -> `F.linear(q_x, W_q, b)` on fp16 tensors
(models_fp_quant_transform_rotate/quant_utils.py:764-769).  Here the quantizer emits (grid value, scale per row and
128-group) -- `PackedCodes` -- and `linear_codes` multiplies two of them on the tensor cores (csrc/fpq_gemm.cu, tcgen05.mma
kind::f8f6f4).  `QuantizedLinearLowBit` is the module form: `from_float(nn.Linear)` packs the weight once, forward packs the
activation and runs the GEMM.  No fallback: without the CUDA library every call raises.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib as L
from .ops import _on_device, _require_cuda, _stream

_DT = {torch.float32: L.FPQ_F32, torch.float16: L.FPQ_F16}
GROUP = 128
FP4_FORMATS = ("e2m1", "e1m2", "e3m0")


def rows_padded(rows: int) -> int:
    return (rows + 127) // 128 * 128


@dataclass
class PackedCodes:
    """rows x k values as one e4m3 byte per element (the grid value, exact) and one fp32 scale per (row, 128-group), in the
    tile order of include/fpq_b200.h: codes [k/128][rows_pad/8][8][8][16] bytes, scales [k/128][rows_pad]."""
    codes: torch.Tensor        # uint8 [rows_pad * k]
    scales: torch.Tensor       # float32 [k / scale_group, rows_pad]
    rows: int
    k: int
    fmt: str
    scale_group: int = GROUP   # 128 (one scale per row and 128-group) or k (one scale per row: per_token / per_channel)

    @property
    def rows_pad(self) -> int:
        return rows_padded(self.rows)

    def check(self, what: str) -> "PackedCodes":
        """The kernels index these buffers from rows / k / scale_group alone: refuse anything that does not match."""
        k, sg = self.k, self.scale_group
        if k <= 0 or k % GROUP != 0 or sg not in (GROUP, k) or self.rows < 0:
            raise L.FpqError(f"{what}: inconsistent PackedCodes (rows {self.rows}, k {k}, scale_group {sg})")
        for t, dt, n, name in ((self.codes, torch.uint8, self.rows_pad * k, "codes"),
                               (self.scales, torch.float32, (k // sg) * self.rows_pad, "scales")):
            if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != dt or t.numel() != n or not t.is_contiguous():
                raise L.FpqError(f"{what}: `{name}` must be a contiguous CUDA {dt} tensor of {n} elements")
        if self.codes.device != self.scales.device:
            raise L.FpqError(f"{what}: codes and scales live on different devices")
        return self

    def dequantize(self, dtype=torch.float16) -> torch.Tensor:
        """The fake-quantized tensor these codes stand for ([rows, k]); bit-identical to ops.fake_quant of the packed input
        when `dtype` is the input's dtype."""
        self.check("dequantize")
        if dtype not in _DT:
            raise L.FpqError(f"dequantize: dtype {dtype} is not supported (float16 / float32 only)")
        out = torch.empty((self.rows, self.k), dtype=dtype, device=self.codes.device)
        with _on_device(self.codes) as dev:
            L.check(L.lib().fpq_unpack_codes(self.codes.data_ptr(), self.scales.data_ptr(), self.rows, self.k, self.scale_group,
                                             _DT[dtype], out.data_ptr(), _stream(dev)), "fpq_unpack_codes")
        return out

    def to_nibbles(self) -> torch.Tensor:
        """4-bit storage (FP4 formats only): uint8 [rows_pad * k / 2]."""
        self.check("to_nibbles")
        nib = torch.empty(self.codes.numel() // 2, dtype=torch.uint8, device=self.codes.device)
        with _on_device(self.codes) as dev:
            L.check(L.lib().fpq_codes_to_nibbles(self.codes.data_ptr(), self.codes.numel(), L.FMT[self.fmt], nib.data_ptr(),
                                                 _stream(dev)), f"fpq_codes_to_nibbles({self.fmt})")
        return nib

    @staticmethod
    def from_nibbles(nib: torch.Tensor, scales: torch.Tensor, rows: int, k: int, fmt: str, scale_group: int = GROUP) -> "PackedCodes":
        _require_cuda(nib, "from_nibbles")
        if nib.dtype != torch.uint8 or not nib.is_contiguous() or nib.numel() * 2 != rows_padded(rows) * k:
            raise L.FpqError(f"from_nibbles: expected a contiguous uint8 tensor of {rows_padded(rows) * k // 2} bytes")
        if fmt not in FP4_FORMATS:
            raise L.FpqError(f"from_nibbles: {fmt} has no 4-bit form (FP4 formats only)")
        codes = torch.empty(nib.numel() * 2, dtype=torch.uint8, device=nib.device)
        with _on_device(nib) as dev:
            L.check(L.lib().fpq_nibbles_to_codes(nib.data_ptr(), codes.numel(), L.FMT[fmt], codes.data_ptr(), _stream(dev)),
                    f"fpq_nibbles_to_codes({fmt})")
        return PackedCodes(codes, scales, rows, k, fmt, scale_group).check("from_nibbles")


def pack_codes(x: torch.Tensor, fmt: str, per_row: bool = False) -> PackedCodes:
    """fp_quant_*_per_group_cuda (groups of 128 along the last dim, kernel tie rule) with the codes kept instead of multiplied
    back; per_row=True: one scale per row, the per_token / per_channel functions (qu.py:503-534).
    x: [..., k] float16 / float32 CUDA tensor; leading dims are flattened into rows."""
    _require_cuda(x, "pack_codes")
    if x.dtype not in _DT:
        raise L.FpqError(f"pack_codes: dtype {x.dtype} is not supported (float16 / float32 only)")
    if fmt not in L.FMT:
        raise ValueError("Unsupported fp_type.")
    k = x.shape[-1]
    if k % GROUP != 0:
        raise L.FpqError(f"pack_codes: last dim {k} is not a multiple of {GROUP}")
    x2 = x.reshape(-1, k)
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    rows = x2.shape[0]
    rp = rows_padded(rows)
    sg = k if per_row else GROUP
    codes = torch.empty(rp * k, dtype=torch.uint8, device=x.device)
    scales = torch.empty((k // sg, rp), dtype=torch.float32, device=x.device)
    with _on_device(x2) as dev:
        L.check(L.lib().fpq_pack_codes(x2.data_ptr(), rows, k, sg, _DT[x2.dtype], L.FMT[fmt], codes.data_ptr(), scales.data_ptr(),
                                       _stream(dev)), f"fpq_pack_codes({fmt})")
    return PackedCodes(codes, scales, rows, k, fmt, sg)


def linear_codes(a: PackedCodes, w: PackedCodes, bias: Optional[torch.Tensor] = None, out_dtype=torch.float16,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """F.linear(a, w, bias) for packed operands: [a.rows, w.rows] in `out_dtype`."""
    a.check("linear_codes(a)")
    w.check("linear_codes(w)")
    if a.k != w.k:
        raise L.FpqError(f"linear_codes: inner sizes differ ({a.k} vs {w.k})")
    if a.codes.device != w.codes.device:
        raise L.FpqError("linear_codes: operands on different devices")
    if (a.scale_group == GROUP) != (w.scale_group == GROUP):
        raise L.FpqError("linear_codes: both operands must be scaled per 128-group, or both per row")
    if out_dtype not in _DT:
        raise L.FpqError(f"linear_codes: output dtype {out_dtype} is not supported")
    m, n = a.rows, w.rows
    if n % 8 != 0:
        raise L.FpqError(f"linear_codes: out_features {n} must be a multiple of 8")
    if out is None:
        out = torch.empty((m, n), dtype=out_dtype, device=a.codes.device)
    elif out.shape != (m, n) or out.dtype != out_dtype or not out.is_contiguous() or out.device != a.codes.device:
        raise L.FpqError("linear_codes: `out` must be a contiguous [m, n] tensor of out_dtype on the operands' device")
    b = None
    if bias is not None:
        _require_cuda(bias, "linear_codes(bias)")
        if bias.numel() != n:
            raise L.FpqError(f"linear_codes: bias has {bias.numel()} entries, expected {n}")
        b = bias.detach().to(device=a.codes.device, dtype=torch.float32).contiguous()
    with _on_device(a.codes) as dev:
        L.check(L.lib().fpq_gemm_codes(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), n, a.k,
                                       a.scale_group, None if b is None else b.data_ptr(), _DT[out_dtype], out.data_ptr(), n,
                                       _stream(dev)), "fpq_gemm_codes")
    return out


def linear_codes_sse(a: PackedCodes, w: PackedCodes, ref: torch.Tensor, bias: Optional[torch.Tensor] = None,
                     sse: Optional[torch.Tensor] = None, row_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """sum_i row_weight[i] * sum_j (ref - F.linear(a, w, bias))[i, j]^2 without materialising the product: the output-level loss
    of the format search (search/search_fp4_format.py:472-476, :798-816).  ref: [a.rows, w.rows] float16 / float32, contiguous;
    row_weight: float64 [a.rows] or None (= 1); returns (and accumulates into) a one-element float64 tensor."""
    _require_cuda(ref, "linear_codes_sse(ref)")
    a.check("linear_codes_sse(a)")
    w.check("linear_codes_sse(w)")
    m, n = a.rows, w.rows
    if a.k != w.k or (a.scale_group == GROUP) != (w.scale_group == GROUP):
        raise L.FpqError("linear_codes_sse: operands do not match")
    if a.codes.device != w.codes.device:
        raise L.FpqError("linear_codes_sse: operands on different devices")
    if ref.dtype not in _DT or ref.shape != (m, n) or not ref.is_contiguous() or n % 8 != 0 or ref.device != a.codes.device:
        raise L.FpqError("linear_codes_sse: ref must be a contiguous float16 / float32 [m, n] tensor on the operands' device, "
                         "n a multiple of 8")
    if sse is None:
        sse = torch.zeros(1, dtype=torch.float64, device=ref.device)
    elif sse.dtype != torch.float64 or not sse.is_cuda or sse.numel() < 1 or sse.device != a.codes.device:
        raise L.FpqError("linear_codes_sse: sse must be a float64 CUDA tensor on the operands' device")
    b = None
    if bias is not None:
        _require_cuda(bias, "linear_codes_sse(bias)")
        if bias.numel() != n:
            raise L.FpqError(f"linear_codes_sse: bias has {bias.numel()} entries, expected {n}")
        b = bias.detach().to(device=a.codes.device, dtype=torch.float32).contiguous()
    if row_weight is not None and (row_weight.dtype != torch.float64 or not row_weight.is_cuda or row_weight.numel() != m
                                   or not row_weight.is_contiguous() or row_weight.device != a.codes.device):
        raise L.FpqError("linear_codes_sse: row_weight must be a contiguous float64 tensor on the operands' device with one "
                         "entry per row")
    with _on_device(a.codes) as dev:
        L.check(L.lib().fpq_gemm_codes_sse(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), n, a.k,
                                           a.scale_group, None if b is None else b.data_ptr(), _DT[ref.dtype], ref.data_ptr(), n,
                                           None if row_weight is None else row_weight.data_ptr(), sse.data_ptr(), _stream(dev)),
                "fpq_gemm_codes_sse")
    return sse


class QuantizedLinearLowBit(torch.nn.Module):
    """QuantizedLinear (qu.py:649-867) with the fake-quantized weight held as codes and the product computed from codes:
    forward(x) = linear_codes(pack_codes(x, act_fmt), weight_codes, bias).  Symmetric per-group formats only (mat_qkv, proj,
    fc1 of the README configuration; the sign-split fc2 input has two scales per group and stays on the fake-quant path)."""

    def __init__(self, weight: PackedCodes, bias: Optional[torch.Tensor], act_fmt: str, out_dtype=torch.float16):
        super().__init__()
        self.in_features, self.out_features = weight.k, weight.rows
        self.weight_fmt, self.act_fmt, self.out_dtype = weight.fmt, act_fmt, out_dtype
        self.per_row = weight.scale_group != GROUP
        self.register_buffer("weight_codes", weight.codes)
        self.register_buffer("weight_scales", weight.scales)
        self.register_buffer("bias", None if bias is None else bias.detach().to(torch.float32).contiguous())

    @classmethod
    def from_float(cls, module: torch.nn.Linear, weight_fmt: str = "e2m1", act_fmt: str = "e2m1", out_dtype=torch.float16,
                   per_row: bool = False):
        """module.weight: [out, in] on a CUDA device; quantized exactly as QuantizedLinear.from_float does for
        weight_quant='per_group' (qu.py:772-813: fp_quant_*_per_group_cuda on the fp32 weight), or, with per_row=True, for
        weight_quant='per_channel' / act_quant='per_token' (the README's W6A6 commands)."""
        w = module.weight.detach()
        _require_cuda(w, "QuantizedLinearLowBit.from_float")
        return cls(pack_codes(w.to(torch.float32), weight_fmt, per_row), module.bias, act_fmt, out_dtype)

    def weight_packed(self) -> PackedCodes:
        return PackedCodes(self.weight_codes, self.weight_scales, self.out_features, self.in_features, self.weight_fmt,
                           self.in_features if self.per_row else GROUP)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        a = pack_codes(x, self.act_fmt, self.per_row)
        y = linear_codes(a, self.weight_packed(), self.bias, self.out_dtype)
        return y.reshape(*x.shape[:-1], self.out_features)

    def extra_repr(self) -> str:
        return (f"{self.in_features}, {self.out_features}, bias={self.bias is not None}, weight={self.weight_fmt} codes, "
                f"act={self.act_fmt} per_group(128), tcgen05 e4m3-container GEMM")
