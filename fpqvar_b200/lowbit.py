"""Packed low-bit operands and the real low-bit linear layer (SURVEY.md section 8 f4).

The reference's QuantizedLinear.forward is `act_quant(x)` -> `F.linear(q_x, W_q, b)` on fp16 tensors
(models_fp_quant_transform_rotate/quant_utils.py:764-769).  Here the quantizer emits (grid value, scale per row and
128-group) -- `PackedCodes` -- and `linear_codes` multiplies two of them on the tensor cores (csrc/fpq_gemm.cu, tcgen05.mma
kind::f8f6f4).  `QuantizedLinearLowBit` is the module form: `from_float(nn.Linear)` packs the weight once, forward packs the
activation and runs the GEMM.  `rotate_pack_codes` emits the codes of a rotated / transformed linear's input (mat_qkv, fc1)
straight out of the fused rotate kernel, for `QuantizedLinearLowBit.forward_packed`.  The sign-split fc2 input
(SPLIT_FORMATS: two scales per 128-group, qu.py:415-452) is a codes operand of depth 2k (`pack_codes`, `gelu_pack_codes`) that
`linear_codes` multiplies with a per-group weight.  No fallback: without the CUDA library every call raises.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib as L
from .ops import _call, _clip_workspace, _ext, _on_device, _require_cuda, _stream

_DT = {torch.float32: L.FPQ_F32, torch.float16: L.FPQ_F16}
GROUP = 128
FP4_FORMATS = ("e2m1", "e1m2", "e3m0")
SPLIT_FORMATS = ("e1m2_neg_e2m1_pos", "afpq_e2m1")      # sign-split formats with a codes form (both half grids inside e4m3)
_NO_CODES = {"int_neg_e2m3_pos": "its negative half grid is the integers 0..32, and 17, 19, ..., 31 are not e4m3 numbers"}


def rows_padded(rows: int) -> int:
    return (rows + 127) // 128 * 128


@dataclass
class PackedCodes:
    """rows x k values as one e4m3 byte per element (the grid value, exact) and one fp32 scale per (row, 128-group), in the
    tile order of include/fpq_b200.h: codes [k/128][rows_pad/8][8][8][16] bytes, scales [k/128][rows_pad].  With `fmt` in
    SPLIT_FORMATS the operand is sign-split, of depth 2k: slab 2t holds group t's negative-half codes, slab 2t+1 its
    positive-half codes, each with its own scale (codes 2 * rows_pad * k bytes, scales [2k/128][rows_pad])."""
    codes: torch.Tensor        # uint8 [rows_pad * k]
    scales: torch.Tensor       # float32 [k / scale_group, rows_pad]
    rows: int
    k: int
    fmt: str
    scale_group: int = GROUP   # 128 (one scale per row and 128-group) or k (one scale per row: per_token / per_channel)

    @property
    def rows_pad(self) -> int:
        return rows_padded(self.rows)

    @property
    def split(self) -> bool:
        return self.fmt in SPLIT_FORMATS

    def check(self, what: str) -> "PackedCodes":
        """The kernels index these buffers from rows / k / scale_group alone: refuse anything that does not match."""
        k, sg = self.k, self.scale_group
        if k <= 0 or k % GROUP != 0 or sg not in (GROUP, k) or self.rows < 0 or (self.split and sg != GROUP):
            raise L.FpqError(f"{what}: inconsistent PackedCodes (rows {self.rows}, k {k}, scale_group {sg}, format {self.fmt})")
        depth = 2 * k if self.split else k
        for t, dt, n, name in ((self.codes, torch.uint8, self.rows_pad * depth, "codes"),
                               (self.scales, torch.float32, (depth // sg) * self.rows_pad, "scales")):
            if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != dt or t.numel() != n or not t.is_contiguous():
                raise L.FpqError(f"{what}: `{name}` must be a contiguous CUDA {dt} tensor of {n} elements")
        if self.codes.device != self.scales.device:
            raise L.FpqError(f"{what}: codes and scales live on different devices")
        return self

    def dequantize(self, dtype=torch.float16) -> torch.Tensor:
        """The fake-quantized tensor these codes stand for ([rows, k]); bit-identical to ops.fake_quant (sign-split:
        ops.fake_quant_signsplit, kernel tie rule, global_clip as packed) of the packed input when `dtype` is the input's dtype."""
        self.check("dequantize")
        if dtype not in _DT:
            raise L.FpqError(f"dequantize: dtype {dtype} is not supported (float16 / float32 only)")
        out = torch.empty((self.rows, self.k), dtype=dtype, device=self.codes.device)
        with _on_device(self.codes) as dev:
            if self.split:
                L.check(L.lib().fpq_unpack_codes_signsplit(self.codes.data_ptr(), self.scales.data_ptr(), self.rows, self.k,
                                                           _DT[dtype], out.data_ptr(), _stream(dev)), "fpq_unpack_codes_signsplit")
                return out
            L.check(L.lib().fpq_unpack_codes(self.codes.data_ptr(), self.scales.data_ptr(), self.rows, self.k, self.scale_group,
                                             _DT[dtype], out.data_ptr(), _stream(dev)), "fpq_unpack_codes")
        return out

    def to_nibbles(self) -> torch.Tensor:
        """4-bit storage (FP4 formats only): uint8 [rows_pad * k / 2]."""
        self.check("to_nibbles")
        if self.split:
            raise L.FpqError(f"to_nibbles: sign-split codes ({self.fmt}) have no 4-bit form")
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


def _split_fmt(fmt: str, per_row: bool, what: str) -> bool:
    """True for a sign-split format with a codes form; refuses the sign-split cases that have none."""
    if fmt in _NO_CODES:
        raise L.FpqError(f"{what}: {fmt} has no codes form: {_NO_CODES[fmt]}")
    if fmt in SPLIT_FORMATS:
        if per_row:
            raise L.FpqError(f"{what}: sign-split codes have scales per 128-group only (per_row=True is not supported)")
        return True
    if fmt not in L.FMT:
        raise ValueError("Unsupported fp_type.")
    return False


def _pack_split(entry, x2: torch.Tensor, fmt: str, global_clip: bool, *dtype) -> PackedCodes:
    rows, k = x2.shape
    rp = rows_padded(rows)
    codes = torch.empty(2 * rp * k, dtype=torch.uint8, device=x2.device)
    scales = torch.empty((2 * k // GROUP, rp), dtype=torch.float32, device=x2.device)
    ws = _clip_workspace(x2.device) if global_clip else None
    with _on_device(x2) as dev:
        L.check(getattr(L.lib(), entry)(x2.data_ptr(), rows, k, *dtype, L.SPLIT[fmt], L.FLAG_GLOBAL_CLIP if global_clip else 0,
                                        None if ws is None else ws.data_ptr(), codes.data_ptr(), scales.data_ptr(), _stream(dev)),
                f"{entry}({fmt})")
    return PackedCodes(codes, scales, rows, k, fmt, GROUP)


def _rows_2d(x: torch.Tensor, what: str) -> torch.Tensor:
    k = x.shape[-1]
    if k % GROUP != 0:
        raise L.FpqError(f"{what}: last dim {k} is not a multiple of {GROUP}")
    x2 = x.reshape(-1, k)
    return x2 if x2.is_contiguous() else x2.contiguous()


def pack_codes(x: torch.Tensor, fmt: str, per_row: bool = False, *, global_clip: bool = True) -> PackedCodes:
    """fp_quant_*_per_group_cuda (groups of 128 along the last dim, kernel tie rule) with the codes kept instead of multiplied
    back; per_row=True: one scale per row, the per_token / per_channel functions (qu.py:503-534).
    fmt in SPLIT_FORMATS: the sign-split quantizer (fp_quant_e1m2_neg_e2m1_pos_per_group_cuda qu.py:415-452, fp4_afpq_per_group_cuda
    qu0.py:498-535) as a depth-2k operand, groups of 128 only; global_clip (sign-split only) applies the whole-tensor clip of
    those functions (qu.py:421-422: a NaN anywhere gives the all-zero operand), as ops.fake_quant_signsplit(global_clip=True).
    x: [..., k] float16 / float32 CUDA tensor; leading dims are flattened into rows."""
    _require_cuda(x, "pack_codes")
    if x.dtype not in _DT:
        raise L.FpqError(f"pack_codes: dtype {x.dtype} is not supported (float16 / float32 only)")
    split = _split_fmt(fmt, per_row, "pack_codes")
    x2 = _rows_2d(x, "pack_codes")
    if split:
        return _pack_split("fpq_pack_codes_signsplit", x2, fmt, global_clip, _DT[x2.dtype])
    k = x2.shape[1]
    rows = x2.shape[0]
    rp = rows_padded(rows)
    sg = k if per_row else GROUP
    codes = torch.empty(rp * k, dtype=torch.uint8, device=x.device)
    scales = torch.empty((k // sg, rp), dtype=torch.float32, device=x.device)
    with _on_device(x2) as dev:
        L.check(L.lib().fpq_pack_codes(x2.data_ptr(), rows, k, sg, _DT[x2.dtype], L.FMT[fmt], codes.data_ptr(), scales.data_ptr(),
                                       _stream(dev)), f"fpq_pack_codes({fmt})")
    return PackedCodes(codes, scales, rows, k, fmt, sg)


def gelu_pack_codes(x_f16: torch.Tensor, fmt: str, global_clip: bool = True) -> PackedCodes:
    """pack_codes(gelu(x_f16, approximate="tanh"), fmt) in one pass (fpq_gelu_pack_codes_signsplit): the fc2 input of the
    reference, `fc2.act_quant(self.act(self.fc1(x)))` (basic_var.py:108,120), as codes.  The codes stand for exactly what
    ops.gelu_fake_quant_signsplit(x_f16, fmt, global_clip) returns.  x_f16: [..., k] float16 CUDA tensor, fmt in SPLIT_FORMATS."""
    _require_cuda(x_f16, "gelu_pack_codes")
    if x_f16.dtype != torch.float16:
        raise L.FpqError("gelu_pack_codes: x must be float16 (the autocast output of fc1)")
    if not _split_fmt(fmt, False, "gelu_pack_codes"):
        raise L.FpqError(f"gelu_pack_codes: {fmt} is not a sign-split format (one of {SPLIT_FORMATS})")
    return _pack_split("fpq_gelu_pack_codes_signsplit", _rows_2d(x_f16, "gelu_pack_codes"), fmt, global_clip)


def rotate_pack_codes(x: torch.Tensor, smooth: Optional[torch.Tensor], sign_bits, fmt: str, scale: Optional[torch.Tensor] = None,
                      shift: Optional[torch.Tensor] = None) -> PackedCodes:
    """ops.transform_rotate_quant (scale / shift given: ops.modulate_transform_rotate_quant) with the quantized activation
    emitted as codes, scales per (row, 128-group), in one launch (fpq_transform_rotate_pack_codes): bit-identical to
    pack_codes(<the same call with fmt=None>, fmt).  x: fp32 [..., C] ([B, ..., C] with [B, 1, C] scale / shift),
    C % 128 == 0; rows = x.numel() // C."""
    _require_cuda(x, "rotate_pack_codes")
    if fmt is None or fmt not in L.FMT:
        raise L.FpqError(f"rotate_pack_codes: a quantizer format is required (one of {sorted(L.FMT)}); got {fmt!r}")
    if (scale is None) != (shift is None):
        raise L.FpqError("rotate_pack_codes: scale and shift go together")
    if x.dtype != torch.float32 or x.dim() < (2 if scale is not None else 1):
        raise L.FpqError("rotate_pack_codes: x must be a float32 tensor" + (" [B, ..., C]" if scale is not None else " [..., C]"))
    c = x.shape[-1]
    if c == 0 or c % GROUP != 0:
        raise L.FpqError(f"rotate_pack_codes: last dim {c} is not a positive multiple of {GROUP}")
    for t, name in ((scale, "scale"), (shift, "shift"), (smooth, "smooth")):
        if t is not None:
            _require_cuda(t, f"rotate_pack_codes({name})")
    bits = list(sign_bits)
    if scale is None:
        codes, scales = _call(_ext().transform_rotate_pack_codes, x, smooth, bits, L.FMT[fmt])
    else:
        codes, scales = _call(_ext().modulate_transform_rotate_pack_codes, x, scale, shift, smooth, bits, L.FMT[fmt])
    return PackedCodes(codes, scales, x.numel() // c, c, fmt, GROUP)


def linear_codes(a: PackedCodes, w: PackedCodes, bias: Optional[torch.Tensor] = None, out_dtype=torch.float16,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """F.linear(a, w, bias) for packed operands: [a.rows, w.rows] in `out_dtype`.  A sign-split `a` (the fc2 input) multiplies a
    weight scaled per 128-group (fpq_gemm_codes_signsplit)."""
    a.check("linear_codes(a)")
    w.check("linear_codes(w)")
    _check_operands(a, w, "linear_codes")
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
        if a.split:
            L.check(L.lib().fpq_gemm_codes_signsplit(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(),
                                                     n, a.k, None if b is None else b.data_ptr(), _DT[out_dtype], out.data_ptr(), n,
                                                     _stream(dev)), "fpq_gemm_codes_signsplit")
            return out
        L.check(L.lib().fpq_gemm_codes(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), n, a.k,
                                       a.scale_group, None if b is None else b.data_ptr(), _DT[out_dtype], out.data_ptr(), n,
                                       _stream(dev)), "fpq_gemm_codes")
    return out


def _check_operands(a: PackedCodes, w: PackedCodes, what: str) -> None:
    if a.k != w.k:
        raise L.FpqError(f"{what}: inner sizes differ ({a.k} vs {w.k})")
    if a.codes.device != w.codes.device:
        raise L.FpqError(f"{what}: operands on different devices")
    if w.split:
        raise L.FpqError(f"{what}: the weight is sign-split ({w.fmt}); only the activation operand may be")
    if (a.scale_group == GROUP) != (w.scale_group == GROUP):
        raise L.FpqError(f"{what}: both operands must be scaled per 128-group, or both per row")


def linear_codes_sse(a: PackedCodes, w: PackedCodes, ref: torch.Tensor, bias: Optional[torch.Tensor] = None,
                     sse: Optional[torch.Tensor] = None, row_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """sum_i row_weight[i] * sum_j (ref - F.linear(a, w, bias))[i, j]^2 without materialising the product: the output-level loss
    of the format search (search/search_fp4_format.py:472-476, :798-816).  ref: [a.rows, w.rows] float16 / float32, contiguous;
    row_weight: float64 [a.rows] or None (= 1); returns (and accumulates into) a one-element float64 tensor."""
    _require_cuda(ref, "linear_codes_sse(ref)")
    a.check("linear_codes_sse(a)")
    w.check("linear_codes_sse(w)")
    m, n = a.rows, w.rows
    _check_operands(a, w, "linear_codes_sse")
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
        if a.split:
            L.check(L.lib().fpq_gemm_codes_signsplit_sse(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(),
                                                         w.scales.data_ptr(), n, a.k, None if b is None else b.data_ptr(),
                                                         _DT[ref.dtype], ref.data_ptr(), n,
                                                         None if row_weight is None else row_weight.data_ptr(), sse.data_ptr(),
                                                         _stream(dev)), "fpq_gemm_codes_signsplit_sse")
            return sse
        L.check(L.lib().fpq_gemm_codes_sse(a.codes.data_ptr(), a.scales.data_ptr(), m, w.codes.data_ptr(), w.scales.data_ptr(), n, a.k,
                                           a.scale_group, None if b is None else b.data_ptr(), _DT[ref.dtype], ref.data_ptr(), n,
                                           None if row_weight is None else row_weight.data_ptr(), sse.data_ptr(), _stream(dev)),
                "fpq_gemm_codes_sse")
    return sse


class QuantizedLinearLowBit(torch.nn.Module):
    """QuantizedLinear (qu.py:649-867) with the fake-quantized weight held as codes and the product computed from codes:
    forward(x) = linear_codes(pack_codes(x, act_fmt), weight_codes, bias).  act_fmt may be a sign-split format (SPLIT_FORMATS)
    when the weight is scaled per 128-group: the fc2 layer of QuantizedLinear_fc2 (qu.py:870-1093), whose input then runs as a
    depth-2k operand; forward_gelu(h) takes the fp16 fc1 output and fuses the GELU into the packing."""

    def __init__(self, weight: PackedCodes, bias: Optional[torch.Tensor], act_fmt: str, out_dtype=torch.float16):
        super().__init__()
        if weight.split:
            raise L.FpqError(f"QuantizedLinearLowBit: the weight is sign-split ({weight.fmt}); only the activation may be")
        if act_fmt in SPLIT_FORMATS or act_fmt in _NO_CODES:
            _split_fmt(act_fmt, weight.scale_group != GROUP, "QuantizedLinearLowBit")
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

    def forward_gelu(self, h: torch.Tensor) -> torch.Tensor:
        """forward(gelu(h, approximate="tanh")) for the fp16 fc1 output h, with the GELU fused into the packing of a sign-split
        act_fmt (gelu_pack_codes): bit-identical to forward of the fp16 GELU output."""
        y = linear_codes(gelu_pack_codes(h, self.act_fmt), self.weight_packed(), self.bias, self.out_dtype)
        return y.reshape(*h.shape[:-1], self.out_features)

    def forward_packed(self, a: PackedCodes) -> torch.Tensor:
        """The product of an activation that is already packed (rotate_pack_codes): [a.rows, out_features].  `a` must carry
        this module's activation format and scale grouping."""
        if a.fmt != self.act_fmt:
            raise L.FpqError(f"forward_packed: activation codes are {a.fmt}, this layer quantizes activations as {self.act_fmt}")
        if (a.scale_group != GROUP) != self.per_row:
            raise L.FpqError("forward_packed: activation scales are " + ("per row" if a.scale_group != GROUP else "per 128-group")
                             + ", this layer expects " + ("per row" if self.per_row else "per 128-group"))
        return linear_codes(a, self.weight_packed(), self.bias, self.out_dtype)

    def extra_repr(self) -> str:
        act = "sign-split per_group(128)" if self.act_fmt in SPLIT_FORMATS else "per_group(128)"
        return (f"{self.in_features}, {self.out_features}, bias={self.bias is not None}, weight={self.weight_fmt} codes, "
                f"act={self.act_fmt} {act}, tcgen05 e4m3-container GEMM")
