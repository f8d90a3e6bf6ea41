"""ctypes loader for libfpq_b200.so (the C ABI declared in include/fpq_b200.h).

There is deliberately no fallback: if the shared library is missing or fails to load, every
operator of this package raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C fpqvar_b200/csrc``.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FPQ_LIB_PATH") or os.path.join(_HERE, "libfpq_b200.so")     # FPQ_LIB_PATH: an alternative BUILD of the same library (csrc: make VARIANT=...)

# mirrors include/fpq_b200.h
FPQ_OK, FPQ_ERR_ARG, FPQ_ERR_UNSUPPORTED, FPQ_ERR_CUDA = 0, -1, -2, -3
FPQ_F32, FPQ_F16 = 0, 1
FMT = {"e2m1": 0, "e1m2": 1, "e3m0": 2, "e2m3": 3, "e3m2": 4}
SPLIT = {"e1m2_neg_e2m1_pos": 0, "int_neg_e2m3_pos": 1, "afpq_e2m1": 2}
TIE = {"kernel": 0, "argmin": 1}
FLAG_CLAMP3, FLAG_GLOBAL_CLIP = 1, 2
MOD_GAIN = 1                                # FPQ_MOD_GAIN (fpq_modulate_transform_rotate_quant flags)

_c = ctypes
SIGNATURES = {
    "fpq_version": (_c.c_char_p, []),
    "fpq_last_cuda_error": (_c.c_char_p, []),
    "fpq_launch_count": (_c.c_uint64, []),
    "fpq_set_tunable": (_c.c_int, [_c.c_char_p, _c.c_longlong]),
    "fpq_rotate_plan": (_c.c_int, [_c.c_int, _c.c_int, _c.c_void_p]),
    "fpq_quant_grid": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int, _c.c_size_t, _c.c_void_p, _c.c_int, _c.c_void_p]),
    "fpq_fake_quant": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t, _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                  _c.c_uint, _c.c_void_p]),
    "fpq_fake_quant_segments": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t, _c.c_size_t, _c.c_size_t, _c.c_size_t,
                                           _c.c_int, _c.c_void_p]),
    "fpq_fake_quant_signsplit": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t, _c.c_int, _c.c_int, _c.c_int,
                                            _c.c_int, _c.c_uint, _c.c_void_p, _c.c_void_p]),
    "fpq_transform_rotate_quant": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t,
                                              _c.c_size_t, _c.c_int, _c.c_void_p]),
    "fpq_modulate_transform_rotate_quant": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_void_p,
                                                       _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t, _c.c_int, _c.c_int,
                                                       _c.c_void_p]),
    "fpq_transform_rotate_pack_codes": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t,
                                                   _c.c_size_t, _c.c_int, _c.c_void_p]),
    "fpq_modulate_transform_rotate_pack_codes": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p,
                                                            _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t, _c.c_int,
                                                            _c.c_int, _c.c_void_p]),
    "fpq_transform_rotate_weight": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t,
                                               _c.c_void_p]),
    "fpq_score_formats": (_c.c_int, [_c.c_void_p, _c.c_size_t, _c.c_size_t, _c.c_int, _c.c_void_p, _c.c_int, _c.c_int,
                                     _c.c_void_p, _c.c_void_p]),
    "fpq_gelu_fake_quant_signsplit": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_int, _c.c_uint, _c.c_void_p, _c.c_void_p]),
    "fpq_selftest_gelu": (_c.c_int, [_c.c_void_p, _c.c_void_p]),
    "fpq_sse_rows": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    "fpq_selftest_rounding": (_c.c_int, [_c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p]),
    "fpq_selftest_f16_flow": (_c.c_int, [_c.c_int, _c.c_void_p, _c.c_void_p]),
    "fpq_codes_rows_padded": (_c.c_size_t, [_c.c_size_t]),
    "fpq_pack_codes": (_c.c_int, [_c.c_void_p, _c.c_size_t, _c.c_size_t, _c.c_size_t, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p,
                                  _c.c_void_p]),
    "fpq_unpack_codes": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t, _c.c_size_t, _c.c_int, _c.c_void_p, _c.c_void_p]),
    "fpq_codes_to_nibbles": (_c.c_int, [_c.c_void_p, _c.c_size_t, _c.c_int, _c.c_void_p, _c.c_void_p]),
    "fpq_nibbles_to_codes": (_c.c_int, [_c.c_void_p, _c.c_size_t, _c.c_int, _c.c_void_p, _c.c_void_p]),
    "fpq_gemm_codes": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t,
                                  _c.c_size_t, _c.c_void_p, _c.c_int, _c.c_void_p, _c.c_size_t, _c.c_void_p]),
    "fpq_gemm_codes_sse": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_size_t,
                                      _c.c_size_t, _c.c_void_p, _c.c_int, _c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
}

_lib = None


class FpqError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """The loaded library (loads on first use; raises if it is not built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FpqError(
                f"{LIB_PATH} is not built. fpqvar_b200 has no CPU or PyTorch fallback: build the CUDA library with "
                "`make -C fpqvar_b200/csrc` (or __graft_entry__.build()).")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(handle, name)    # AttributeError here = header and library out of sync
            except AttributeError:
                if os.environ.get("FPQ_LIB_PATH") and name in ("fpq_set_tunable", "fpq_rotate_plan", "fpq_fake_quant_segments", "fpq_sse_rows", "fpq_gelu_fake_quant_signsplit", "fpq_selftest_gelu"):
                    continue                  # an older build selected for an A/B measurement (tools/): it has no tunables
                raise
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def set_tunable(name: str, value: int) -> None:
    """fpq_set_tunable: move a measured launch-geometry choice at run time (measurement tools and tests only)."""
    check(lib().fpq_set_tunable(name.encode(), int(value)), f"fpq_set_tunable({name!r}, {value})")


def check(rc: int, what: str) -> None:
    if rc == FPQ_OK:
        return
    if rc == FPQ_ERR_CUDA:
        raise FpqError(f"{what}: CUDA error: {lib().fpq_last_cuda_error().decode()}")
    name = {FPQ_ERR_ARG: "invalid argument", FPQ_ERR_UNSUPPORTED: "unsupported configuration"}.get(rc, f"error {rc}")
    raise FpqError(f"{what}: {name}")
