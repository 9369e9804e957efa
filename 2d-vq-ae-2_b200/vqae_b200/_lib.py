"""ctypes binding of ``libvqae_b200.so`` (the C-ABI declared in include/vqae_b200.h).

This is the only place the Python host code touches the native library.  There is no
fallback: if the library is missing and cannot be built, or a call returns an error code,
an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

PKG = Path(__file__).resolve().parent
LIB_NAME = "libvqae_b200.so"

OK, ERR_BAD_ARG, ERR_UNSUPPORTED, ERR_DIM_MISMATCH, ERR_CUDA, ERR_SCRATCH = range(6)
LAYOUT_NCHW, LAYOUT_NHWC = 0, 1
DT_F32, DT_BF16, DT_U8, DT_F16 = 0, 1, 2, 3
QUANT_AUTO, QUANT_CUDA_CORE, QUANT_TENSOR_CORE = 0, 1, 2
MODE_SAME, MODE_DOWN, MODE_UP = 0, 1, 2
CONV_1x1, CONV_2x2S2, CONV_3x3_CIRC = 0, 1, 2
STEM_OUT_EXACT, STEM_OUT_TENSOR_CORE = 0, 1


class VqaeError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str = ""):
        self.code = code
        super().__init__(f"{where}: vqae error {code}: {detail}")


class FixupParams(C.Structure):
    """struct vqae_fixup_params"""
    _fields_ = [
        ("mode", C.c_int), ("c_in", C.c_int), ("c_out", C.c_int), ("c_branch", C.c_int),
        ("w1", C.c_void_p), ("w2", C.c_void_p), ("w3", C.c_void_p), ("w_skip", C.c_void_p),
        ("bias1a", C.c_float), ("bias1b", C.c_float), ("bias2a", C.c_float),
        ("bias2b", C.c_float), ("bias3a", C.c_float), ("bias3b", C.c_float),
        ("bias4", C.c_float), ("scale", C.c_float), ("bias1c", C.c_float),
        ("bias1d", C.c_float),
    ]


class PackDesc(C.Structure):
    """struct vqae_pack_desc"""
    _fields_ = [("kind", C.c_int32), ("c_in", C.c_int32), ("c_out", C.c_int32), ("taps", C.c_int32),
                ("scale", C.c_float), ("n_elems", C.c_int32), ("src", C.c_void_p * 4),
                ("dst", C.c_void_p), ("premul", C.c_float * 4)]


PACK_F32_CONV, PACK_SAME_F16, PACK_RESIDENT_F16, PACK_DOWN_F16, PACK_SAME_MMA_F16 = 0, 1, 2, 3, 4
PACK_DOWN_MMA_F16, PACK_UP_MMA_F16 = 5, 6
PACK_LO = 0x100


class QuantizerParams(C.Structure):
    """struct vqae_quantizer_params"""
    _fields_ = [
        ("num_codes", C.c_int), ("dim", C.c_int), ("c", C.c_int),
        ("embed", C.c_void_p), ("w_in", C.c_void_p), ("b_in", C.c_void_p),
        ("table", C.c_void_p), ("commitment_cost", C.c_float),
    ]


_vp, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
_fp = C.POINTER(C.c_float)

# name -> (restype, argtypes); every symbol include/vqae_b200.h declares
SIGNATURES = {
    "vqae_abi_version": (_i, []),
    "vqae_error_string": (C.c_char_p, [_i]),
    "vqae_last_cuda_error": (C.c_char_p, []),
    "vqae_launch_count": (C.c_uint64, []),
    "vqae_normalize_u8": (_i, [_vp, _vp, _i64, _i, _i, _fp, _fp, _i, _vp]),
    "vqae_pack_conv_weight_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "vqae_pack_elems": (_sz, [_i, _i, _i, _i]),
    "vqae_pack_batched": (_i, [_vp, _i, _i, _vp]),
    "vqae_stem_in_f32": (_i, [_vp, _i, _i, _vp, _vp, _vp, _i64, _i, _i, _i, _fp, _fp, _vp]),
    "vqae_stem_in": (_i, [_vp, _i, _i, _vp, _vp, _vp, _i, _i64, _i, _i, _i, _fp, _fp, _vp]),
    "vqae_stem_out_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _i, _i, _i, _vp]),
    "vqae_stem_out_u8_supported": (_i, [_i, _i, _i, _i]),
    "vqae_stem_out_u8": (_i, [_vp, _vp, _vp, _fp, _fp, _vp, _i64, _i64, _i64, _i, _i64, _i, _i, _i, _i,
                              _vp]),
    "vqae_conv_f32": (_i, [_i, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _f, _i, _f, _f, _f, _vp]),
    "vqae_bicubic_up2_f32": (_i, [_vp, _vp, _i64, _i, _i, _i, _f, _vp]),
    "vqae_fixup_block_scratch_bytes": (_sz, [C.POINTER(FixupParams), _i64, _i, _i]),
    "vqae_fixup_block_f32": (_i, [C.POINTER(FixupParams), _vp, _vp, _vp, _sz, _i64, _i, _i, _vp]),
    "vqae_quantizer_prepare_f32": (_i, [_vp, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "vqae_quantizer_scratch_bytes": (_sz, [_i64]),
    "vqae_quantize_f32": (_i, [C.POINTER(QuantizerParams), _vp, _i, _vp, _i, _vp, _vp, _vp, _f,
                               _vp, _vp, _sz, _i64, _i64, _vp]),
    "vqae_quantize_supported": (_i, [C.POINTER(QuantizerParams), _i, _i, _i, _i, _i, _i]),
    "vqae_quantize": (_i, [C.POINTER(QuantizerParams), _vp, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _f,
                           _vp, _vp, _sz, _i64, _i64, _i, _vp]),
    "vqae_quantize_tc_supported": (_i, [C.POINTER(QuantizerParams), _i, _i, _i]),
    "vqae_quantize_tc_f32": (_i, [C.POINTER(QuantizerParams), _vp, _vp, _vp, _vp, _vp, _f, _vp,
                                  _vp, _vp, _sz, _i64, _i64, _vp]),
    "vqae_embed_codes_f32": (_i, [_vp, _i, _vp, _i, _i, _vp, _i, _i64, _i64, _vp]),
    "vqae_embed_codemap_f32": (_i, [_vp, _i, _i64, _i64, _i, _i, _i64, _i64, _i64, _i64, _i64, _vp, _i,
                                    _i, _vp, _vp]),
    "vqae_codemap_place_u8": (_i, [_vp, _i64, _i, _i, _i64, _i, _vp, _i64, _i64, _vp]),
    "vqae_codemap_place_i64": (_i, [_vp, _i64, _i, _i, _i64, _i, _vp, _i64, _i64, _vp]),
    "vqae_ema_scratch_bytes": (_sz, [_i64, _i, _i]),
    "vqae_ema_accumulate_f32": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "vqae_ema_update_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _f, _vp]),
    "vqae_column_stats_f32": (_i, [_vp, _i64, _i, _vp, _vp, _vp, _sz, _vp]),
    "vqae_ema_init_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "vqae_add_f32": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "vqae_pointwise_conv_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _i, _i, _vp]),
    "vqae_depthwise_conv_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp]),
    "vqae_se_gate_f32": (_i, [_vp, _i64, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "vqae_quality_u8_scratch_bytes": (_sz, [_i64, _i, _i]),
    "vqae_quality_u8": (_i, [_vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _i64, _i64, _i64,
                             _i64, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "vqae_codemap_histogram": (_i, [_vp, _i, _i64, _i64, _i64, _i64, _i64, _i64, _i, _vp, _vp]),
    "vqae_codemap_pack_scratch_bytes": (_sz, [_i64, _i, _i]),
    "vqae_codemap_pack_worst_bytes": (_i64, [_i64, _i, _i]),
    "vqae_codemap_pack": (_i, [_vp, _i, _i64, _i64, _i, _i, _vp, _i, _i, _vp, _vp, _i64, _vp, _sz, _vp]),
    "vqae_codemap_unpack": (_i, [_vp, _i64, _vp, _vp, _i64, _i64, _i, _i, _vp, _i, _i, _i64, _i64, _i64, _i64,
                                 _vp, _i, _vp, _vp]),
    "vqae_residual_stats": (_i, [_vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _i64, _i64, _i64,
                                 _i64, _i, _i, _i, _vp, _vp, _vp]),
    "vqae_residual_tables": (_i, [_vp, _i64, _vp, _vp]),
    "vqae_residual_encode_scratch_bytes": (_sz, [_i64, _i, _i]),
    "vqae_residual_encode": (_i, [_vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _i64, _i64, _i64,
                                  _i64, _i, _i, _i, _vp, _vp, _vp, _i64, _vp, _sz, _vp]),
    "vqae_residual_apply": (_i, [_vp, _i64, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _i64, _i64,
                                 _i64, _i64, _i64, _i64, _i64, _i, _i, _i, _vp, _vp]),
    "vqae_pyramid_u8_scratch_bytes": (_sz, [_i64, _i, _i, _i]),
    "vqae_pyramid_u8": (_i, [_vp, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i, _i, _i, _vp, _vp, _vp, _i64, _i64,
                             _i64, _i64, _vp, _sz, _vp]),
    "vqae_jpeg_tiles_scratch_bytes": (_sz, [_i64, _i64, _i, _i, _i64, _i64, _i, _i]),
    "vqae_jpeg_tiles_worst_bytes": (_i64, [_i64, _i64, _i, _i, _i64, _i64, _i, _i]),
    "vqae_jpeg_tiles": (_i, [_vp, _i64, _i64, _i64, _i, _i, _i64, _i64, _i, _i, _vp, _i, _vp, _vp, _vp, _i64, _vp,
                             _sz, _vp]),
}

_lib: Optional[C.CDLL] = None


def library_path() -> Path:
    return Path(os.environ.get("VQAE_B200_LIB", PKG / LIB_NAME))


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if the .so is absent and nvcc exists) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if "VQAE_B200_LIB" not in os.environ:
        # rebuild when the sources changed (no-op when the stamp matches); a prebuilt .so
        # without nvcc around is used as is
        try:
            from .csrc.build import build_library
            path = build_library()
        except FileNotFoundError:      # no nvcc: fall through to the prebuilt library
            if not path.exists() or not build_if_missing:
                raise
    if not path.exists():
        raise FileNotFoundError(
            f"{path} not built; run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(str(path))
    declared = dict(SIGNATURES)
    from . import _lib_tc  # optional tensor-core entry points share the same .so
    declared.update(_lib_tc.SIGNATURES)
    for name, (res, args) in declared.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.vqae_abi_version() != 4:
        raise RuntimeError(f"{path}: ABI version {lib.vqae_abi_version()} != 4")
    _lib = lib
    return lib


_aids: Optional[C.CDLL] = None


def load_testaids() -> C.CDLL:
    """libvqae_b200_testaids.so (include/vqae_b200_testaids.h): self test, MMA microbenchmarks and
    profiling hooks -- for tests/ and profiles/, never used by the product path."""
    global _aids
    if _aids is not None:
        return _aids
    load()                                   # builds both libraries; the aids link against the first
    from . import _lib_tc
    lib = C.CDLL(str(PKG / "libvqae_b200_testaids.so"))
    for name, (res, args) in _lib_tc.AIDS_SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _aids = lib
    return lib


def check(code: int, where: str) -> None:
    if code == OK:
        return
    lib = load()
    detail = lib.vqae_error_string(code).decode()
    if code == ERR_CUDA:
        detail += " -- " + lib.vqae_last_cuda_error().decode()
    if code == ERR_DIM_MISMATCH:
        # same exception type as the reference (vq_ae/layers/vq.py:100-104)
        raise NotImplementedError(f"{where}: {detail}")
    raise VqaeError(code, where, detail)


def f3(values) -> "C.Array":
    return (C.c_float * 3)(*[float(v) for v in values])
