"""Loads libjxlb200.so and declares the C ABI of include/jxlb200.h for ctypes.

There is no CPU fallback: if the library is missing it is built with nvcc (jxlatte_b200/build.py); if that fails, or
the library cannot be loaded, importing the product path raises.
"""
import ctypes as C
import os

from .params import FrameParams

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("JXLB200_LIB") or os.path.join(_HERE, "libjxlb200.so")   # override: kernel-variant experiments

OK, E_ARG, E_STREAM, E_UNSUPPORTED, E_CUDA = 0, -1, -2, -3, -4
QM_FLOATS = 3 * 131584
HALO_ROWS = 8
OPT_STAGE2 = 1
OPT_OVERLAP_ROWS = 2
OPT_PIPE_ROWS, OPT_PIPE_FANOUT = 3, 4
STAGE2_AUTO, STAGE2_STAGED, STAGE2_FUSED, STAGE2_PAIR, STAGE2_STREAM, STAGE2_TILE = 0, 1, 2, 3, 5, 6


class QmParams(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("n_dct", C.c_int32), ("n_param", C.c_int32), ("n_4x4", C.c_int32),
        ("denominator", C.c_float),
        ("dct_param", (C.c_float * 17) * 3), ("param", (C.c_float * 9) * 3), ("params4x4", (C.c_float * 17) * 3),
        ("raw", C.POINTER(C.c_float) * 3),
    ]


class Slab(C.Structure):
    _fields_ = [("y0", C.c_int32), ("rows", C.c_int32), ("frame_height", C.c_int32),
                ("has_top", C.c_int32), ("has_bottom", C.c_int32)]


# every symbol include/jxlb200.h declares: name -> (restype, argtypes)
_vp = C.c_void_p
_i32 = C.c_int32
_P3 = C.POINTER(_vp)   # const T *const planes[3]
_FP = C.POINTER(FrameParams)
SYMBOLS = {
    "jxlb200_create": (_i32, [_i32, C.POINTER(_vp)]),
    "jxlb200_destroy": (None, [_vp]),
    "jxlb200_last_error": (C.c_char_p, [_vp]),
    "jxlb200_set_stream": (_i32, [_vp, _vp]),
    "jxlb200_sync": (_i32, [_vp]),
    "jxlb200_launch_count": (C.c_int64, [_vp]),
    "jxlb200_set_option": (_i32, [_vp, _i32, _i32]),
    "jxlb200_host_register": (_i32, [_vp, _vp, C.c_uint64]),
    "jxlb200_host_unregister": (_i32, [_vp, _vp]),
    "jxlb200_selftest_divide": (_i32, [_vp, C.c_int64, _i32, C.POINTER(C.c_int64)]),
    "jxlb200_stage1_plan": (_i32, [_vp, _vp, _vp]),
    "jxlb200_qm_default_params": (_i32, [C.POINTER(QmParams)]),
    "jxlb200_qm_generate": (_i32, [C.POINTER(QmParams), _vp, _vp]),
    "jxlb200_set_qm_weights": (_i32, [_vp, _vp, _vp]),
    "jxlb200_vardct_reconstruct": (_i32, [_vp, _FP, _P3, _P3, _vp, _vp, _vp, _vp, _vp, _vp, _P3]),
    "jxlb200_vardct_reconstruct_i16": (_i32, [_vp, _FP, _P3, _P3, _vp, _vp, _vp, _vp, _vp, _vp, _P3]),
    "jxlb200_vardct_reconstruct_packed": (_i32, [_vp, _FP, _P3, _i32, _P3, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "jxlb200_comm_unique_id": (_i32, [_vp]),
    "jxlb200_comm_init": (_i32, [_vp, _vp, _i32, _i32]),
    "jxlb200_comm_destroy": (_i32, [_vp]),
    "jxlb200_vardct_reconstruct_split_dev": (_i32, [_vp, _FP, C.POINTER(Slab), _P3, _P3, _vp, _vp, _vp, _vp, _vp, _vp, _P3]),
    "jxlb200_vardct_invert_dev": (_i32, [_vp, _FP, _P3, _P3, _vp, _vp, _vp, _vp, _vp, _P3, C.c_int64]),
    "jxlb200_restore_dev": (_i32, [_vp, _FP, C.POINTER(Slab), _P3, C.c_int64, _vp, _vp, _P3]),
    "jxlb200_vardct_reconstruct_dev": (_i32, [_vp, _FP, _P3, _P3, _vp, _vp, _vp, _vp, _vp, _vp, _P3]),
    "jxlb200_vardct_reconstruct_batch_dev": (_i32, [_vp, _FP, _i32, _P3, _P3, _vp, _vp, _vp, _vp, _vp, _vp, _P3]),
    "jxlb200_host_slab_schedule": (_i32, [_i32, _vp, _i32]),
    "jxlb200_host_stage2_ranges": (_i32, [_i32, _vp, _vp, _i32]),
    "jxlb200_gaborish": (_i32, [_vp, _FP, _P3, _P3]),
    "jxlb200_restore_uniform": (_i32, [_vp, _FP, C.c_float, _P3, _P3]),
    "jxlb200_epf": (_i32, [_vp, _FP, _P3, _vp, _vp, _P3]),
    "jxlb200_color_transform": (_i32, [_vp, _FP, _P3, _P3]),
    "jxlb200_vardct_invert": (_i32, [_vp, _FP, _P3, _P3, _vp, _vp, _vp, _vp, _vp, _P3]),
    "jxlb200_modular_rct": (_i32, [_vp, _P3, _i32, _i32, _i32]),
    "jxlb200_modular_palette": (_i32, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _P3]),
    "jxlb200_modular_squeeze": (_i32, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp]),
    "jxlb200_modular_rct_dev": (_i32, [_vp, _P3, _i32, _i32, _i32]),
    "jxlb200_modular_palette_dev": (_i32, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _P3]),
    "jxlb200_modular_squeeze_dev": (_i32, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp]),
    "jxlb200_upsample": (_i32, [_vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "jxlb200_noise": (_i32, [_vp, _P3, _i32, _i32, _i32, C.c_int64, _vp, C.c_float, C.c_float]),
    "jxlb200_splines": (_i32, [_vp, _P3, _i32, _i32, _i32, _vp, _vp, _vp, _i32, C.c_float, C.c_float]),
    "jxlb200_pack_samples": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "jxlb200_lf_dequant": (_i32, [_vp, _i32, _i32, _vp, C.c_float, C.c_float, _i32, _i32, _P3, _vp, _P3]),
    "jxlb200_blend_batch": (_i32, [_vp, _i32, C.POINTER(_vp), _vp, _vp, _vp, _i32, _vp]),
    "jxlb200_blend": (_i32, [_vp, _vp, _i32, _i32, _vp, C.c_int64, _vp, C.c_int64, _vp, C.c_int64, _vp, C.c_int64, _vp, C.c_int64]),
    "jxlb200_lf_dequant_dev": (_i32, [_vp, _i32, _i32, _vp, C.c_float, C.c_float, _i32, _i32, _P3, _vp, _P3]),
    "jxlb200_restore_uniform_dev": (_i32, [_vp, _FP, C.c_float, _P3, _P3]),
    "jxlb200_color_transform_dev": (_i32, [_vp, _FP, _P3, _P3]),
    "jxlb200_upsample_dev": (_i32, [_vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "jxlb200_noise_dev": (_i32, [_vp, _P3, _i32, _i32, _i32, C.c_int64, _vp, C.c_float, C.c_float]),
    "jxlb200_splines_dev": (_i32, [_vp, _P3, _i32, _i32, _i32, _vp, _vp, _vp, _i32, C.c_float, C.c_float]),
    "jxlb200_blend_batch_dev": (_i32, [_vp, _i32, C.POINTER(_vp), _vp, _vp, _i32, _vp]),
    "jxlb200_pack_samples_dev": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "jxlb200_cast_to_float_dev": (_i32, [_vp, _vp, C.c_int64, C.c_float, _vp]),
    "jxlb200_modular_xyb_dev": (_i32, [_vp, _P3, C.c_int64, _vp, _P3]),
    "jxlb200_lf_preview": (_i32, [_vp, _FP, _vp, C.c_float, C.c_float, _i32, _P3, _vp, _i32, _i32, _i32, _P3]),
    "jxlb200_lf_preview_dev": (_i32, [_vp, _FP, _vp, C.c_float, C.c_float, _i32, _P3, _vp, _i32, _i32, _i32, _P3]),
    "jxlb200_area_mean8": (_i32, [_vp, _i32, _P3, _vp, _vp, _i32, _i32, _P3]),
    "jxlb200_area_mean8_dev": (_i32, [_vp, _i32, _P3, _vp, _vp, _i32, _i32, _P3]),
    "jxlb200_pack_batch_dev": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp]),
}


class BlendOp(C.Structure):
    _fields_ = [("mode", C.c_int32), ("is_int", C.c_int32), ("is_alpha", C.c_int32), ("has_extra", C.c_int32),
                ("clamp", C.c_int32), ("premult", C.c_int32)]

class BlendItem(C.Structure):
    _fields_ = [("op", BlendOp), ("h", C.c_int32), ("w", C.c_int32), ("plane", C.c_int32 * 5), ("y", C.c_int32 * 5), ("x", C.c_int32 * 5)]


class BatchItem(C.Structure):
    _fields_ = [("plane", _vp * 4), ("is_int", C.c_int32 * 4), ("depth", C.c_int32 * 4), ("h", C.c_int32), ("w", C.c_int32),
                ("pitch", C.c_int32 * 4), ("orientation", C.c_int32), ("linear", C.c_int32)]


_LIB = None


def lib():
    """The loaded library.  Raises if it cannot be built or loaded (no silent fallback)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            from . import build
            build.build()
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)   # AttributeError here = header and library drifted apart
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def planes(ptrs):
    """int/ctypes pointers -> `const T *const p[n]` argument."""
    return (_vp * len(ptrs))(*[_vp(int(p)) if not isinstance(p, _vp) else p for p in ptrs])
