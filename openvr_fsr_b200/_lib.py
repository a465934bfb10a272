"""ctypes binding of the C ABI (include/ovrfsr.h).  There is no fallback: if libovrfsr.so is missing the
import of the symbols raises, and any call that needs the GPU returns OVRFSR_ERR_CUDA without one."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

PKG = Path(__file__).resolve().parent
# OVRFSR_LIB: dev-only override used by tools/ A/B measurements against an older build of the library
LIB_PATH = Path(os.environ["OVRFSR_LIB"]) if os.environ.get("OVRFSR_LIB") else PKG / "libovrfsr.so"

OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_NOMEM, PASSTHROUGH = range(6)
FORMAT_RGBA8, FORMAT_BGRA8, FORMAT_RGBA16F, FORMAT_RGBA32F, FORMAT_RGB10A2, FORMAT_AUTO = 0, 1, 2, 3, 4, -1
FORMAT_BGRX8, FORMAT_RGB32F = 5, 6
FORMAT_SRGB_BIT, FORMAT_TYPELESS_BIT, FORMAT_LAYOUT_MASK = 0x100, 0x200, 0xff
MATH_FAST, MATH_STRICT = 0, 1
FLAG_FUSED_FSR = 1


class Image(C.Structure):
    _fields_ = [("data", C.c_void_p), ("width", C.c_uint32), ("height", C.c_uint32), ("pitch", C.c_uint32),
                ("format", C.c_int32), ("array_slices", C.c_uint32), ("slice_pitch", C.c_uint32),
                ("sample_count", C.c_uint32)]


class Bounds(C.Structure):
    _fields_ = [("u_min", C.c_float), ("v_min", C.c_float), ("u_max", C.c_float), ("v_max", C.c_float)]


class Rect(C.Structure):
    _fields_ = [("x", C.c_uint32), ("y", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32)]


class Config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("fsr_enabled", C.c_int32), ("use_nis", C.c_int32),
                ("render_scale", C.c_float), ("sharpness", C.c_float), ("radius", C.c_float),
                ("debug_mode", C.c_int32), ("proj_centre", C.c_float * 4), ("device", C.c_int32),
                ("output_format", C.c_int32), ("math_mode", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32 * 4)]


# every entry point include/ovrfsr.h declares: (restype, argtypes)
_u32p, _f32p, _imgp, _cfgp, _vp = C.POINTER(C.c_uint32), C.POINTER(C.c_float), C.POINTER(Image), C.POINTER(Config), C.c_void_p
SYMBOLS = {
    "ovrfsr_config_default": (None, [_cfgp]),
    "ovrfsr_create": (C.c_int, [C.POINTER(_vp), _cfgp]),
    "ovrfsr_destroy": (None, [_vp]),
    "ovrfsr_reset": (C.c_int, [_vp]),
    "ovrfsr_set_config": (C.c_int, [_vp, _cfgp]),
    "ovrfsr_get_config": (C.c_int, [_vp, _cfgp]),
    "ovrfsr_apply": (C.c_int, [_vp, C.c_int, _imgp, C.c_int, _imgp, _vp]),
    "ovrfsr_apply_host": (C.c_int, [_vp, C.c_int, _imgp, C.c_int, _imgp, _vp]),
    "ovrfsr_apply_pair": (C.c_int, [_vp, _imgp, _imgp, C.c_int, _imgp, _vp]),
    "ovrfsr_apply_bounds": (C.c_int, [_vp, C.c_int, _imgp, C.POINTER(Bounds), _imgp, C.POINTER(Rect), _vp]),
    "ovrfsr_bounds_rects": (C.c_int, [C.c_uint32] * 4 + [C.POINTER(Bounds), C.POINTER(Rect), C.POINTER(Rect)]),
    "ovrfsr_dispatch_fsr_easu": (C.c_int, [_imgp, _imgp, _u32p, C.c_int, _vp]),
    "ovrfsr_dispatch_fsr_rcas": (C.c_int, [_imgp, _imgp, _u32p, C.c_int, _vp]),
    "ovrfsr_dispatch_fsr_fused": (C.c_int, [_imgp, _imgp, _u32p, _u32p, C.c_int, _vp]),
    "ovrfsr_dispatch_nis_scaler": (C.c_int, [_imgp, _imgp, _vp, C.c_int, _vp]),
    "ovrfsr_dispatch_nis_sharpen": (C.c_int, [_imgp, _imgp, _vp, C.c_int, _vp]),
    "ovrfsr_output_size": (None, [C.c_uint32, C.c_uint32, C.c_float, _u32p, _u32p]),
    "ovrfsr_fsr_easu_con": (None, [_u32p] + [C.c_float] * 6),
    "ovrfsr_fsr_rcas_con": (None, [_u32p, C.c_float]),
    "ovrfsr_make_upscale_constants": (None, [_u32p, _cfgp, C.c_int, C.c_int] + [C.c_uint32] * 4),
    "ovrfsr_make_sharpen_constants": (None, [_u32p, _cfgp, C.c_int, C.c_int] + [C.c_uint32] * 2),
    "ovrfsr_make_nis_config": (C.c_int, [_vp, _cfgp, C.c_int, C.c_int, C.c_int] + [C.c_uint32] * 4),
    "ovrfsr_nis_coef_scale": (_f32p, []),
    "ovrfsr_nis_coef_usm": (_f32p, []),
    "ovrfsr_get_upscale_constants": (C.c_int, [_vp, C.c_int, _u32p]),
    "ovrfsr_get_sharpen_constants": (C.c_int, [_vp, C.c_int, _u32p]),
    "ovrfsr_selftest_rcp": (C.c_int, [_u32p, _u32p]),
    "ovrfsr_selftest_div": (C.c_int, [_u32p, _u32p]),
    "ovrfsr_kernel_launches": (C.c_uint64, []),
    "ovrfsr_get_gpu_time_ms": (C.c_int, [_vp, _f32p]),
    "ovrfsr_last_error": (C.c_char_p, [_vp]),
    "ovrfsr_status_string": (C.c_char_p, [C.c_int]),
    "ovrfsr_version": (C.c_uint32, []),
    "ovrfsr_image_alloc": (C.c_int, [_imgp, C.c_uint32, C.c_uint32, C.c_int32]),
    "ovrfsr_image_free": (None, [_imgp]),
    "ovrfsr_cas_setup": (None, [_u32p] + [C.c_float] * 6),
    "ovrfsr_dispatch_cas": (C.c_int, [_imgp, _imgp, _u32p, C.c_int, C.c_int, _vp]),
    "ovrfsr_resolve_msaa": (C.c_int, [_imgp, _imgp, _vp]),
    "ovrfsr_expand_rgb32f": (C.c_int, [_imgp, _imgp, _vp]),
    "ovrfsr_format_considered_srgb": (C.c_int, [C.c_int32]),
    "ovrfsr_recommended_render_size": (None, [_cfgp, _u32p, _u32p]),
    "ovrfsr_mip_lod_bias": (C.c_float, [C.c_uint32, C.c_uint32]),
    "ovrfsr_sampler_lod_bias": (C.c_float, [C.c_float, C.c_uint32, C.c_float]),
    "ovrfsr_request_capture": (C.c_int, [_vp, C.c_char_p]),
    "ovrfsr_last_capture_path": (C.c_char_p, [_vp]),
    "ovrfsr_capture_filename": (C.c_int, [_cfgp, C.c_int64, C.c_char_p, C.c_uint32]),
    "ovrfsr_dds_write": (C.c_int, [C.c_char_p, _imgp]),
    "ovrfsr_dds_read": (C.c_int, [C.c_char_p, _imgp]),
    "ovrfsr_host_free": (None, [_vp]),
}

_lib = None


def lib():
    """Load libovrfsr.so (built in-tree by openvr_fsr_b200.build).  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -m openvr_fsr_b200.build` "
                               "(there is no CPU fallback for the CUDA path)")
        l = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SYMBOLS.items():
            if os.environ.get("OVRFSR_LIB") and not hasattr(l, name):
                continue  # an older build under A/B measurement
            fn = getattr(l, name)  # AttributeError if the library does not export it
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


class OvrFsrError(RuntimeError):
    def __init__(self, status: int, what: str = ""):
        self.status = status
        msg = lib().ovrfsr_status_string(status).decode()
        super().__init__(f"{what}: {msg}" if what else msg)


def check(status: int, what: str = "", ctx=None):
    if status != OK:
        detail = what
        if ctx is not None:
            err = lib().ovrfsr_last_error(ctx)
            if err:
                detail = f"{what} ({err.decode()})"
        raise OvrFsrError(status, detail)
