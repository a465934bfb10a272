"""ctypes bindings for the CPU checkers (oracle/libovrfsr_oracle.so, oracle/_ref/libovrfsr_ref.so).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package (openvr_fsr_b200) never imports this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
FMT_RGBA8, FMT_BGRA8, FMT_RGBA16F, FMT_RGBA32F, FMT_RGB10A2, FMT_BGRX8, FMT_RGB32F = 0, 1, 2, 3, 4, 5, 6


class Image(C.Structure):
    _fields_ = [("data", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32),
                ("pitch", C.c_int32), ("format", C.c_int32)]


class UpscaleConstants(C.Structure):
    _fields_ = [("const0", C.c_uint32 * 4), ("const1", C.c_uint32 * 4), ("const2", C.c_uint32 * 4),
                ("const3", C.c_uint32 * 4), ("imageCentre", C.c_uint32 * 4), ("radius", C.c_uint32 * 4)]

    def words(self):
        return np.frombuffer(bytes(self), dtype=np.uint32).copy()


class SharpenConstants(C.Structure):
    _fields_ = [("const0", C.c_uint32 * 4), ("imageCentre", C.c_uint32 * 4), ("radius", C.c_uint32 * 4)]

    def words(self):
        return np.frombuffer(bytes(self), dtype=np.uint32).copy()


class NISConfig(C.Structure):
    _fields_ = [(n, C.c_float) for n in (
        "kDetectRatio", "kDetectThres", "kMinContrastRatio", "kRatioNorm", "kContrastBoost", "kEps",
        "kSharpStartY", "kSharpScaleY", "kSharpStrengthMin", "kSharpStrengthScale", "kSharpLimitMin",
        "kSharpLimitScale", "kScaleX", "kScaleY", "kDstNormX", "kDstNormY", "kSrcNormX", "kSrcNormY")] + \
        [(n, C.c_uint32) for n in (
            "kInputViewportOriginX", "kInputViewportOriginY", "kInputViewportWidth", "kInputViewportHeight",
            "kOutputViewportOriginX", "kOutputViewportOriginY", "kOutputViewportWidth", "kOutputViewportHeight")] + \
        [("reserved0", C.c_float), ("reserved1", C.c_float), ("imageCentre", C.c_uint32 * 4),
         ("radius", C.c_uint32 * 4), ("pad_", C.c_uint32 * 28)]

    def words(self):
        return np.frombuffer(bytes(self), dtype=np.uint32).copy()


class CasConstants(C.Structure):
    """cb of src/cas/cas.compute.h:1-4"""
    _fields_ = [("const0", C.c_uint32 * 4), ("const1", C.c_uint32 * 4)]

    def words(self):
        return np.frombuffer(bytes(self), dtype=np.uint32).copy()


assert C.sizeof(UpscaleConstants) == 96 and C.sizeof(SharpenConstants) == 48 and C.sizeof(NISConfig) == 256


def build(force: bool = False) -> None:
    """Compile the restated oracle (always) and oracle/_ref (only where /root/reference exists)."""
    so = HERE / "libovrfsr_oracle.so"
    srcs = [p for p in HERE.iterdir() if p.suffix in (".c", ".h", ".inc")]
    if force or not so.exists() or any(p.stat().st_mtime > so.stat().st_mtime for p in srcs):
        subprocess.check_call(["make", "-C", str(HERE), "libovrfsr_oracle.so"], stdout=subprocess.DEVNULL)
    ref_root = Path(os.environ.get("OVRFSR_REFERENCE", "/root/reference"))
    ref_so = HERE / "_ref" / "libovrfsr_ref.so"
    try:
        have_ref = (ref_root / "src/fsr/ffx_fsr1.h").exists()
    except OSError:  # a parent directory this user may not search: the sources are not available to it
        have_ref = False
    if have_ref:
        shim = list((HERE / "ref_shim").glob("*.cpp")) + [HERE / "build_ref.sh", HERE / "ovr_glue.h",
                                                           HERE / "fsr_entry.inc"]
        if force or not ref_so.exists() or any(p.stat().st_mtime > ref_so.stat().st_mtime for p in shim if p.exists()):
            subprocess.check_call(["bash", str(HERE / "build_ref.sh")], stdout=subprocess.DEVNULL)


_PI = C.POINTER(Image)


def _sig(lib, prefix):
    for name, ctype in (("fsr_easu", UpscaleConstants), ("fsr_rcas", SharpenConstants),
                        ("nis_scaler", NISConfig), ("nis_sharpen", NISConfig)):
        fn = getattr(lib, prefix + name, None)
        if fn is not None:
            fn.argtypes = [_PI, _PI, C.POINTER(ctype), C.c_int]
            fn.restype = C.c_int


_oracle = None
_ref = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        build()
        lib = C.CDLL(str(HERE / "libovrfsr_oracle.so"))
        _sig(lib, "ovo_")
        u32p, f32p = C.POINTER(C.c_uint32), C.POINTER(C.c_float)
        lib.ovo_output_size.argtypes = [C.c_uint32, C.c_uint32, C.c_float, u32p, u32p]
        lib.ovo_fsr_easu_con.argtypes = [u32p] + [C.c_float] * 6
        lib.ovo_fsr_rcas_con.argtypes = [u32p, C.c_float]
        lib.ovo_make_upscale_constants.argtypes = [C.POINTER(UpscaleConstants), C.c_int, C.c_int, C.c_uint32,
                                                   C.c_uint32, C.c_uint32, C.c_uint32, f32p, C.c_float]
        lib.ovo_make_sharpen_constants.argtypes = [C.POINTER(SharpenConstants), C.c_int, C.c_int, C.c_uint32,
                                                   C.c_uint32, f32p, C.c_float, C.c_float, C.c_int]
        if hasattr(lib, "ovo_make_nis_config"):
            lib.ovo_make_nis_config.argtypes = [C.POINTER(NISConfig), C.c_int, C.c_int, C.c_int, C.c_uint32,
                                                C.c_uint32, C.c_uint32, C.c_uint32, f32p, C.c_float, C.c_float,
                                                C.c_int]
            lib.ovo_make_nis_config.restype = C.c_int
            lib.ovo_nis_coef_scale.restype = f32p
            lib.ovo_nis_coef_usm.restype = f32p
        lib.ovo_group_inside.argtypes = [C.c_uint32] * 4 + [u32p, C.c_uint32]
        lib.ovo_group_inside.restype = C.c_int
        lib.ovo_cas_setup.argtypes = [C.POINTER(CasConstants)] + [C.c_float] * 6
        lib.ovo_cas.argtypes = [_PI, _PI, C.POINTER(CasConstants), C.c_int, C.c_int]
        lib.ovo_cas.restype = C.c_int
        _oracle = lib
    return _oracle


DXGI_OF_FORMAT = {FMT_RGBA8: 28, FMT_BGRA8: 87, FMT_RGBA16F: 10, FMT_RGBA32F: 2, FMT_RGB10A2: 24}  # dxgiformat.h values


def ref_dds_header(width: int, height: int, fmt: int, bytes_per_texel: int) -> bytes:
    """The DDS file header SaveDDSTextureToFile writes (ScreenGrab11.cpp:72-208,819-906 compiled from the reference's own
    lines, oracle/ref_shim/dds_ref.cpp) for an uncompressed texture of ovrfsr format `fmt` with tight rows."""
    buf = (C.c_uint8 * 148)()
    n = ref_lib().ref_dds_header(buf, width, height, DXGI_OF_FORMAT[fmt], width * bytes_per_texel)
    if n <= 0:
        raise RuntimeError(f"reference rejects the format (rc={n})")
    return bytes(buf[:n])


def ref_available() -> bool:
    build()
    return (HERE / "_ref" / "libovrfsr_ref.so").exists()


def ref_lib():
    global _ref
    if _ref is None:
        build()
        lib = C.CDLL(str(HERE / "_ref" / "libovrfsr_ref.so"))
        _sig(lib, "ref_")
        u32p, f32p = C.POINTER(C.c_uint32), C.POINTER(C.c_float)
        lib.ref_FsrEasuCon.argtypes = [u32p] + [C.c_float] * 6
        lib.ref_FsrRcasCon.argtypes = [u32p, C.c_float]
        lib.ref_AClampF1.argtypes = [C.c_float] * 3
        lib.ref_AClampF1.restype = C.c_float
        lib.ref_NVScalerUpdateConfig.argtypes = [C.c_void_p, C.c_float] + [C.c_uint32] * 4
        lib.ref_NVSharpenUpdateConfig.argtypes = [C.c_void_p, C.c_float] + [C.c_uint32] * 2
        lib.ref_coef_scale.restype = f32p
        lib.ref_coef_usm.restype = f32p
        lib.ref_cas_setup.argtypes = [u32p, u32p] + [C.c_float] * 6
        lib.ref_cas.argtypes = [_PI, _PI, C.POINTER(CasConstants), C.c_int, C.c_int]
        lib.ref_cas.restype = C.c_int
        _ref = lib
    return _ref


# ---------------------------------------------------------------------------------------------
# numpy-level helpers
# ---------------------------------------------------------------------------------------------
def _np_format(arr: np.ndarray, fmt: int | None) -> int:
    if fmt is not None:
        return fmt
    return {np.dtype(np.float16): FMT_RGBA16F, np.dtype(np.float32): FMT_RGBA32F}.get(arr.dtype, FMT_RGBA8)


def as_image(arr: np.ndarray, fmt: int | None = None) -> Image:
    """arr: (H, W, 4) uint8, float16 or float32, C-contiguous rows (row pitch = arr.strides[0])."""
    if fmt == FMT_RGB32F:  # R32G32B32_FLOAT source: (H, W, 3) float32
        assert arr.ndim == 3 and arr.shape[2] == 3 and arr.dtype == np.float32 and arr.strides[1] == 12
        return Image(arr.ctypes.data, arr.shape[1], arr.shape[0], arr.strides[0], fmt)
    assert arr.ndim == 3 and arr.shape[2] == 4 and arr.dtype in (np.uint8, np.float16, np.float32)
    assert arr.strides[2] == arr.itemsize and arr.strides[1] == 4 * arr.itemsize
    return Image(arr.ctypes.data, arr.shape[1], arr.shape[0], arr.strides[0], _np_format(arr, fmt))


def output_size(in_w: int, in_h: int, render_scale: float) -> tuple[int, int]:
    w, h = C.c_uint32(), C.c_uint32()
    oracle_lib().ovo_output_size(in_w, in_h, render_scale, C.byref(w), C.byref(h))
    return w.value, h.value


def _proj(proj):
    return (C.c_float * 4)(*proj)


def upscale_constants(eye, only_one_eye, in_w, in_h, out_w, out_h, proj=(.5, .5, .5, .5), radius=0.5):
    c = UpscaleConstants()
    oracle_lib().ovo_make_upscale_constants(C.byref(c), eye, int(only_one_eye), in_w, in_h, out_w, out_h,
                                            _proj(proj), radius)
    return c


def sharpen_constants(eye, only_one_eye, out_w, out_h, proj=(.5, .5, .5, .5), radius=0.5, sharpness=0.9,
                      debug=False):
    c = SharpenConstants()
    oracle_lib().ovo_make_sharpen_constants(C.byref(c), eye, int(only_one_eye), out_w, out_h, _proj(proj),
                                            radius, sharpness, int(debug))
    return c


def nis_config(sharpen_only, eye, only_one_eye, in_w, in_h, out_w, out_h, proj=(.5, .5, .5, .5), radius=0.5,
               sharpness=0.9, debug=False):
    c = NISConfig()
    ok = oracle_lib().ovo_make_nis_config(C.byref(c), int(sharpen_only), eye, int(only_one_eye), in_w, in_h, out_w,
                                          out_h, _proj(proj), radius, sharpness, int(debug))
    return c, bool(ok)


def _run(fn, src: np.ndarray, out_shape, consts, out_dtype, nthreads, src_fmt=None, dst_fmt=None):
    dst = np.zeros((out_shape[0], out_shape[1], 4), dtype=out_dtype)
    s, d = as_image(src, src_fmt), as_image(dst, dst_fmt)
    rc = fn(C.byref(s), C.byref(d), C.byref(consts), nthreads)
    if rc != 0:
        raise RuntimeError(f"oracle pass failed rc={rc}")
    return dst


def _lib(which):
    return ref_lib() if which == "ref" else oracle_lib()


def _pfx(which):
    return "ref_" if which == "ref" else "ovo_"


def easu(src, out_w, out_h, consts, which="oracle", out_dtype=np.uint8, nthreads=1, src_fmt=None, dst_fmt=None):
    return _run(getattr(_lib(which), _pfx(which) + "fsr_easu"), src, (out_h, out_w), consts, out_dtype, nthreads,
                src_fmt, dst_fmt)


def rcas(src, consts, which="oracle", out_dtype=np.uint8, nthreads=1, src_fmt=None, dst_fmt=None):
    return _run(getattr(_lib(which), _pfx(which) + "fsr_rcas"), src, src.shape[:2], consts, out_dtype, nthreads,
                src_fmt, dst_fmt)


def nis_scaler(src, out_w, out_h, cfg, which="oracle", out_dtype=np.uint8, nthreads=1, src_fmt=None, dst_fmt=None):
    return _run(getattr(_lib(which), _pfx(which) + "nis_scaler"), src, (out_h, out_w), cfg, out_dtype, nthreads,
                src_fmt, dst_fmt)


def nis_sharpen(src, cfg, which="oracle", out_dtype=np.uint8, nthreads=1, src_fmt=None, dst_fmt=None):
    return _run(getattr(_lib(which), _pfx(which) + "nis_sharpen"), src, src.shape[:2], cfg, out_dtype, nthreads,
                src_fmt, dst_fmt)


# ---- legacy CAS path (src/cas) ---------------------------------------------------------------------------
def cas_setup(sharpness, max_color_delta, in_w, in_h, out_w, out_h, which="oracle") -> CasConstants:
    """CasSetup, src/cas/ffx_cas.h:375-397"""
    c = CasConstants()
    if which == "ref":
        ref_lib().ref_cas_setup(c.const0, c.const1, sharpness, max_color_delta, in_w, in_h, out_w, out_h)
    else:
        oracle_lib().ovo_cas_setup(C.byref(c), sharpness, max_color_delta, in_w, in_h, out_w, out_h)
    return c


def cas(src, out_w, out_h, consts, sharpen_only, which="oracle", out_dtype=np.uint8, nthreads=1, src_fmt=None, dst_fmt=None):
    """cas.sharpen.hlsl (sharpen_only) / cas.upscale.hlsl over the whole output, src/cas/cas.compute.h:25-47"""
    dst = np.zeros((out_h, out_w, 4), dtype=out_dtype)
    s, d = as_image(src, src_fmt), as_image(dst, dst_fmt)
    fn = ref_lib().ref_cas if which == "ref" else oracle_lib().ovo_cas
    rc = fn(C.byref(s), C.byref(d), C.byref(consts), int(bool(sharpen_only)), nthreads)
    if rc != 0:
        raise RuntimeError(f"CAS oracle pass failed rc={rc}")
    return dst
