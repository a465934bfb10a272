"""Python mirror of the reference's post-process surface, over the C ABI.

`PostProcessor.apply / reset` keep the names and argument meaning of vr::PostProcessor::Apply / Reset
(/root/reference/src/postprocess/PostProcessor.h:12-13); `Config` carries the fields of the reference's
Config singleton that steer this path (src/postprocess/Config.h:11-17).  Images are torch CUDA tensors
(H, W, 4) uint8 or float16 -- torch only provides device memory and streams here.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _lib as L


@dataclass
class Config:
    """src/postprocess/Config.h:11-17 plus the projection centres the reference reads from IVRSystem."""
    fsrEnabled: bool = False
    useNis: bool = False
    renderScale: float = 1.0
    sharpness: float = 0.75
    radius: float = 0.5
    debugMode: bool = False
    projCentre: tuple = (0.5, 0.5, 0.5, 0.5)
    device: int = -1
    outputFormat: int = L.FORMAT_AUTO
    mathMode: int = L.MATH_STRICT
    fusedFsr: bool = False  # OVRFSR_FLAG_FUSED_FSR: one fused EASU->RCAS kernel instead of the two dispatches (slower on B200)

    def to_c(self) -> L.Config:
        c = L.Config()
        L.lib().ovrfsr_config_default(C.byref(c))
        c.fsr_enabled, c.use_nis = int(self.fsrEnabled), int(self.useNis)
        c.render_scale, c.sharpness, c.radius = self.renderScale, self.sharpness, self.radius
        c.debug_mode = int(self.debugMode)
        c.proj_centre = (C.c_float * 4)(*self.projCentre)
        c.device, c.output_format, c.math_mode = self.device, self.outputFormat, self.mathMode
        c.flags = L.FLAG_FUSED_FSR if self.fusedFsr else 0
        return c


@dataclass
class TextureBounds:
    """VRTextureBounds_t, headers/openvr.h:609-613"""
    uMin: float = 0.0
    vMin: float = 0.0
    uMax: float = 1.0
    vMax: float = 1.0


EYE_LEFT, EYE_RIGHT = 0, 1


def _format_of(t) -> int:
    import torch
    if t.dtype == torch.uint8:
        return L.FORMAT_RGBA8
    if t.dtype == torch.float16:
        return L.FORMAT_RGBA16F
    if t.dtype == torch.float32:
        return L.FORMAT_RGBA32F
    raise TypeError("eye textures are uint8 (RGBA8/BGRA8), float16 (RGBA16F) or float32 (RGBA32F) tensors (H, W, 4)")


def image_of(t, fmt: int | None = None, samples: int = 1) -> L.Image:
    """Describe a (H, W, 4) tensor (CUDA or pinned host) as an ovrfsr_image; rows may be strided.  With
    samples > 1 the tensor is (H, W * samples, 4): the samples of one texel are consecutive (multisampled source)."""
    if fmt is not None and (fmt & L.FORMAT_LAYOUT_MASK) == L.FORMAT_RGB32F and fmt >= 0:
        # R32G32B32_FLOAT: (H, W, 3) float32, 12-byte texels
        if t.dim() != 3 or t.shape[2] != 3 or t.stride(2) != 1 or t.stride(1) != 3:
            raise ValueError("an RGB32F image is a (H, W, 3) float32 tensor with packed pixels")
        return L.Image(t.data_ptr(), t.shape[1], t.shape[0], t.stride(0) * t.element_size(), fmt, 1, 0, 0)
    if t.dim() != 3 or t.shape[2] != 4 or t.stride(2) != 1 or t.stride(1) != 4:
        raise ValueError("expected a (H, W, 4) tensor with packed pixels")
    if samples > 1 and t.shape[1] % samples:
        raise ValueError("row length is not a multiple of the sample count")
    return L.Image(t.data_ptr(), t.shape[1] // max(samples, 1), t.shape[0], t.stride(0) * t.element_size(),
                   _format_of(t) if fmt is None else fmt, 1, 0, samples if samples > 1 else 0)


def alloc_image(width: int, height: int, dtype=None, device="cuda", align: int = 256):
    """A (H, W, 4) device tensor whose row pitch is a multiple of `align` bytes -- what cudaMallocPitch /
    ovrfsr_image_alloc give, and what the TMA tile loader needs (base and pitch 16-byte aligned).  The padding
    bytes are never read or written by the kernels."""
    import torch
    dtype = dtype or torch.uint8
    esize = torch.empty((), dtype=dtype).element_size()
    row = width * 4 * esize
    pitch = (row + align - 1) // align * align
    buf = torch.zeros((height, pitch // esize), dtype=dtype, device=device)
    return buf[:, : width * 4].view(height, width, 4) if pitch == row else torch.as_strided(
        buf, (height, width, 4), (pitch // esize, 4, 1))


def to_image(array, device="cuda", align: int = 256):
    """Copy a numpy (H, W, 4) array into a pitch-aligned device image."""
    import torch
    src = torch.from_numpy(array)
    img = alloc_image(array.shape[1], array.shape[0], src.dtype, device, align)
    img.copy_(src)
    return img


def output_size(in_w: int, in_h: int, render_scale: float) -> tuple[int, int]:
    """PrepareResources, PostProcessor.cpp:509-518"""
    w, h = C.c_uint32(), C.c_uint32()
    L.lib().ovrfsr_output_size(in_w, in_h, render_scale, C.byref(w), C.byref(h))
    return w.value, h.value


def _stream_ptr(stream) -> int:
    import torch
    if stream is None:
        if not torch.cuda.is_available():
            return 0  # the C ABI then reports OVRFSR_ERR_CUDA itself (no device)
        stream = torch.cuda.current_stream()
    return stream.cuda_stream


class PostProcessor:
    """Drop-in for vr::PostProcessor on this path: apply(eye, texture, bounds) returns the texture the hook
    would hand on to the real Submit (the ctx-owned upscaled/sharpened eye), or the input itself when
    post-processing is disabled -- the reference's pass-through behaviour (PostProcessor.cpp:124,145-152)."""

    def __init__(self, config: Config):
        self._ctx = C.c_void_p()
        self.config = config
        L.check(L.lib().ovrfsr_create(C.byref(self._ctx), C.byref(config.to_c())), "ovrfsr_create")

    def close(self):
        if self._ctx:
            L.lib().ovrfsr_destroy(self._ctx)
            self._ctx = C.c_void_p()

    __del__ = close

    def reset(self):
        """vr::PostProcessor::Reset"""
        L.check(L.lib().ovrfsr_reset(self._ctx), "ovrfsr_reset", self._ctx)

    def set_config(self, config: Config):
        """What the hotkeys do: mutate Config, then Reset (PostProcessor.cpp:670-704)."""
        self.config = config
        L.check(L.lib().ovrfsr_set_config(self._ctx, C.byref(config.to_c())), "ovrfsr_set_config", self._ctx)

    def apply(self, eye: int, texture, bounds: TextureBounds | None = None, fmt: int | None = None, stream=None,
              samples: int = 1):
        """vr::PostProcessor::Apply.  Returns a torch tensor VIEW of the ctx-owned output (valid until the next
        apply for this eye / reset), or `texture` itself on pass-through.  samples > 1: `texture` is a multisampled
        source (see image_of) and is resolved first, as GetInputView does."""
        import torch
        bounds = bounds or TextureBounds()
        only_one_eye = int(abs(bounds.uMax - bounds.uMin) > 0.5)  # PostProcessor.cpp:146
        src, out = image_of(texture, fmt, samples), L.Image()
        rc = L.lib().ovrfsr_apply(self._ctx, eye, C.byref(src), only_one_eye, C.byref(out), _stream_ptr(stream))
        if rc == L.PASSTHROUGH:
            return texture
        L.check(rc, "ovrfsr_apply", self._ctx)
        self.last_output_format = out.format  # RGBA8, or RGB10A2 for a 10-bit source (bytes of the packed u32 texels)
        return _wrap_device(out, texture.device)

    def apply_pair(self, left, right, bounds: TextureBounds | None = None, fmt: int | None = None, stream=None):
        """Both eyes of a frame in one call (ovrfsr_apply_pair): the same outputs as apply(0, left) then apply(1, right)
        on `stream`, with the right eye's passes forked onto a ctx-owned stream and joined back before returning.
        Returns (left_out, right_out), or the inputs on pass-through."""
        bounds = bounds or TextureBounds()
        only_one_eye = int(abs(bounds.uMax - bounds.uMin) > 0.5)
        sl, sr, outs = image_of(left, fmt), image_of(right, fmt), (L.Image * 2)()
        rc = L.lib().ovrfsr_apply_pair(self._ctx, C.byref(sl), C.byref(sr), only_one_eye, outs, _stream_ptr(stream))
        if rc == L.PASSTHROUGH:
            return left, right
        L.check(rc, "ovrfsr_apply_pair", self._ctx)
        self.last_output_format = outs[0].format
        return _wrap_device(outs[0], left.device), _wrap_device(outs[1], right.device)

    def apply_bounds(self, eye: int, texture, bounds: TextureBounds | None = None, fmt: int | None = None, stream=None,
                     samples: int = 1):
        """ovrfsr_apply_bounds: post-process only the `bounds` rectangle of the eye texture, as if it had been cut out
        as a texture of its own, and write the result at the matching rectangle of the full-size output.  Returns
        (output view, (x, y, w, h) of the output rectangle), or (`texture`, None) on pass-through."""
        b = bounds or TextureBounds()
        cb, rect = L.Bounds(b.uMin, b.vMin, b.uMax, b.vMax), L.Rect()
        src, out = image_of(texture, fmt, samples), L.Image()
        rc = L.lib().ovrfsr_apply_bounds(self._ctx, eye, C.byref(src), C.byref(cb), C.byref(out), C.byref(rect),
                                         _stream_ptr(stream))
        if rc == L.PASSTHROUGH:
            return texture, None
        L.check(rc, "ovrfsr_apply_bounds", self._ctx)
        self.last_output_format = out.format
        return _wrap_device(out, texture.device), (rect.x, rect.y, rect.width, rect.height)

    def apply_host(self, eye: int, src_host, dst_host, bounds: TextureBounds | None = None, fmt: int | None = None,
                   stream=None, dst_fmt: int | None = None):
        """End-to-end entry: host (pinned) tensors in and out, copies included, asynchronous on `stream`."""
        bounds = bounds or TextureBounds()
        only_one_eye = int(abs(bounds.uMax - bounds.uMin) > 0.5)
        s, d = image_of(src_host, fmt), image_of(dst_host, dst_fmt)
        L.check(L.lib().ovrfsr_apply_host(self._ctx, eye, C.byref(s), only_one_eye, C.byref(d), _stream_ptr(stream)),
                "ovrfsr_apply_host", self._ctx)

    def request_capture(self, directory: str = ""):
        """The F7 hotkey (PostProcessor.cpp:699-702): the next left-eye apply writes its output as a DDS file."""
        L.check(L.lib().ovrfsr_request_capture(self._ctx, directory.encode()), "ovrfsr_request_capture", self._ctx)

    def last_capture_path(self) -> str:
        return L.lib().ovrfsr_last_capture_path(self._ctx).decode()

    def upscale_constants(self, eye: int) -> np.ndarray:
        w = (C.c_uint32 * 24)()
        L.check(L.lib().ovrfsr_get_upscale_constants(self._ctx, eye, w), "get_upscale_constants")
        return np.array(w, dtype=np.uint32)

    def sharpen_constants(self, eye: int) -> np.ndarray:
        w = (C.c_uint32 * 12)()
        L.check(L.lib().ovrfsr_get_sharpen_constants(self._ctx, eye, w), "get_sharpen_constants")
        return np.array(w, dtype=np.uint32)

    def gpu_time_ms(self):
        ms = C.c_float()
        n = L.lib().ovrfsr_get_gpu_time_ms(self._ctx, C.byref(ms))
        return (ms.value, n) if n else (None, 0)


def _wrap_device(img: L.Image, device):
    """torch view over a ctx-owned device image (no copy)."""
    import torch
    elem = {L.FORMAT_RGBA16F: 2, L.FORMAT_RGBA32F: 4}.get(img.format, 1)
    nbytes = img.pitch * img.height

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (img.data, False), "version": 2}
    flat = torch.as_tensor(h, device=device)
    if elem == 2:
        return torch.as_strided(flat.view(torch.float16), (img.height, img.width, 4), (img.pitch // 2, 4, 1))
    if elem == 4:
        return torch.as_strided(flat.view(torch.float32), (img.height, img.width, 4), (img.pitch // 4, 4, 1))
    return torch.as_strided(flat, (img.height, img.width, 4), (img.pitch, 4, 1))


# ---- the individual dispatches (ApplyUpscaling / ApplySharpening) on tensors ---------------------------
def _dispatch(fn, src, dst, consts, math_mode, stream, src_fmt=None, dst_fmt=None):
    s, d = image_of(src, src_fmt), image_of(dst, dst_fmt)
    L.check(fn(C.byref(s), C.byref(d), consts, math_mode, _stream_ptr(stream)), fn.__name__)
    return dst


def fsr_easu(src, dst, consts24, math_mode=L.MATH_FAST, stream=None, src_fmt=None, dst_fmt=None):
    c = (C.c_uint32 * 24)(*[int(x) for x in consts24])
    return _dispatch(L.lib().ovrfsr_dispatch_fsr_easu, src, dst, c, math_mode, stream, src_fmt, dst_fmt)


def fsr_rcas(src, dst, consts12, math_mode=L.MATH_FAST, stream=None, src_fmt=None, dst_fmt=None):
    c = (C.c_uint32 * 12)(*[int(x) for x in consts12])
    return _dispatch(L.lib().ovrfsr_dispatch_fsr_rcas, src, dst, c, math_mode, stream, src_fmt, dst_fmt)


def fsr_fused(src, dst, consts24, consts12, math_mode=L.MATH_STRICT, stream=None, src_fmt=None, dst_fmt=None):
    """ApplyUpscaling + ApplySharpening (FSR) as one kernel: bit-identical to fsr_easu followed by fsr_rcas."""
    cu = (C.c_uint32 * 24)(*[int(x) for x in consts24])
    cs = (C.c_uint32 * 12)(*[int(x) for x in consts12])
    s, d = image_of(src, src_fmt), image_of(dst, dst_fmt)
    L.check(L.lib().ovrfsr_dispatch_fsr_fused(C.byref(s), C.byref(d), cu, cs, math_mode, _stream_ptr(stream)),
            "ovrfsr_dispatch_fsr_fused")
    return dst


def nis_scaler(src, dst, cfg256: bytes, math_mode=L.MATH_FAST, stream=None, src_fmt=None, dst_fmt=None):
    buf = C.create_string_buffer(bytes(cfg256), 256)
    return _dispatch(L.lib().ovrfsr_dispatch_nis_scaler, src, dst, C.cast(buf, C.c_void_p), math_mode, stream, src_fmt, dst_fmt)


def nis_sharpen(src, dst, cfg256: bytes, math_mode=L.MATH_FAST, stream=None, src_fmt=None, dst_fmt=None):
    buf = C.create_string_buffer(bytes(cfg256), 256)
    return _dispatch(L.lib().ovrfsr_dispatch_nis_sharpen, src, dst, C.cast(buf, C.c_void_p), math_mode, stream, src_fmt, dst_fmt)


def cas_setup(sharpness, max_color_delta, in_w, in_h, out_w, out_h) -> np.ndarray:
    """CasSetup, src/cas/ffx_cas.h:375-397: const0 and const1 as 8 words"""
    w = (C.c_uint32 * 8)()
    L.lib().ovrfsr_cas_setup(w, sharpness, max_color_delta, in_w, in_h, out_w, out_h)
    return np.array(w, dtype=np.uint32)


def cas(src, dst, consts8, sharpen_only: bool, math_mode=L.MATH_STRICT, stream=None, src_fmt=None, dst_fmt=None):
    """The legacy CAS shaders (src/cas/cas.compute.h:25-47): sharpen in place size or adaptive upscale"""
    c = (C.c_uint32 * 8)(*[int(x) for x in consts8])
    s, d = image_of(src, src_fmt), image_of(dst, dst_fmt)
    L.check(L.lib().ovrfsr_dispatch_cas(C.byref(s), C.byref(d), c, int(bool(sharpen_only)), math_mode, _stream_ptr(stream)),
            "ovrfsr_dispatch_cas")
    return dst


def resolve_msaa(src_samples, dst, samples: int, stream=None, fmt=None):
    """GetInputView's ResolveSubresource (PostProcessor.cpp:219-226): (H, W*samples, 4) -> (H, W, 4) mean."""
    s, d = image_of(src_samples, fmt, samples), image_of(dst, fmt)
    L.check(L.lib().ovrfsr_resolve_msaa(C.byref(s), C.byref(d), _stream_ptr(stream)), "ovrfsr_resolve_msaa")
    return dst


def expand_rgb32f(src, dst, stream=None):
    """R32G32B32_FLOAT (H, W, 3) float32 -> RGBA32F (H, W, 4) with alpha 1 (PostProcessor.cpp:34-35: such a view reads 1 in .w)."""
    s, d = image_of(src, L.FORMAT_RGB32F), image_of(dst, L.FORMAT_RGBA32F)
    L.check(L.lib().ovrfsr_expand_rgb32f(C.byref(s), C.byref(d), _stream_ptr(stream)), "ovrfsr_expand_rgb32f")
    return dst


def format_considered_srgb(tagged_format: int) -> bool:
    """IsConsideredSrgbByOpenVR, PostProcessor.cpp:76-92, on a tagged ovrfsr_format"""
    return bool(L.lib().ovrfsr_format_considered_srgb(int(tagged_format)))


def recommended_render_size(cfg: Config, width: int, height: int) -> tuple[int, int]:
    """IVRSystem_GetRecommendedRenderTargetSize detour, VrHooks.cpp:37-48"""
    w, h = C.c_uint32(width), C.c_uint32(height)
    L.lib().ovrfsr_recommended_render_size(C.byref(cfg.to_c()), C.byref(w), C.byref(h))
    return w.value, h.value


def mip_lod_bias(input_width: int, output_width: int) -> float:
    """PostProcessor.cpp:537-538"""
    return L.lib().ovrfsr_mip_lod_bias(input_width, output_width)


def sampler_lod_bias(sampler_bias: float, max_anisotropy: int, bias: float) -> float:
    """VrHooks.cpp:123-128"""
    return L.lib().ovrfsr_sampler_lod_bias(sampler_bias, max_anisotropy, bias)


def capture_filename(cfg: Config, unix_time: int) -> str:
    """PostProcessor.cpp:641-652"""
    buf = C.create_string_buffer(96)
    L.check(L.lib().ovrfsr_capture_filename(C.byref(cfg.to_c()), int(unix_time), buf, 96), "ovrfsr_capture_filename")
    return buf.value.decode()


def save_dds(path: str, array: np.ndarray, fmt: int | None = None):
    """Write a HOST (H, W, 4) array as the DDS file the F7 capture produces (ScreenGrab11.cpp:815-935)."""
    a = np.ascontiguousarray(array)
    f = fmt if fmt is not None else {np.dtype(np.float16): L.FORMAT_RGBA16F, np.dtype(np.float32): L.FORMAT_RGBA32F}.get(a.dtype, L.FORMAT_RGBA8)
    img = L.Image(a.ctypes.data, a.shape[1], a.shape[0], a.strides[0], f, 1, 0, 0)
    L.check(L.lib().ovrfsr_dds_write(str(path).encode(), C.byref(img)), "ovrfsr_dds_write")


def load_dds(path: str) -> tuple[np.ndarray, int]:
    """Read such a file back: ((H, W, 4) array, ovrfsr_format)."""
    img = L.Image()
    L.check(L.lib().ovrfsr_dds_read(str(path).encode(), C.byref(img)), "ovrfsr_dds_read")
    try:
        dt = {L.FORMAT_RGBA16F: np.float16, L.FORMAT_RGBA32F: np.float32}.get(img.format, np.uint8)
        n = img.pitch * img.height
        raw = np.frombuffer(C.string_at(img.data, n), dtype=np.uint8).copy()
        return raw.view(dt).reshape(img.height, img.width, 4), img.format
    finally:
        L.lib().ovrfsr_host_free(img.data)


def bounds_rects(width: int, height: int, out_w: int, out_h: int, bounds: TextureBounds | None = None):
    """The source and output rectangles ovrfsr_apply_bounds uses, each (x, y, w, h); raises OvrFsrError
    (ERR_INVALID) for an empty rectangle."""
    b = bounds or TextureBounds()
    cb, s, d = L.Bounds(b.uMin, b.vMin, b.uMax, b.vMax), L.Rect(), L.Rect()
    L.check(L.lib().ovrfsr_bounds_rects(width, height, out_w, out_h, C.byref(cb), C.byref(s), C.byref(d)),
            "ovrfsr_bounds_rects")
    return (s.x, s.y, s.width, s.height), (d.x, d.y, d.width, d.height)


def make_upscale_constants(cfg: Config, eye, only_one_eye, in_w, in_h, out_w, out_h) -> np.ndarray:
    w = (C.c_uint32 * 24)()
    L.lib().ovrfsr_make_upscale_constants(w, C.byref(cfg.to_c()), eye, int(only_one_eye), in_w, in_h, out_w, out_h)
    return np.array(w, dtype=np.uint32)


def make_sharpen_constants(cfg: Config, eye, only_one_eye, out_w, out_h) -> np.ndarray:
    w = (C.c_uint32 * 12)()
    L.lib().ovrfsr_make_sharpen_constants(w, C.byref(cfg.to_c()), eye, int(only_one_eye), out_w, out_h)
    return np.array(w, dtype=np.uint32)


def make_nis_config(cfg: Config, sharpen_only, eye, only_one_eye, in_w, in_h, out_w, out_h):
    buf = C.create_string_buffer(256)
    ok = L.lib().ovrfsr_make_nis_config(C.cast(buf, C.c_void_p), C.byref(cfg.to_c()), int(sharpen_only), eye,
                                        int(only_one_eye), in_w, in_h, out_w, out_h)
    return buf.raw, bool(ok)


def kernel_launches() -> int:
    return int(L.lib().ovrfsr_kernel_launches())
