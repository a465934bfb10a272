"""ovrfsr_apply_bounds on the GPU: an eye submitted with texture bounds is processed exactly as if its rectangle had
been cut out as a texture of its own (the crop rule of include/ovrfsr.h), checked against the oracle on the numpy
crop, plus isolation from the texels / pixels outside the rectangles, dynamic resolution, side-by-side eyes and
consistency with ovrfsr_apply."""
import ctypes as C
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H = 203, 157
# source rectangles (x, y, w, h) in a W x H texture: every edge inside; x0 % 4 = 1, 2, 3; odd sizes; smaller than a
# tile; touching the right and bottom edges; the whole texture
RECTS = [(25, 31, 131, 97), (26, 8, 101, 139), (71, 50, 132, 107), (90, 60, 13, 7), (0, 0, W, H)]


def _bounds(r, w=W, h=H):
    import openvr_fsr_b200 as ovr
    x, y, rw, rh = r
    f = np.float32
    return ovr.TextureBounds(float(f(x) / f(w)), float(f(y) / f(h)), float(f(x + rw) / f(w)), float(f(y + rh) / f(h)))


def _crop(a, r):
    x, y, w, h = r
    return np.ascontiguousarray(a[y:y + h, x:x + w])


def _oracle(img, cfg, eye, s, d, src_fmt=None):
    """the oracle's passes on the cropped source, with the constants for the rectangle sizes and only_one_eye = 1"""
    from oracle import pyoracle as po
    crop = _crop(img, s)
    ten = src_fmt == po.FMT_RGB10A2
    ofmt = po.FMT_RGB10A2 if ten else None
    mid_fmt = po.FMT_RGB10A2 if ten else po.FMT_RGBA8
    kw = dict(proj=cfg.projCentre, radius=cfg.radius, sharpness=cfg.sharpness, debug=cfg.debugMode)
    if cfg.useNis:
        nc, _ = po.nis_config(cfg.renderScale == 1.0, eye, True, s[2], s[3], d[2], d[3], **kw)
        if cfg.renderScale == 1.0:
            return po.nis_sharpen(crop, nc, src_fmt=src_fmt, dst_fmt=ofmt)
        return po.nis_scaler(crop, d[2], d[3], nc, src_fmt=src_fmt, dst_fmt=ofmt)
    sc = po.sharpen_constants(eye, True, d[2], d[3], **kw)
    if cfg.renderScale == 1.0:
        return po.rcas(crop, sc, src_fmt=src_fmt, dst_fmt=ofmt)
    uc = po.upscale_constants(eye, True, s[2], s[3], d[2], d[3], proj=cfg.projCentre, radius=cfg.radius)
    mid = po.easu(crop, d[2], d[3], uc, src_fmt=src_fmt, dst_fmt=mid_fmt)
    return po.rcas(mid, sc, src_fmt=mid_fmt, dst_fmt=ofmt)


def _rects(cfg, r, w=W, h=H):
    import openvr_fsr_b200 as ovr
    ow, oh = ovr.output_size(w, h, cfg.renderScale)
    s, d = ovr.bounds_rects(w, h, ow, oh, _bounds(r, w, h))
    assert s == tuple(r)
    return s, d


def _apply(pp, eye, tex, r, fmt=None, w=W, h=H, samples=1):
    out, d = pp.apply_bounds(eye, tex, _bounds(r, w, h), fmt=fmt, samples=samples)
    return out, d


@pytest.mark.parametrize("use_nis", [False, True])
@pytest.mark.parametrize("scale", [0.75, 0.59, 1.0, 1.3])
def test_crop_equivalence_strict(cuda, use_nis, scale):
    import torch
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    img = synth.natural_rgba8(W, H, 31)
    for i, r in enumerate(RECTS):
        radius = (0.5, 2.0)[i % 2]
        cfg = ovr.Config(fsrEnabled=True, useNis=use_nis, renderScale=scale, sharpness=0.85, radius=radius,
                         projCentre=(0.41, 0.57, 0.62, 0.45), debugMode=(i == 2))
        s, d = _rects(cfg, r)
        for tex in (ovr.to_image(img, cuda), torch.from_numpy(img).to(cuda)):  # TMA / plain-load source reads
            pp = ovr.PostProcessor(cfg)
            for eye in (0, 1):
                out, got_d = _apply(pp, eye, tex, r)
                assert got_d == d
                got = _crop(out.cpu().numpy(), d)
                assert np.array_equal(got, _oracle(img, cfg, eye, s, d)), (r, eye)
            pp.close()


@pytest.mark.parametrize("fmt", ["rgba8", "bgra8", "bgrx8", "rgba16f", "rgba32f", "rgb10a2"])
@pytest.mark.parametrize("use_nis,scale", [(False, 0.75), (False, 1.0), (True, 0.75), (True, 1.0)])
def test_crop_equivalence_formats(cuda, fmt, use_nis, scale):
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    from oracle import pyoracle as po
    img, f, pf = {
        "rgba8": (synth.natural_rgba8(W, H, 5), ovr.FORMAT_RGBA8, None),
        "bgra8": (synth.natural_rgba8(W, H, 6), ovr.FORMAT_BGRA8, po.FMT_BGRA8),
        "bgrx8": (synth.natural_rgba8(W, H, 7), ovr.FORMAT_BGRX8, po.FMT_BGRX8),
        "rgba16f": (synth.natural_rgba16f(W, H, 8), ovr.FORMAT_RGBA16F, None),
        "rgba32f": (synth.natural_rgba16f(W, H, 9).astype(np.float32), ovr.FORMAT_RGBA32F, None),
        "rgb10a2": (synth.natural_rgb10a2(W, H, 10), ovr.FORMAT_RGB10A2, po.FMT_RGB10A2),
    }[fmt]
    cfg = ovr.Config(fsrEnabled=True, useNis=use_nis, renderScale=scale, sharpness=0.9, radius=0.5,
                     projCentre=(0.45, 0.52, 0.55, 0.5))
    pp = ovr.PostProcessor(cfg)
    tex = ovr.to_image(img, cuda)
    for r in RECTS[:4]:
        s, d = _rects(cfg, r)
        out, _ = _apply(pp, 0, tex, r, fmt=f)
        assert np.array_equal(_crop(out.cpu().numpy(), d), _oracle(img, cfg, 0, s, d, src_fmt=pf)), r
    pp.close()


@pytest.mark.parametrize("use_nis,scale", [(False, 0.75), (False, 1.0), (True, 0.75), (True, 1.0)])
def test_crop_equivalence_fast(cuda, use_nis, scale):
    """fast math: bit-equal to the stateless dispatches on a freshly allocated, aligned copy of the crop, and within
    the per-pass fast-math tolerances of the oracle (1 LSB per pass; <= 4 LSB for EASU -> RCAS composed)"""
    import torch
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    img = synth.natural_rgba8(W, H, 12)
    cfg = ovr.Config(fsrEnabled=True, useNis=use_nis, renderScale=scale, sharpness=0.9, radius=0.5,
                     projCentre=(0.45, 0.52, 0.55, 0.5), mathMode=ovr.MATH_FAST)
    pp = ovr.PostProcessor(cfg)
    tex = ovr.to_image(img, cuda)
    for r in RECTS[:4]:
        s, d = _rects(cfg, r)
        out, _ = _apply(pp, 0, tex, r)
        got = _crop(out.cpu().numpy(), d)
        crop = ovr.to_image(_crop(img, s), cuda)
        ref = ovr.alloc_image(d[2], d[3], torch.uint8, cuda)
        if use_nis:
            nc, _ = ovr.make_nis_config(cfg, scale == 1.0, 0, True, s[2], s[3], d[2], d[3])
            (ovr.nis_sharpen if scale == 1.0 else ovr.nis_scaler)(crop, ref, nc, ovr.MATH_FAST)
        elif scale == 1.0:
            ovr.fsr_rcas(crop, ref, ovr.make_sharpen_constants(cfg, 0, True, d[2], d[3]), ovr.MATH_FAST)
        else:
            mid = ovr.alloc_image(d[2], d[3], torch.uint8, cuda)
            ovr.fsr_easu(crop, mid, ovr.make_upscale_constants(cfg, 0, True, s[2], s[3], d[2], d[3]), ovr.MATH_FAST)
            ovr.fsr_rcas(mid, ref, ovr.make_sharpen_constants(cfg, 0, True, d[2], d[3]), ovr.MATH_FAST)
        torch.cuda.synchronize()
        assert np.array_equal(got, ref.cpu().numpy()), r
        strict = _oracle(img, cfg, 0, s, d)
        tol = 4 if (not use_nis and scale != 1.0) else 1
        assert np.abs(got.astype(np.int16) - strict.astype(np.int16)).max() <= tol, r
    pp.close()


@pytest.mark.parametrize("use_nis,scale", [(False, 0.75), (False, 1.0), (True, 0.75), (True, 1.0)])
def test_isolation(cuda, use_nis, scale):
    """texels outside the source rectangle never influence the result; pixels outside the output rectangle are not
    written"""
    import torch
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    img = synth.natural_rgba8(W, H, 14)
    cfg = ovr.Config(fsrEnabled=True, useNis=use_nis, renderScale=scale, sharpness=0.9, radius=0.5,
                     projCentre=(0.45, 0.52, 0.55, 0.5))
    rng = np.random.default_rng(3)
    for r in RECTS[:4]:
        s, d = _rects(cfg, r)
        outs = []
        for fill in ("garbage", "zeros"):
            a = rng.integers(0, 256, img.shape, dtype=np.uint8) if fill == "garbage" else np.zeros_like(img)
            a[s[1]:s[1] + s[3], s[0]:s[0] + s[2]] = _crop(img, s)
            pp = ovr.PostProcessor(cfg)
            out, _ = _apply(pp, 0, ovr.to_image(a, cuda), r)
            outs.append(_crop(out.cpu().numpy(), d))
            # sentinel everywhere, apply again: only the output rectangle changes
            out.fill_(0xA5)
            out2, _ = _apply(pp, 0, ovr.to_image(a, cuda), r)
            assert out2.data_ptr() == out.data_ptr()
            full = out2.cpu().numpy()
            mask = np.ones(full.shape[:2], bool)
            mask[d[1]:d[1] + d[3], d[0]:d[0] + d[2]] = False
            assert (full[mask] == 0xA5).all(), r
            assert np.array_equal(_crop(full, d), outs[-1])
            pp.close()
        assert np.array_equal(outs[0], outs[1]), r


@pytest.mark.parametrize("use_nis", [False, True])
def test_dynamic_resolution(cuda, use_nis):
    """one ctx, a rectangle that changes every frame at a fixed texture size: each frame matches the oracle and the
    output image is never reallocated"""
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    img = synth.natural_rgba8(W, H, 15)
    cfg = ovr.Config(fsrEnabled=True, useNis=use_nis, renderScale=0.75, sharpness=0.9, radius=0.6,
                     projCentre=(0.45, 0.52, 0.55, 0.5))
    pp = ovr.PostProcessor(cfg)
    tex = ovr.to_image(img, cuda)
    ptr = None
    for frame in range(8):
        sc = 1.0 - 0.07 * frame
        r = (frame * 3, frame, int(W * sc) - frame * 3, int(H * sc) - frame)
        s, d = _rects(cfg, r)
        out, _ = _apply(pp, frame % 2, tex, r)
        if frame % 2 == 0:
            ptr = out.data_ptr() if ptr is None else ptr
            assert out.data_ptr() == ptr
        assert np.array_equal(_crop(out.cpu().numpy(), d), _oracle(img, cfg, frame % 2, s, d)), frame
    pp.close()


@pytest.mark.parametrize("use_nis", [False, True])
def test_side_by_side_eyes(cuda, use_nis):
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    w2 = 2 * W
    img = synth.natural_rgba8(w2, H, 16)
    cfg = ovr.Config(fsrEnabled=True, useNis=use_nis, renderScale=0.75, sharpness=0.9, radius=0.5,
                     projCentre=(0.45, 0.52, 0.55, 0.5))
    ow, oh = ovr.output_size(w2, H, cfg.renderScale)
    pp = ovr.PostProcessor(cfg)
    tex = ovr.to_image(img, cuda)
    for eye, b in ((0, ovr.TextureBounds(0.0, 0.0, 0.5, 1.0)), (1, ovr.TextureBounds(0.5, 0.0, 1.0, 1.0))):
        s, d = ovr.bounds_rects(w2, H, ow, oh, b)
        assert s == (eye * W, 0, W, H)
        out, got_d = pp.apply_bounds(eye, tex, b)
        assert got_d == d
        assert np.array_equal(_crop(out.cpu().numpy(), d), _oracle(img, cfg, eye, s, d)), eye
    pp.close()


@pytest.mark.parametrize("use_nis,scale", [(False, 0.75), (False, 1.0), (True, 0.75), (True, 1.0)])
def test_consistency_with_apply(cuda, use_nis, scale):
    """full bounds = ovrfsr_apply; apply and apply_bounds alternated on one ctx each give their standalone results"""
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    img = synth.natural_rgba8(W, H, 17)
    cfg = ovr.Config(fsrEnabled=True, useNis=use_nis, renderScale=scale, sharpness=0.9, radius=0.5,
                     projCentre=(0.45, 0.52, 0.55, 0.5))
    tex = ovr.to_image(img, cuda)
    pp = ovr.PostProcessor(cfg)
    full = pp.apply(0, tex).cpu().numpy()
    pp.close()
    pp = ovr.PostProcessor(cfg)
    out, d = pp.apply_bounds(0, tex, None)
    assert d == (0, 0, full.shape[1], full.shape[0]) and np.array_equal(out.cpu().numpy(), full)
    pp.close()
    r = RECTS[0]
    s, d = _rects(cfg, r)
    want = _oracle(img, cfg, 0, s, d)
    pp = ovr.PostProcessor(cfg)
    for _ in range(2):
        assert np.array_equal(pp.apply(0, tex).cpu().numpy(), full)
        out, _ = _apply(pp, 0, tex, r)
        assert np.array_equal(_crop(out.cpu().numpy(), d), want)
    pp.close()


def test_fused_flag_gives_the_same_bits(cuda):
    import dataclasses
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    img = synth.natural_rgba8(W, H, 18)
    cfg = ovr.Config(fsrEnabled=True, renderScale=0.75, sharpness=0.9, radius=0.5, projCentre=(0.45, 0.52, 0.55, 0.5))
    tex = ovr.to_image(img, cuda)
    for r in (RECTS[0], RECTS[4]):
        got = []
        for fused in (False, True):
            pp = ovr.PostProcessor(dataclasses.replace(cfg, fusedFsr=fused))
            out, d = _apply(pp, 0, tex, r)
            got.append(_crop(out.cpu().numpy(), d))
            pp.close()
        assert np.array_equal(got[0], got[1]), r


def test_msaa_source_with_bounds(cuda):
    import torch
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    samples = 4
    rng = np.random.default_rng(19)
    base = synth.natural_rgba8(W, H, 19)
    ms = np.repeat(base, samples, axis=1).astype(np.int16) + rng.integers(-6, 7, (H, W * samples, 4))
    ms = np.clip(ms, 0, 255).astype(np.uint8)
    src = torch.from_numpy(ms).to(cuda)
    resolved = ovr.alloc_image(W, H, torch.uint8, cuda)
    ovr.resolve_msaa(src, resolved, samples)
    torch.cuda.synchronize()
    res = resolved.cpu().numpy()
    for use_nis in (False, True):
        cfg = ovr.Config(fsrEnabled=True, useNis=use_nis, renderScale=0.75, sharpness=0.9, radius=0.5)
        pp = ovr.PostProcessor(cfg)
        r = RECTS[1]
        s, d = _rects(cfg, r)
        out, _ = _apply(pp, 0, src, r, samples=samples)
        assert np.array_equal(_crop(out.cpu().numpy(), d), _oracle(res, cfg, 0, s, d))
        pp.close()


def test_array_texture_right_eye_with_bounds(cuda):
    import torch
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import _lib as L, synth
    left, right = synth.stereo_pair("natural", W, H, 20)
    arr = torch.from_numpy(np.stack([left, right])).to(cuda)
    cfg = ovr.Config(fsrEnabled=True, renderScale=0.75, sharpness=0.9, radius=0.5, projCentre=(0.45, 0.52, 0.55, 0.5))
    ctx = C.c_void_p()
    L.check(L.lib().ovrfsr_create(C.byref(ctx), C.byref(cfg.to_c())))
    src = L.Image(arr.data_ptr(), W, H, W * 4, L.FORMAT_RGBA8, 2, W * H * 4)
    r = RECTS[2]
    s, d = _rects(cfg, r)
    b = _bounds(r)
    out, rect = L.Image(), L.Rect()
    L.check(L.lib().ovrfsr_apply_bounds(ctx, 1, C.byref(src), C.byref(L.Bounds(b.uMin, b.vMin, b.uMax, b.vMax)),
                                        C.byref(out), C.byref(rect), C.c_void_p(torch.cuda.current_stream().cuda_stream)), "apply_bounds")
    assert (rect.x, rect.y, rect.width, rect.height) == d
    torch.cuda.synchronize()
    from openvr_fsr_b200.api import _wrap_device
    got = _wrap_device(out, cuda).cpu().numpy()
    assert np.array_equal(_crop(got, d), _oracle(right, cfg, 1, s, d))
    L.lib().ovrfsr_destroy(ctx)


@pytest.mark.parametrize("scale,kernel,arg", [(0.75, "easu_kernel", 3), (1.0, "rcas_kernel", 2)])
def test_tma_kept_for_unaligned_origin(cuda, tmp_path, scale, kernel, arg):
    """a rectangle at x0 % 4 != 0 still reads the user texture through the TMA instantiation"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    img = synth.natural_rgba8(W, H, 21)
    tex = ovr.to_image(img, cuda)
    cfg = ovr.Config(fsrEnabled=True, renderScale=scale, sharpness=0.9, radius=2.0)
    pp = ovr.PostProcessor(cfg)
    for r in RECTS[:3]:
        assert r[0] % 4 != 0
        _apply(pp, 0, tex, r)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for r in RECTS[:3]:
            _apply(pp, 0, tex, r)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if kernel in e.key]
    pp.close()
    assert names, [e.key for e in prof.key_averages()]
    for n in names:
        m = re.search(kernel + r"<([^>]*)>", n)
        assert m, n
        assert [t.strip() for t in m.group(1).split(",")][arg] == "true", n
