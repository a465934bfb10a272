"""ovrfsr_bounds_rects (the rectangles of ovrfsr_apply_bounds) against a numpy restatement of the rule in
include/ovrfsr.h, and the constant blocks built for a rectangle.  Pure host code: no GPU needed."""
import numpy as np
import pytest

f32 = np.float32


def _rects_np(w, h, ow, oh, b):
    """u0 = clamp(min(uMin, uMax), 0, 1) ...; x = (uint32)(u * (float)W + 0.5f) in single precision."""
    def lo_hi(a, c):
        a, c = f32(a), f32(c)
        return np.clip(np.minimum(a, c), f32(0), f32(1)), np.clip(np.maximum(a, c), f32(0), f32(1))

    def edge(t, n):
        return int(f32(f32(t) * f32(n)) + f32(0.5))

    (u0, u1), (v0, v1) = lo_hi(b[0], b[2]), lo_hi(b[1], b[3])
    s = (edge(u0, w), edge(v0, h), edge(u1, w) - edge(u0, w), edge(v1, h) - edge(v0, h))
    d = (edge(u0, ow), edge(v0, oh), edge(u1, ow) - edge(u0, ow), edge(v1, oh) - edge(v0, oh))
    return None if 0 in (s[2], s[3], d[2], d[3]) else (s, d)


def _cases():
    rng = np.random.default_rng(20261017)
    for i in range(400):
        w, h = int(rng.integers(1, 4097)), int(rng.integers(1, 4097))
        scale = float(rng.choice([0.59, 0.75, 0.77, 1.0, 1.3]))
        kind = i % 6
        if kind == 0:    # anywhere, including outside [0, 1]
            b = tuple(float(x) for x in rng.uniform(-0.3, 1.3, 4))
        elif kind == 1:  # flipped (OpenGL-style vMin > vMax, or u)
            u0, v0 = rng.uniform(0, 0.5, 2)
            u1, v1 = rng.uniform(0.5, 1, 2)
            b = (float(u1), float(v1), float(u0), float(v0)) if i % 12 == 1 else (float(u0), float(v1), float(u1), float(v0))
        elif kind == 2:  # side-by-side halves
            b = (0.0, 0.0, 0.5, 1.0) if i % 12 == 2 else (0.5, 0.0, 1.0, 1.0)
        elif kind == 3:  # one texel
            x, y = int(rng.integers(0, w)), int(rng.integers(0, h))
            b = (float(f32(x) / f32(w)), float(f32(y) / f32(h)), float(f32(x + 1) / f32(w)), float(f32(y + 1) / f32(h)))
        elif kind == 4:  # empty in one dimension
            u = float(rng.uniform(0, 1))
            b = (u, 0.1, u, 0.9) if i % 12 == 4 else (0.1, u, 0.9, u)
        else:            # dynamic resolution: a shrinking view at the origin
            s = float(rng.uniform(0.05, 1.0))
            b = (0.0, 0.0, s, s)
        yield w, h, scale, b


def test_bounds_rects_match_the_rule(built_lib):
    import openvr_fsr_b200 as ovr
    checked = empty = 0
    for w, h, scale, b in _cases():
        ow, oh = ovr.output_size(w, h, scale)
        want = _rects_np(w, h, ow, oh, b)
        tb = ovr.TextureBounds(*b)
        if want is None:
            with pytest.raises(ovr.OvrFsrError) as e:
                ovr.bounds_rects(w, h, ow, oh, tb)
            assert e.value.status == ovr.ERR_INVALID, (w, h, b)
            empty += 1
            continue
        got = ovr.bounds_rects(w, h, ow, oh, tb)
        assert got == want, (w, h, scale, b)
        s, d = got
        assert s[0] + s[2] <= w and s[1] + s[3] <= h and d[0] + d[2] <= ow and d[1] + d[3] <= oh
        if scale == 1.0:
            assert s == d
        checked += 1
    assert checked > 250 and empty > 30


def test_bounds_rects_special_values(built_lib):
    import ctypes as C
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import _lib as L
    # NULL bounds = the whole texture; flipped bounds = the same rectangle
    s, d = L.Rect(), L.Rect()
    assert L.lib().ovrfsr_bounds_rects(640, 480, 853, 640, None, C.byref(s), C.byref(d)) == ovr.OK
    assert (s.x, s.y, s.width, s.height, d.x, d.y, d.width, d.height) == (0, 0, 640, 480, 0, 0, 853, 640)
    assert ovr.bounds_rects(640, 480, 853, 640, ovr.TextureBounds(0.1, 0.9, 0.6, 0.2)) == \
        ovr.bounds_rects(640, 480, 853, 640, ovr.TextureBounds(0.6, 0.2, 0.1, 0.9))
    # NaN bounds are rejected
    with pytest.raises(ovr.OvrFsrError):
        ovr.bounds_rects(640, 480, 853, 640, ovr.TextureBounds(float("nan"), 0, 1, 1))


@pytest.mark.parametrize("use_nis", [False, True])
def test_rectangle_constants_follow_the_view(built_lib, use_nis):
    """What ovrfsr_apply_bounds builds for a rectangle is the existing builders called with the rectangle sizes and
    only_one_eye = 1; the reference's own constant code (the oracle) gives the same words, so the foveation centre and
    radius are placed for the view, not for the texture."""
    import openvr_fsr_b200 as ovr
    from oracle import pyoracle as po
    proj, radius, sharp = (0.42, 0.55, 0.61, 0.47), 0.5, 0.8
    cfg = ovr.Config(fsrEnabled=True, useNis=use_nis, renderScale=0.75, radius=radius, sharpness=sharp, projCentre=proj)
    w, h = 1683, 1869
    ow, oh = ovr.output_size(w, h, 0.75)
    for eye in (0, 1):
        s, d = ovr.bounds_rects(w, h, ow, oh, ovr.TextureBounds(0.0, 0.0, 0.8, 0.8))
        if use_nis:
            got, _ = ovr.make_nis_config(cfg, False, eye, True, s[2], s[3], d[2], d[3])
            want, _ = po.nis_config(False, eye, True, s[2], s[3], d[2], d[3], proj=proj, radius=radius, sharpness=sharp)
            assert got[:144] == bytes(want)[:144]  # NISConfig, the centres and the radius words
        else:
            uc = ovr.make_upscale_constants(cfg, eye, True, s[2], s[3], d[2], d[3])
            sc = ovr.make_sharpen_constants(cfg, eye, True, d[2], d[3])
            assert np.array_equal(uc, np.array(po.upscale_constants(eye, True, s[2], s[3], d[2], d[3], proj=proj, radius=radius).words(), dtype=np.uint32))
            assert np.array_equal(sc, np.array(po.sharpen_constants(eye, True, d[2], d[3], proj=proj, radius=radius, sharpness=sharp).words(), dtype=np.uint32))
            # the circle is centred in the view and sized from its height
            cx = proj[2 * eye] * d[2]
            assert uc[16] == int(f32(d[2]) * f32(proj[2 * eye])) and abs(int(uc[16]) - cx) < 1
            assert uc[20] == int(f32(0.5) * f32(radius) * f32(d[3]))
