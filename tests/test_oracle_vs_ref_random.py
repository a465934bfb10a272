"""Seeded random sweep: the restated oracle against the reference's own lines compiled on the host (oracle/_ref), over
random sizes, scales, radii, projection centres, sharpness, formats, eyes and debug tint -- FSR, NIS and CAS.  CPU only;
skipped where /root/reference (hence oracle/_ref) is absent."""
import numpy as np
import pytest

from oracle import pyoracle as po
from openvr_fsr_b200 import synth

pytestmark = pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref not built: the original project's sources are absent")


def _image(rng, w, h, fmt):
    if fmt == po.FMT_RGBA16F:
        return synth.natural_rgba16f(w, h, int(rng.integers(0, 1000)))
    if fmt == po.FMT_RGB10A2:
        return synth.uniform_rgb10a2(w, h, int(rng.integers(0, 1000)))
    return (synth.natural_rgba8 if rng.integers(0, 2) else synth.uniform_rgba8)(w, h, int(rng.integers(0, 1000)))


@pytest.mark.parametrize("seed", range(16))
def test_fsr_random(seed):
    rng = np.random.default_rng(7000 + seed)
    iw, ih = int(rng.integers(5, 90)), int(rng.integers(5, 70))
    scale = float(rng.choice([0.5, 0.59, 0.67, 0.75, 0.77, 0.9, 1.0, 1.3, 1.7]))
    fmt = int(rng.choice([po.FMT_RGBA8, po.FMT_BGRA8, po.FMT_RGBA16F, po.FMT_RGB10A2]))
    eye, one = int(rng.integers(0, 2)), bool(rng.integers(0, 3))
    kw = dict(proj=tuple(float(x) for x in rng.uniform(0.3, 0.7, 4)), radius=float(rng.choice([0.0, 0.3, 0.5, 0.8, 2.0])))
    sharp, debug = float(rng.uniform(0, 1.2)), bool(rng.integers(0, 2))
    src = _image(rng, iw, ih, fmt)
    ow, oh = po.output_size(iw, ih, scale)
    uc = po.upscale_constants(eye, one, iw, ih, ow, oh, **kw)
    sc = po.sharpen_constants(eye, one, ow, oh, sharpness=sharp, debug=debug, **kw)
    ten = fmt == po.FMT_RGB10A2
    for odt in ((np.uint8,) if ten else (np.uint8, np.float32)):
        f = dict(src_fmt=None if fmt == po.FMT_RGBA16F else fmt, dst_fmt=po.FMT_RGB10A2 if ten else None, out_dtype=odt)
        a, b = po.easu(src, ow, oh, uc, **f), po.easu(src, ow, oh, uc, which="ref", **f)
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), ("easu", seed)
        g = dict(src_fmt=po.FMT_RGB10A2 if ten else None, dst_fmt=po.FMT_RGB10A2 if ten else None, out_dtype=odt)
        c, d = po.rcas(a, sc, **g), po.rcas(a, sc, which="ref", **g)
        assert np.array_equal(c.view(np.uint8), d.view(np.uint8)), ("rcas", seed)


@pytest.mark.parametrize("seed", range(10))
def test_nis_random(seed):
    rng = np.random.default_rng(8000 + seed)
    iw, ih = int(rng.integers(8, 80)), int(rng.integers(8, 60))
    scale = float(rng.choice([0.5, 0.59, 0.67, 0.75, 0.77, 0.9, 1.0]))
    sharpen_only = scale == 1.0
    eye, one = int(rng.integers(0, 2)), bool(rng.integers(0, 3))
    src = _image(rng, iw, ih, int(rng.choice([po.FMT_RGBA8, po.FMT_RGBA16F])))
    ow, oh = po.output_size(iw, ih, scale)
    cfg, _ = po.nis_config(sharpen_only, eye, one, iw, ih, ow, oh, proj=tuple(float(x) for x in rng.uniform(0.3, 0.7, 4)),
                           radius=float(rng.choice([0.0, 0.4, 0.7, 2.0])), sharpness=float(rng.uniform(0, 1)),
                           debug=bool(rng.integers(0, 2)))
    for odt in (np.uint8, np.float32):
        if sharpen_only:
            a, b = po.nis_sharpen(src, cfg, out_dtype=odt), po.nis_sharpen(src, cfg, which="ref", out_dtype=odt)
        else:
            a, b = po.nis_scaler(src, ow, oh, cfg, out_dtype=odt), po.nis_scaler(src, ow, oh, cfg, which="ref", out_dtype=odt)
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), seed


@pytest.mark.parametrize("seed", range(10))
def test_cas_random(seed):
    rng = np.random.default_rng(9000 + seed)
    iw, ih = int(rng.integers(4, 90)), int(rng.integers(4, 70))
    sharpen_only = bool(rng.integers(0, 2))
    scale = 1.0 if sharpen_only else float(rng.choice([0.5, 0.59, 0.67, 0.75, 0.9, 1.0]))
    ow, oh = po.output_size(iw, ih, scale)
    src = _image(rng, iw, ih, int(rng.choice([po.FMT_RGBA8, po.FMT_BGRA8, po.FMT_RGBA16F])))
    fmt = None if src.dtype != np.uint8 else int(rng.choice([po.FMT_RGBA8, po.FMT_BGRA8]))
    sharp, mcd = float(rng.uniform(-0.2, 1.3)), float(rng.choice([1.0, 0.3, 0.05]))
    k, kr = po.cas_setup(sharp, mcd, iw, ih, ow, oh), po.cas_setup(sharp, mcd, iw, ih, ow, oh, which="ref")
    assert np.array_equal(k.words(), kr.words())
    for odt in (np.uint8, np.float32):
        a = po.cas(src, ow, oh, k, sharpen_only, out_dtype=odt, src_fmt=fmt)
        b = po.cas(src, ow, oh, k, sharpen_only, which="ref", out_dtype=odt, src_fmt=fmt)
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), seed
