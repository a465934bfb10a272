"""Legacy CAS path (src/cas, SURVEY 8f row 4): the restated oracle against the reference's own CasSetup / CasFilter
lines compiled on the host (oracle/_ref), bit for bit."""
from pathlib import Path

import numpy as np
import pytest

from oracle import pyoracle as po
from openvr_fsr_b200 import synth

needs_ref = pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref not built: the original project's sources are absent")


@needs_ref
@pytest.mark.parametrize("sharp", [0.0, 0.3, 0.75, 1.0, 1.7, -0.5])
@pytest.mark.parametrize("mcd", [1.0, 0.25, 0.0])
def test_cas_setup_matches_reference(sharp, mcd):
    for iw, ih, ow, oh in ((1683, 1869, 2244, 2492), (960, 1080, 1920, 2160), (100, 50, 100, 50), (1512, 1680, 2016, 2240)):
        a = po.cas_setup(sharp, mcd, iw, ih, ow, oh)
        b = po.cas_setup(sharp, mcd, iw, ih, ow, oh, which="ref")
        assert np.array_equal(a.words(), b.words()), (sharp, mcd, iw, ih, a.words(), b.words())


@pytest.mark.parametrize("name,sharp,mcd", [("sharpen_natural_57x41", 0.8, 1.0), ("sharpen_clamped_57x41", 1.0, 0.06),
                                            ("upscale_natural_57x41_s067", 0.9, 1.0), ("upscale_fp16_33x27_s05", 0.5, 1.0)])
def test_cas_setup_matches_golden(name, sharp, mcd):
    """The words the reference's own CasSetup produced for the pass_cas_* fixtures (tests/golden/make_golden_more.py),
    checked where the reference's sources are absent: the oracle's and the library's CasSetup must reproduce them."""
    import openvr_fsr_b200 as ovr
    g = np.load(Path(__file__).parent / "golden" / f"pass_cas_{name}.npz")
    (ih, iw), (oh, ow) = g["src"].shape[:2], g["out"].shape[:2]
    assert np.array_equal(po.cas_setup(sharp, mcd, iw, ih, ow, oh).words(), g["consts"])
    assert np.array_equal(ovr.cas_setup(sharp, mcd, iw, ih, ow, oh), g["consts"])


@needs_ref
@pytest.mark.parametrize("w,h", [(37, 29), (64, 64), (129, 65)])
@pytest.mark.parametrize("sharp,mcd", [(0.0, 1.0), (0.8, 1.0), (1.0, 0.1)])
def test_cas_sharpen_bit_identical(w, h, sharp, mcd):
    k = po.cas_setup(sharp, mcd, w, h, w, h)
    for src in (synth.natural_rgba8(w, h, 3), synth.uniform_rgba8(w, h, 4)):
        for odt in (np.uint8, np.float32):
            a = po.cas(src, w, h, k, True, out_dtype=odt)
            b = po.cas(src, w, h, k, True, which="ref", out_dtype=odt)
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
            assert (a[..., 3] == (255 if odt == np.uint8 else 1.0)).all()
    f16 = synth.natural_rgba16f(w, h, 5)
    assert np.array_equal(po.cas(f16, w, h, k, True, out_dtype=np.float16).view(np.uint8),
                          po.cas(f16, w, h, k, True, which="ref", out_dtype=np.float16).view(np.uint8))


@needs_ref
@pytest.mark.parametrize("iw,ih,scale", [(37, 29, 0.75), (48, 40, 0.5), (100, 70, 0.77), (64, 64, 1.0), (33, 47, 0.59)])
@pytest.mark.parametrize("sharp", [0.0, 0.9])
def test_cas_upscale_bit_identical(iw, ih, scale, sharp):
    ow, oh = po.output_size(iw, ih, scale)
    k = po.cas_setup(sharp, 1.0, iw, ih, ow, oh)
    for src in (synth.natural_rgba8(iw, ih, 6), synth.uniform_rgba8(iw, ih, 7)):
        for odt in (np.uint8, np.float32):
            a = po.cas(src, ow, oh, k, False, out_dtype=odt)
            b = po.cas(src, ow, oh, k, False, which="ref", out_dtype=odt)
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), int((a != b).sum())


def test_cas_known_properties():
    """A constant image stays constant (sharpen and upscale); maxColorDelta 0 makes the sharpen pass the identity."""
    w, h = 40, 24
    flat = np.full((h, w, 4), 128, np.uint8)
    k = po.cas_setup(0.8, 1.0, w, h, w, h)
    out = po.cas(flat, w, h, k, True)
    assert (out[2:-2, 2:-2, :3] == 128).all()  # the 1-px border sees the zero Load outside the image
    img = synth.natural_rgba8(w, h, 1)
    k0 = po.cas_setup(0.8, 0.0, w, h, w, h)
    out0 = po.cas(img, w, h, k0, True)
    assert np.array_equal(out0[..., :3], img[..., :3])
    ow, oh = po.output_size(w, h, 0.5)
    ku = po.cas_setup(0.5, 1.0, w, h, ow, oh)
    up = po.cas(flat, ow, oh, ku, False)
    assert (up[4:-4, 4:-4, :3] == 128).all()


@pytest.mark.parametrize("sharp", [0.0, 0.3, 0.75, 1.0, 1.7, -0.5])
@pytest.mark.parametrize("mcd", [1.0, 0.25, 0.0])
def test_library_cas_setup_matches_oracle(sharp, mcd):
    """ovrfsr_cas_setup is host code: checked without a GPU."""
    import openvr_fsr_b200 as ovr
    for iw, ih, ow, oh in ((1683, 1869, 2244, 2492), (960, 1080, 1920, 2160), (100, 50, 100, 50)):
        assert np.array_equal(ovr.cas_setup(sharp, mcd, iw, ih, ow, oh), po.cas_setup(sharp, mcd, iw, ih, ow, oh).words())
