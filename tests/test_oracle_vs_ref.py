"""Pins the restated oracle (oracle/*.c) to the reference's OWN lines compiled on the host (oracle/_ref).

The reference ships no tests or golden vectors for this path (SURVEY.md section 4), so the pin is the
reference itself run here: every case must be BIT-IDENTICAL between the two checkers.  Those comparisons are
skipped where oracle/_ref cannot be built (the original's sources are absent); tests/test_golden.py then still pins
the oracle against the committed fixtures that oracle/_ref generated.  The known-answer words and the thread-count
check need the oracle alone and run everywhere.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as po
from tests.cases import SMALL, corner_images

needs_ref = pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref not built: the original project's sources are absent")


@needs_ref
@pytest.mark.parametrize("iw,ih,scale", SMALL)
def test_fsr_bit_identical(iw, ih, scale):
    ow, oh = po.output_size(iw, ih, scale)
    for radius in (2.0, 0.5, 0.2):
        uc = po.upscale_constants(0, True, iw, ih, ow, oh, radius=radius)
        for debug in (False, True):
            sc = po.sharpen_constants(0, True, ow, oh, radius=radius, sharpness=0.9, debug=debug)
            for name, src in corner_images(iw, ih).items():
                a = po.easu(src, ow, oh, uc)
                b = po.easu(src, ow, oh, uc, which="ref")
                assert np.array_equal(a, b), (name, radius)
                assert np.array_equal(po.rcas(a, sc), po.rcas(a, sc, which="ref")), (name, radius, debug)


@needs_ref
def test_fsr_formats_bit_identical():
    iw, ih, scale = 37, 29, 0.75
    ow, oh = po.output_size(iw, ih, scale)
    uc = po.upscale_constants(1, True, iw, ih, ow, oh, radius=0.4, proj=(0.45, 0.52, 0.55, 0.48))
    sc = po.sharpen_constants(1, True, ow, oh, radius=0.4, sharpness=0.6, proj=(0.45, 0.52, 0.55, 0.48))
    from openvr_fsr_b200 import synth
    src8 = synth.natural_rgba8(iw, ih, 5)
    src16 = synth.natural_rgba16f(iw, ih, 5)
    for src, fmt in ((src8, po.FMT_RGBA8), (src8, po.FMT_BGRA8), (src16, po.FMT_RGBA16F)):
        for odt in (np.uint8, np.float16):
            a = po.easu(src, ow, oh, uc, out_dtype=odt, src_fmt=fmt)
            b = po.easu(src, ow, oh, uc, which="ref", out_dtype=odt, src_fmt=fmt)
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
            c, d = po.rcas(a, sc, out_dtype=odt), po.rcas(a, sc, which="ref", out_dtype=odt)
            assert np.array_equal(c.view(np.uint8), d.view(np.uint8))


@needs_ref
def test_fsr_rgb10a2_bit_identical():
    """10-bit sources keep a 10-bit target (DetermineOutputFormat, PostProcessor.cpp:63-74)."""
    iw, ih, scale = 41, 33, 0.75
    ow, oh = po.output_size(iw, ih, scale)
    uc = po.upscale_constants(0, True, iw, ih, ow, oh, radius=0.45)
    sc = po.sharpen_constants(0, True, ow, oh, radius=0.45, sharpness=0.8)
    from openvr_fsr_b200 import synth
    src = synth.natural_rgb10a2(iw, ih, 6)
    kw = dict(src_fmt=po.FMT_RGB10A2, dst_fmt=po.FMT_RGB10A2)
    a, b = po.easu(src, ow, oh, uc, **kw), po.easu(src, ow, oh, uc, which="ref", **kw)
    assert np.array_equal(a, b)
    assert (synth.unpack_rgb10a2(a)[..., 3] == 3).all()  # EASU writes alpha 1
    assert ((synth.unpack_rgb10a2(a)[..., 0] * 255) % 1023 != 0).any()  # codes that no 8-bit value maps to
    assert np.array_equal(po.rcas(a, sc, **kw), po.rcas(a, sc, which="ref", **kw))


def test_threads_do_not_change_results():
    iw, ih = 65, 43
    ow, oh = po.output_size(iw, ih, 0.75)
    uc = po.upscale_constants(0, True, iw, ih, ow, oh, radius=0.5)
    src = corner_images(iw, ih)["natural"]
    assert np.array_equal(po.easu(src, ow, oh, uc, nthreads=1), po.easu(src, ow, oh, uc, nthreads=5))


@needs_ref
def test_constants_match_reference_functions():
    lib, ref = po.oracle_lib(), po.ref_lib()
    rng = np.random.default_rng(7)
    for _ in range(200):
        iw, ih = int(rng.integers(8, 4000)), int(rng.integers(8, 4000))
        ow, oh = int(rng.integers(iw, 2 * iw + 1)), int(rng.integers(ih, 2 * ih + 1))
        a, b = (C.c_uint32 * 16)(), (C.c_uint32 * 16)()
        lib.ovo_fsr_easu_con(a, iw, ih, iw, ih, ow, oh)
        ref.ref_FsrEasuCon(b, iw, ih, iw, ih, ow, oh)
        assert list(a) == list(b)
    for stops in np.linspace(0, 2, 81):
        a, b = (C.c_uint32 * 4)(), (C.c_uint32 * 4)()
        lib.ovo_fsr_rcas_con(a, float(stops))
        ref.ref_FsrRcasCon(b, float(stops))
        assert list(a) == list(b), stops


def test_known_answer_words():
    """SURVEY.md section 4: words obtained by compiling ffx_fsr1.h with A_CPU."""
    uc = po.upscale_constants(0, True, 1683, 1869, 2244, 2492, radius=0.5).words()
    assert [hex(x) for x in uc[:8]] == ["0x3f400000", "0x3f400000", "0xbe000000", "0xbe000000",
                                       "0x3a1bc28c", "0x3a0c424b", "0x3a1bc28c", "0xba0c424b"]
    assert list(uc[16:24]) == [1122, 1246, 1122, 1246, 623, 388129, 2244, 2492]
    sc = po.sharpen_constants(0, True, 2244, 2492, sharpness=0.9).words()
    assert hex(sc[0]) == "0x3f5edc66" and hex(sc[1]) == "0x3af63af6"
