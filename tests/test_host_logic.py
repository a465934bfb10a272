"""Host-side logic of the product (no GPU): constant blocks against the oracle and the reference's own
functions, the ABI surface, the pass-through / failure behaviour of PostProcessor."""
import ctypes as C
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import openvr_fsr_b200 as ovr
from openvr_fsr_b200 import _lib as L
from oracle import pyoracle as po

ROOT = Path(__file__).resolve().parents[1]


def test_library_exports_every_declared_symbol(built_lib):
    header = (ROOT / "include" / "ovrfsr.h").read_text()
    declared = set(re.findall(r"OVRFSR_API\s+[\w\s\*]+?\b(ovrfsr_\w+)\s*\(", header))
    assert len(declared) >= 25
    exported = set(re.findall(r" T (ovrfsr_\w+)", subprocess.check_output(["nm", "-D", "--defined-only", str(built_lib)], text=True)))
    assert declared <= exported, f"missing: {sorted(declared - exported)}"
    assert declared == set(L.SYMBOLS), "python binding and header disagree"
    assert L.lib().ovrfsr_version() == 0x00010000
    # the library must load without a CUDA driver: no libcuda / libcudart DT_NEEDED
    needed = subprocess.check_output(["readelf", "-d", str(built_lib)], text=True)
    assert "libcuda" not in needed


def test_sm100a_only(built_lib):
    out = subprocess.check_output(["cuobjdump", "-lelf", str(built_lib)], text=True)
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


@pytest.mark.parametrize("iw,ih,scale", [(1683, 1869, 0.75), (960, 1080, 0.5), (2244, 2492, 1.3), (1512, 1680, 0.75),
                                         (1000, 999, 0.77), (641, 479, 0.59), (300, 200, 1.0)])
def test_output_size_and_constants_match_oracle(iw, ih, scale):
    ow, oh = ovr.output_size(iw, ih, scale)
    assert (ow, oh) == po.output_size(iw, ih, scale)
    for radius in (0.5, 2.0, 0.0, 0.37):
        for proj in ((.5, .5, .5, .5), (.46, .51, .54, .49)):
            for one_eye in (True, False):
                for eye in (0, 1):
                    cfg = ovr.Config(fsrEnabled=True, renderScale=scale, sharpness=0.9, radius=radius, projCentre=proj,
                                     debugMode=bool(eye))
                    got = ovr.make_upscale_constants(cfg, eye, one_eye, iw, ih, ow, oh)
                    want = po.upscale_constants(eye, one_eye, iw, ih, ow, oh, proj=proj, radius=radius).words()
                    assert np.array_equal(got, want)
                    got = ovr.make_sharpen_constants(cfg, eye, one_eye, ow, oh)
                    want = po.sharpen_constants(eye, one_eye, ow, oh, proj=proj, radius=radius, sharpness=0.9,
                                                debug=bool(eye)).words()
                    assert np.array_equal(got, want)


def test_c3_output_size_is_the_codes_not_the_readmes():
    # PostProcessor.cpp:515-517: uint32(2244*1.3f) = 2917, uint32(2492*1.3f) = 3239 (README says 2915x3240)
    assert ovr.output_size(2244, 2492, 1.3) == (2917, 3239)
    assert ovr.output_size(1683, 1869, 0.75) == (2244, 2492)
    assert ovr.output_size(960, 1080, 0.5) == (1920, 2160)
    assert ovr.output_size(1512, 1680, 0.75) == (2016, 2240)


def test_rcas_con_sweep_matches_oracle():
    lib, olib = L.lib(), po.oracle_lib()
    for s in np.linspace(-0.5, 3.0, 141):
        a, b = (C.c_uint32 * 4)(), (C.c_uint32 * 4)()
        lib.ovrfsr_fsr_rcas_con(a, float(s))
        olib.ovo_fsr_rcas_con(b, float(s))
        assert list(a) == list(b)


@pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref not built: the original project's sources are absent")
def test_constants_match_reference_functions():
    lib, ref = L.lib(), po.ref_lib()
    rng = np.random.default_rng(11)
    for _ in range(100):
        iw, ih = int(rng.integers(8, 4000)), int(rng.integers(8, 4000))
        ow, oh = int(rng.integers(iw, 2 * iw + 1)), int(rng.integers(ih, 2 * ih + 1))
        a, b = (C.c_uint32 * 16)(), (C.c_uint32 * 16)()
        lib.ovrfsr_fsr_easu_con(a, iw, ih, iw, ih, ow, oh)
        ref.ref_FsrEasuCon(b, iw, ih, iw, ih, ow, oh)
        assert list(a) == list(b)
    for stops in np.linspace(0, 2, 41):
        a, b = (C.c_uint32 * 4)(), (C.c_uint32 * 4)()
        lib.ovrfsr_fsr_rcas_con(a, float(stops))
        ref.ref_FsrRcasCon(b, float(stops))
        assert list(a) == list(b)
    # NISConfig against NVScalerUpdateConfig / NVSharpenUpdateConfig compiled as shipped
    for sharp in (0.0, 0.25, 0.5, 0.75, 0.9, 1.0, 1.4):
        for (iw, ih, ow, oh) in ((1512, 1680, 2016, 2240), (960, 1080, 1920, 2160), (1683, 1869, 2244, 2492), (100, 100, 300, 300)):
            cfg = ovr.Config(fsrEnabled=True, useNis=True, renderScale=iw / ow, sharpness=sharp)
            got, ok = ovr.make_nis_config(cfg, False, 0, True, iw, ih, ow, oh)
            buf = C.create_string_buffer(256)
            rok = ref.ref_NVScalerUpdateConfig(C.cast(buf, C.c_void_p), sharp, iw, ih, ow, oh)
            assert bool(rok) == ok
            if ok:
                assert got[:112] == buf.raw[:112]
            got, ok = ovr.make_nis_config(cfg, True, 0, True, ow, oh, ow, oh)
            rok = ref.ref_NVSharpenUpdateConfig(C.cast(buf, C.c_void_p), sharp, ow, oh)
            assert ok and rok and got[:112] == buf.raw[:112]
    n = 64 * 8
    assert np.array_equal(np.ctypeslib.as_array(lib.ovrfsr_nis_coef_scale(), (n,)).view(np.uint32),
                          np.ctypeslib.as_array(ref.ref_coef_scale(), (n,)).view(np.uint32))
    assert np.array_equal(np.ctypeslib.as_array(lib.ovrfsr_nis_coef_usm(), (n,)).view(np.uint32),
                          np.ctypeslib.as_array(ref.ref_coef_usm(), (n,)).view(np.uint32))


def _round_f32(fr):
    """Correctly rounded (nearest-even) float32 of an exact Fraction, as a Fraction."""
    import math
    from fractions import Fraction as F
    if fr == 0:
        return F(0)
    e = math.floor(math.log2(fr))
    while F(2) ** e > fr:
        e -= 1
    while F(2) ** (e + 1) <= fr:
        e += 1
    sc = F(2) ** (23 - e)
    m = fr * sc
    fl = m.numerator // m.denominator
    rem = m - fl
    if rem > F(1, 2) or (rem == F(1, 2) and fl % 2 == 1):
        fl += 1
    return F(fl) / sc


def test_unorm8_decode_recipe_is_exact():
    """device_common.cuh unorm8(): fma(v, clo, v * chi) with chi = 0x3b808080 (the float below 1/255) and
    clo = 0x2f808081 (float(1/255 - chi)) must equal the correctly rounded v/255 for all 256 inputs -- checked in exact
    rational arithmetic with one rounding per device operation."""
    from fractions import Fraction as F
    chi = F(float(np.uint32(0x3b808080).view(np.float32)))
    clo = F(float(np.uint32(0x2f808081).view(np.float32)))
    assert chi < F(1, 255) and clo == _round_f32(F(1, 255) - chi)
    got = []
    for v in range(256):
        q = _round_f32(v * chi)          # FMUL
        got.append(_round_f32(v * clo + q))  # FFMA: exact product and sum, one rounding
        assert got[-1] == _round_f32(F(v, 255)), v
    q2 = np.array([float(g) for g in got], dtype=np.float32)
    assert np.array_equal(q2, (np.arange(256, dtype=np.float32) / np.float32(255.0)))
    # and encode(decode(v)) == v, which makes RCAS's outside-radius copy an identity on RGBA8
    assert np.array_equal((np.clip(q2, 0, 1) * np.float32(255.0) + np.float32(0.5)).astype(np.uint8), np.arange(256))


def test_unorm10_decode_recipe_is_exact():
    """device_common.cuh unorm10()/unorm2(): the same residual-corrected multiply must give the correctly rounded
    v/1023 (v/3) for all 1024 (4) codes, and encode(decode(v)) == v (RCAS's raw pass-through on RGB10A2)."""
    for maxv in (1023, 3):
        v = np.arange(maxv + 1, dtype=np.float64)
        r = np.float64(np.float32(1.0) / np.float32(maxv))
        q = (v * r).astype(np.float32).astype(np.float64)
        e = (v - maxv * q).astype(np.float32).astype(np.float64)
        q2 = (e * r + q).astype(np.float32)
        assert np.array_equal(q2, np.arange(maxv + 1, dtype=np.float32) / np.float32(maxv))
        assert np.array_equal((np.clip(q2, 0, 1) * np.float32(maxv) + np.float32(0.5)).astype(np.uint32), np.arange(maxv + 1))


def test_rgb10a2_pack_roundtrip_and_oracle_decode():
    """synth's R10G10B10A2 packing is the layout the oracle decodes: an RCAS whose radius mask excludes every group
    is the identity on 10-bit texels (decode -> x1 -> encode), alpha included."""
    from openvr_fsr_b200 import synth
    from oracle import pyoracle as po
    img = synth.uniform_rgb10a2(40, 24, 3)
    codes = synth.unpack_rgb10a2(img)
    assert codes[..., :3].max() <= 1023 and codes[..., 3].max() <= 3
    assert np.array_equal(synth.pack_rgb10a2(codes[..., :3], codes[..., 3]), img)
    sc = po.sharpen_constants(0, True, 40, 24, radius=0.0, sharpness=0.9, proj=(5.0, 5.0, 5.0, 5.0))
    out = po.rcas(img, sc, src_fmt=po.FMT_RGB10A2, dst_fmt=po.FMT_RGB10A2)
    assert np.array_equal(out, img)
    # and a float view of the same texels: code / 1023, alpha / 3
    f = po.rcas(img, sc, out_dtype=np.float32, src_fmt=po.FMT_RGB10A2)
    assert np.array_equal(f[..., :3], codes[..., :3].astype(np.float32) / np.float32(1023.0))
    assert np.array_equal(f[..., 3], codes[..., 3].astype(np.float32) / np.float32(3.0))


def test_passthrough_and_loud_failure_without_gpu():
    import torch
    tex = torch.zeros((8, 8, 4), dtype=torch.uint8)
    pp = ovr.PostProcessor(ovr.Config(fsrEnabled=False))
    assert pp.apply(0, tex) is tex  # Config::fsrEnabled == false -> untouched (PostProcessor.cpp:134)
    pp.close()
    if not torch.cuda.is_available():
        pp = ovr.PostProcessor(ovr.Config(fsrEnabled=True, renderScale=0.5))
        with pytest.raises(ovr.OvrFsrError):
            pp.apply(0, tex)  # no device: fails loudly, never computes on the CPU
        # the reference disables itself after a failed resource creation (PostProcessor.cpp:148-152)
        assert pp.apply(0, tex) is tex
        pp.reset()  # Reset re-enables
        with pytest.raises(ovr.OvrFsrError):
            pp.apply(0, tex)
        pp.close()
    with pytest.raises(ovr.OvrFsrError):
        ovr.PostProcessor(ovr.Config(fsrEnabled=True, renderScale=0.0))


def test_group_mask_matches_reference_rule():
    """the wrapping-u32 radius test at 16x16 granularity (fsr_easu.hlsl:40-44)"""
    olib = po.oracle_lib()
    centre = (C.c_uint32 * 4)(1122, 1246, 1122, 1246)
    inside = sum(olib.ovo_group_inside(gx, gy, 16, 16, centre, 388129) for gy in range(156) for gx in range(141))
    assert 0.20 < inside / (141 * 156) < 0.24  # SURVEY.md 8d: EASU area fraction 0.218 at radius 0.5
    assert olib.ovo_group_inside(70, 77, 16, 16, centre, 0) == 0
    big = (C.c_uint32 * 4)(0, 0, 0, 0)
    assert olib.ovo_group_inside(0, 0, 16, 16, big, 128) == 1  # (0-8)^2*2 = 128 with wraparound


def test_both_math_modes_are_distinct_kernels(built_lib):
    """Regression: the strict and fast builds of the same kernel template must not fold into one symbol."""
    out = subprocess.check_output(["cuobjdump", "-elf", str(built_lib)], text=True, stderr=subprocess.DEVNULL)
    for kernel in ("easu_kernel", "rcas_kernel"):
        assert re.search(rf"strict_math\d+{kernel}", out), kernel
        assert re.search(rf"fast_math\d+{kernel}", out), kernel
