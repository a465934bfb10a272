"""The C++ drop-in with Config::honourTextureBounds: vr::PostProcessor::Apply submits each eye's bounds rectangle
through ovrfsr_apply_bounds (tests/cpp/pp_bounds.cpp); the output rectangle must match the oracle on the crop."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def bounds_exe(built_lib, tmp_path_factory):
    exe = tmp_path_factory.mktemp("cpp") / "pp_bounds"
    pkg = ROOT / "openvr_fsr_b200"
    subprocess.check_call(["nvcc", "-O2", "-std=c++17", "-I", str(pkg / "csrc"), "-I", str(ROOT / "include"),
                           str(ROOT / "tests/cpp/pp_bounds.cpp"), "-o", str(exe), "-L", str(pkg), "-lovrfsr",
                           "-Xlinker", f"-rpath={pkg}"])
    return exe


@pytest.mark.parametrize("use_nis,scale", [(0, 0.75), (1, 0.75), (0, 1.0), (1, 1.0)])
def test_cpp_postprocessor_honours_bounds(cuda, bounds_exe, tmp_path, use_nis, scale):
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import synth
    from oracle import pyoracle as po
    iw, ih, sharp, radius = 180, 132, 0.9, 0.5
    bounds = (0.1, 0.15, 0.85, 0.9)
    img = synth.natural_rgba8(iw, ih, 23)
    (tmp_path / "in.rgba").write_bytes(img.tobytes())
    out = tmp_path / "out.rgba"
    subprocess.check_call([str(bounds_exe), str(tmp_path / "in.rgba"), str(iw), str(ih), str(scale), str(sharp),
                           str(radius), str(use_nis), *map(str, bounds), str(out)])
    ow, oh = po.output_size(iw, ih, scale)
    (sx, sy, sw, sh), (dx, dy, dw, dh) = ovr.bounds_rects(iw, ih, ow, oh, ovr.TextureBounds(*bounds))
    crop = np.ascontiguousarray(img[sy:sy + sh, sx:sx + sw])
    both = np.frombuffer(out.read_bytes(), dtype=np.uint8).reshape(2, oh, ow, 4)
    for eye in (0, 1):  # the right eye is submitted with the bounds flipped vertically: the same rectangle
        if use_nis:
            cfg, _ = po.nis_config(scale == 1.0, eye, True, sw, sh, dw, dh, radius=radius, sharpness=sharp)
            want = po.nis_sharpen(crop, cfg) if scale == 1.0 else po.nis_scaler(crop, dw, dh, cfg)
        else:
            sc = po.sharpen_constants(eye, True, dw, dh, radius=radius, sharpness=sharp)
            mid = crop if scale == 1.0 else po.easu(crop, dw, dh, po.upscale_constants(eye, True, sw, sh, dw, dh, radius=radius))
            want = po.rcas(mid, sc)
        assert np.array_equal(both[eye][dy:dy + dh, dx:dx + dw], want), eye
