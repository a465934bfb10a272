"""bench.py's command-line contract, as far as a box without a GPU can check it: the reference arm (the reference's own
lines on the host cores) prints ONE JSON line with the keys the driver reads, on the same config object as the product
arm; the product arm refuses to run without a CUDA device instead of falling back to anything.  On a GPU:
--dump-outputs writes what the timed path computed."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def _run(*args, timeout=600):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    from oracle import pyoracle as po
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("stereo eye-pairs/sec") and d["unit"] == "pairs/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and abs(d["value"] * d["ms_per_step"] * 1e-3 - 1.0) < 1e-6  # one pair per step
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["config"]["workload"].startswith("C2: stereo 1683x1869->2244x2492") and d["config"]["radius"] == 2.0
    cb = d["cpu_baseline"]
    # without the original's sources (no oracle/_ref) the arm runs the restated oracle and says so
    assert cb["kind"] == ("reference" if po.ref_available() else "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "pair" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0  # nothing of the product runs on this arm


@pytest.mark.gpu
def test_dump_outputs_are_the_last_steps_outputs(cuda, tmp_path):
    """--dump-outputs: float32 samples, within 64 MB, of the eye textures the last timed step handed back (the last
    frame of each of the 2 contexts at --streams 4), equal to the oracle's EASU+RCAS of the same pool frames."""
    import os

    import numpy as np

    import bench
    from openvr_fsr_b200 import synth
    from oracle import pyoracle as po
    r = _run("--steps", "2", "--no-extras", "--no-e2e", "--no-cpu-baseline", "--no-ncu", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])["steps"] == 2
    files = sorted(tmp_path.glob("*.npy"))
    assert {f.stem for f in files} == {f"frame{bench.POOL - k}_{e}" for k in (1, 2) for e in ("left", "right")}
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    base = synth.stereo_pair("natural", bench.IN_W, bench.IN_H, 1)
    idx = np.sort(np.random.default_rng(0).choice(bench.OUT_W * bench.OUT_H, bench.DUMP_PIXELS, replace=False))
    for f in files:
        frame, eye = int(f.stem.split("_")[0][5:]), ("left", "right").index(f.stem.split("_")[1])
        got = np.load(f)
        assert got.dtype == np.float32 and got.shape == (bench.DUMP_PIXELS, 4)
        src = np.roll(base[eye], 37 * frame, axis=0)  # bench.build_pool's frame of rank 0
        uc = po.upscale_constants(eye, True, bench.IN_W, bench.IN_H, bench.OUT_W, bench.OUT_H, radius=2.0)
        sc = po.sharpen_constants(eye, True, bench.OUT_W, bench.OUT_H, radius=2.0, sharpness=bench.SHARPNESS)
        n = os.cpu_count() or 1
        want = po.rcas(po.easu(src, bench.OUT_W, bench.OUT_H, uc, nthreads=n), sc, nthreads=n)
        assert np.array_equal(got, want.reshape(-1, 4)[idx].astype(np.float32)), f.name


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = _run("--steps", "1", "--warmup", "3", "--no-cpu-baseline", timeout=300)
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stdout + r.stderr)
    assert not [l for l in r.stdout.splitlines() if l.startswith('{"metric"')]
