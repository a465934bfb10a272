"""Dev/measurement tool: per-eye time of ovrfsr_apply_bounds against ovrfsr_apply on the C2 FSR workload (1683x1869
-> 2244x2492 RGBA8, strict, sharpness 0.9, radius 2.0 and 0.5) and the C4 NIS one (1512x1680 -> 2016x2240, NVScaler,
radius 2.0).  Eyes alternate over a pool of 8 distinct textures per eye (C2: 201 MB, more than the 126 MB L2), the two
eyes on one stream, CUDA events around each timed window.  Cases: full bounds through ovrfsr_apply and through
ovrfsr_apply_bounds; views of 0.9, 0.8 and 0.7 of the texture at the origin; a 0.8 view at an origin with x0 % 4 != 0;
a 0.8-ish view whose rectangle changes every frame (dynamic resolution).  The C ABI is called directly through ctypes
so that the host side stays ahead of the GPU.
usage: python tools/bench_bounds.py [--reps N] [--out FILE]"""
import argparse
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import openvr_fsr_b200 as ovr  # noqa: E402
from openvr_fsr_b200 import _lib as L, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=6, help="passes over the pool per timed window")
ap.add_argument("--windows", type=int, default=5)
ap.add_argument("--out", default=None)
a = ap.parse_args()
dev = torch.device("cuda:0")
lib = L.lib()
stream = torch.cuda.current_stream()
sp = C.c_void_p(stream.cuda_stream)

WORKLOADS = {
    "C2_fsr_r2.0": dict(iw=1683, ih=1869, cfg=ovr.Config(fsrEnabled=True, renderScale=0.75, sharpness=0.9, radius=2.0)),
    "C2_fsr_r0.5": dict(iw=1683, ih=1869, cfg=ovr.Config(fsrEnabled=True, renderScale=0.75, sharpness=0.9, radius=0.5)),
    "C4_nis_r2.0": dict(iw=1512, ih=1680, cfg=ovr.Config(fsrEnabled=True, useNis=True, renderScale=0.75, sharpness=0.9, radius=2.0)),
}


def cases(iw):
    x1 = 5.0 / iw  # 5 texels: x0 % 4 == 1
    dyn = [L.Bounds(k * 3.0 / iw, k * 2.0 / iw, 0.78 + 0.02 * (k % 4), 0.8 - 0.01 * k) for k in range(8)]
    return {
        "apply_full": None,
        "bounds_full": [L.Bounds(0, 0, 1, 1)],
        "bounds_0.9": [L.Bounds(0, 0, 0.9, 0.9)],
        "bounds_0.8": [L.Bounds(0, 0, 0.8, 0.8)],
        "bounds_0.7": [L.Bounds(0, 0, 0.7, 0.7)],
        "bounds_0.8_x0mod4=1": [L.Bounds(x1, x1, x1 + 0.8, x1 + 0.8)],
        "bounds_dynamic_0.8": dyn,
    }


def run(ctx, pool, bounds, n):
    """n eyes, alternating left / right over the pool; `bounds` (a list cycled per frame) or None for ovrfsr_apply"""
    out, rect = L.Image(), L.Rect()
    for i in range(n):
        eye, k = i & 1, (i >> 1) % len(pool[0])
        src = C.byref(pool[eye][k])
        if bounds is None:
            rc = lib.ovrfsr_apply(ctx, eye, src, 1, C.byref(out), sp)
        else:
            rc = lib.ovrfsr_apply_bounds(ctx, eye, src, C.byref(bounds[(i >> 1) % len(bounds)]), C.byref(out), C.byref(rect), sp)
        if rc != 0:
            raise RuntimeError(lib.ovrfsr_last_error(ctx).decode())


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else None}


res = {"tool": "tools/bench_bounds.py", **gpu_info(), "pool_per_eye": 8, "reps": a.reps, "windows": a.windows, "results": {}}
for wname, w in WORKLOADS.items():
    iw, ih, cfg = w["iw"], w["ih"], w["cfg"]
    gen = synth.natural_rgba8
    keep, pool = [], [[], []]
    for eye in (0, 1):
        for k in range(8):
            t = ovr.to_image(np.roll(gen(iw, ih, 1 + eye), 37 * k + 11 * eye, axis=0), dev)
            keep.append(t)
            pool[eye].append(ovr.image_of(t))
    ctx = C.c_void_p()
    L.check(lib.ovrfsr_create(C.byref(ctx), C.byref(cfg.to_c())))
    n = 2 * 8 * a.reps
    out = {}
    allcases = cases(iw)
    for cname, b in allcases.items():  # warm up every shape
        run(ctx, pool, b, 32)
    torch.cuda.synchronize()
    times = {c: [] for c in allcases}
    for _ in range(a.windows):  # the cases alternate window by window
        for cname, b in allcases.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            run(ctx, pool, b, n)
            e1.record(stream)
            e1.synchronize()
            times[cname].append(e0.elapsed_time(e1) * 1000.0 / n)
    for cname, ts in times.items():
        us = float(np.median(ts))
        out[cname] = {"us_per_eye": round(us, 2), "us_per_eye_spread": [round(min(ts), 2), round(max(ts), 2)],
                      "pairs_per_s": round(1e6 / (2 * us), 1)}
    lib.ovrfsr_destroy(ctx)
    res["results"][wname] = out
    del keep, pool
    torch.cuda.empty_cache()
print(json.dumps(res, indent=1))
if a.out:
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
