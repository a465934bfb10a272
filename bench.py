#!/usr/bin/env python
"""bench.py -- stereo eye-pairs/s of the FSR1 EASU+RCAS pass (BASELINE.json metric) on N B200s.

Workload (config.workload): BASELINE.json configs[1] = SURVEY.md C2: stereo 1683x1869 -> 2244x2492 RGBA8,
renderScale 0.75, sharpness 0.9, FSR path, radius 2.0 (mask off: EVERY pixel takes EASU+RCAS; the reference's
default radius 0.5 is reported beside it as `masked_r0.5`).  A "step" is one pass of the hot path over
PAIRS_PER_STEP = 256 stereo pairs per GPU (BASELINE.json configs[4]'s batch): 32 passes over a pool of 8 distinct
pairs (201 MB of input, larger than the 126 MB L2, so no step re-reads inputs from L2).  At ~4.5 k pairs/s a step
is ~55 ms, so the driver's `--steps 20` gives a timed region above one second and the clock samples are taken
inside it.

  value     : whole-job pairs/s, inputs resident in HBM, CUDA-event timed, max over ranks.  --streams (default 4):
              streams/2 PostProcessor contexts = frames in flight, one CUDA stream per eye of each; 1 = everything
              strictly back to back on one stream (`value_one_stream` reports that beside the headline)
  pipeline  : "two-pass" (default) = the reference's two dispatches per eye; "fused" (--fused) = ONE kernel per eye does
              EASU -> RGBA8 -> RCAS with the intermediate in shared memory.  Same output bits; the other one is
              measured beside the headline (`value_fused` / `value_two_pass`) -- the fused kernel is slower on B200
              because the pass is issue-bound, not traffic-bound (DESIGN.md section 5)
  e2e       : same metric through PostProcessor.apply_host with pinned HOST buffers (H2D + kernels + D2H timed),
              3 contexts in flight, the rank bound to its GPU's NUMA node before the pinned allocation
  roofline  : the dominant kernel's ALGORITHMIC bytes (SURVEY.md 8d: fused = source in + output out = 34,950,300 B per
              eye; two-pass EASU the same figure, RCAS 44,736,384 B) / its mean launch time (CUDA events on the launch
              stream, the kernel alone on its stream) against MEASURED_PEAKS.json hbm_gbs; `traffic` and
              `instr_per_output_px` are measured in this run by an `ncu` child over steady-state launches
              (--cache-control none, so earlier launches' outputs are evicted while later ones run); null if ncu is
              not usable on the box
  clocks    : nvidia-smi SM clock / throttle reasons sampled every 20 ms inside the timed region
  cpu_baseline : the reference's own lines (oracle/_ref, kind "reference") or the restated oracle ("port") on the
              box's host cores, a bounded sample of the same workload, rank 0 at N=1 only
  c5_strong : BASELINE.json configs[4] as written: 256 C2 frames sharded frame f -> rank f mod N, wall = max over
              ranks between two barriers (strong scaling: the driver compares N = 1, 2, 4, 8)
  c4_eye_sharded : (N = 2 only) BASELINE.json configs[3]: NIS NVScaler 1512x1680 -> 2016x2240, one eye per GPU, with an
              all-gathered checksum against both eyes computed on one GPU
  --impl reference : the CPU reference arm (same metric / config), rank 0 only under torchrun; a step = one stereo
              pair (a bounded sample of the 256-pair step)
  --dump-outputs DIR : after the timed steps, rank 0 writes the eye textures its last step handed back as
              DIR/frame<i>_<eye>.npy (float32 texel codes at a fixed, seeded sample of pixels), so that two builds can be
              compared output for output on the same inputs

Multi-GPU: frames are independent (SURVEY.md 8e) -> each rank processes its own pool, no data-path
collective; NCCL only broadcasts the constant block from rank 0 and forms the barriers.  scaling = weak.
"""
from __future__ import annotations

import argparse
import csv
import io
import json
import os
import shutil
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

IN_W, IN_H, RENDER_SCALE, SHARPNESS = 1683, 1869, 0.75, 0.9
OUT_W, OUT_H = 2244, 2492
EASU_BYTES_PER_EYE = IN_W * IN_H * 4 + OUT_W * OUT_H * 4          # 34,950,300 (SURVEY.md 8d)
RCAS_BYTES_PER_EYE = 2 * OUT_W * OUT_H * 4                          # 44,736,384
FUSED_BYTES_PER_EYE = EASU_BYTES_PER_EYE                            # in + out: the intermediate is not traffic
PAIR_BYTES_TWO_PASS = 2 * (EASU_BYTES_PER_EYE + RCAS_BYTES_PER_EYE)  # 159,373,368
PAIR_BYTES_FUSED = 2 * FUSED_BYTES_PER_EYE                          # 69,900,600
METRIC = "stereo eye-pairs/sec EASU+RCAS @2244x2492"
WORKLOAD = "C2: stereo 1683x1869->2244x2492 RGBA8, renderScale=0.75, sharpness=0.9, FSR EASU+RCAS"
POOL = 8               # distinct stereo pairs resident per GPU
PASSES = 32            # passes over the pool per step
PAIRS_PER_STEP = POOL * PASSES  # 256
C5_FRAMES = 256
C4 = dict(iw=1512, ih=1680, scale=0.75)


def make_config(args, world):
    """The `config` object of the JSON line; built from the arguments only, so both arms print the same one."""
    return {"workload": WORKLOAD, "radius": args.radius, "math": args.math,
            "pipeline": "fused" if args.fused else "two-pass",
            "pairs_per_step_per_gpu": PAIRS_PER_STEP,
            "pool": f"{POOL} distinct pairs per GPU cycled {PASSES}x per step",
            "l2": f"inputs larger than L2 ({POOL} distinct pairs = {POOL * 2 * IN_W * IN_H * 4 / 1e6:.0f} MB per GPU)",
            "source_pitch": "256-byte aligned rows (TMA tile loads)",
            "streams": f"{args.streams} CUDA streams per GPU: {max(1, args.streams // 2)} frame(s) in flight, one stream per eye",
            "parallelism": f"frames sharded {world}x, no data-path collective"}


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed workload runs (B200_PROFILING.md recipe).  The sampler
    is started before the warm-up (nvidia-smi needs ~100 ms to produce its first row); rows are time-stamped on
    arrival and only those inside the marked window [mark_begin, mark_end] count."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.t0, self.t1 = index, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if self.t0 is None or ts < self.t0 or (self.t1 is not None and ts > self.t1):
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons),
                "note": "sampled inside the timed region (nvidia-smi -lms 20)"}


# ------------------------------------------------------------------------------------------------------
# CPU reference arm / baseline
# ------------------------------------------------------------------------------------------------------
def cpu_pair_seconds(left, right, radius, which, threads):
    """One stereo pair (EASU+RCAS, both eyes) on the host with `threads` threads."""
    from oracle import pyoracle as po
    t0 = time.perf_counter()
    for eye, img in ((0, left), (1, right)):
        uc = po.upscale_constants(eye, True, IN_W, IN_H, OUT_W, OUT_H, radius=radius)
        sc = po.sharpen_constants(eye, True, OUT_W, OUT_H, radius=radius, sharpness=SHARPNESS)
        po.rcas(po.easu(img, OUT_W, OUT_H, uc, which=which, nthreads=threads), sc, which=which, nthreads=threads)
    return time.perf_counter() - t0


def cpu_threads():
    """Threads this process may really use, and how many physical cores that is (SMT siblings share one)."""
    cpus = sorted(os.sched_getaffinity(0))
    cores = set()
    for c in cpus:
        try:
            sib = Path(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read_text().strip()
        except Exception:
            sib = str(c)
        cores.add(sib)
    return len(cpus), len(cores)


def pick_cpu_threads(left, right, radius, which):
    """Best of {all usable threads, one per physical core}: SMT pairs sharing an FP unit are not always a win for this
    arithmetic-bound loop.  One untimed pair each."""
    t_all, t_cores = cpu_threads()
    cands = sorted({t_all, max(1, t_cores)}, reverse=True)
    best = min(cands, key=lambda t: cpu_pair_seconds(left, right, radius, which, t))
    return best, t_all, t_cores


def cpu_arm_inputs():
    from oracle import pyoracle as po
    from openvr_fsr_b200 import synth
    which, kind = ("ref", "reference") if po.ref_available() else ("oracle", "port")
    left, right = synth.stereo_pair("natural", IN_W, IN_H, 1)
    return which, kind, left, right


def cpu_baseline(radius, pairs=12):
    which, kind, left, right = cpu_arm_inputs()
    threads, t_all, t_cores = pick_cpu_threads(left, right, radius, which)
    t0 = time.perf_counter()
    for _ in range(pairs):
        cpu_pair_seconds(left, right, radius, which, threads)
    sec = (time.perf_counter() - t0) / pairs
    return {"value": 1.0 / sec, "unit": "pairs/s", "cores": threads, "kind": kind, "physical_cores": t_cores,
            "usable_threads": t_all,
            "sample": f"{pairs} stereo pairs of the same workload (both eyes EASU+RCAS each), {threads} threads "
                      f"(best of {t_all} threads / {t_cores} physical cores), work units of 16 groups"}


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores."""
    if rank != 0:
        return
    which, kind, left, right = cpu_arm_inputs()
    threads, t_all, t_cores = pick_cpu_threads(left, right, args.radius, which)
    for _ in range(args.warmup):
        cpu_pair_seconds(left, right, args.radius, which, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_pair_seconds(left, right, args.radius, which, threads)
    dt = time.perf_counter() - t0
    val = args.steps / dt
    sample = (f"each step = 1 stereo pair of the {PAIRS_PER_STEP}-pair step (bounded sample), {threads} host threads "
              f"(best of {t_all} threads / {t_cores} physical cores)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": make_config(args, world),
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": threads, "kind": kind, "physical_cores": t_cores,
                         "usable_threads": t_all, "sample": sample},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
def build_pool(ovr, synth, dev, rank):
    pool = []
    base_l, base_r = synth.stereo_pair("natural", IN_W, IN_H, 1)
    for i in range(POOL):
        sh = 37 * (i + rank * POOL)
        # device images with a 256-byte-aligned row pitch (what cudaMallocPitch / ovrfsr_image_alloc return): the
        # TMA tile loader needs a 16-byte-aligned pitch; algorithmic bytes are counted without the padding
        pool.append((ovr.to_image(np.roll(base_l, sh, axis=0), dev), ovr.to_image(np.roll(base_r, sh, axis=0), dev)))
    return pool


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--radius", type=float, default=2.0, help="Config::radius; 2.0 = mask off (headline)")
    ap.add_argument("--math", default="strict", choices=["fast", "strict"],
                    help="strict = bit-identical to the reference lines end to end (headline); fast = <=1 LSB per pass")
    ap.add_argument("--streams", type=int, default=4, choices=[1, 2, 4, 6, 8],
                    help="1 = everything on one stream; 2 = one stream per eye; 4+ = streams/2 frames in flight, one context each")
    ap.add_argument("--fused", action="store_true", help="one fused EASU->RCAS kernel per eye instead of the two dispatches")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline + roofline only")
    ap.add_argument("--no-ncu", action="store_true", help="skip the ncu child that measures DRAM traffic / instructions")
    ap.add_argument("--traffic-probe", action="store_true", help=argparse.SUPPRESS)  # the ncu child's workload
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last step as DIR/<name>.npy (float32, sampled)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm has none")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import openvr_fsr_b200 as ovr
    from openvr_fsr_b200 import numa, sharding, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    if args.warmup < 3:
        args.warmup = 3
    # host placement first: pinned buffers allocated later land on the GPU's own NUMA node
    props = torch.cuda.get_device_properties(local_rank)
    pci = None
    if all(hasattr(props, a) for a in ("pci_domain_id", "pci_bus_id", "pci_device_id")):
        pci = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
    host = numa.bind_to_gpu_node(local_rank, pci_bus_id=pci)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.traffic_probe:
        traffic_probe_workload(ovr, torch, synth, dev, args)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    math_mode = ovr.MATH_STRICT if args.math == "strict" else ovr.MATH_FAST
    cfg = ovr.Config(fsrEnabled=True, renderScale=RENDER_SCALE, sharpness=SHARPNESS, radius=args.radius,
                     mathMode=math_mode, device=local_rank, fusedFsr=args.fused)

    # north_star: NCCL only as barrier / broadcast of the shared FSR constants (96 + 48 bytes), root 0
    consts = sharding.broadcast_constants(cfg, IN_W, IN_H, OUT_W, OUT_H, dev if world > 1 else None)
    pool = build_pool(ovr, synth, dev, rank)
    runner = EyeStreams(ovr, torch, cfg, dev, args.streams)
    assert np.array_equal(pp_consts_after_first(runner.pps[0], pool[0][0]), consts["upscale"][0]), "rank constants differ from root's"

    def step():
        for _ in range(PASSES):
            runner.pass_over(pool)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    barrier()
    sampler.mark_begin()
    launches0 = ovr.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    runner.fork()
    for _ in range(args.steps):
        step()
    runner.join()
    ev1.record()
    barrier()
    sampler.mark_end()
    launches = ovr.kernel_launches() - launches0
    elapsed_ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    elapsed_ms = float(elapsed_ms.item())
    clocks = sampler.stop() if rank == 0 else None
    pairs = world * PAIRS_PER_STEP * args.steps
    value = pairs / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(runner, args.dump_outputs)
    runner.close()

    # ---- instrumented pass: per-kernel CUDA events on the launch stream (roofline of the dominant kernel)
    kt = per_kernel_times(ovr, torch, pool, consts, math_mode, 4)
    peak, peak_src = _peaks()
    sm_clock_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    prof = {}
    if rank == 0 and world == 1 and not args.no_ncu:
        prof = ncu_child(args)

    def roof(kernel, nbytes, ms, key):
        p = prof.get(key, {})
        r = {"bound": "hbm", "kernel": kernel, "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
             "frac": nbytes / (ms * 1e-3) / 1e9 / peak, "traffic": p.get("traffic"), "peak_source": peak_src,
             "algorithmic_bytes_per_launch": nbytes, "ms_per_launch": ms,
             "instr_per_output_px": p.get("instr_per_px")}
        if p.get("instr_per_px"):
            # executed warp-instructions / s against 4 issue slots / SM / clock: the bound that applies when the mask is off
            r["fp32_issue_frac"] = p["instr_per_px"] * OUT_W * OUT_H / 32 / (ms * 1e-3) / (148 * 4 * sm_clock_mhz * 1e6)
        return r

    dominant = ("fsr_fused_kernel", FUSED_BYTES_PER_EYE, kt["fused"], "fused") if args.fused else \
        ("easu_kernel", EASU_BYTES_PER_EYE, kt["easu"], "easu")
    roofline = roof(*dominant)
    roofline["timing"] = ("ms_per_launch = this kernel alone on its stream (CUDA events); inside the step, kernels of the other "
                          "eye / frame run concurrently, so ms_per_step is below the sum of launch times")
    roofline["traffic_note"] = prof.get("note", "ncu child skipped (multi-GPU rank or --no-ncu)")
    roofline["note"] = ("unmasked EASU+RCAS is FP32-issue-bound, not HBM-bound (DESIGN.md section 5): fp32_issue_frac = executed "
                        "warp-instructions/s (ncu count of this run x live launch rate) / issue peak")
    rooflines_other = {"fused": roof("fsr_fused_kernel", FUSED_BYTES_PER_EYE, kt["fused"], "fused"),
                       "easu": roof("easu_kernel", EASU_BYTES_PER_EYE, kt["easu"], "easu"),
                       "rcas": roof("rcas_kernel", RCAS_BYTES_PER_EYE, kt["rcas"], "rcas")}

    extras = {}
    if not args.no_extras:
        import dataclasses
        n = 6  # passes over the pool per sub-measurement (48 pairs, >= 10 ms each)
        extras["masked_r0.5"] = {"value": world * quick_value(ovr, torch, dataclasses.replace(cfg, radius=0.5), pool, n, args.streams),
                                 "unit": "pairs/s", "note": "reference default radius 0.5 (EASU/RCAS inside the radius only)"}
        other_mode = "fast" if args.math == "strict" else "strict"
        extras[f"value_{other_mode}_math"] = {
            "value": world * quick_value(ovr, torch, dataclasses.replace(cfg, mathMode=ovr.MATH_FAST if other_mode == "fast" else ovr.MATH_STRICT), pool, n, args.streams),
            "unit": "pairs/s", "note": ("FMA-contracted kernels: each pass <= 1 LSB from the reference lines on identical inputs"
                                        if other_mode == "fast" else "reference operation order: bit-identical to the reference lines end to end")}
        other_pipe = "two_pass" if args.fused else "fused"
        extras[f"value_{other_pipe}"] = {
            "value": world * quick_value(ovr, torch, dataclasses.replace(cfg, fusedFsr=not args.fused), pool, n, args.streams),
            "masked_r0.5": world * quick_value(ovr, torch, dataclasses.replace(cfg, fusedFsr=not args.fused, radius=0.5), pool, n, args.streams),
            "unit": "pairs/s", "note": "the other pipeline (same output bits): " + ("the reference's two dispatches per eye" if args.fused else "one fused EASU->RCAS kernel per eye")}
        extras["value_one_stream"] = {"value": world * quick_value(ovr, torch, cfg, pool, n, 1),
                                      "masked_r0.5": world * quick_value(ovr, torch, dataclasses.replace(cfg, radius=0.5), pool, n, 1),
                                      "unit": "pairs/s", "note": "everything strictly back to back on ONE stream (a VR render thread)"}
        extras["value_one_stream_pair"] = {"value": world * quick_value(ovr, torch, cfg, pool, n, 1, pair=True),
                                           "masked_r0.5": world * quick_value(ovr, torch, dataclasses.replace(cfg, radius=0.5), pool, n, 1, pair=True),
                                           "unit": "pairs/s", "note": "ONE caller stream, both eyes per call (ovrfsr_apply_pair: the right eye forked onto a ctx-owned stream and joined back)"}
        extras["c5_strong"] = c5_strong(ovr, torch, dist, cfg, pool, dev, rank, world, args.streams)
        if world == 2:
            extras["c4_eye_sharded"] = c4_eye_sharded(ovr, torch, dist, synth, sharding, dev, rank, math_mode)

    # ---- end to end: host buffers through the public API, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = e2e_run(ovr, torch, dist, cfg, pool, dev, world)
        if e2e is not None:
            e2e["numa"] = host

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args.radius)

    if rank == 0:
        pair_bytes = PAIR_BYTES_FUSED if args.fused else PAIR_BYTES_TWO_PASS
        out = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args, world),
            "hbm_gbs_whole_pass": value / world * pair_bytes / 1e9,
            "hbm_frac_whole_pass": value / world * pair_bytes / 1e9 / peak,
            "algorithmic_bytes_per_pair": pair_bytes,
            "roofline": roofline, "rooflines_per_kernel": rooflines_other, "clocks": clocks, "gpu_launches": int(launches),
            "host": host,
        }
        ipp = {k: v.get("instr_per_px") for k, v in prof.items() if isinstance(v, dict)}
        step_ipp = ipp.get("fused") if args.fused else ((ipp.get("easu") or 0) + (ipp.get("rcas") or 0) or None)
        if step_ipp:
            wi = step_ipp * OUT_W * OUT_H * 2 / 32 * (value / world)
            out["issue_roofline_whole_step"] = {
                "achieved": wi / 1e12, "peak": 148 * 4 * sm_clock_mhz * 1e6 / 1e12, "unit": "T warp-instr/s",
                "frac": wi / (148 * 4 * sm_clock_mhz * 1e6),
                "note": "executed warp-instructions per pair (ncu count of this run) x pairs/s, against 148 SMs x 4 schedulers "
                        "x the SM clock sampled during the run: utilisation of the kernel's own instruction stream"}
        out.update(extras)
        if e2e is not None:
            out["e2e"] = e2e
        if cpu is not None:
            out["cpu_baseline"] = cpu
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def pp_consts_after_first(pp, tex):
    import torch
    pp.apply(0, tex)
    torch.cuda.synchronize()
    c = pp.upscale_constants(0)
    pp.reset()
    return c


def per_kernel_times(ovr, torch, pool, consts, math_mode, reps):
    """Mean device time of one launch (per eye) of the fused kernel and of the two dispatches it replaces; events
    recorded on the launching stream, nothing synchronises inside the loops, so the GPU stays busy."""
    dev = pool[0][0].device
    mid = ovr.alloc_image(OUT_W, OUT_H, torch.uint8, dev)
    dst = ovr.alloc_image(OUT_W, OUT_H, torch.uint8, dev)
    marks, fmarks = [], []
    for _ in range(reps):
        for left, right in pool:
            for eye, tex in ((0, left), (1, right)):
                evs = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                evs[0].record()
                ovr.fsr_easu(tex, mid, consts["upscale"][eye], math_mode)
                evs[1].record()
                ovr.fsr_rcas(mid, dst, consts["sharpen"][eye], math_mode)
                evs[2].record()
                marks.append(evs)
    for _ in range(reps):
        for left, right in pool:
            for eye, tex in ((0, left), (1, right)):
                evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                evs[0].record()
                ovr.fsr_fused(tex, dst, consts["upscale"][eye], consts["sharpen"][eye], math_mode)
                evs[1].record()
                fmarks.append(evs)
    torch.cuda.synchronize()
    skip = min(len(marks) // 4, 8)
    return {"easu": statistics.mean(m[0].elapsed_time(m[1]) for m in marks[skip:]),
            "rcas": statistics.mean(m[1].elapsed_time(m[2]) for m in marks[skip:]),
            "fused": statistics.mean(m[0].elapsed_time(m[1]) for m in fmarks[skip:])}


class EyeStreams:
    """The device-resident workload driver: n_streams // 2 PostProcessor contexts (frames in flight), one CUDA stream
    per eye of each.  A context keeps one output set per eye, so its two eyes can run concurrently; frame i goes to
    context i % n_ctx.  Kernels of different eyes / frames then share the SMs: a persistent grid's last wave no
    longer leaves SMs idle."""

    def __init__(self, ovr, torch, cfg, dev, n_streams, pair=False):
        self.pair = pair  # one caller stream, both eyes handed over in one PostProcessor.apply_pair call
        self.last = {}  # context -> (pool index, (left out, right out)) of the last frame it processed
        self.main = torch.cuda.current_stream(dev)
        self.pps = [ovr.PostProcessor(cfg) for _ in range(max(1, n_streams // 2))]
        if n_streams == 1:
            self.streams = [[self.main, self.main]]
        else:
            self.streams = [[torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)] for _ in self.pps]

    def pass_over(self, pool, frames=None):
        n = len(self.pps)
        for i in (range(len(pool)) if frames is None else frames):
            left, right = pool[i % len(pool)]
            if self.pair:
                outs = self.pps[i % n].apply_pair(left, right, stream=self.streams[i % n][0])
            else:
                outs = (self.pps[i % n].apply(0, left, stream=self.streams[i % n][0]),
                        self.pps[i % n].apply(1, right, stream=self.streams[i % n][1]))
            # the returned views stay valid until the context's next apply of the same eye
            self.last[i % n] = (i % len(pool), outs)

    def fork(self):
        for pair in self.streams:
            for s in pair:
                if s is not self.main:
                    s.wait_stream(self.main)

    def join(self):
        for pair in self.streams:
            for s in pair:
                if s is not self.main:
                    self.main.wait_stream(s)

    def close(self):
        for p in self.pps:
            p.close()


DUMP_PIXELS = 1 << 18  # 4 MiB of float32 per eye texture; --streams 8 leaves 8 of them: 32 MiB in all


def dump_outputs(runner, directory):
    """--dump-outputs: the eye textures the last step handed back that the contexts still hold (the last frame each
    context processed, both eyes; the earlier frames' outputs were overwritten inside the step), once the step has
    finished.  A 2244x2492 RGBA8 eye is 89 MB as float32, so each file holds the texel codes of the same DUMP_PIXELS
    pixels, drawn without replacement with seed 0 and sorted (row-major index): shape (DUMP_PIXELS, 4)."""
    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    idx = None
    for frame, eyes in sorted(runner.last.values(), key=lambda fe: fe[0]):
        for name, t in zip(("left", "right"), eyes):
            px = t.contiguous().cpu().numpy().reshape(-1, 4)
            if idx is None:
                idx = np.sort(np.random.default_rng(0).choice(px.shape[0], DUMP_PIXELS, replace=False))
            np.save(out / f"frame{frame}_{name}.npy", px[idx].astype(np.float32))


def quick_value(ovr, torch, cfg, pool, passes, n_streams, pair=False):
    """pairs/s of `passes` passes over the pool with the given configuration (one rank)."""
    dev = pool[0][0].device
    r = EyeStreams(ovr, torch, cfg, dev, n_streams, pair)
    for _ in range(2):
        r.pass_over(pool)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r.fork()
    for _ in range(passes):
        r.pass_over(pool)
    r.join()
    e1.record()
    torch.cuda.synchronize()
    v = len(pool) * passes / (e0.elapsed_time(e1) * 1e-3)
    r.close()
    return v


def c5_strong(ovr, torch, dist, cfg, pool, dev, rank, world, n_streams):
    """BASELINE.json configs[4] as written: 256 independent C2 stereo frames, frame f -> rank f mod N, inputs
    resident (the 8-pair pool cycled), wall = max over ranks between two barriers.  Strong scaling: the total is fixed."""
    from openvr_fsr_b200 import sharding
    frames = sharding.frames_for_rank(C5_FRAMES, rank, world)
    r = EyeStreams(ovr, torch, cfg, dev, n_streams)
    r.pass_over(pool)
    times = []
    for _ in range(3):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r.fork()
        r.pass_over(pool, frames)
        r.join()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        times.append(float(ms.item()))
    r.close()
    best = min(times)
    return {"frames": C5_FRAMES, "frames_per_gpu": len(frames), "ms_total": best, "value": C5_FRAMES / (best * 1e-3),
            "unit": "pairs/s", "scaling": "strong", "ms_all": times,
            "note": "256 C2 frames sharded frame f -> rank f mod N; wall = max over ranks between two barriers, best of 3"}


def c4_eye_sharded(ovr, torch, dist, synth, sharding, dev, rank, math_mode):
    """BASELINE.json configs[3]: NIS NVScaler 1512x1680 -> 2016x2240, 2 GPUs, one eye per GPU (VrHooks.cpp:53 calls
    Apply per eye).  Each rank runs its eye of 8 frames; the output checksums are all-gathered and rank 0 checks them
    against BOTH eyes computed on its own GPU: sharding does not change a bit."""
    iw, ih, scale = C4["iw"], C4["ih"], C4["scale"]
    eye = sharding.eye_for_rank(rank, 2)[0]
    cfg = ovr.Config(fsrEnabled=True, useNis=True, renderScale=scale, sharpness=SHARPNESS, radius=2.0, mathMode=math_mode,
                     device=dev.index)
    left, right = synth.stereo_pair("natural", iw, ih, 1)
    frames = [[ovr.to_image(np.roll(e, 31 * i, axis=0), dev) for e in (left, right)] for i in range(8)]

    def checksum(t):
        v = t.contiguous().view(torch.uint8).to(torch.int64).flatten()
        return int((v * (torch.arange(v.numel(), device=v.device) % 65521 + 1)).sum().item())

    pp = ovr.PostProcessor(cfg)
    mine = [checksum(pp.apply(eye, f[eye])) for f in frames]
    torch.cuda.synchronize()
    dist.barrier()
    reps = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        for f in frames:
            pp.apply(eye, f[eye])
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    sums = torch.tensor(mine, dtype=torch.int64, device=dev)
    gathered = [torch.zeros_like(sums) for _ in range(2)]
    dist.all_gather(gathered, sums)
    ok = None
    if rank == 0:
        both = [[checksum(pp.apply(e, f[e])) for f in frames] for e in (0, 1)]
        ok = all(gathered[e].tolist() == both[e] for e in (0, 1))
    pp.close()
    return {"workload": "C4: stereo 1512x1680->2016x2240 RGBA8, NIS NVScaler, sharpness 0.9, radius 2.0, one eye per GPU",
            "value": reps * len(frames) / (float(ms.item()) * 1e-3), "unit": "pairs/s",
            "bit_equal_to_single_gpu": ok, "algorithmic_bytes_per_eye": iw * ih * 4 + 2016 * 2240 * 4,
            "note": "each rank runs its eye of every frame; pairs/s = frames / max-over-ranks time"}


def e2e_run(ovr, torch, dist, cfg, pool, dev, world, passes=160, contexts=3):
    """Same metric through the reference-facing call with HOST buffers: per eye, pinned host -> device copy,
    EASU+RCAS, device -> pinned host copy, all inside the timed region.  `contexts` PostProcessor contexts are cycled
    (frame i uses context i % contexts, each with one stream per eye) so that uploads, kernels and downloads of
    neighbouring frames overlap: a context owns its staging / output images, so frames in flight need one each."""
    pps = [ovr.PostProcessor(cfg) for _ in range(contexts)]
    n = len(pool)
    h_in = [(l.cpu().contiguous().pin_memory(), r.cpu().contiguous().pin_memory()) for l, r in pool]
    h_out = [(torch.empty((OUT_H, OUT_W, 4), dtype=torch.uint8).pin_memory(),
              torch.empty((OUT_H, OUT_W, 4), dtype=torch.uint8).pin_memory()) for _ in range(n)]
    streams = [[torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)] for _ in pps]

    def one_pass():
        for i in range(n):
            for eye in (0, 1):
                pps[i % contexts].apply_host(eye, h_in[i][eye], h_out[i][eye], stream=streams[i % contexts][eye])

    for _ in range(2):
        one_pass()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(streams[0][0])
    for _ in range(passes):
        one_pass()
    for pair in streams:
        for s in pair:
            if s is not streams[0][0]:
                streams[0][0].wait_stream(s)
    e1.record(streams[0][0])
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = torch.tensor([max(e0.elapsed_time(e1), 0.0)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    for p in pps:
        p.close()
    pairs = world * n * passes
    return {"value": pairs / (float(ms.item()) * 1e-3), "unit": "pairs/s",
            "h2d_bytes_per_step": PAIRS_PER_STEP * 2 * IN_W * IN_H * 4, "d2h_bytes_per_step": PAIRS_PER_STEP * 2 * OUT_W * OUT_H * 4,
            "pairs_timed_per_gpu": n * passes, "seconds_timed": float(ms.item()) * 1e-3, "wall_value": pairs / wall,
            "note": f"pinned host -> H2D -> EASU+RCAS -> D2H per eye via ovrfsr_apply_host; {contexts} contexts x 2 streams in flight; "
                    "byte counts are per 256-pair step per GPU"}


# ------------------------------------------------------------------------------------------------------
# DRAM traffic / executed instructions of the kernels, measured in THIS run by an ncu child
# ------------------------------------------------------------------------------------------------------
def traffic_probe_workload(ovr, torch, synth, dev, args):
    """What the ncu child runs: steady-state launches of the fused kernel and of the two dispatches over the pool
    (inputs > L2, outputs cycling over 4 images so that earlier outputs are evicted by later launches)."""
    math_mode = ovr.MATH_STRICT if args.math == "strict" else ovr.MATH_FAST
    cfg = ovr.Config(fsrEnabled=True, renderScale=RENDER_SCALE, sharpness=SHARPNESS, radius=args.radius, mathMode=math_mode)
    pool = build_pool(ovr, synth, dev, 0)
    uc = [ovr.make_upscale_constants(cfg, e, True, IN_W, IN_H, OUT_W, OUT_H) for e in (0, 1)]
    sc = [ovr.make_sharpen_constants(cfg, e, True, OUT_W, OUT_H) for e in (0, 1)]
    outs = [ovr.alloc_image(OUT_W, OUT_H, torch.uint8, dev) for _ in range(4)]
    mids = [ovr.alloc_image(OUT_W, OUT_H, torch.uint8, dev) for _ in range(4)]
    k = 0
    for _ in range(3):
        for left, right in pool:
            for eye, tex in ((0, left), (1, right)):
                ovr.fsr_fused(tex, outs[k % 4], uc[eye], sc[eye], math_mode)
                ovr.fsr_easu(tex, mids[k % 4], uc[eye], math_mode)
                ovr.fsr_rcas(mids[k % 4], outs[(k + 1) % 4], sc[eye], math_mode)
                k += 1
    torch.cuda.synchronize()


def ncu_child(args):
    """Run `bench.py --traffic-probe` under ncu (two metrics passes, no cache flush between launches) and average
    dram bytes and executed instructions per launch over the steady-state launches of each kernel."""
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not Path(ncu).exists():
        return {"note": "ncu not found on this box"}
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum,smsp__inst_executed.sum",
           "--cache-control", "none", "--clock-control", "none", "-k", "regex:fsr_fused_kernel|easu_kernel|rcas_kernel",
           "--launch-skip", "48", "--launch-count", "96", "--csv", sys.executable, str(ROOT / "bench.py"), "--traffic-probe",
           "--radius", str(args.radius), "--math", args.math]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=240).stdout
    except Exception as e:  # noqa: BLE001
        return {"note": f"ncu child failed: {type(e).__name__}"}
    start = out.find('"ID"')
    if start < 0:
        return {"note": "ncu produced no CSV (permissions?)"}
    acc = {}
    for row in csv.DictReader(io.StringIO(out[start:])):
        name = row.get("Kernel Name", "")
        key = "fused" if "fsr_fused" in name else ("easu" if "easu_kernel" in name else ("rcas" if "rcas_kernel" in name else None))
        if key is None:
            continue
        try:
            v = float(row["Metric Value"].replace(",", ""))
        except Exception:
            continue
        unit = row.get("Metric Unit", "")
        mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1.0)
        acc.setdefault(key, {}).setdefault(row["Metric Name"], []).append(v * mult)
    res = {"note": "ncu child over steady-state launches (--cache-control none): per-launch mean of dram__bytes_read.sum + "
                   "dram__bytes_write.sum and of smsp__inst_executed.sum x 32 / output pixels"}
    for key, m in acc.items():
        rd, wr, inst = m.get("dram__bytes_read.sum", []), m.get("dram__bytes_write.sum", []), m.get("smsp__inst_executed.sum", [])
        if rd and wr:
            res[key] = {"traffic": statistics.mean(rd) + statistics.mean(wr), "dram_read": statistics.mean(rd),
                        "dram_write": statistics.mean(wr), "launches": len(rd),
                        "instr_per_px": (statistics.mean(inst) * 32 / (OUT_W * OUT_H)) if inst else None}
    return res


if __name__ == "__main__":
    main()
