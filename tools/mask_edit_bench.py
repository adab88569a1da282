"""3-D mask editor timing on a 512^3 mask (phantom.ct((512,)*3, seed=2) thresholded at 226..3071):
the polygon cut (three 64-vertex polygons on a 1920x1080 screen, depth_val 0.5 and 1.0, both
modes) and 100 brush strokes of radius 15 (BRUSH_SIZE 30 / 2). Prints one JSON line.

Device times come from CUDA events around the kernels only; every repetition starts from a
fresh device copy of the mask, made outside the timed window. The 128 MiB mask is larger than
the B200's 126 MB L2, so the cut reads it from HBM. Shim times are host wall clock around the
numpy entry points (transfers included). The CPU numbers are the C restatement on one thread;
the reference crate runs the same loops with rayon on every core."""
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from invesalius3_b200 import device as dev, mask_edit as me, phantom  # noqa: E402
from oracle import mask_edit as oracle_me  # noqa: E402
from test_gpu_mask_edit import _camera, _polygons  # noqa: E402

SCREEN = (1920, 1080)
SPACING = (0.48, 0.48, 0.9)
RADIUS = 15.0


def _events_ms(fn, reps, reset):
    times = []
    for _ in range(reps):
        reset()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.min(times))


def _card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, power = (s.strip() for s in r.stdout.strip().split(","))
    except Exception as e:                                  # the card name still comes from torch
        name, power = torch.cuda.get_device_name(0), f"unavailable ({type(e).__name__})"
    return name, power


def main(reps=5):
    dev.require_cuda()
    t0 = time.perf_counter()
    ct = phantom.ct((512,) * 3, seed=2)
    mask = ((ct >= 226) & (ct <= 3071)).astype(np.uint8) * np.uint8(255)
    del ct
    padded = np.zeros((513,) * 3, np.uint8)
    padded[1:, 1:, 1:] = mask
    setup_s = time.perf_counter() - t0
    n = mask.size
    master = torch.from_numpy(mask).cuda()
    work = torch.empty_like(master)
    polys = _polygons(SCREEN, 4, k=3, n=64)
    res = {"workload": "512^3 mask (phantom seed 2, 226..3071), 1920x1080 screen, 3 x 64-vertex polygons",
           "mask_bytes": n, "l2_note": "128 MiB mask > 126 MB L2: every cut reads the mask from HBM",
           "voxels_over_127": int((mask > 127).sum()), "setup_s": round(setup_s, 1), "cut": [], "brush": {}}

    def reset():
        work.copy_(master)

    for depth_val in (0.5, 1.0):
        for mode in (0, 1):
            M, MV, near, far = _camera(mask.shape, SPACING, SCREEN, "outside")
            depth = near + (far - near) * depth_val
            filt = me._raster(polys, SCREEN[0], SCREEN[1], True, mode == 0, work.device)

            def fused():
                me.cut_from_polygons_device(work, SPACING, depth, polys, M, MV, mode, SCREEN)

            def cut_only():
                me.mask_cut_device(work, SPACING, depth, filt, M, MV, mode)

            def raster_only():
                me._raster(polys, SCREEN[0], SCREEN[1], True, mode == 0, work.device)

            for f in (fused, cut_only, raster_only):             # warm-up
                reset(); f()
            torch.cuda.synchronize()
            reset(); cut_only(); torch.cuda.synchronize()
            zeroed = int((work == 0).sum().item()) - int((master == 0).sum().item())
            fused_ms = _events_ms(fused, reps, reset)
            cut_ms = _events_ms(cut_only, reps, reset)
            raster_ms = _events_ms(raster_only, reps, reset)
            # the staged numpy shims: polygon2mask_rs x 3 + logical_or + mask_cut, and the fused shim
            host_filter = np.logical_or.reduce([me.polygon2mask_rs(SCREEN, p) for p in polys]).T
            if mode == 0:
                np.logical_not(host_filter, out=host_filter)
            shim = []
            for _ in range(3):
                out = padded.copy()
                t = time.perf_counter()
                me.mask_cut(mask, *SPACING, depth, host_filter, M, MV, out[1:, 1:, 1:], mode)
                shim.append(time.perf_counter() - t)
            fshim = []
            for _ in range(3):
                out = padded.copy()
                t = time.perf_counter()
                me.cut_from_polygons(out[1:, 1:, 1:], SPACING, depth, polys, M, MV, mode, SCREEN)
                fshim.append(time.perf_counter() - t)
            res["cut"].append({
                "depth_val": depth_val, "edit_mode": mode, "voxels_zeroed": zeroed,
                "device_fused_ms_median_min": fused_ms, "device_cut_kernel_ms_median_min": cut_ms,
                "device_raster_ms_median_min": raster_ms,
                "algorithmic_bytes_cut": n + zeroed, "hbm_gbps_cut_median": round((n + zeroed) / cut_ms[0] / 1e6, 1),
                "shim_mask_cut_wall_ms_median": round(1e3 * float(np.median(shim)), 2),
                "shim_cut_from_polygons_wall_ms_median": round(1e3 * float(np.median(fshim)), 2),
                "pcie_bytes_per_mask_cut_call": 2 * n + host_filter.size,
            })
    # one cut of the C restatement (1 thread)
    M, MV, near, far = _camera(mask.shape, SPACING, SCREEN, "outside")
    out = padded.copy()
    t = time.perf_counter()
    oracle_me.mask_cut(mask, *SPACING, near + (far - near) * 1.0, host_filter, M, MV, out[1:, 1:, 1:], 1)
    res["cpu_cut_s"] = round(time.perf_counter() - t, 2)
    res["cpu_label"] = "C restatement, 1 thread; the reference uses rayon"

    # brush: 100 strokes along a path through the volume, alternating reveal (from orig) and erase
    ext = np.array([512 * SPACING[0], 512 * SPACING[1], 512 * SPACING[2]])
    strokes = []
    for i in range(100):
        t_ = i / 99.0
        c = tuple(float(v) for v in ext * np.array([0.15 + 0.7 * t_, 0.5 + 0.3 * np.sin(5 * t_), 0.5 + 0.3 * np.cos(3 * t_)]))
        strokes.append((c, 0 if (i // 10) % 2 else 1))
    orig_dev = master.clone()

    def strokes_dev():
        for c, mode in strokes:
            me.brush_device(work, orig_dev if mode == 0 else None, SPACING, c, RADIUS, mode)

    reset(); strokes_dev(); torch.cuda.synchronize()
    ms = _events_ms(strokes_dev, reps, reset)
    boxes = [me.brush_box(mask.shape, SPACING, c, RADIUS) for c, _ in strokes]
    box_bytes = [int(np.prod(b[3:])) for b in boxes]
    pcie = [2 * b + (b if mode == 0 else 0) for b, (_, mode) in zip(box_bytes, strokes)]
    out = padded.copy()
    orig = padded.copy()
    me.brush_mask_rs(out[1:, 1:, 1:], orig[1:, 1:, 1:], SPACING, strokes[0][0], RADIUS, 0)      # warm-up
    t = time.perf_counter()
    for c, mode in strokes:
        me.brush_mask_rs(out[1:, 1:, 1:], orig[1:, 1:, 1:] if mode == 0 else None, SPACING, c, RADIUS, mode)
    shim_s = time.perf_counter() - t
    cpu = padded.copy()
    t = time.perf_counter()
    for c, mode in strokes[:3]:
        oracle_me.brush_mask_rs(cpu[1:, 1:, 1:], orig[1:, 1:, 1:] if mode == 0 else None, SPACING, c, RADIUS, mode)
    cpu_stroke_s = (time.perf_counter() - t) / 3
    res["brush"] = {"strokes": 100, "radius_mm": RADIUS, "box_voxels_median": int(np.median(box_bytes)),
                    "device_100_strokes_ms_median_min": ms,
                    "device_per_stroke_us_median": round(1e3 * ms[0] / 100, 1),
                    "shim_brush_mask_rs_wall_ms_per_call": round(1e3 * shim_s / 100, 3),
                    "pcie_bytes_per_call_median": int(np.median(pcie)),
                    "cpu_per_stroke_s": round(cpu_stroke_s, 3),
                    "cpu_label": "C restatement, 1 thread, visits every voxel as the reference does; the reference uses rayon"}
    name, power = _card()
    res.update(card=name, power_limit=power, torch=torch.__version__)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
