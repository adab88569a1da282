#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json configs[1]):
threshold -> seeded flood-fill region grow -> marching cubes on a 512^3 int16 CT phantom.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).

`value`     Mvoxel/s of the whole job with inputs resident in HBM (CUDA-event timed, max over
            ranks). At N > 1 the job is ONE (N*512) x 512 x 512 volume, Z-sharded (weak scaling),
            region-grown from ONE seed in its middle slice: the wave has to cross every shard —
            the honest multi-GPU version of "the user clicks once". The easier workload (one
            seed per shard, waves meet at the boundaries) is timed too and reported in
            `config.seeding`.
`e2e`       N = 1: the same three ops through the reference-shaped numpy API (slice_ops /
            invesalius_rs / surface_process) on pinned HOST buffers, copies inside the timed
            region. N > 1: the sharded pipeline fed from / drained to pinned host buffers (image
            uploaded once per step; stated in `e2e.api`).
`verified`  the GPU results are checked in this run: N = 1 against the CPU restatement of the
            reference on the same 512^3 volume (reached-voxel count, mask equality, V, T, the
            triangle array and the vertices); N > 1 against a single-GPU run of the whole
            gathered volume on rank 0 (count, V, T, order-independent checksums of both arrays).
`roofline`  the dominant stage against the measured HBM peak.
`cpu_baseline` / `--impl reference`  the CPU restatement of the reference path timed on this
            box's host cores on the SAME 512^3 volume (full, not a slab).
`extra`     (N = 1) driver-visible secondary results: 1024^3 threshold / MaxIP x3 / MIDA with
            their roofline fractions, 512^3 watershed times + agreement with the CPU checker.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "Mvoxels/s threshold+floodfill+MC on 512^3 int16"
UNIT = "Mvoxel/s"
THR = (226, 3071)          # presets.py "Bone"
SPACING = (1.0, 1.0, 1.0)
FILL = 254


def workload_desc(n, world):
    vol = f"{n}^3" if world == 1 else f"{n * world}x{n}x{n}"
    return (f"{vol} synthetic int16 CT phantom (seed 2){'' if world == 1 else f', Z-sharded {n}^3 per GPU'}: "
            f"threshold [226,3071] -> 6-connected flood fill from ONE seed in the middle slice -> marching cubes "
            f"iso 127 on the grown mask")


def measured_peak():
    try:
        return float(json.load(open(ROOT / "MEASURED_PEAKS.json"))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def global_seed(n, world):
    """(x, y, z) of the first in-range voxel (raveled order) of the volume's middle slice."""
    from invesalius3_b200 import phantom
    DZ = n * world
    zmid = DZ // 2
    mid = phantom.ct((DZ, n, n), seed=2, zrange=(zmid, zmid + 1))
    sx, sy, _ = phantom.first_seed_in_range(mid, 0, *THR)
    return (sx, sy, zmid)


def shard_seed(own, z0):
    """One seed inside this shard: the first in-range voxel of the plane closest to the shard's
    middle that has one (the shards at the ends of a long volume hold mostly air). None if the
    shard has no in-range voxel at all."""
    nz = own.shape[0]
    order = sorted(range(nz), key=lambda z: abs(z - nz // 2))
    for z in order:
        idx = np.flatnonzero((own[z] >= THR[0]) & (own[z] <= THR[1]))
        if idx.size:
            yy, xx = divmod(int(idx[0]), own.shape[2])
            return (xx, yy, z0 + z)
    return None


# ------------------------------------------------------------------ CPU reference path
def cpu_step(vol, seed, threads, want_arrays=False):
    """The reference's CPU path restated (oracle/): NumPy threshold statements verbatim
    (single thread, as in the reference), serial stack flood fill, marching cubes over
    20(+1)-slice Z pieces on a thread pool (surface.py:1360-1381 uses a process pool).
    Returns (reached voxels, triangles[, mask, out])."""
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    from scipy.ndimage import generate_binary_structure
    dz, dy, dx = vol.shape
    mm = np.zeros((dz + 1, dy + 1, dx + 1), np.uint8)
    oracle.set_mask_threshold_numpy(vol, mm, THR)
    out = np.zeros(vol.shape, np.uint8)
    oracle.floodfill_threshold(vol, [seed], THR[0], THR[1], FILL, generate_binary_structure(3, 1), out)
    n_pieces = int(round(dz / 20 + 0.5))
    rois = [slice(i * 20, min(dz, (i + 1) * 20 + 1)) for i in range(n_pieces) if i * 20 < dz]

    def piece(roi):
        a = np.ascontiguousarray(out[roi])
        if a.shape[0] < 2:
            return 0
        v, f = oracle.marching_cubes(a, 127, SPACING, (0, 0, roi.start), True)
        return len(f)

    with ThreadPoolExecutor(max_workers=max(1, min(threads, len(rois)))) as ex:
        ntri = sum(ex.map(piece, rois))
    count = int(np.count_nonzero(out == FILL))
    if want_arrays:
        return count, ntri, mm, out
    return count, ntri


DUMP_KEEP = 1 << 20


def dump_outputs(dirname, outputs, suffix=""):
    """--dump-outputs: each output of the last timed step as DIR/<name><suffix>.npy, masks and vertices
    as float32, triangle indices as float64 (exact). An output with more than DUMP_KEEP voxels (masks)
    or rows (mesh arrays) keeps DUMP_KEEP of them at fixed, seeded positions, in index order; each mask
    also gets its exact per-plane sums (<name>_plane_sums), which catch what the sample misses. About
    44 MiB in all."""
    import torch
    d = Path(dirname)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in outputs.items():
        flat = t.reshape(-1) if t.dim() == 3 else t
        if flat.shape[0] > DUMP_KEEP:
            idx = np.sort(np.random.default_rng(0).choice(flat.shape[0], DUMP_KEEP, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        wide = t.dtype in (torch.int32, torch.int64)
        np.save(d / f"{name}{suffix}.npy", flat.to(torch.float64 if wide else torch.float32).cpu().numpy())
        if t.dim() == 3:
            sums = t.sum(dim=(1, 2), dtype=torch.int64).to(torch.float64)
            np.save(d / f"{name}_plane_sums{suffix}.npy", sums.cpu().numpy())


def crossing_edges(mask_u8, iso=127):
    """Number of iso-crossing grid edges = number of marching-cubes vertices (independent of any
    case table)."""
    ins = mask_u8 >= iso
    return int(np.count_nonzero(ins[:, :, 1:] != ins[:, :, :-1]) + np.count_nonzero(ins[:, 1:] != ins[:, :-1]) +
               np.count_nonzero(ins[1:] != ins[:-1]))


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock and throttle reasons of one GPU, sampled DURING the warm-up and the timed region.

    In-process NVML (the library behind nvidia-smi) on a background thread: an `nvidia-smi -lms`
    child stalls this process's host-synchronous CUDA calls for milliseconds at every poll (measured:
    +0.3 .. +0.6 ms per step on a 1.3 ms step), which a 13 ms timed region cannot absorb. The
    subprocess remains as the fallback when pynvml is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, pci_bus_id=None, period=0.01, force_smi=False):
        self.samples = []        # (sm MHz, reasons bitmask)
        self.max_mhz = None
        self.skip = 0
        self.p = self.f = self.thread = None
        try:
            if force_smi:
                raise RuntimeError("nvidia-smi requested")
            import threading
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByPciBusId(pci_bus_id.encode() if isinstance(pci_bus_id, str) else pci_bus_id) \
                if pci_bus_id else nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                         "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                         "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                         "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            self.stop_flag = False

            def loop():
                while not self.stop_flag:
                    try:
                        self.samples.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                             int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))))
                    except Exception:
                        pass
                    time.sleep(period)

            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            self.source = "nvml"
            return
        except Exception:
            self.thread = None
        self.source = "nvidia-smi"
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def rows(self):
        if self.thread is not None:
            return len(self.samples)
        try:
            return sum(1 for r in open(self.f.name).read().splitlines() if r.count(",") >= 8)
        except Exception:
            return 0

    def wait_ready(self, timeout=15.0):
        """Wait for the first sample BEFORE the load starts (nvidia-smi needs up to a second to attach
        on a fresh box); samples taken up to here are idle ones and are dropped."""
        t0 = time.perf_counter()
        alive = lambda: self.thread is not None or (self.p is not None and self.p.poll() is None)
        while alive() and self.rows() == 0 and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)
        self.skip = self.rows()

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            rows = self.samples[self.skip:] or self.samples
            if not rows:
                return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples"], "source": "nvml"}
            sm = sorted(r[0] for r in rows)
            reasons = sorted(k for k, bit in self.bits.items() if any(r[1] & bit for r in rows))
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(rows),
                    "source": "nvml"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        if len(rows) > self.skip:
            rows = rows[self.skip:]      # under load only (warm-up + timed region)
        os.unlink(self.f.name)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if "Active" in v and "Not" not in v:
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                "samples": len(rows), "source": "nvidia-smi"}


def bind_to_gpu_numa(local_rank):
    """Best effort: run this process on the CPUs of the NUMA node the GPU hangs off, so that
    first-touch puts the pinned host buffers next to the GPU's PCIe root (cross-socket DMA and
    memset are several times slower). Returns a short description for the JSON line."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local_rank), "pci_domain_id", 0)
        dev_id = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev_id:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return "numa: single node"
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, ids)
        return f"numa: bound to node {node} ({len(ids)} cpus)"
    except Exception as e:   # noqa: BLE001
        return f"numa: not bound ({type(e).__name__})"


def checksums(verts, tris):
    """Order-independent exact checksums of a mesh on the device: int64 sums of the triangle
    indices and of the vertex coordinates' bit patterns."""
    import torch
    tsum = int(tris.to(torch.int64).sum().item()) if tris.numel() else 0
    vsum = int(verts.contiguous().view(torch.int32).to(torch.int64).sum().item()) if verts.numel() else 0
    return tsum, vsum


# ------------------------------------------------------------------ secondary results (N = 1)
def extra_results(peak):
    """1024^3 threshold / MaxIP on three axes / MIDA, and the 512^3 watershed (BASELINE configs
    [2], [3]) — device-timed like the headline (CUDA events, median of 5, inputs >> L2)."""
    import torch
    from invesalius3_b200 import device as dev, projection
    res = {}

    def timeit(fn, iters=5, warmup=2):
        for _ in range(warmup):
            fn()
        ts = []
        for _ in range(iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2]

    n = 1024
    try:
        g = torch.Generator(device="cuda").manual_seed(0)
        vol = torch.randint(-1024, 3072, (n, n, n), dtype=torch.int16, device="cuda", generator=g)
        N = vol.numel()
        out = torch.empty((n, n, n), dtype=torch.uint8, device="cuda")
        ms = timeit(lambda: dev.threshold(vol, 226, 3071, out=out))
        res["threshold_1024"] = {"ms": round(ms, 4), "GBs": round(3 * N / ms / 1e6, 1), "frac": round(3 * N / ms / 1e6 / peak, 4)}
        del out
        tot = 0.0
        for axis in (0, 1, 2):
            o = dev.mip(vol, axis, "max")
            ms = timeit(lambda: dev.mip(vol, axis, "max", out=o))
            tot += ms
            res[f"maxip_1024_axis{axis}"] = {"ms": round(ms, 4), "GBs": round(2 * N / ms / 1e6, 1),
                                             "frac": round(2 * N / ms / 1e6 / peak, 4)}
        t = res["threshold_1024"]["ms"] + tot
        res["threshold_plus_3mip_1024"] = {"ms": round(t, 4), "alg_bytes_per_voxel": 9,
                                           "frac": round(9 * N / t / 1e6 / peak, 4)}
        for axis in (0, 1, 2):
            o = projection.mida(vol, axis, 32000, 2)    # opacity 0 everywhere: no ray terminates early
            ms = timeit(lambda: projection.mida(vol, axis, 32000, 2, out=o), iters=3)
            res[f"mida_fullrays_1024_axis{axis}"] = {"ms": round(ms, 4), "GBs": round(4 * N / ms / 1e6, 1),
                                                      "frac": round(4 * N / ms / 1e6 / peak, 4)}
        # contour-MIP (n = 2): contour volume (2 B read + 2 B written per voxel) + projection of it (2 B/voxel)
        for tmip, name in ((0, "max"), (2, "mida")):
            for axis in (0, 2):
                o = projection.fast_countour_mip(vol, 2.0, axis, 300, 300, tmip)
                ms = timeit(lambda: projection.fast_countour_mip(vol, 2.0, axis, 300, 300, tmip, out=o), iters=3)
                res[f"contour_{name}_1024_axis{axis}"] = {"ms": round(ms, 4), "GBs_2B_per_voxel": round(2 * N / ms / 1e6, 1),
                                                          "frac_2B_per_voxel": round(2 * N / ms / 1e6 / peak, 4),
                                                          "frac_moved_bytes": round((6 if tmip == 0 else 8) * N / ms / 1e6 / peak, 4)}
        del vol
        torch.cuda.empty_cache()
    except Exception as e:   # noqa: BLE001
        res["error_1024"] = f"{type(e).__name__}: {e}"
    try:
        res["label_512"] = label_results(timeit)
    except Exception as e:   # noqa: BLE001
        res["label_512"] = {"error": f"{type(e).__name__}: {e}"}
    try:
        res["view_transform_512"] = view_transform_results(timeit)
    except Exception as e:   # noqa: BLE001
        res["view_transform_512"] = {"error": f"{type(e).__name__}: {e}"}
    try:
        res["watershed_512"] = watershed_results()
    except Exception as e:   # noqa: BLE001
        res["watershed_512"] = {"error": f"{type(e).__name__}: {e}"}
    return res


def label_results(timeit):
    """SURVEY 8f-3: scipy.ndimage.label of the 512^3 bone-threshold mask and of its complement (what
    Mask.fill_holes_auto labels), 6-connected, device-resident; SciPy timed on a 64-plane slab."""
    import torch
    from scipy import ndimage
    from invesalius3_b200 import labeling, phantom
    vol = phantom.ct((512, 512, 512), seed=2)
    img = (vol >= THR[0]) & (vol <= THR[1])
    st = ndimage.generate_binary_structure(3, 1)
    res = {}
    for name, a in (("bone_mask", img), ("complement", ~img)):
        t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).cuda()
        ms = timeit(lambda: labeling.label_device(t, st), iters=3, warmup=1)
        lab, n = labeling.label_device(t, st)
        slab = np.ascontiguousarray(a[224:288])
        t0 = time.perf_counter()
        w, nw = ndimage.label(slab, st, output=np.uint32)
        cpu = time.perf_counter() - t0
        g, ng = labeling.label(slab, st)
        res[name] = {"ms": round(ms, 3), "Mvoxel/s": round(a.size / ms / 1e3, 1), "labels": n,
                     "scipy_slab64_Mvoxel/s": round(slab.size / cpu / 1e6, 1), "slab_equals_scipy": bool(ng == nw and np.array_equal(g, w))}
    return res


def view_transform_results(timeit):
    """SURVEY 8f-1: apply_view_matrix_transform of a whole 512^3 int16 volume (apply_reorientation,
    slice_.py:1980) through a rotation about its centre, device-resident, per interpolator; algorithmic
    bytes 2 read + 2 written per voxel (the gathers hit L1 / L2)."""
    import ctypes as C
    import torch
    from invesalius3_b200 import _lib, device as dev, phantom
    n = 512
    vol = torch.from_numpy(phantom.ct((n, n, n), seed=2)).cuda()
    out = torch.empty_like(vol)
    ws = dev._workspace(256, vol.device)
    a = 0.3
    c = n / 2.0
    R = np.array([[1, 0, 0, 0], [0, np.cos(a), -np.sin(a), 0], [0, np.sin(a), np.cos(a), 0], [0, 0, 0, 1.0]])
    T0 = np.eye(4); T0[:3, 3] = -c
    T1 = np.eye(4); T1[:3, 3] = c
    M = np.ascontiguousarray(T1 @ R @ T0)
    sp = np.ones(3)
    res = {}
    for interp, name in ((0, "nearest"), (1, "trilinear"), (2, "tricubic"), (3, "lanczos4")):
        fn = lambda: _lib.call("b2v_apply_view_matrix_transform", dev._p(vol), _lib.I16, n, n, n, C.c_void_p(sp.ctypes.data),
                               C.c_void_p(M.ctypes.data), 0, 0, interp, -1024.0, dev._p(out), n, n, n, dev._p(ws), dev._stream())
        ms = timeit(fn, iters=3, warmup=1)
        res[name] = {"ms": round(ms, 3), "Mvoxel/s": round(n ** 3 / ms / 1e3, 1), "GBs_4B_per_voxel": round(4 * n ** 3 / ms / 1e6, 1)}
    return res


def ws_markers(vol, seed):
    rng = np.random.default_rng(seed)
    m = np.zeros(vol.shape, np.uint8)
    zz, yy, xx = np.ogrid[:vol.shape[0], :vol.shape[1], :vol.shape[2]]
    ins, outs = np.argwhere(vol > 600), np.argwhere(vol < -900)
    for lab, pool in ((1, ins), (2, outs)):
        for _ in range(4):
            c = pool[rng.integers(len(pool))]
            m[(zz - c[0]) ** 2 + (yy - c[1]) ** 2 + (xx - c[2]) ** 2 <= 16] = lab
    return m


def watershed_results():
    """BASELINE configs[3]: 512^3, 8 marker balls, ww 406 / wl -18, mg_size 3, 6-connected, both
    algorithms; agreement with the CPU checker (SciPy itself for IFT) on a 96^3 phantom, overall
    and on the voxels whose label does not depend on the queue order."""
    import torch
    from scipy.ndimage import generate_binary_structure
    from invesalius3_b200 import phantom, watershed_process as wp
    from oracle import watershed as W
    st = generate_binary_structure(3, 1)
    n = 512
    vol = phantom.ct((n, n, n), seed=4)
    mk = ws_markers(vol, 4)
    t_vol, t_mk = torch.from_numpy(vol).cuda(), torch.from_numpy(mk).cuda()
    res = {}
    for alg in ("Watershed", "Watershed IFT"):
        wp.watershed_device(t_vol, t_mk, st, alg, 3, True, -18, 406)
        ts = []
        for _ in range(2):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); wp.watershed_device(t_vol, t_mk, st, alg, 3, True, -18, 406); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        res[alg] = {"ms": round(min(ts), 2), "Mvoxel/s": round(vol.size / min(ts) / 1e3, 1)}
    del t_vol, t_mk
    m = 96
    v2 = phantom.ct((m, m, m), seed=4)
    mk2 = ws_markers(v2, 4)
    for alg in ("Watershed", "Watershed IFT"):
        want = W.do_watershed_array(v2, mk2, st, alg, 3, True, -18, 406)
        r = wp.watershed_device(torch.from_numpy(v2).cuda(), torch.from_numpy(mk2).cuda(), st, alg, 3, True, -18, 406,
                                return_ambiguous=True)
        got, amb = r[0].cpu().numpy(), r[1].cpu().numpy().astype(bool)
        res[alg].update(agreement_96=round(float((got == want).mean()), 5),
                        order_independent_fraction_96=round(float((~amb).mean()), 5),
                        exact_on_order_independent_96=bool(np.array_equal(got[~amb], want[~amb])))
    return res


# ------------------------------------------------------------------ GPU arm
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from scipy.ndimage import generate_binary_structure
    from invesalius3_b200 import _lib, device as dev, invesalius_rs, phantom, slice_ops, surface_process
    from invesalius3_b200.mesh import marching_cubes
    from invesalius3_b200 import dist as zd

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev.require_cuda()
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa(local)
    torch.set_num_threads(16)   # host memset of the out mask: 128 OpenMP threads make it erratic (0.3 .. 25 ms)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()
    n = args.size
    shard = zd.ZShard(n * world, rank, world)
    ext_np = phantom.ct((n * world, n, n), seed=2, zrange=(shard.ze0, shard.ze1))   # own planes + halo planes
    vol = shard.interior(torch.from_numpy(ext_np)).numpy()          # this rank's n^3 shard
    gseed = global_seed(n, world)
    if world > 1:
        got = [None] * world
        dist.all_gather_object(got, shard_seed(vol, shard.z0))
        pseeds = [s for s in got if s is not None]
    else:
        pseeds = [gseed]
    seedings = {"global": [gseed], "per_shard": pseeds}
    strct = generate_binary_structure(3, 1)
    N = vol.size
    nz_ext = ext_np.shape[0]
    link = zd.peer_link(shard, n, n) if world > 1 else None   # NVLink peer mappings for the fused exchange kernels

    # pinned host buffers for the e2e leg (numpy views of torch pinned tensors)
    h_ext = torch.from_numpy(ext_np).pin_memory()
    h_vol = shard.interior(h_ext)
    h_mask = torch.zeros((n + 1, n + 1, n + 1), dtype=torch.uint8).pin_memory()
    h_out = torch.zeros((nz_ext, n, n), dtype=torch.uint8).pin_memory()
    np_vol, np_mask, np_out = h_vol.numpy(), h_mask.numpy(), h_out.numpy()

    d_ext = h_ext.cuda(non_blocking=True)
    d_vol = shard.interior(d_ext)
    d_mask = torch.empty((n, n, n), dtype=torch.uint8, device="cuda")
    d_out = torch.empty((nz_ext, n, n), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    info = {}

    def do_flood(data_ext, out_ext, seeds):
        if world == 1:
            info["rounds"] = dev.floodfill_threshold(data_ext, seeds, THR[0], THR[1], FILL, strct, out_ext)
        else:
            info["exchanges"] = zd.floodfill_threshold(data_ext, seeds, THR[0], THR[1], FILL, strct, out_ext, shard,
                                                       link=link)
            info["rounds"] = link.last_rounds if link is not None else info["exchanges"]

    def do_surface(out_ext):
        if world == 1:
            v, f = marching_cubes(out_ext, 127, SPACING, (0, 0, 0), True, _events=info.get("mc_events"))
            info["V"], info["T"] = int(v.shape[0]), int(f.shape[0])
        else:
            v, f, _, info["V"], info["T"] = zd.marching_cubes(out_ext[int(shard.has_lo):], 127, SPACING, (0, 0, 0),
                                                              True, shard, link=link)
        return v, f

    def step_device(seeds, ev=None):
        if ev: ev[0].record()
        dev.threshold(d_vol, THR[0], THR[1], out=d_mask)
        if ev: ev[1].record()
        d_out.zero_()
        do_flood(d_ext, d_out, seeds)
        if ev: ev[2].record()
        v, f = do_surface(d_out)
        if ev: ev[3].record()
        return v, f

    e2e_min = {}
    e2e_calls = {"set_mask_threshold": 0.0, "zero_out_mask": 0.0, "floodfill_threshold": 0.0, "contour": 0.0}

    def step_e2e_session():
        """The same action through the device-resident session (image uploaded once, results into
        the same pinned host arrays)."""
        from invesalius3_b200.session import VolumeSession
        with VolumeSession(np_vol) as s:
            s.set_mask_threshold(np_mask, THR)
            s.floodfill_threshold([gseed], THR[0], THR[1], FILL, strct, np_out)
            return s.contour([127], SPACING, 0, True)

    def step_e2e():
        if world == 1:
            t0 = time.perf_counter()
            slice_ops.set_mask_threshold(np_vol, np_mask, THR)
            t1 = time.perf_counter()
            h_out.zero_()      # the reference allocates out_mask = np.zeros_like(mask) here (styles.py:3183)
            t2 = time.perf_counter()
            invesalius_rs.floodfill_threshold(np_vol, [gseed], THR[0], THR[1], FILL, strct, np_out)
            t3 = time.perf_counter()
            v, f = surface_process.contour(np_out, [127], SPACING, 0, True)
            t4 = time.perf_counter()
            for k, dt in zip(e2e_calls, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
                e2e_calls[k] += dt
                e2e_min[k] = min(e2e_min.get(k, 1e9), dt)
            return v, f
        # N > 1: the sharded pipeline fed from / drained to pinned host memory (image uploaded once)
        t_ext = dev.to_device(h_ext.numpy())
        m = dev.threshold(shard.interior(t_ext), THR[0], THR[1])
        dev.to_host(m, np_mask[1:, 1:, 1:])
        np_mask[1:, 0, 0] = 1
        o_ext = torch.zeros((nz_ext, n, n), dtype=torch.uint8, device="cuda")
        do_flood(t_ext, o_ext, seedings["global"])
        v, f = do_surface(o_ext)
        dev.to_host(shard.interior(o_ext), shard.interior(h_out).numpy())
        return dev.to_numpy(v), dev.to_numpy(f)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(*xs):
        t = torch.tensor(list(xs), dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [int(v) for v in t.tolist()]

    # ---- device-resident leg, both seedings (the headline is the single global seed)
    timed = {}
    clocks = None
    launches = 0
    for name in ("per_shard", "global") if world > 1 else ("global",):
        seeds = seedings[name]
        head = name == "global"
        sampler = None
        if rank == 0 and head:
            try:
                bus = torch.cuda.get_device_properties(local)
                bus_id = f"{getattr(bus, 'pci_domain_id', 0):08x}:{bus.pci_bus_id:02x}:{bus.pci_device_id:02x}.0"
            except Exception:
                bus_id = None
            sampler = ClockSampler(local, bus_id, force_smi=bool(os.environ.get("B2V_BENCH_SMI")))
        if sampler:
            sampler.wait_ready()
        v = f = None
        for _ in range(max(args.warmup, 3)):
            v, f = step_device(seeds)     # results stay bound as in the timed loop: the caching allocator
        barrier()                         # reaches its steady state (two sets of output blocks) here
        lib.b2v_launch_count_reset()
        stage_ms = np.zeros(3)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        dbg = []
        if os.environ.get("B2V_BENCH_DEBUG"):
            info["mc_events"] = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        for _ in range(args.steps):
            v, f = step_device(seeds, ev)
            torch.cuda.synchronize()
            stage_ms += [ev[i].elapsed_time(ev[i + 1]) for i in range(3)]
            if info.get("mc_events"):
                me = info["mc_events"]
                dbg.append([round(x, 3) for x in (ev[2].elapsed_time(me[0]), me[0].elapsed_time(me[1]),
                                                  me[1].elapsed_time(me[2]), me[2].elapsed_time(ev[3]))])
        if dbg:
            sys.stderr.write("mc [ws alloc, count, out alloc, emit] per step: " + json.dumps(dbg) + "\n")
        e1.record()
        barrier()
        if head:
            launches = int(lib.b2v_launch_count())
        total_ms = max_over_ranks(e0.elapsed_time(e1))
        if sampler:
            clocks = sampler.stop()
        count = int((shard.interior(d_out) == FILL).sum().item())
        tsum, vsum = checksums(v, f)
        gc, gt, gv = sum_over_ranks(count, tsum, vsum)
        timed[name] = {"ms_per_step": total_ms / args.steps, "stage_ms": stage_ms / args.steps,
                       "rounds": info["rounds"], "exchanges": info.get("exchanges", 0), "V": info["V"], "T": info["T"], "reached": gc, "tsum": gt, "vsum": gv,
                       "nseeds": len(seeds)}
        if head and args.dump_outputs:
            dump_outputs(args.dump_outputs, {"threshold_mask": d_mask, "flood_mask": shard.interior(d_out),
                                             "vertices": v, "triangles": f}, "" if world == 1 else f"_rank{rank}")
    head = timed["global"]
    ms_per_step = head["ms_per_step"]
    value = world * N / (ms_per_step * 1e-3) / 1e6
    stage_ms = head["stage_ms"]
    info.update(V=head["V"], T=head["T"], rounds=head["rounds"])

    # ---- verification (outside every timed region)
    verified = {"ok": False}
    if world == 1:
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        t0 = time.perf_counter()
        c_count, c_tri, c_mm, c_out = cpu_step(vol, gseed, cores, want_arrays=True)
        cpu_s = time.perf_counter() - t0
        import oracle
        ov, of = oracle.marching_cubes(c_out, 127, SPACING, (0, 0, 0), True)
        v, f = step_device(seedings["global"])
        g_mask, g_out = d_mask.cpu().numpy(), d_out.cpu().numpy()
        gv, gf = v.cpu().numpy(), f.cpu().numpy()
        checks = {
            "threshold_mask_equal": bool(np.array_equal(g_mask, c_mm[1:, 1:, 1:])),
            "flood_mask_equal": bool(np.array_equal(g_out, c_out)),
            "reached_voxels": [head["reached"], c_count],
            "triangles": [head["T"], c_tri, int(of.shape[0])],
            "vertices": [head["V"], int(ov.shape[0]), crossing_edges(c_out)],
            "triangle_array_equal": bool(gf.shape == of.shape and np.array_equal(gf, of)),
            "vertex_max_abs_diff": float(np.abs(gv - ov).max()) if gv.shape == ov.shape and gv.size else None,
        }
        ok = (checks["threshold_mask_equal"] and checks["flood_mask_equal"] and head["reached"] == c_count and
              head["T"] == c_tri == of.shape[0] and head["V"] == ov.shape[0] == checks["vertices"][2] and
              checks["triangle_array_equal"] and checks["vertex_max_abs_diff"] is not None and
              checks["vertex_max_abs_diff"] <= 1e-5)
        verified = {"ok": bool(ok), "against": "CPU restatement of the reference (oracle/) on the same 512^3 volume",
                    **checks}
        cpu_baseline = {"value": round(vol.size / cpu_s / 1e6, 2), "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"the full {n}^3 volume, one step ({cpu_s:.2f} s): NumPy threshold (1 thread) + serial "
                                  f"flood fill (1 thread) + marching cubes over 21-slice pieces on {cores} threads"}
        del c_mm, c_out, g_mask, g_out
    else:
        cpu_baseline = None
        # gather the whole volume on rank 0 and run the single-GPU path there
        own = d_vol.contiguous()
        if rank == 0:
            whole = torch.empty((n * world, n, n), dtype=torch.int16, device="cuda")
            whole[:n].copy_(own)
            for r in range(1, world):
                dist.recv(whole[r * n:(r + 1) * n].view(torch.uint8), src=r)
        else:
            dist.send(own.view(torch.uint8), dst=0)
        if rank == 0:
            res = {}
            for name, seeds in seedings.items():
                o = torch.zeros((n * world, n, n), dtype=torch.uint8, device="cuda")
                dev.floodfill_threshold(whole, seeds, THR[0], THR[1], FILL, strct, o)
                v1, f1 = marching_cubes(o, 127, SPACING, (0, 0, 0), True)
                ts, vs = checksums(v1, f1)
                one = {"reached": int((o == FILL).sum().item()), "V": int(v1.shape[0]), "T": int(f1.shape[0]),
                       "tsum": ts, "vsum": vs}
                shd = {k: timed[name][k] for k in one}
                res[name] = {"sharded": shd, "single_gpu": one, "equal": shd == one}
                del o, v1, f1
            del whole
            verified = {"ok": all(r["equal"] for r in res.values()),
                        "against": "single-GPU run of the whole gathered volume on rank 0 (reached count, V, T, "
                                   "int64 checksums of the triangle indices and of the vertex bit patterns)", **res}
        barrier()

    # ---- e2e leg: reference-shaped numpy API on pinned host buffers
    e2e_steps = max(1, min(args.steps, 5))
    v, f = step_e2e()
    v, f = step_e2e()   # results stay bound across calls, as in the timed loop: the pinned result
    v, f = step_e2e()   # pool reaches its steady state (two sets of blocks in flight)
    for k in e2e_calls:
        e2e_calls[k] = 0.0
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        v, f = step_e2e()
    barrier()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    sess = None
    if world == 1:
        vs, fs = step_e2e_session()
        vs, fs = step_e2e_session()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            vs, fs = step_e2e_session()
        torch.cuda.synchronize()
        sess_s = (time.perf_counter() - t0) / e2e_steps
        same = bool(vs.shape == v.shape and fs.shape == f.shape and np.array_equal(fs, f) and np.array_equal(vs, v))
        sess = {"value": round(N / sess_s / 1e6, 1), "unit": UNIT, "ms_per_step": round(sess_s * 1e3, 3),
                "h2d_bytes_per_step": int(2 * N), "d2h_bytes_per_step": int(2 * N + vs.nbytes + fs.nbytes),
                "same_results_as_numpy_api": same,
                "api": "session.VolumeSession: image uploaded once per step, mask / grown mask / mesh read back"}
    if world == 1:
        h2d = 2 * N * 2 + 2 * N            # image twice (threshold, flood fill), out in, out again for MC
    else:
        h2d = ext_np.nbytes                # the extended slab once; the pipeline stays on the device
    d2h = 2 * N + v.nbytes + f.nbytes  # mask, out, mesh
    e2e_value = world * N / e2e_s / 1e6

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_kind = measured_peak()
    # dominant stage and its roofline (algorithmic bytes: SURVEY.md 8d / DESIGN.md)
    alg = {"threshold": 3.0 * N, "floodfill": 4.0 * N,
           "marching_cubes": 1.0 * N + (12.0 * info["V"] + 12.0 * info["T"]) / world}
    names = list(alg)
    dom = int(np.argmax(stage_ms))
    achieved = alg[names[dom]] / (stage_ms[dom] * 1e-3) / 1e9
    traffic, traffic_src = None, None
    for cand in ("r02_traffic.json", "r01_traffic.json"):
        try:   # DRAM bytes per launch of that stage from the committed ncu capture (profiles/)
            traffic = json.load(open(ROOT / "profiles" / cand))["stages"][names[dom]]["traffic"]
            traffic_src = f"profiles/{cand}"
            break
        except Exception:
            pass
    seeding = {}
    for name, t in timed.items():
        seeding[name] = {"ms_per_step": round(t["ms_per_step"], 4),
                         "Mvoxel/s": round(world * N / (t["ms_per_step"] * 1e-3) / 1e6, 1), "seeds": t["nseeds"],
                         "flood_rounds": t["rounds"], "flood_exchanges": t["exchanges"],
                         "stage_ms": {k: round(float(m), 4) for k, m in zip(names, t["stage_ms"])}}
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": {"workload": workload_desc(n, world),
                   "volume": f"{n * world}x{n}x{n} (Z-sharded, one halo plane per inner side)",
                   "shard": f"{n}^3 voxels per GPU", "l2": "inputs (256 MiB int16 + 128 MiB uint8) exceed the 126 MB L2",
                   "host": numa, "flood_rounds": info["rounds"], "vertices": info["V"], "triangles": info["T"],
                   "stage_ms": {k: round(float(m), 4) for k, m in zip(names, stage_ms)},
                   "seeding": seeding, "exchange": (link.describe() if link is not None else
                                                    ("none (one GPU)" if world == 1 else "NCCL send/recv + all_reduce"))},
        "verified": verified,
        "clocks": clocks, "gpu_launches": launches,
        "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": round(e2e_s * 1e3, 3),
                "ms_per_call": {k: round(v / e2e_steps * 1e3, 3) for k, v in e2e_calls.items()} if world == 1 else None,
                "ms_per_call_min": {k: round(v * 1e3, 3) for k, v in e2e_min.items()} if world == 1 else None,
                "api": ("slice_ops.set_mask_threshold + invesalius_rs.floodfill_threshold + surface_process.contour "
                        "on pinned numpy buffers (image uploaded by each call, as the numpy API implies)") if world == 1 else
                       "dist.* sharded pipeline fed from / drained to pinned host buffers (image uploaded once per step)",
                "session": sess},
        "roofline": {"bound": "hbm", "kernel": names[dom], "achieved": round(achieved, 1), "peak": peak,
                     "peak_kind": peak_kind, "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
                     "traffic_source": traffic_src,
                     "note": "stage-level: algorithmic bytes of the dominant stage / its CUDA-event time; the flood's "
                             "rounds are L2/latency-bound, see DESIGN.md",
                     "per_stage_GBs": {k: round(alg[k] / (m * 1e-3) / 1e9, 1) for k, m in zip(names, stage_ms)},
                     "per_stage_frac": {k: round(alg[k] / (m * 1e-3) / 1e9 / peak, 4) for k, m in zip(names, stage_ms)}},
        "cpu_baseline": cpu_baseline,
    }
    if world == 1 and not args.no_extra:
        del d_ext, d_mask, d_out
        torch.cuda.empty_cache()
        line["extra"] = extra_results(peak)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from invesalius3_b200 import phantom
    n = args.size
    vol = phantom.ct((n, n, n), seed=2)
    seed = global_seed(n, 1)
    cores = os.cpu_count() or 1
    if args.cpu_slices and args.cpu_slices < n:     # optional bounded slab (not the default)
        z0 = max(0, min(n - args.cpu_slices, seed[2] - args.cpu_slices // 2))
        vol, seed = np.ascontiguousarray(vol[z0:z0 + args.cpu_slices]), (seed[0], seed[1], seed[2] - z0)
    for _ in range(min(args.warmup, 1)):
        cpu_step(vol, seed, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        count, ntri = cpu_step(vol, seed, cores)
    s = (time.perf_counter() - t0) / args.steps
    v = vol.size / s / 1e6
    sample = (f"the full {vol.shape[0]}x{vol.shape[1]}x{vol.shape[2]} volume per step: NumPy threshold (1 thread) + serial "
              f"flood fill (1 thread) + marching cubes over 21-slice pieces on {cores} threads")
    emit({
        "impl": "reference", "metric": METRIC, "value": round(v, 2), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": round(s * 1e3, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": {"workload": workload_desc(n, 1), "reached_voxels": count, "triangles": ntri},
        "cpu_baseline": {"value": round(v, 2), "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(v, 2), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


_REAL_STDOUT = None


def claim_stdout():
    """Exactly ONE line may reach stdout (the JSON result). Libraries print there too (NCCL's version
    banner, for one): point fd 1 at stderr for the life of the process and keep the real stdout for
    the result line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--cpu-slices", type=int, default=0, help="reference arm: time a slab of this many slices instead "
                                                              "of the full volume (0 = full volume, the default)")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary 1024^3 / watershed measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the threshold mask, grown mask and mesh of the last "
                                                          "timed step to DIR/*.npy (sampled, see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
