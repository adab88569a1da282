"""CPU restatement of the 3-D mask editor — TEST INFRASTRUCTURE ONLY.

invesalius_rs.mask_cut, brush_mask_rs and polygon2mask_rs (imported by
invesalius/data/mask3d_editor_state.py:14), restated in oracle/mask_edit.c and built by
oracle/mask_edit.mk into libmask_edit.so. The names and argument order are the crate's. The
reference holds no test for these functions: PARITY UNPINNED (restated, not pinned).
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from . import _estrides, _ptr, _suffix

_HERE = Path(__file__).resolve().parent
_LIB = None


def build(force: bool = False) -> Path:
    r = subprocess.run(["make", "-C", str(_HERE), "-f", "mask_edit.mk", *(["-B"] if force else [])],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"build of libmask_edit.so failed:\n{r.stdout}\n{r.stderr}")
    return _HERE / "libmask_edit.so"


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        so = _HERE / "libmask_edit.so"
        if not so.exists() or so.stat().st_mtime < (_HERE / "mask_edit.c").stat().st_mtime:
            build()
        _LIB = C.CDLL(str(so))
    return _LIB


def mask_cut(image, sx, sy, sz, max_depth, mask, m, mv, out, edit_mode):
    """invesalius_rs.mask_cut (mask_cut.rs:7-62). `image` only selects the dtype; `out` (uint8,
    any strides) is edited in place; `mask` is the bool (h, w) screen filter, any strides."""
    _suffix(image)
    assert out.dtype == np.uint8 and out.ndim == 3 and mask.dtype == np.bool_ and mask.ndim == 2
    mm = np.ascontiguousarray(m, dtype=np.float64).reshape(16)
    vv = np.ascontiguousarray(mv, dtype=np.float64).reshape(16)
    mk = mask.view(np.uint8)
    lib().orc_mask_cut(_ptr(out), _estrides(out), *map(C.c_int64, out.shape), C.c_double(sx), C.c_double(sy),
                       C.c_double(sz), C.c_double(max_depth), _ptr(mk), _estrides(mk), *map(C.c_int64, mask.shape),
                       _ptr(mm), _ptr(vv), C.c_int(int(edit_mode)))


def brush_mask_rs(out, orig, spacing, center, radius, edit_mode):
    """invesalius_rs.brush_mask_rs (brush_mask.rs:5-71). `out` / `orig` uint8 3-D, any strides;
    orig is read only where the reference reads it (a read outside orig panics there: ValueError
    here)."""
    assert out.dtype == np.uint8 and out.ndim == 3
    sp = np.ascontiguousarray([float(v) for v in spacing], dtype=np.float64)
    ce = np.ascontiguousarray([float(v) for v in center], dtype=np.float64)
    if orig is None:
        og, gs, gshape = None, None, (0, 0, 0)
    else:
        assert orig.dtype == np.uint8 and orig.ndim == 3
        og, gs, gshape = _ptr(orig), _estrides(orig), orig.shape
    rc = lib().orc_brush_mask(_ptr(out), _estrides(out), *map(C.c_int64, out.shape), og, gs, *map(C.c_int64, gshape),
                              _ptr(sp), _ptr(ce), C.c_double(radius), C.c_int(int(edit_mode)))
    if rc:
        raise ValueError("orig is indexed outside its shape (the reference panics)")


def polygon2mask_rs(shape, polygon):
    """invesalius_rs.polygon2mask_rs (polygon_mask.rs:4-79): bool (w, h) for shape = (w, h),
    element [r, c] = even-odd inside(px=r, py=c)."""
    w, h = (int(v) for v in shape)
    pts = np.asarray(polygon)
    assert pts.dtype == np.float64 and pts.ndim == 2 and (pts.shape[0] == 0 or pts.shape[1] >= 2)
    out = np.zeros((w, h), np.uint8)
    lib().orc_polygon2mask(C.c_int64(w), C.c_int64(h), _ptr(pts), _estrides(pts), C.c_int64(pts.shape[0]), _ptr(out))
    return out.view(np.bool_)
