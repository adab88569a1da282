"""The 3-D mask editor on the device (invesalius/data/mask3d_editor_state.py).

InVesalius imports three native functions for it from the `invesalius_rs` crate:
`mask_cut` (cut the mask with screen polygons seen through the camera), `brush_mask_rs`
(the sphere brush, called on every mouse move) and `polygon2mask_rs` (even-odd polygon
rasteriser). This module provides them with the crate's names, argument order, in-place
output convention and error behaviour (numpy in, numpy out), plus device-tensor forms and
a fused `cut_from_polygons` that rasterises every polygon straight into the cut's screen
filter without a host round trip. Results equal the crate's bit for bit: float64 in its
operation order, see csrc/mask_edit.cu.

Transfers: `brush_mask_rs` moves only the sphere's bounding box of `out` (and of `orig`)
to the device and back, straight from a view such as `mask.matrix[1:, 1:, 1:]`;
`mask_cut` moves `out` up and back and the bool filter once, never `image`.

Error mapping (crate -> here), all raised before any device work:
  argument extraction (dtype, dimensions, tuple shapes) -> TypeError
  an integer that does not fit i32 / usize               -> OverflowError
  a Rust panic (m / mv not 16 contiguous values, a polygon with fewer than two columns,
  orig too small for the brush's box)                    -> ValueError
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from . import device as dev

_IMAGE_DTYPES = (np.dtype(np.int16), np.dtype(np.uint8), np.dtype(np.float64))


# ----------------------------------------------------------------------------- argument extraction
def _int(v, lo, hi):
    if isinstance(v, (float, np.floating)):
        raise TypeError("'float' object cannot be interpreted as an integer")
    v = int(v)
    if not lo <= v <= hi:
        raise OverflowError("out of range integral type conversion attempted")
    return v


def _i32(v):
    return _int(v, -(2 ** 31), 2 ** 31 - 1)


def _f64(v):
    if isinstance(v, (str, bytes)):
        raise TypeError("must be real number, not str")
    return float(v)


def _triple(v, name):
    try:
        t = tuple(v)
    except TypeError:
        raise TypeError(f"{name} must be a tuple of 3 floats") from None
    if len(t) != 3:
        raise TypeError(f"{name} must be a tuple of 3 floats")
    return np.array([_f64(x) for x in t], dtype=np.float64)


def _mat16(m, name):
    """PyReadonlyArray2<f64> + as_slice().unwrap() + Matrix4::from_row_slice."""
    if not isinstance(m, np.ndarray) or m.dtype != np.float64 or m.ndim != 2:
        raise TypeError(f"{name} must be a 2-D float64 array")
    if not m.flags.c_contiguous or m.size != 16:
        raise ValueError(f"{name} must hold 16 contiguous float64 values (a C-order 4x4 matrix)")
    return np.ascontiguousarray(m).reshape(16)


def _out_u8(out):
    if not isinstance(out, np.ndarray) or out.dtype != np.uint8 or out.ndim != 3:
        raise TypeError("Invalid mask type: out must be a 3-D uint8 array")
    if not out.flags.writeable:
        raise ValueError("out is read-only")


def _polygon(p):
    if not isinstance(p, np.ndarray) or p.dtype != np.float64 or p.ndim != 2:
        raise TypeError("polygon must be a 2-D float64 array")
    if p.shape[0] > 0 and p.shape[1] < 2:
        raise ValueError("polygon rows need an x and a y column")
    return p


def _screen(shape):
    t = tuple(shape)
    if len(t) != 2:
        raise TypeError("shape must be a (w, h) tuple")
    w, h = t
    return _int(w, 0, 2 ** 63 - 1), _int(h, 0, 2 ** 63 - 1)


def brush_box(shape, spacing, center, radius):
    """(z0, y0, x0, nz, ny, nx): the voxels brush_mask_rs visits in a volume of `shape` (all zero
    when none). Host only, the same definition the kernel launch uses (b2v_brush_bbox)."""
    sp, ce = _triple(spacing, "spacing"), _triple(center, "center")
    box = (C.c_int64 * 6)()
    _lib.call("b2v_brush_bbox", *[int(s) for s in shape], C.c_void_p(sp.ctypes.data), C.c_void_p(ce.ctypes.data),
              _f64(radius), box)
    return tuple(box)


# ----------------------------------------------------------------------------- device tensors
def _dense_u8(t, name, ndim):
    dev._dense(t, name)
    if t.dtype not in (torch.uint8, torch.bool) or t.dim() != ndim:
        raise TypeError(f"{name} must be a {ndim}-D uint8 tensor")
    return t


def _raster(polygons, w, h, transpose, negate, device):
    pts = [p[:, :2] if len(p) else np.zeros((0, 2)) for p in polygons]
    offs = np.zeros(len(pts) + 1, np.int64)
    offs[1:] = np.cumsum([len(p) for p in pts])
    flat = np.ascontiguousarray(np.concatenate(pts) if offs[-1] else np.zeros((0, 2)), dtype=np.float64)
    out = torch.empty((h, w) if transpose else (w, h), dtype=torch.uint8, device=device)
    dpts, doffs = dev.to_device(flat, device), dev.to_device(offs, device)
    ws = dev._workspace(_lib.load().b2v_polygons_workspace_bytes(len(pts)), device)
    with torch.cuda.device(device):
        _lib.call("b2v_polygons_raster", dev._p(dpts), dev._p(doffs), len(pts), w, h, int(transpose), int(negate),
                  dev._p(out), dev._p(ws), dev._stream())
    return out


def polygon2mask_device(shape, polygon, device=None) -> torch.Tensor:
    """polygon2mask_rs on the device: uint8 (w, h) tensor, [r, c] = even-odd inside(px=r, py=c)."""
    w, h = _screen(shape)
    p = _polygon(polygon)
    dev.require_cuda()
    return _raster([p], w, h, False, False, torch.device("cuda" if device is None else device))


def mask_cut_device(out: torch.Tensor, spacing, max_depth, filt: torch.Tensor, m, mv, edit_mode) -> torch.Tensor:
    """mask_cut on the device: `out` (dense uint8 [dz][dy][dx]) edited in place through the
    dense (h, w) uint8 / bool screen `filt`; spacing = (sx, sy, sz). Does not synchronise."""
    _dense_u8(out, "out", 3)
    _dense_u8(filt, "filt", 2)
    sp, mm, vv = _triple(spacing, "spacing"), _mat16(m, "m"), _mat16(mv, "mv")
    mode, depth = _i32(edit_mode), _f64(max_depth)
    h, w = filt.shape
    with torch.cuda.device(out.device):
        _lib.call("b2v_mask_cut", dev._p(out), *out.shape, C.c_void_p(sp.ctypes.data), depth, dev._p(filt), h, w,
                  C.c_void_p(mm.ctypes.data), C.c_void_p(vv.ctypes.data), mode, dev._stream())
    return out


def cut_from_polygons_device(out: torch.Tensor, spacing, max_depth, polygons, m, mv, edit_mode, resolution) -> torch.Tensor:
    """CutMaskFromPolygons (mask3d_editor_state.py:196-221) in one device call: the K >= 1
    polygons (float64 (N, 2) screen points) are rasterised on the (w, h) = `resolution` screen
    straight into the cut's (h, w) filter: OR over the polygons, transposed, negated when
    edit_mode == 0; then mask_cut runs on `out`. Equals polygon2mask_rs + logical_or.reduce + .T
    (+ logical_not) + mask_cut bit for bit. Does not synchronise."""
    polys = [_polygon(p) for p in polygons]
    if not polys:
        raise ValueError("cut_from_polygons needs at least one polygon")
    w, h = _screen(resolution)
    _dense_u8(out, "out", 3)
    _triple(spacing, "spacing")
    _mat16(m, "m")
    _mat16(mv, "mv")
    _f64(max_depth)
    mode = _i32(edit_mode)
    filt = _raster(polys, w, h, True, mode == 0, out.device)
    return mask_cut_device(out, spacing, max_depth, filt, m, mv, mode)


def brush_device(out: torch.Tensor, orig: torch.Tensor | None, spacing, center, radius, edit_mode,
                 origin=(0, 0, 0), volume_shape=None) -> torch.Tensor:
    """brush_mask_rs on the device. `out` (and `orig`, or None) are dense uint8 copies of the box
    of the volume that starts at `origin` (z, y, x); `volume_shape` is the whole volume's shape
    (default: out's, i.e. `out` is the whole volume). Only voxels inside both the box and the
    brush's bounding box are visited. Does not synchronise."""
    _dense_u8(out, "out", 3)
    if orig is not None:
        _dense_u8(orig, "orig", 3)
        if orig.shape != out.shape or orig.device != out.device:
            raise ValueError("orig must be a box of the shape of out on the same device")
    sp, ce = _triple(spacing, "spacing"), _triple(center, "center")
    mode, r = _i32(edit_mode), _f64(radius)
    vol = tuple(out.shape) if volume_shape is None else tuple(int(v) for v in volume_shape)
    with torch.cuda.device(out.device):
        _lib.call("b2v_brush_mask", dev._p(out), dev._p(orig), *out.shape, *[int(o) for o in origin], *vol,
                  C.c_void_p(sp.ctypes.data), C.c_void_p(ce.ctypes.data), r, mode, dev._stream())
    return out


# ----------------------------------------------------------------------------- the crate's numpy surface
def mask_cut(image, sx, sy, sz, max_depth, mask, m, mv, out, edit_mode):
    """invesalius_rs.mask_cut (mask_cut_py.rs:8-69 -> mask_cut.rs:7-62); `image` only selects the
    dtype (int16, uint8, float64) and is never read or transferred. `out` is edited in place."""
    if not isinstance(image, np.ndarray) or image.dtype not in _IMAGE_DTYPES or image.ndim != 3:
        raise TypeError("Invalid image or mask type")
    sp = np.array([_f64(sx), _f64(sy), _f64(sz)])
    depth = _f64(max_depth)
    if not isinstance(mask, np.ndarray) or mask.dtype != np.bool_ or mask.ndim != 2:
        raise TypeError("mask must be a 2-D bool array")
    _mat16(m, "m")
    _mat16(mv, "mv")
    _out_u8(out)
    mode = _i32(edit_mode)
    o = dev.to_device(out)
    filt = dev.to_device(np.ascontiguousarray(mask).view(np.uint8), o.device)
    mask_cut_device(o, sp, depth, filt, m, mv, mode)
    dev.to_host(o, out)


def cut_from_polygons(out, spacing, max_depth, polygons, m, mv, edit_mode, resolution):
    """cut_from_polygons_device on a host mask (e.g. `mask_data[1:, 1:, 1:]`), edited in place:
    `out` goes up and back once, the polygons' points once, the filter never leaves the device."""
    polys = [_polygon(p) for p in polygons]
    if not polys:
        raise ValueError("cut_from_polygons needs at least one polygon")
    _screen(resolution)
    _triple(spacing, "spacing")
    _mat16(m, "m")
    _mat16(mv, "mv")
    _f64(max_depth)
    _i32(edit_mode)
    _out_u8(out)
    o = dev.to_device(out)
    cut_from_polygons_device(o, spacing, max_depth, polys, m, mv, edit_mode, resolution)
    dev.to_host(o, out)


def polygon2mask_rs(shape, polygon):
    """invesalius_rs.polygon2mask_rs (polygon_mask_py.rs:6-27 -> polygon_mask.rs:4-79): bool (w, h)
    array for shape = (w, h); element [r, c] is the even-odd inside(px=r, py=c)."""
    w, h = _screen(shape)
    p = _polygon(polygon)
    if w == 0 or h == 0 or p.shape[0] == 0:
        return np.zeros((w, h), dtype=np.bool_)
    return dev.to_numpy(polygon2mask_device((w, h), p)).view(np.bool_)


def brush_mask_rs(out, orig, spacing, center, radius, edit_mode):
    """invesalius_rs.brush_mask_rs (brush_mask_py.rs:7-28 -> brush_mask.rs:5-71), `out` edited in
    place. Only the brush's bounding box of `out` (and of `orig` in mode 0) crosses to the device.
    `orig` may share memory with `out`: it is read as it was before the stroke."""
    _out_u8(out)
    if orig is not None and (not isinstance(orig, np.ndarray) or orig.dtype != np.uint8 or orig.ndim != 3):
        raise TypeError("Invalid mask type: orig must be None or a 3-D uint8 array")
    sp, ce = _triple(spacing, "spacing"), _triple(center, "center")
    r, mode = _f64(radius), _i32(edit_mode)
    box = brush_box(out.shape, sp, ce, r)
    lo, n = box[:3], box[3:]
    if mode not in (0, 1) or 0 in n:
        return
    sl = tuple(slice(a, a + b) for a, b in zip(lo, n))
    src = orig if mode == 0 else None
    if src is not None and any(g < a + b for g, a, b in zip(src.shape, lo, n)):
        raise ValueError("orig is smaller than the brush's box in out (the crate panics on the index)")
    ob = dev.to_device(out[sl])
    gb = None if src is None else dev.to_device(src[sl], ob.device)
    brush_device(ob, gb, sp, ce, r, mode, origin=lo, volume_shape=out.shape)
    dev.to_host(ob, out[sl])
