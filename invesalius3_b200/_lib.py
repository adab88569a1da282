"""ctypes binding of libb2v.so — the C ABI declared in include/b2v.h.

The library is mandatory: there is no CPU fallback. A missing or stale build raises
ImportError-style RuntimeError at first use, loudly.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libb2v.so"

OK, ERR_ARG, ERR_CUDA, ERR_RANGE, ERR_NOCONV = 0, 1, 2, 3, 4
I16, U8, F64 = 0, 1, 2
MIP_MAX, MIP_MIN, MIP_MEAN = 0, 1, 2

i64, i32, vp, cint = C.c_int64, C.c_int32, C.c_void_p, C.c_int
dbl, u8, u32, f32 = C.c_double, C.c_uint8, C.c_uint32, C.c_float

# name -> (restype, argtypes). Must list every symbol of include/b2v.h (tests check).
PROTOTYPES = {
    "b2v_last_error": (C.c_char_p, []),
    "b2v_version": (cint, []),
    "b2v_launch_count": (i64, []),
    "b2v_launch_count_reset": (None, []),
    "b2v_copy3d_h2d": (cint, [vp, vp, i64, i64, i64, i64, i64, i64, vp]),
    "b2v_copy3d_d2h": (cint, [vp, vp, i64, i64, i64, i64, i64, i64, vp]),
    "b2v_threshold_i16": (cint, [vp, i64, i32, i32, vp, cint, vp]),
    "b2v_threshold_i16_masklayout": (cint, [vp, i64, i64, i64, i32, i32, vp, cint, cint, vp]),
    "b2v_mip_workspace_bytes": (i64, [cint, i64, i64, i64, cint, cint]),
    "b2v_mip": (cint, [vp, cint, i64, i64, i64, cint, cint, vp, vp, vp]),
    "b2v_minmax_workspace_bytes": (i64, [i64]),
    "b2v_minmax_f32": (cint, [vp, cint, i64, vp, vp, vp]),
    "b2v_floodfill_workspace_bytes": (i64, [i64, i64, i64, i64]),
    "b2v_floodfill_set_engine": (None, [cint]),
    "b2v_floodfill_threshold": (cint, [vp, cint, i64, i64, i64, vp, i64, dbl, dbl, u8, vp, i64, i64, i64, vp, vp, vp,
                                       C.POINTER(cint)]),
    "b2v_floodfill_threshold_inplace": (cint, [vp, cint, i64, i64, i64, vp, i64, dbl, dbl, dbl, vp, i64, i64, i64, vp,
                                               vp, C.POINTER(cint)]),
    "b2v_floodfill_equal": (cint, [vp, cint, i64, i64, i64, i64, i64, i64, dbl, u8, vp, vp, vp, C.POINTER(cint)]),
    "b2v_fill_holes_workspace_bytes": (i64, [u32]),
    "b2v_fill_holes_staged": (cint, [cint, vp, vp, i64, u32, u32, vp, vp, C.POINTER(cint)]),
    "b2v_fill_holes": (cint, [vp, vp, i64, u32, u32, vp, vp, C.POINTER(cint)]),
    "b2v_proj_workspace_bytes": (i64, [i64]),
    "b2v_proj_set_tma": (None, [cint]),
    "b2v_mida": (cint, [vp, cint, i64, i64, i64, cint, dbl, dbl, vp, cint, vp, vp]),
    "b2v_mida_minmax": (cint, [vp, cint, i64, i64, i64, cint, dbl, dbl, vp, vp, cint, vp, vp]),
    "b2v_lmip": (cint, [vp, cint, i64, i64, i64, cint, dbl, dbl, vp, vp, vp]),
    "b2v_fcm_workspace_bytes": (i64, [cint, i64, i64, i64, cint, cint]),
    "b2v_fcm_volume": (cint, [vp, cint, i64, i64, i64, f32, cint, vp, vp, vp]),
    "b2v_fast_countour_mip": (cint, [vp, cint, i64, i64, i64, f32, cint, dbl, dbl, cint, vp, vp, vp]),
    "b2v_ca_smoothing_workspace_bytes": (i64, [i64, i64]),
    "b2v_ca_smoothing": (cint, [vp, i64, vp, i64, vp, vp, dbl, dbl, dbl, u32, vp, vp]),
    "b2v_boolean_op": (cint, [vp, vp, i64, cint, vp, vp]),
    "b2v_convolve_non_zero": (cint, [vp, i64, i64, i64, vp, i64, i64, i64, dbl, vp, vp]),
    "b2v_median_filter_i16": (cint, [vp, i64, i64, i64, cint, vp, vp]),
    "b2v_uniform_filter_i16": (cint, [vp, i64, i64, i64, cint, vp, vp, vp]),
    "b2v_correlate1d": (cint, [vp, cint, i64, i64, i64, cint, vp, cint, cint, vp, cint, vp]),
    "b2v_sharpen_i16": (cint, [vp, vp, i64, dbl, dbl, dbl, vp, vp]),
    "b2v_sobel_magnitude": (cint, [vp, vp, vp, i64, vp]),
    "b2v_rescale_cast_i16": (cint, [vp, i64, cint, dbl, dbl, dbl, dbl, vp, vp]),
    "b2v_label_workspace_bytes": (i64, [i64]),
    "b2v_label": (cint, [vp, i64, i64, i64, vp, i64, i64, i64, vp, vp, vp, C.POINTER(i64)]),
    "b2v_count_regions": (cint, [vp, cint, i64, u32, vp, vp, vp]),
    "b2v_apply_view_matrix_transform": (cint, [vp, cint, i64, i64, i64, vp, vp, i64, cint, cint, dbl, vp, i64, i64, i64, vp,
                                               vp]),
    "b2v_mask_cut": (cint, [vp, i64, i64, i64, vp, dbl, vp, i64, i64, vp, vp, cint, vp]),
    "b2v_brush_bbox": (cint, [i64, i64, i64, vp, vp, dbl, vp]),
    "b2v_brush_mask": (cint, [vp, vp, i64, i64, i64, i64, i64, i64, i64, i64, i64, vp, vp, dbl, cint, vp]),
    "b2v_polygons_workspace_bytes": (i64, [i64]),
    "b2v_polygons_raster": (cint, [vp, vp, i64, i64, i64, cint, cint, vp, vp, vp]),
    "b2v_mc_workspace_bytes": (i64, [i64, i64, i64]),
    "b2v_mc_count": (cint, [vp, cint, i64, i64, i64, dbl, vp, vp, C.POINTER(i64), C.POINTER(i64)]),
    "b2v_mc_emit": (cint, [vp, cint, i64, i64, i64, dbl, vp, f32, f32, f32, i32, i32, i32, cint, vp, vp, vp]),
    "b2v_ws_lut_i16": (cint, [vp, i64, dbl, dbl, vp, vp]),
    "b2v_ws_shift_i16": (cint, [vp, i64, vp, vp, vp]),
    "b2v_ws_morph_gradient_u16": (cint, [vp, i64, i64, i64, cint, cint, cint, vp, vp]),
    "b2v_ws_workspace_bytes": (i64, [i64, i64, i64]),
    "b2v_ws_flood_staged": (cint, [cint, vp, vp, i64, i64, i64, cint, cint, cint, vp, vp, vp, vp, C.POINTER(cint)]),
    "b2v_ws_plane_bytes": (i64, [i64, i64, cint]),
    "b2v_ws_plane": (cint, [cint, cint, i64, i64, i64, cint, cint, cint, i64, vp, vp, vp, C.POINTER(cint)]),
    "b2v_ws_shift_i16_with": (cint, [vp, i64, vp, vp, vp]),
    "b2v_ws_stats": (cint, [C.POINTER(cint), cint]),
    "b2v_ws_flood": (cint, [vp, vp, i64, i64, i64, vp, i64, i64, i64, cint, vp, vp, vp, vp, C.POINTER(cint)]),
    "b2v_floodfill_threshold_staged": (cint, [cint, vp, cint, i64, i64, i64, vp, i64, dbl, dbl, u8, vp, i64, i64, i64,
                                              vp, vp, vp, C.POINTER(cint)]),
    "b2v_floodfill_layout": (cint, [i64, i64, i64, i64, C.POINTER(i64)]),
    "b2v_floodfill_merge_plane": (cint, [i64, i64, i64, i64, vp, i64, vp, cint, vp]),
    "b2v_mc_count_shard": (cint, [vp, cint, i64, i64, i64, dbl, cint, vp, vp, C.POINTER(i64), C.POINTER(i64)]),
    "b2v_mc_emit_shard": (cint, [vp, cint, i64, i64, i64, dbl, vp, f32, f32, f32, i32, i32, i32, cint, cint, i32, vp,
                                 i32, vp, vp, vp]),
    "b2v_mc_layout": (cint, [i64, i64, i64, C.POINTER(i64)]),
    "b2v_peer_mailbox_bytes": (i64, [i64, i64]),
    "b2v_peer_alloc": (cint, [i64, C.POINTER(vp), vp]),
    "b2v_peer_open": (cint, [vp, C.POINTER(vp)]),
    "b2v_peer_close": (cint, [vp]),
    "b2v_peer_free": (cint, [vp]),
    "b2v_peer_barrier": (cint, [cint, cint, vp, i64, u32, vp]),
    "b2v_floodfill_threshold_peer": (cint, [vp, cint, i64, i64, i64, vp, i64, dbl, dbl, u8, vp, i64, i64, i64, vp, vp,
                                            vp, cint, cint, vp, i64, u32, C.POINTER(cint), C.POINTER(cint)]),
    "b2v_mc_count_shard_peer": (cint, [vp, cint, i64, i64, i64, dbl, cint, vp, vp, cint, cint, vp, i64, u32, vp]),
    "b2v_peer_mc_inbox_offset": (i64, [i64, u32]),
    "b2v_mida_z_partial": (cint, [vp, cint, i64, i64, i64, dbl, dbl, vp, vp, cint, cint, vp, cint, vp, vp]),
    "b2v_lmip_z_partial": (cint, [vp, cint, i64, i64, i64, dbl, dbl, vp, cint, cint, vp, vp, vp]),
}

_lib = None


class B2VError(RuntimeError):
    pass


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension is mandatory (no CPU fallback). "
            "Build it with `python -m invesalius3_b200._build` or __graft_entry__.build()."
        )
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here = stale build
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    """Map a B2V_* status to the exception the reference boundary would raise."""
    if rc == OK:
        return
    msg = load().b2v_last_error().decode("utf-8", "replace")
    if rc == ERR_ARG:
        raise ValueError(msg)
    if rc == ERR_RANGE:
        raise ValueError(msg)
    raise B2VError(f"b2v status {rc}: {msg}")


def call(name: str, *args):
    fn = getattr(load(), name)
    check(fn(*args))
