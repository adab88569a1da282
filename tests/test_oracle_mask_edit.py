"""The CPU restatement of the 3-D mask editor (oracle/mask_edit.c) against an independent NumPy
restatement written here: elementwise float64 with explicit left-to-right sums (no matmul), on
hand-built cases for every branch of mask_cut, brush_mask_rs and polygon2mask_rs."""
import math

import numpy as np
import pytest


@pytest.fixture(scope="module")
def ome():
    """The CPU restatement of the mask editor (oracle/mask_edit.c)."""
    from oracle import mask_edit
    mask_edit.lib()
    return mask_edit


# ----------------------------------------------------------------------------- NumPy restatements
def _row(m, i, p0, p1, p2):
    return ((m[i, 0] * p0 + m[i, 1] * p1) + m[i, 2] * p2) + m[i, 3] * 1.0


def np_mask_cut(sx, sy, sz, depth, mask, M, MV, out, mode):
    h, w = mask.shape
    wm1 = float((w - 1) % 2 ** 64)
    hm1 = float((h - 1) % 2 ** 64)
    z, y, x = np.nonzero(out > 127)
    p0, p1, p2 = x.astype(np.float64) * sx, y.astype(np.float64) * sy, z.astype(np.float64) * sz
    with np.errstate(all="ignore"):
        q3 = _row(M, 3, p0, p1, p2)
        q0, q1 = _row(M, 0, p0, p1, p2) / q3, _row(M, 1, p0, p1, p2) / q3
        c3 = _row(MV, 3, p0, p1, p2)
        c0, c1, c2 = (_row(MV, i, p0, p1, p2) / c3 for i in range(3))
        dist = np.sqrt((c0 * c0 + c1 * c1) + c2 * c2)
        px, py = (q0 / 2.0 + 0.5) * wm1, (q1 / 2.0 + 0.5) * hm1
        live = (q3 > 0.0) & (dist <= depth)
        on = (px >= 0.0) & (px < w) & (py >= 0.0) & (py < h)
        hit = np.zeros(len(x), bool)
        k = live & on
        hit[k] = mask[py[k].astype(np.int64), px[k].astype(np.int64)]
    cut = hit | (live & ~on & (mode == 0))
    out[z[cut], y[cut], x[cut]] = 0


def _rmax(a, b):
    return b if math.isnan(a) else (a if math.isnan(b) else max(a, b))


def _rmin(a, b):
    return b if math.isnan(a) else (a if math.isnan(b) else min(a, b))


def _usize(v):
    return 0 if math.isnan(v) or v <= 0 else (2 ** 64 - 1 if v >= 2.0 ** 64 else int(v))


def np_brush(out, orig, spacing, center, radius, mode):
    d, h, w = out.shape
    if 0 in out.shape:
        return
    lo, hi = [], []
    for c, s, n in zip(center, spacing, (w, h, d)):
        lo.append(_usize(_rmax(math.floor((c - radius) / s) if math.isfinite((c - radius) / s) else (c - radius) / s, 0.0)))
        e = (c + radius) / s
        hi.append(_usize(_rmin(_rmax(math.ceil(e) if math.isfinite(e) else e, 0.0), float(n - 1))))
    if any(a > b for a, b in zip(lo, hi)) or mode not in (0, 1):
        return
    sl = (slice(lo[2], hi[2] + 1), slice(lo[1], hi[1] + 1), slice(lo[0], hi[0] + 1))
    zz, yy, xx = np.meshgrid(*[np.arange(s.start, s.stop, dtype=np.float64) for s in sl], indexing="ij")
    dx, dy, dz = xx * spacing[0] - center[0], yy * spacing[1] - center[1], zz * spacing[2] - center[2]
    inside = (dx * dx + dy * dy) + dz * dz <= radius * radius
    box = out[sl]
    if mode == 1:
        box[inside & (box > 0)] = 0
    elif orig is None:
        box[inside] = 255
    else:
        g = orig[sl]
        take = inside & (g > 0)
        box[take] = g[take]


def _isize(v):
    return 0 if math.isnan(v) else (2 ** 63 - 1 if v >= 2.0 ** 63 else (-(2 ** 63) if v <= -(2.0 ** 63) else int(v)))


def _wrap(v):
    return (v + 2 ** 63) % 2 ** 64 - 2 ** 63


def np_polygon2mask(shape, pts):
    w, h = shape
    out = np.zeros((w, h), bool)
    n = len(pts)
    if n == 0 or w == 0 or h == 0:
        return out
    xs, ys = pts[:, 0], pts[:, 1]
    mn = [np.finfo(np.float64).max] * 2
    mx = [np.finfo(np.float64).min] * 2
    for a in range(2):
        for v in (xs, ys)[a]:
            if v < mn[a]:
                mn[a] = v
            if v > mx[a]:
                mx[a] = v
    rng = []
    for a, n_ in enumerate((w, h)):
        f, c = math.floor(mn[a]) if math.isfinite(mn[a]) else mn[a], math.ceil(mx[a]) if math.isfinite(mx[a]) else mx[a]
        rng.append((min(max(_wrap(_isize(f) - 1), 0), n_), min(max(_wrap(_isize(c) + 1), 0), n_)))
    (r0, r1), (c0, c1) = rng
    if r0 > r1 or c0 > c1:
        return out
    px, py = np.meshgrid(np.arange(r0, min(r1, w - 1) + 1, dtype=np.float64),
                         np.arange(c0, min(c1, h - 1) + 1, dtype=np.float64), indexing="ij")
    inside = np.zeros(px.shape, bool)
    j = n - 1
    with np.errstate(all="ignore"):
        for i in range(n):
            xi, yi, xj, yj = xs[i], ys[i], xs[j], ys[j]
            cross = (yi > py) != (yj > py)
            inside ^= cross & (px < (xj - xi) * (py - yi) / (yj - yi) + xi)
            j = i
    out[r0:r0 + px.shape[0], c0:c0 + px.shape[1]] = inside
    return out


# ----------------------------------------------------------------------------- mask_cut
def _cut_both(ome, out, sp, depth, mask, M, MV, mode):
    a, b = out.copy(), out.copy()
    ome.mask_cut(np.zeros((1, 1, 1), np.int16), *sp, depth, mask, M, MV, a, mode)
    np_mask_cut(*sp, depth, mask, M, MV, b, mode)
    assert np.array_equal(a, b)
    return a


def _screen_map(w, h):
    """q0 = x / 2 - 1 and q1 = y / 2 - 1, so px = x (w - 1) / 4 and py = y (h - 1) / 4 land on integers."""
    M = np.zeros((4, 4))
    M[0, 0], M[0, 3], M[1, 1], M[1, 3], M[3, 3] = 0.5, -1.0, 0.5, -1.0, 1.0
    return M


def test_cut_truncates_on_a_pixel_edge(ome):
    out = np.full((1, 5, 5), 200, np.uint8)
    mask = np.zeros((5, 5), bool)
    mask[2, 3] = True                       # px = x, py = y exactly (w = h = 5)
    got = _cut_both(ome, out, (1.0, 1.0, 1.0), 1e9, mask, _screen_map(5, 5), np.eye(4), 1)
    assert list(zip(*np.nonzero(got == 0))) == [(0, 2, 3)]
    mask = np.zeros((5, 5), bool)
    mask[1, 1] = True                       # px = 1.5 -> column 1 (w = 4: px = x * 3 / 4)
    mask4 = mask[:5, :4]
    got = _cut_both(ome, np.full((1, 5, 4), 255, np.uint8), (2.0, 1.0, 1.0), 1e9, mask4, _screen_map(4, 5), np.eye(4), 1)
    assert (got == 0).sum() >= 1


def test_cut_behind_the_camera_is_untouched(ome):
    out = np.full((2, 3, 6), 255, np.uint8)
    M = _screen_map(8, 8)
    M[3] = (1.0, 0.0, 0.0, -2.0)            # q3 = x - 2: x <= 2 has q3 <= 0
    got = _cut_both(ome, out, (1.0, 1.0, 1.0), 1e9, np.ones((8, 8), bool), M, np.eye(4), 0)
    assert (got[..., :3] == 255).all() and (got[..., 3:] == 0).all()


def test_cut_depth_bound_is_inclusive(ome):
    out = np.full((1, 1, 4), 255, np.uint8)
    dist = math.sqrt(2.0 * 2.0)             # voxel x = 2 at (2, 0, 0)
    mask = np.ones((3, 3), bool)
    M = _screen_map(3, 3)
    at = _cut_both(ome, out, (1.0, 1.0, 1.0), dist, mask, M, np.eye(4), 1)
    below = _cut_both(ome, out, (1.0, 1.0, 1.0), np.nextafter(dist, 0.0), mask, M, np.eye(4), 1)
    assert at[0, 0, 2] == 0 and below[0, 0, 2] == 255 and at[0, 0, 3] == 255


def test_cut_off_screen_depends_on_the_mode(ome):
    out = np.full((1, 2, 12), 250, np.uint8)
    M = _screen_map(4, 4)                   # px = 3x / 4 >= 4 from x = 6 on
    mask = np.zeros((4, 4), bool)
    m0 = _cut_both(ome, out, (1.0, 1.0, 1.0), 1e9, mask, M, np.eye(4), 0)
    m1 = _cut_both(ome, out, (1.0, 1.0, 1.0), 1e9, mask, M, np.eye(4), 1)
    assert (m0[..., 6:] == 0).all() and (m0[..., :6] == 250).all()
    assert (m1 == 250).all()


def test_cut_never_touches_values_up_to_127(ome):
    rng = np.random.default_rng(0)
    out = rng.integers(0, 256, (5, 6, 7)).astype(np.uint8)
    out[0, 0, :4] = (126, 127, 128, 255)
    got = _cut_both(ome, out, (0.9, 1.1, 1.5), 1e9, np.ones((3, 3), bool), _screen_map(3, 3), np.eye(4), 0)
    low = out <= 127
    assert np.array_equal(got[low], out[low]) and (got[~low] == 0).all()


def test_cut_random_cameras(ome):
    rng = np.random.default_rng(1)
    out = (rng.random((9, 10, 11)) * 256).astype(np.uint8)
    for seed in range(6):
        r = np.random.default_rng(seed)
        M, MV = r.normal(size=(4, 4)), r.normal(size=(4, 4))
        MV[3] = (0, 0, 0, 1) if seed % 2 else MV[3]
        mask = r.random((13, 17)) < 0.5
        for mode in (0, 1):
            _cut_both(ome, out, (0.7, 1.3, 2.0), r.uniform(1, 20), mask.T.copy().T if seed % 3 else mask, M, MV, mode)


# ----------------------------------------------------------------------------- brush
def _brush_both(ome, out, orig, sp, ce, r, mode):
    a, b = out.copy(), out.copy()
    ome.brush_mask_rs(a, orig, sp, ce, r, mode)
    np_brush(b, orig, sp, ce, r, mode)
    assert np.array_equal(a, b), (sp, ce, r, mode)
    return a


def test_brush_box_can_exclude_what_the_sphere_includes(ome):
    out = np.zeros((3, 3, 6), np.uint8)
    # spacing -1 on x: the sphere covers x = 1..3, but floor/ceil of (c -/+ r) / s give min 3 > max 1
    got = _brush_both(ome, out, None, (-1.0, 1.0, 1.0), (-2.0, 1.0, 1.0), 1.0, 0)
    assert (got == 0).all()
    x = np.arange(6) * -1.0
    assert ((x - -2.0) ** 2 <= 1.0).any()


def test_brush_cases(ome):
    rng = np.random.default_rng(4)
    base = (rng.random((8, 9, 10)) < 0.5).astype(np.uint8) * 255
    orig = (rng.random((8, 9, 10)) * 3).astype(np.uint8) * 100
    nan = float("nan")
    cases = [((1.0, 1.0, 1.0), (4.0, 4.0, 3.0), 2.5),
             ((0.5, 0.7, 1.5), (2.3, 3.1, 5.0), 2.0),
             ((1.0, 1.0, 1.0), (-2.0, 4.0, 4.0), 3.0),        # centre outside the volume, sphere reaches in
             ((1.0, 1.0, 1.0), (-9.0, 4.0, 4.0), 3.0),        # centre outside, sphere stays out
             ((1.0, 1.0, 1.0), (40.0, 4.0, 4.0), 3.0),
             ((1.0, 1.0, 1.0), (3.0, 4.0, 5.0), 0.0),         # radius 0 on a voxel centre
             ((1.0, 1.0, 1.0), (nan, 4.0, 5.0), 3.0),         # NaN centre
             ((1.0, 1.0, 1.0), (3.0, 4.0, 5.0), nan)]
    for sp, ce, r in cases:
        for mode in (0, 1, 2):
            for g in (None, orig):
                got = _brush_both(ome, base, g, sp, ce, r, mode)
                if mode == 2:
                    assert np.array_equal(got, base)
    got = _brush_both(ome, base, None, (1.0, 1.0, 1.0), (3.0, 4.0, 5.0), 0.0, 0)
    assert (got != base).sum() <= 1 and got[5, 4, 3] == 255
    assert np.array_equal(_brush_both(ome, base, None, (1.0, 1.0, 1.0), (-9.0, 4.0, 4.0), 3.0, 0), base)


def test_brush_orig_too_small_panics(ome):
    out = np.zeros((6, 6, 6), np.uint8)
    with pytest.raises(ValueError):
        ome.brush_mask_rs(out, np.zeros((6, 6, 2), np.uint8), (1.0, 1.0, 1.0), (3.0, 3.0, 3.0), 2.0, 0)
    ome.brush_mask_rs(out, np.zeros((6, 6, 2), np.uint8), (1.0, 1.0, 1.0), (3.0, 3.0, 3.0), 2.0, 1)


# ----------------------------------------------------------------------------- rasteriser
def _raster_both(ome, shape, pts):
    pts = np.asarray(pts, dtype=np.float64).reshape(-1, 2) if not isinstance(pts, np.ndarray) else pts
    a = ome.polygon2mask_rs(shape, pts)
    b = np_polygon2mask(shape, pts)
    assert a.shape == tuple(shape) and a.dtype == np.bool_
    assert np.array_equal(a, b), (shape, pts)
    return a


def test_raster_degenerate_polygons(ome):
    assert not _raster_both(ome, (7, 5), []).any()
    assert not _raster_both(ome, (7, 5), [(2.0, 2.0)]).any()
    assert not _raster_both(ome, (7, 5), [(1.0, 1.0), (5.0, 4.0)]).any()
    assert _raster_both(ome, (0, 5), [(1.0, 1.0), (5.0, 4.0), (0, 4)]).shape == (0, 5)


def test_raster_nan_vertex_and_off_screen(ome):
    nan = float("nan")
    _raster_both(ome, (9, 8), [(1.0, 1.0), (7.0, 1.5), (nan, 4.0), (2.0, 6.0)])
    _raster_both(ome, (9, 8), [(nan, nan), (nan, nan), (nan, nan)])
    got = _raster_both(ome, (20, 15), [(-5.0, -3.0), (30.0, 2.0), (12.0, 40.0)])
    assert got.any()
    _raster_both(ome, (20, 15), [(-1e300, 2.0), (10.0, 2.0), (10.0, 12.0)])      # floor -> isize::MIN, wraps
    _raster_both(ome, (20, 15), [(1.0, 2.0), (1e300, 2.0), (10.0, 12.0)])


def test_raster_even_odd_star(ome):
    t = np.arange(5) * 4 * np.pi / 5
    star = np.stack([15 + 12 * np.sin(t), 15 + 12 * np.cos(t)], 1)
    got = _raster_both(ome, (31, 31), star)
    assert not got[15, 15]                  # the pentagon in the middle is crossed twice
    assert got[15, 25] or got[15, 5] or got[25, 15] or got[5, 15] or got.sum() > 50


def test_raster_integer_vertices_and_horizontal_edges(ome):
    got = _raster_both(ome, (10, 10), [(2.0, 2.0), (7.0, 2.0), (7.0, 6.0), (2.0, 6.0)])
    assert got[2:7, 2:6].all() and not got[7].any() and not got[:, 6].any()


def test_raster_orientation(ome):
    got = _raster_both(ome, (12, 5), [(1.0, 1.0), (10.0, 1.0), (10.0, 3.0)])   # wide in x: rows are x
    assert got.shape == (12, 5) and got[8, 1] and not got[1, 3]
    strided = np.asfortranarray(np.array([[1.0, 1.0, 9.0], [10.0, 1.0, 9.0], [10.0, 3.0, 9.0]]))
    assert np.array_equal(_raster_both(ome, (12, 5), strided), got)
