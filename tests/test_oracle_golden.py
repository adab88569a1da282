"""Pins the CPU oracle against every known-answer the reference holds for the hot path:
  - tests/test_bone_thresholding.py:51-185 and tests/test_segmentation_tools.py:137-160 (threshold)
  - samples/Cranium.inv3 mask_0/mask_1 (thresholds produced by the reference itself;
    crop, whole masks and slice counts in tests/golden/cranium_crop.npz, a lattice and the
    threshold-bound voxels of the whole matrix in tests/golden/cranium_sample.npz, generator
    tools/make_golden_cranium.py)
  - tests/test_segmentation_tools.py:17-51, :54-102 (flood fill), :105-134 (fill holes)
MIP/MIDA/LMIP/contour-MIP have no reference test or golden: parity unpinned (checked
here only against independent NumPy restatements of the same formulas).
"""
import numpy as np
import pytest
from scipy import ndimage
from scipy.ndimage import generate_binary_structure


# ------------------------------------------------------------------ threshold
def test_threshold_cranium_crop(orc, cranium):
    img = cranium["matrix_crop"]
    for i in (0, 1):
        lo, hi = cranium[f"thr_{i}"]
        want = np.unpackbits(cranium[f"mask_{i}_crop_bits"])[: img.size].reshape(img.shape) * np.uint8(255)
        got = np.zeros(img.shape, np.uint8)
        orc.threshold(img, lo, hi, got, False)
        assert np.array_equal(got, want)
        assert 0 < int((got == 255).sum()) < got.size


def test_threshold_cranium_whole_volume_sample(orc, cranium):
    """Whole-volume check against the shipped masks, on the stored sample of the matrix: a
    lattice over every slice, and every voxel on (or one past) a bound of either threshold."""
    from pathlib import Path
    smp = np.load(Path(__file__).resolve().parent / "golden" / "cranium_sample.npz")
    shape = tuple(int(v) for v in cranium["full_shape"])
    lat, step = smp["lattice"], tuple(int(s) for s in smp["lattice_step"])
    on_lattice = tuple(slice(None, None, s) for s in step)
    # the sample comes from the same matrix as the stored crop
    crop = tuple(slice(int(a), int(b)) for a, b in cranium["crop"])
    assert all(c.start % s == 0 for c, s in zip(crop, step))
    in_crop = tuple(slice(c.start // s, -(-c.stop // s)) for c, s in zip(crop, step))
    assert np.array_equal(lat[in_crop], cranium["matrix_crop"][on_lattice])
    idx, val = smp["bound_index"], smp["bound_value"]
    for i in (0, 1):
        thr = cranium[f"thr_{i}"]
        m = np.unpackbits(cranium[f"mask_{i}_bits_full"])[: int(np.prod(shape))].reshape(shape) * np.uint8(255)
        assert int((m == 255).sum()) == int(cranium[f"mask_{i}_count_full"])
        assert np.array_equal((m == 255).sum(axis=(1, 2)), cranium[f"mask_{i}_slice_counts"])
        got = np.zeros(lat.shape, np.uint8)
        orc.threshold(lat, thr[0], thr[1], got, False)
        assert np.array_equal(got, m[on_lattice])
        assert 0 < int((got == 255).sum()) < got.size
        # the voxels on the bounds, as one row
        got = np.zeros((1, 1, idx.size), np.uint8)
        orc.threshold(val.reshape(got.shape), thr[0], thr[1], got, False)
        assert np.array_equal(got.reshape(-1), m.reshape(-1)[idx])
        assert (val == thr[0]).any() and (val == thr[0] - 1).any()
        # the reference's NumPy statements give the same thing
        mm = np.zeros(tuple(s + 1 for s in lat.shape), np.uint8)
        orc.set_mask_threshold_numpy(lat, mm, thr)
        assert np.array_equal(mm[1:, 1:, 1:], m[on_lattice]) and (mm[1:, 0, 0] == 1).all()


def test_threshold_reference_known_answers(orc):
    bone_min, bone_max = 226, 3071  # presets.py:35-52, test_bone_thresholding.py:42
    rng = np.random.default_rng(0)
    # test_do_threshold_to_a_slice (test_bone_thresholding.py:92-118)
    sl = rng.integers(0, bone_min - 1, (10, 10), dtype=np.int16)
    sl[5:8, 5:8] = (bone_min + bone_max) // 2
    m0 = np.zeros((10, 10), np.uint8)
    m0[0:2, 0:2] = 1; m0[2:4, 2:4] = 2; m0[4:6, 4:6] = 253; m0[6:8, 6:8] = 254
    expected = np.zeros((10, 10), np.uint8)
    expected[5:8, 5:8] = 255
    expected[0:2, 0:2] = 1; expected[2:4, 2:4] = 2; expected[4:6, 4:6] = 253; expected[6:8, 6:8] = 254
    got = m0.copy()[None]
    orc.threshold(sl[None], bone_min, bone_max, got, True)
    assert np.array_equal(got[0], expected)
    assert np.array_equal(orc.do_threshold_to_a_slice_numpy(sl, m0, (bone_min, bone_max)), expected)
    # edge cases (test_bone_thresholding.py:156-185): bounds are inclusive
    e = np.zeros((1, 10, 10), np.int16)
    e[0, 0, :4] = [226, 3071, 225, 3072]
    got = np.zeros(e.shape, np.uint8)
    orc.threshold(e, bone_min, bone_max, got, False)
    assert got[0, 0, :4].tolist() == [255, 255, 0, 0] and got.sum() == 510
    # test_do_threshold_to_all_slices (:121-153) on the padded Mask layout
    vol = rng.integers(0, bone_min - 1, (10, 10, 10), dtype=np.int16)
    vol[5:8, 5:8, 5:8] = (bone_min + bone_max) // 2
    mm = np.zeros((11, 11, 11), np.uint8)
    orc.do_threshold_to_all_slices_numpy(vol, mm, (bone_min, bone_max))
    exp = np.zeros((10, 10, 10), np.uint8); exp[5:8, 5:8, 5:8] = 255
    assert np.array_equal(mm[1:, 1:, 1:], exp)
    got = np.zeros(vol.shape, np.uint8)
    orc.threshold(vol, bone_min, bone_max, got, True)
    assert np.array_equal(got, exp)
    # test_threshold_and_density_measure (test_segmentation_tools.py:137-160)
    image = np.zeros((5, 5, 5), np.int16); image[2, 2, 2] = 100; image[3, 3, 3] = 200
    got = np.zeros(image.shape, np.uint8)
    orc.threshold(image, 100, 200, got, True)
    exp = np.zeros((5, 5, 5), np.uint8); exp[2, 2, 2] = 255; exp[3, 3, 3] = 255
    assert np.array_equal(got, exp)


# ------------------------------------------------------------------ flood fill
def test_region_growing_threshold(orc):
    """tests/test_segmentation_tools.py:17-51."""
    image = np.array([[[1, 1, 1, 5, 5], [1, 2, 2, 5, 5], [1, 2, 3, 5, 5], [1, 2, 2, 5, 5], [1, 1, 1, 5, 5]]],
                     dtype=np.int16)
    out_mask = np.zeros((1, 5, 5), dtype=np.uint8)
    orc.floodfill_threshold(image, [[2, 2, 0]], 2, 3, 1, generate_binary_structure(3, 1), out_mask)
    expected = np.array([[0, 0, 0, 0, 0], [0, 1, 1, 0, 0], [0, 1, 1, 0, 0], [0, 1, 1, 0, 0], [0, 0, 0, 0, 0]],
                        dtype=np.uint8)
    assert np.array_equal(out_mask[0], expected)


def test_region_growing_strct_disconnected(orc):
    """tests/test_segmentation_tools.py:54-102."""
    image = np.array([[[2, 2, 0], [0, 2, 0], [0, 0, 2]]], dtype=np.int16)
    out8 = np.zeros((1, 3, 3), dtype=np.uint8)
    orc.floodfill_threshold(image, [[0, 0, 0]], 2, 2, 1, generate_binary_structure(3, 2), out8)
    assert np.array_equal(out8, np.array([[[1, 1, 0], [0, 1, 0], [0, 0, 1]]], dtype=np.uint8))
    out4 = np.zeros((1, 3, 3), dtype=np.uint8)
    orc.floodfill_threshold(image, [[0, 0, 0]], 2, 2, 1, generate_binary_structure(3, 1), out4)
    assert np.array_equal(out4, np.array([[[1, 1, 0], [0, 1, 0], [0, 0, 0]]], dtype=np.uint8))


def test_fill_holes_automatically(orc):
    """tests/test_segmentation_tools.py:105-134."""
    mask_2d = np.ones((7, 7), dtype=np.uint8)
    mask_2d[3, 3] = 0
    mask = mask_2d[np.newaxis, ...]
    labels_2d, nlabels = ndimage.label(mask_2d == 0, structure=np.ones((3, 3), np.uint8), output=np.uint32)
    border = set(labels_2d[:, 0]) | set(labels_2d[:, -1]) | set(labels_2d[0, :]) | set(labels_2d[-1, :])
    for bl in border:
        labels_2d[labels_2d == bl] = 0
    labels = labels_2d[np.newaxis, ...]
    ret = orc.fill_holes_automatically(mask, labels, int(labels.max()), 1)
    expected = np.ones((1, 7, 7), dtype=np.uint8)
    expected[0, 3, 3] = 254
    assert ret and np.array_equal(mask, expected)


def test_floodfill_walls_seeds_and_inplace(orc):
    rng = np.random.default_rng(3)
    data = rng.integers(0, 4, (6, 7, 8)).astype(np.int16)
    st = generate_binary_structure(3, 1)
    # independent restatement via scipy.ndimage.label on the passable set
    out = np.zeros(data.shape, np.uint8)
    out[2, :, :] = 1  # pre-filled plane acts as a wall (floodfill.rs:154)
    seeds = [(1, 1, 0), (3, 3, 5), (0, 0, 2)]
    ref = out.copy()
    passable = (data >= 1) & (data <= 2) & (ref != 1)
    for (x, y, z) in seeds:
        if 1 <= data[z, y, x] <= 2:
            passable[z, y, x] = True
    lab, _ = ndimage.label(passable, st)
    keep = {lab[z, y, x] for (x, y, z) in seeds if 1 <= data[z, y, x] <= 2}
    ref[np.isin(lab, list(keep)) & (lab > 0)] = 1
    orc.floodfill_threshold(data, seeds, 1, 2, 1, st, out)
    assert np.array_equal(out, ref)
    # in-place twin on a uint8 mask (styles.py:2450-2458 usage)
    m = rng.integers(0, 3, (5, 6, 7)).astype(np.uint8) * 127
    m2 = m.copy()
    orc.floodfill_threshold_inplace(m2, [(0, 0, 0)], int(m[0, 0, 0]), int(m[0, 0, 0]), 200, st)
    lab, _ = ndimage.label(m == m[0, 0, 0], st)
    want = m.copy(); want[lab == lab[0, 0, 0]] = 200
    assert np.array_equal(m2, want)
    with pytest.raises(OverflowError):
        orc.floodfill_threshold(data, seeds, 1, 40000, 1, st, out)
    with pytest.raises(IndexError):
        orc.floodfill_threshold(data, [(99, 0, 0)], 1, 2, 1, st, out)


def test_floodfill_equal(orc):
    data = np.zeros((3, 4, 5), np.int16); data[1] = 7; data[2, 0, 0] = 7
    out = np.zeros(data.shape, np.uint8)
    orc.floodfill(data, 2, 2, 1, 7, 9, out)
    want = np.zeros(data.shape, np.uint8); want[1] = 9; want[2, 0, 0] = 9
    assert np.array_equal(out, want)
    out = np.zeros(data.shape, np.uint8)
    orc.floodfill(data, 0, 0, 0, 7, 9, out)  # seed marked unconditionally, grows into 7s
    assert out[0, 0, 0] == 9 and out[1, 0, 0] == 9


# ------------------------------------------------------------------ projections (unpinned)
def _mida_numpy(img, axis, wl, ww):
    f = np.float32
    a = np.moveaxis(img, axis, 0).astype(f)
    mn, mx = f(a.min()), f(a.max())
    rng = f(mx - mn)
    inv = f(f(1.0) / rng)
    out = np.zeros(a.shape[1:], f)
    lo, hi = f(f(wl) - f(f(ww) / f(2))), f(f(wl) + f(f(ww) / f(2)))
    for idx in np.ndindex(*a.shape[1:]):
        fmax = ap = cp = fc = f(0)
        for v in a[(slice(None),) + idx]:
            fpi = f(inv * f(v - mn))
            dl = f(0)
            if fpi > fmax:
                dl = f(fpi - fmax); fmax = fpi
            bt = f(f(1) - dl)
            al = f(0) if v < lo else (f(1) if v > hi else f(f(v - lo) / f(hi - lo)))
            one_m = f(f(1) - f(bt * ap))
            c = f(f(bt * cp) + f(f(one_m * fpi) * al))
            ca = f(f(bt * ap) + f(one_m * al))
            cp, ap, fc = c, ca, c
            if ca >= 1:
                break
        out[idx] = f(f(rng * fc) + mn)
    return np.trunc(out).astype(img.dtype)


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_mida_matches_numpy_restatement(orc, axis):
    rng = np.random.default_rng(axis)
    img = rng.integers(-1000, 2000, (5, 6, 7)).astype(np.int16)
    out = np.zeros([(6, 7), (5, 7), (5, 6)][axis], np.int16)
    orc.mida(img, axis, 300, 600, out)
    assert np.array_equal(out, _mida_numpy(img, axis, 300, 600))
    with pytest.raises(TypeError):
        orc.mida(img, axis, 300, 600, out.astype(np.uint8))
    with pytest.raises(ValueError):
        orc.mida(np.zeros((2, 2, 2), np.int16), axis, 1, 1, np.zeros((2, 2), np.int16))  # range == 0 -> NaN


def test_lmip_small(orc):
    img = np.array([0, 800, 900, 850, 2000], np.int16).reshape(5, 1, 1)
    out = np.zeros((1, 1), np.int16)
    orc.lmip(img, 0, 700, 3033, out)
    assert out[0, 0] == 900  # first local max after entering [tmin, tmax]
    orc.lmip(img, 0, 3000, 3033, out)
    assert out[0, 0] == 2000  # never entered the window: plain max


# ---- wider independent cross-checks of the unpinned projections (no reference test exists for them):
# second restatements written from mips.rs in vectorised NumPy float32, compared on larger volumes,
# every dtype pair and axis
def _lmip_numpy(img, axis, tmin, tmax):
    a = np.moveaxis(img, axis, 0)
    tmin, tmax = a.dtype.type(tmin), a.dtype.type(tmax)
    mv = a[0].copy()
    start = (a[0] >= tmin) & (a[0] <= tmax)
    done = np.zeros(mv.shape, bool)
    for v in a:                      # mips.rs:40-66, all rays of a plane at once
        act = ~done
        gt = v > mv
        stop = act & ~gt & (v < mv) & start
        mv = np.where(act & gt, v, mv)
        done |= stop
        start |= act & ~stop & (v >= tmin) & (v <= tmax)
    return mv


def _fcm_numpy(img, n, axis):
    f = np.float32
    def diff(hi, lo):
        if img.dtype == np.float64:
            return (hi - lo).astype(f)
        return (hi.astype(np.int64) - lo.astype(np.int64)).astype(img.dtype).astype(f)   # wraps like the release build
    p = np.pad(img, 1, mode="edge")
    gz = diff(p[2:, 1:-1, 1:-1], p[:-2, 1:-1, 1:-1]) / f(2)
    gy = diff(p[1:-1, 2:, 1:-1], p[1:-1, :-2, 1:-1]) / f(2)
    gx = diff(p[1:-1, 1:-1, 2:], p[1:-1, 1:-1, :-2]) / f(2)
    gm = np.sqrt(((gx * gx).astype(f) + (gy * gy).astype(f)).astype(f) + (gz * gz).astype(f)).astype(f)
    d = [gz, gy, gx][axis]
    with np.errstate(invalid="ignore", divide="ignore"):
        base = (f(1) - np.abs((d / gm).astype(f))).astype(f)
        sf = base if n == 1 else (base * base).astype(f)
        val = np.where(gm == 0, f(0), (gm * sf).astype(f))
    return val.astype(img.dtype) if img.dtype != np.float64 else val.astype(np.float64)


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_projections_against_second_restatements(orc, axis):
    rng = np.random.default_rng(10 + axis)
    shape = (9, 11, 13)
    smooth = ndimage.gaussian_filter(rng.normal(size=shape), 1.0)
    i16 = (smooth / np.abs(smooth).max() * 1800 + 500).astype(np.int16)
    u8 = ((i16.astype(np.int32) + 1400) // 16).clip(0, 255).astype(np.uint8)
    f64 = i16.astype(np.float64) * 0.37
    oshape = [(shape[1], shape[2]), (shape[0], shape[2]), (shape[0], shape[1])][axis]
    # MIDA: (int16,int16) and (uint8,uint8)
    for img, wl, ww in ((i16, 300, 600), (u8, 100, 60)):
        out = np.zeros(oshape, img.dtype)
        orc.mida(img, axis, wl, ww, out)
        assert np.array_equal(out, _mida_numpy(img, axis, wl, ww)), img.dtype
    # LMIP: every image dtype
    for img, tmin, tmax in ((i16, 700, 3033), (u8, 90, 200), (f64, 100.0, 900.0)):
        out = np.zeros(oshape, img.dtype)
        orc.lmip(img, axis, tmin, tmax, out)
        assert np.array_equal(out, _lmip_numpy(img, axis, tmin, tmax)), img.dtype
    # contour volume (mips.rs:170-242) for the exact exponents, every dtype; then its projections
    for img in (i16, u8, f64):
        for n in (1, 2):
            got, want = orc.fcm_volume(img, float(n), axis), _fcm_numpy(img, n, axis)
            if n == 2 and img.dtype == np.float64:
                # powf(x, 2) of glibc (what the reference's f32::powf calls) is faithfully, not correctly,
                # rounded: a few values per thousand sit one float32 ulp from x * x
                ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
                assert (np.abs(got - want) <= ulp).all() and (got != want).mean() < 0.01
            else:
                assert np.array_equal(got, want), (img.dtype, n)
    tmp = _fcm_numpy(i16, 2, axis)
    out = np.zeros(oshape, np.int16)
    orc.fast_countour_mip(i16, 2.0, axis, 300, 600, 0, out)
    assert np.array_equal(out, tmp.max(axis))
    orc.fast_countour_mip(i16, 2.0, axis, 300, 600, 1, out)
    assert np.array_equal(out, _lmip_numpy(tmp, axis, 700, 3033))
    orc.fast_countour_mip(i16, 2.0, axis, 300, 600, 2, out)
    assert np.array_equal(out, _mida_numpy(tmp, axis, 300, 600))


@pytest.mark.parametrize("shape", [(1, 5, 7), (4, 1, 3), (3, 4, 1), (2, 2, 2), (17, 3, 29)])
def test_projection_restatements_agree_on_thin_and_ragged_volumes(orc, shape):
    """Single-plane, single-row, single-column and ragged volumes: the ray loops, the clamped
    differences of the contour volume and the output shapes for every axis."""
    rng = np.random.default_rng(sum(shape))
    i16 = rng.integers(-1000, 3000, shape).astype(np.int16)
    for axis in (0, 1, 2):
        oshape = tuple(s for a, s in enumerate(shape) if a != axis)
        out = np.zeros(oshape, np.int16)
        orc.lmip(i16, axis, 700, 3033, out)
        assert np.array_equal(out, _lmip_numpy(i16, axis, 700, 3033))
        orc.mida(i16, axis, 300, 600, out)
        assert np.array_equal(out, _mida_numpy(i16, axis, 300, 600))
        for n in (1, 2):
            assert np.array_equal(orc.fcm_volume(i16, float(n), axis), _fcm_numpy(i16, n, axis))
