"""CPU-only checks of invesalius3_b200.mask_edit: every argument error the crate raises (or
panics on) comes out as the mapped exception before any device work, and the brush's box is
computed on the host."""
import numpy as np
import pytest


@pytest.fixture
def me(monkeypatch):
    from invesalius3_b200 import device, mask_edit

    def no_device(*a, **k):
        raise AssertionError("device work before the argument checks")

    for name in ("to_device", "to_host", "to_numpy", "require_cuda"):
        monkeypatch.setattr(device, name, no_device)
    return mask_edit


def _cut_args(**kw):
    a = dict(image=np.zeros((2, 3, 4), np.int16), sx=1.0, sy=1.0, sz=1.0, max_depth=10.0,
             mask=np.zeros((5, 6), bool).T, m=np.eye(4), mv=np.eye(4), out=np.zeros((3, 4, 5), np.uint8)[1:, 1:, 1:],
             edit_mode=0)
    a.update(kw)
    return a


@pytest.mark.parametrize("kw, exc", [
    (dict(out=np.zeros((2, 3, 4), np.int16)), TypeError),
    (dict(out=np.zeros((2, 3), np.uint8)), TypeError),
    (dict(out=np.zeros((2, 3, 4), np.uint8)[None]), TypeError),
    (dict(mask=np.zeros((5, 6), np.uint8)), TypeError),
    (dict(mask=np.zeros((5, 6, 1), bool)), TypeError),
    (dict(m=np.eye(4, dtype=np.float32)), TypeError),
    (dict(m=np.eye(4).reshape(16)), TypeError),
    (dict(m=np.eye(4).T), ValueError),                 # as_slice().unwrap() on a non-standard layout
    (dict(mv=np.eye(3)), ValueError),                  # from_row_slice needs 16 values
    (dict(mv=np.zeros((4, 5))[:, :4]), ValueError),
    (dict(edit_mode=2 ** 31), OverflowError),
    (dict(edit_mode=-(2 ** 31) - 1), OverflowError),
    (dict(edit_mode=0.5), TypeError),
    (dict(image=np.zeros((2, 3, 4), np.float32)), TypeError),
    (dict(image=np.zeros((2, 3), np.int16)), TypeError),
    (dict(sx="1"), TypeError),
])
def test_mask_cut_argument_errors(me, kw, exc):
    with pytest.raises(exc):
        me.mask_cut(**_cut_args(**kw))


def test_mask_cut_read_only_out(me):
    out = np.zeros((3, 4, 5), np.uint8)
    out.flags.writeable = False
    with pytest.raises(ValueError):
        me.mask_cut(**_cut_args(out=out))


@pytest.mark.parametrize("shape, poly, exc", [
    ((-1, 4), np.zeros((3, 2)), OverflowError),
    ((4, -1), np.zeros((3, 2)), OverflowError),
    ((4.0, 4), np.zeros((3, 2)), TypeError),
    ((4, 4, 4), np.zeros((3, 2)), TypeError),
    ((4, 4), np.zeros((3, 1)), ValueError),            # r[1] panics
    ((4, 4), np.zeros((3, 2), np.float32), TypeError),
    ((4, 4), np.zeros(6), TypeError),
    ((4, 4), [[0.0, 1.0]], TypeError),
])
def test_polygon2mask_argument_errors(me, shape, poly, exc):
    with pytest.raises(exc):
        me.polygon2mask_rs(shape, poly)


def test_polygon2mask_trivial_results_need_no_device(me):
    assert me.polygon2mask_rs((3, 4), np.zeros((0, 2))).shape == (3, 4)
    assert me.polygon2mask_rs((3, 4), np.zeros((0, 1))).dtype == np.bool_     # no row: no panic
    assert me.polygon2mask_rs((0, 4), np.ones((3, 2))).shape == (0, 4)


def _brush_args(**kw):
    a = dict(out=np.zeros((9, 9, 9), np.uint8)[1:, 1:, 1:], orig=None, spacing=(1.0, 1.0, 1.0), center=(4.0, 4.0, 4.0),
             radius=2.0, edit_mode=0)
    a.update(kw)
    return a


@pytest.mark.parametrize("kw, exc", [
    (dict(out=np.zeros((8, 8, 8), np.int16)), TypeError),
    (dict(out=np.zeros((8, 8), np.uint8)), TypeError),
    (dict(orig=np.zeros((8, 8, 8), np.int16)), TypeError),
    (dict(orig=np.zeros((8, 8), np.uint8)), TypeError),
    (dict(orig=np.zeros((8, 8, 5), np.uint8)), ValueError),      # box reaches x = 6
    (dict(spacing=(1.0, 1.0)), TypeError),
    (dict(center=(1.0, 1.0, 1.0, 1.0)), TypeError),
    (dict(center=5.0), TypeError),
    (dict(edit_mode=2 ** 40), OverflowError),
    (dict(edit_mode=1.0), TypeError),
])
def test_brush_argument_errors(me, kw, exc):
    with pytest.raises(exc):
        me.brush_mask_rs(**_brush_args(**kw))


def test_brush_without_work_stays_on_the_host(me):
    a = _brush_args()
    me.brush_mask_rs(**{**a, "edit_mode": 2})                         # any other mode: nothing
    me.brush_mask_rs(**{**a, "center": (50.0, 4.0, 4.0)})             # empty box
    me.brush_mask_rs(**{**a, "spacing": (-1.0, 1.0, 1.0), "center": (-4.0, 4.0, 4.0)})   # min 6 > max 2
    me.brush_mask_rs(**{**a, "out": np.zeros((0, 4, 4), np.uint8)})
    assert not a["out"].any()


def test_brush_box_matches_the_crate_arithmetic():
    from invesalius3_b200.mask_edit import brush_box
    assert brush_box((10, 20, 30), (1.0, 1.0, 2.0), (5.0, 5.0, 5.0), 3.0) == (1, 2, 2, 4, 7, 7)
    assert brush_box((10, 20, 30), (1.0, 1.0, 1.0), (float("nan"), 5.0, 5.0), 3.0)[5] == 1   # NaN -> [0, 0]
    assert brush_box((10, 20, 30), (1.0, 1.0, 1.0), (1e30, 5.0, 5.0), 3.0) == (0,) * 6       # saturates: empty
    assert brush_box((10, 20, 30), (1.0, 1.0, 1.0), (28.5, 18.5, 9.5), 3.0) == (6, 15, 25, 4, 5, 5)
    assert brush_box((0, 20, 30), (1.0, 1.0, 1.0), (5.0, 5.0, 5.0), 3.0) == (0,) * 6


@pytest.mark.parametrize("polys, exc", [
    ([], ValueError),
    ([np.zeros((3, 1))], ValueError),
    ([np.zeros((3, 2), np.float32)], TypeError),
])
def test_fused_cut_argument_errors(me, polys, exc):
    a = _cut_args()
    with pytest.raises(exc):
        me.cut_from_polygons(a["out"], (1.0, 1.0, 1.0), 1.0, polys, a["m"], a["mv"], 0, (6, 5))
