"""The 3-D mask editor on the device against the CPU restatement (oracle/mask_edit.c), bit for bit:
mask_cut, brush_mask_rs, polygon2mask_rs and the fused cut_from_polygons, on strided
[1:, 1:, 1:] views of padded masks written in place, through perspective cameras composed the
way ReceiveVolumeViewerActiveCamera does (perspective . look-at . flip-Y)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ome():
    """The CPU restatement of the mask editor (oracle/mask_edit.c)."""
    from oracle import mask_edit
    mask_edit.lib()
    return mask_edit

SCREENS = [(641, 479), (1920, 1080)]


# ----------------------------------------------------------------------------- scene
def _look_at(eye, target, up):
    f = target - eye
    f = f / np.linalg.norm(f)
    s = np.cross(f, up)
    s = s / np.linalg.norm(s)
    u = np.cross(s, f)
    V = np.eye(4)
    V[0, :3], V[1, :3], V[2, :3] = s, u, -f
    V[:3, 3] = -V[:3, :3] @ eye
    return V


def _perspective(fovy_deg, aspect, near, far):
    t = 1.0 / np.tan(np.radians(fovy_deg) / 2)
    P = np.zeros((4, 4))
    P[0, 0], P[1, 1] = t / aspect, t
    P[2, 2], P[2, 3] = -(far + near) / (far - near), -2 * far * near / (far - near)
    P[3, 2] = -1.0
    return P


def _camera(shape, sp, screen, kind):
    """(world_to_screen, world_to_camera, near, far) for a volume [dz][dy][dx] with spacing (sx, sy, sz).
    'outside': the whole volume in view; 'inside': the eye sits in the volume, part of it behind
    the camera; 'narrow': a small field of view, part of the volume projects off screen."""
    w, h = screen
    ext = np.array([shape[2] * sp[0], -shape[1] * sp[1], shape[0] * sp[2]])
    centre = ext / 2
    size = np.abs(ext).max()
    direction = np.array([0.6, -0.5, 0.62])
    direction /= np.linalg.norm(direction)
    if kind == "inside":
        eye, fov = centre + 0.2 * size * direction, 70.0
    else:
        eye, fov = centre + 2.2 * size * direction, (35.0 if kind == "outside" else 12.0)
    V = _look_at(eye, centre, np.array([0.0, 0.0, 1.0]))
    near, far = 0.01 * size, 4.0 * size
    inv_y = np.eye(4)
    inv_y[1, 1] = -1
    M = _perspective(fov, w / float(h), near, far) @ V
    return np.ascontiguousarray(M @ inv_y), np.ascontiguousarray(V @ inv_y), near, far


def _polygons(screen, seed, k=3, n=64):
    """k star-shaped screen polygons in display pixels, one of them partly off screen."""
    w, h = screen
    rng = np.random.default_rng(seed)
    out = []
    for i in range(k):
        t = np.sort(rng.uniform(0, 2 * np.pi, n))
        r = rng.uniform(0.08, 0.3, n) * min(w, h)
        cx, cy = (rng.uniform(0.3, 0.7) * w, rng.uniform(0.3, 0.7) * h) if i else (0.05 * w, 0.9 * h)
        out.append(np.stack([cx + r * np.cos(t), cy + r * np.sin(t)], 1))
    return out


def _padded(mask, border=255):
    dz, dy, dx = mask.shape
    a = np.full((dz + 1, dy + 1, dx + 1), border, np.uint8)
    a[1:, 1:, 1:] = mask
    return a


def _volumes(cranium, big=False):
    from invesalius3_b200 import phantom
    rng = np.random.default_rng(7)
    yield "7x9x11", _padded((rng.random((7, 9, 11)) < 0.6).astype(np.uint8) * 255), (1.0, 1.2, 1.5)
    v = (rng.random((33, 65, 129)) * 256).astype(np.uint8)
    yield "33x65x129", _padded(v), (0.5, 0.7, 2.0)
    img, sp = cranium["matrix_crop"], tuple(float(s) for s in cranium["spacing"])
    for i in (0, 1):
        lo, hi = cranium[f"thr_{i}"]
        yield f"cranium{i}", _padded(((img >= lo) & (img <= hi)).astype(np.uint8) * 255), sp
    if big:
        ct = phantom.ct((256, 512, 512), seed=3)
        yield "phantom256", _padded(((ct >= 226) & (ct <= 3071)).astype(np.uint8) * 255), (0.48, 0.48, 0.9)


# ----------------------------------------------------------------------------- rasteriser
def test_polygon2mask_matches_checker(ome):
    from invesalius3_b200 import mask_edit as me
    for screen in SCREENS:
        polys = _polygons(screen, 1)
        nan = float("nan")
        polys += [np.array([[10.0, 10.0], [600.0, 12.0], [nan, 400.0], [20.0, 470.0]]),
                  np.array([[-50.0, -20.0], [3000.0, 40.0], [900.0, 2000.0]]),
                  np.array([[100.0, 100.0], [300.0, 100.0], [300.0, 300.0], [100.0, 300.0]]),
                  np.array([[5.0, 5.0], [9.0, 7.0]]),
                  np.asfortranarray(np.array([[40.0, 30.0, 1.0], [400.0, 60.0, 1.0], [120.0, 300.0, 1.0]]))[:, :]]
        t = np.arange(5) * 4 * np.pi / 5
        polys.append(np.stack([320 + 200 * np.sin(t), 240 + 200 * np.cos(t)], 1)[::-1])   # negative strides
        for p in polys:
            got = me.polygon2mask_rs(screen, p)
            want = ome.polygon2mask_rs(screen, p)
            assert got.shape == tuple(screen) and got.dtype == np.bool_
            assert np.array_equal(got, want), (screen, p[:3])


# ----------------------------------------------------------------------------- mask_cut
def _cut_pair(ome, me, padded, sp, screen, kind, mode, depth_val, polys):
    M, MV, near, far = _camera(padded[1:, 1:, 1:].shape, sp, screen, kind)
    depth = near + (far - near) * depth_val
    filt = np.logical_or.reduce([ome.polygon2mask_rs(screen, p) for p in polys]).T
    if mode == 0:
        np.logical_not(filt, out=filt)
    want, got = padded.copy(), padded.copy()
    image = np.zeros((1, 1, 1), np.int16)
    ome.mask_cut(image, *sp, depth, filt, M, MV, want[1:, 1:, 1:], mode)
    me.mask_cut(image, *sp, depth, filt, M, MV, got[1:, 1:, 1:], mode)
    assert np.array_equal(got, want), (screen, kind, mode, depth_val)
    return want, (M, MV, depth)


def test_mask_cut_matches_checker(ome, cranium):
    from invesalius3_b200 import mask_edit as me
    for name, padded, sp in _volumes(cranium):
        changed = 0
        for screen in SCREENS:
            polys = _polygons(screen, 2)
            for kind in ("outside", "inside", "narrow"):
                for mode in (0, 1):
                    want, _ = _cut_pair(ome, me, padded, sp, screen, kind, mode, 0.5 if mode else 1.0, polys)
                    changed += int((want != padded).any())
        assert changed >= 6, name                           # the cameras really cut


def test_mask_cut_large_slab(ome, cranium):
    from invesalius3_b200 import mask_edit as me
    name, padded, sp = list(_volumes(cranium, big=True))[-1]
    assert name == "phantom256"
    for kind, mode in (("inside", 1), ("narrow", 0)):
        want, _ = _cut_pair(ome, me, padded, sp, (1920, 1080), kind, mode, 0.7, _polygons((1920, 1080), 5))
        assert (want != padded).any()
    # brush strokes on the same slab
    rng = np.random.default_rng(9)
    want, got = padded.copy(), padded.copy()
    for mode in (0, 1):
        c = tuple(float(v) for v in rng.uniform(0, 200, 3))
        ome.brush_mask_rs(want[1:, 1:, 1:], None, sp, c, 15.0, mode)
        me.brush_mask_rs(got[1:, 1:, 1:], None, sp, c, 15.0, mode)
    assert np.array_equal(got, want)


def test_fused_cut_equals_the_three_shims(ome, cranium):
    import torch
    from invesalius3_b200 import device as dev, mask_edit as me
    for name, padded, sp in list(_volumes(cranium))[1:3]:
        for screen in SCREENS:
            polys = _polygons(screen, 3) + [np.zeros((0, 2))]
            for kind, mode in (("outside", 0), ("narrow", 1), ("inside", 0)):
                M, MV, near, far = _camera(padded[1:, 1:, 1:].shape, sp, screen, kind)
                depth = near + (far - near) * 0.8
                filt = np.logical_or.reduce([me.polygon2mask_rs(screen, p) for p in polys]).T
                if mode == 0:
                    np.logical_not(filt, out=filt)
                want = padded.copy()
                me.mask_cut(np.zeros((1, 1, 1), np.uint8), *sp, depth, filt, M, MV, want[1:, 1:, 1:], mode)
                o = dev.to_device(padded[1:, 1:, 1:])
                me.cut_from_polygons_device(o, sp, depth, polys, M, MV, mode, screen)
                got = padded.copy()
                dev.to_host(o, got[1:, 1:, 1:])
                assert np.array_equal(got, want), (name, screen, kind, mode)
                host = padded.copy()
                me.cut_from_polygons(host[1:, 1:, 1:], sp, depth, polys, M, MV, mode, screen)
                assert np.array_equal(host, want)
                ref = padded.copy()
                ome.mask_cut(np.zeros((1, 1, 1), np.uint8), *sp, depth, filt, M, MV, ref[1:, 1:, 1:], mode)
                assert np.array_equal(ref, want)
    torch.cuda.synchronize()


def test_mask_cut_device_on_unaligned_and_ragged_buffers(ome):
    import torch
    from invesalius3_b200 import mask_edit as me
    rng = np.random.default_rng(11)
    vol = (rng.random((6, 7, 13)) * 256).astype(np.uint8)                  # 546 voxels: a ragged tail
    M, MV, near, far = _camera(vol.shape, (1.0, 1.0, 1.0), (64, 48), "inside")
    filt = rng.random((48, 64)) < 0.5
    want = vol.copy()
    ome.mask_cut(vol, 1.0, 1.0, 1.0, far, filt, M, MV, want, 0)
    flat = torch.zeros(vol.size + 3, dtype=torch.uint8, device="cuda")
    view = flat[3:].view(vol.shape)                                        # 3 bytes off 16-byte alignment
    view.copy_(torch.from_numpy(vol).cuda())
    me.mask_cut_device(view, (1.0, 1.0, 1.0), far, torch.from_numpy(filt).cuda(), M, MV, 0)
    assert np.array_equal(view.cpu().numpy(), want)


# ----------------------------------------------------------------------------- brush
def test_brush_matches_checker(ome, cranium):
    from invesalius3_b200 import mask_edit as me
    rng = np.random.default_rng(5)
    for name, padded, sp in _volumes(cranium):
        shape = padded[1:, 1:, 1:].shape
        base = _padded((rng.random(shape) * 3).astype(np.uint8) * 120, border=0)
        ext = np.array([shape[2] * sp[0], shape[1] * sp[1], shape[0] * sp[2]])
        centres = [tuple(rng.uniform(-0.1, 1.1, 3) * ext) for _ in range(4)] + [(-30.0, 2.0, 2.0), (float("nan"), 1.0, 1.0)]
        for c in centres:
            for r in (0.0, 2.5, 15.0):
                for mode in (0, 1, 2):
                    for orig in (None, base[1:, 1:, 1:]):
                        want, got = padded.copy(), padded.copy()
                        ome.brush_mask_rs(want[1:, 1:, 1:], orig, sp, c, r, mode)
                        me.brush_mask_rs(got[1:, 1:, 1:], orig, sp, c, r, mode)
                        assert np.array_equal(got, want), (name, c, r, mode, orig is None)


def test_brush_orig_aliasing_out(ome):
    """orig sharing memory with out reads orig as it was before the stroke."""
    from invesalius3_b200 import mask_edit as me
    rng = np.random.default_rng(6)
    a = (rng.random((20, 21, 22)) * 4).astype(np.uint8) * 60
    for orig_of in (lambda x: x[1:, 1:, 1:], lambda x: x[:-1, :-1, :-1]):
        want, got = a.copy(), a.copy()
        snap = orig_of(want).copy()
        ome.brush_mask_rs(want[1:, 1:, 1:], snap, (1.0, 1.0, 1.0), (9.0, 8.0, 10.0), 6.0, 0)
        me.brush_mask_rs(got[1:, 1:, 1:], orig_of(got), (1.0, 1.0, 1.0), (9.0, 8.0, 10.0), 6.0, 0)
        assert np.array_equal(got, want)


def test_brush_moves_only_the_box(ome, monkeypatch):
    from invesalius3_b200 import device as dev, mask_edit as me
    moved = []
    up, down = dev.to_device, dev.to_host

    def spy_up(a, device=None):
        moved.append(("up", a.shape))
        return up(a, device)

    def spy_down(t, out):
        moved.append(("down", out.shape))
        return down(t, out)

    monkeypatch.setattr(dev, "to_device", spy_up)
    monkeypatch.setattr(dev, "to_host", spy_down)
    padded = _padded(np.full((60, 90, 100), 255, np.uint8), border=7)
    orig = _padded(np.full((60, 90, 100), 200, np.uint8), border=0)
    sp, c, r = (0.9, 0.9, 1.5), (40.0, 35.0, 30.0), 15.0
    box = me.brush_box((60, 90, 100), sp, c, r)
    for mode, g in ((1, None), (0, orig[1:, 1:, 1:])):
        moved.clear()
        want = padded.copy()
        ome.brush_mask_rs(want[1:, 1:, 1:], g, sp, c, r, mode)
        me.brush_mask_rs(padded[1:, 1:, 1:], g, sp, c, r, mode)
        assert np.array_equal(padded, want)
        assert moved == [("up", box[3:])] * (1 + (g is not None)) + [("down", box[3:])], moved
        assert np.prod(box[3:]) < 0.1 * 60 * 90 * 100


def test_brush_stroke_path(ome, cranium):
    """100 strokes of radius 15 along a path, alternating reveal (from orig) and erase."""
    from invesalius3_b200 import mask_edit as me
    img, sp = cranium["matrix_crop"], tuple(float(s) for s in cranium["spacing"])
    lo, hi = cranium["thr_1"]
    mask = _padded(((img >= lo) & (img <= hi)).astype(np.uint8) * 255)
    orig = mask.copy()
    mask[1:, 1:, 1:] = 0
    want, got = mask.copy(), mask.copy()
    ext = np.array([img.shape[2] * sp[0], img.shape[1] * sp[1], img.shape[0] * sp[2]])
    for i in range(100):
        t = i / 99.0
        c = tuple(float(v) for v in ext * np.array([0.1 + 0.8 * t, 0.5 + 0.35 * np.sin(6 * t), 0.5 + 0.3 * np.cos(4 * t)]))
        mode = 0 if (i // 10) % 3 else 1
        ome.brush_mask_rs(want[1:, 1:, 1:], orig[1:, 1:, 1:], sp, c, 15.0, mode)
        me.brush_mask_rs(got[1:, 1:, 1:], orig[1:, 1:, 1:], sp, c, 15.0, mode)
    assert np.array_equal(got, want)
    assert (want[1:, 1:, 1:] == 255).sum() > 1000 and (want[0] == 255).all()
