"""CPU suite: the offscreen renderer's source (render.cuh), compiled as plain C++ by tests/hostcheck/render.py, in float64.

It is compared with an independent numpy ray caster built from the oracle's geom_xpos / geom_xmat / geom_size, pinned in closed form
on tests/models/render_pins.xml, and its camera construction, geom_rgba loading and argument checks are covered."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.hostcheck import build as HC
from tests.hostcheck import render as HR
from ur3e_b200 import _lib
from ur3e_b200.batch import default_geoms, make_camera
from ur3e_b200.model import Model

PINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "models", "render_pins.xml")
PLANE, BOX = 0, 6


def _cam(pos, xyaxes, fovy=45.0, znear=0.01, zfar=50.0, objtype=-1, objid=0):
    return make_camera(None, dict(pos=pos, xyaxes=xyaxes, fovy=fovy, znear=znear, zfar=zfar)) if objtype == -1 else _anchored(pos, xyaxes, fovy, znear, zfar, objtype, objid)


def _anchored(pos, xyaxes, fovy, znear, zfar, objtype, objid):
    c = make_camera(None, dict(pos=pos, xyaxes=xyaxes, fovy=fovy, znear=znear, zfar=zfar))
    c.objtype, c.objid = objtype, objid
    return c


def _frame(xyaxes):
    """Camera rotation (columns x, y, z) from MJCF xyaxes."""
    x = np.asarray(xyaxes[:3], float); x = x / np.linalg.norm(x)
    y = np.asarray(xyaxes[3:], float); y = y - (x @ y) * x; y = y / np.linalg.norm(y)
    return np.column_stack([x, y, np.cross(x, y)])


def _reference(gpos, gmat, gsize, gtype, grgb, ids, cpos, cR, fovy, W, H, znear, zfar, jitter=(0.0, 0.0)):
    """Independent numpy ray caster: (rgb, depth, seg) of the geoms `ids` (ascending) from a camera at cpos with rotation cR."""
    ty = np.tan(np.radians(fovy) / 2); tx = ty * W / H
    px, py = np.meshgrid(np.arange(W), np.arange(H))
    xs = (2 * (px + 0.5) / W - 1) * tx + jitter[0]; ys = (1 - 2 * (py + 0.5) / H) * ty + jitter[1]
    d = np.stack([xs, ys, -np.ones_like(xs)], -1) @ cR.T          # t along d is the z-depth
    best = np.full((H, W), float(zfar)); seg = np.full((H, W), -1); cosang = np.zeros((H, W))
    for g in ids:
        R, p, s = gmat[g].reshape(3, 3), gpos[g], gsize[g]
        ol = R.T @ (cpos - p); dl = d @ R
        with np.errstate(divide="ignore", invalid="ignore"):
            if gtype[g] == PLANE:
                t = -ol[2] / dl[..., 2]
                x = ol[0] + t * dl[..., 0]; y = ol[1] + t * dl[..., 1]
                ok = (dl[..., 2] < 0) & ((s[0] <= 0) | (np.abs(x) <= s[0])) & ((s[1] <= 0) | (np.abs(y) <= s[1]))
                nd = -dl[..., 2]
            else:
                t1 = (-s - ol) / dl; t2 = (s - ol) / dl
                lo = np.where(dl == 0, -np.inf, np.minimum(t1, t2)); hi = np.where(dl == 0, np.inf, np.maximum(t1, t2))
                inside = np.all((dl != 0) | (np.abs(ol) <= s), -1)
                ax = np.argmax(lo, -1); t = np.take_along_axis(lo, ax[..., None], -1)[..., 0]
                ok = inside & (t <= hi.min(-1))
                nd = np.abs(np.take_along_axis(dl, ax[..., None], -1)[..., 0])
        ok &= (t >= znear) & (t <= best) & ((seg < 0) | (t < best))
        best = np.where(ok, t, best); seg = np.where(ok, g, seg); cosang = np.where(ok, nd, cosang)
    shade = 0.3 + 0.7 * cosang / np.sqrt(xs ** 2 + ys ** 2 + 1)
    rgb = np.floor(255 * np.clip(grgb[np.maximum(seg, 0)] * shade[..., None], 0, 1) + 0.5).astype(np.uint8)
    rgb[seg < 0] = 0
    return rgb, best, seg


def _oracle_scene(path, qpos):
    m = O.Model(path); d = O.Data(m)
    d.reset(); d.set_state(qpos, np.zeros(m.nv)); d.forward()
    return m, d, d.arr("geom_xpos").reshape(-1, 3), d.arr("geom_xmat").reshape(-1, 9), np.asarray(m.py["geom_size"]).reshape(-1, 3), np.asarray(m.py["geom_type"])


def _compare(path, qpos, cam, cpos, cR, ids, W, H, rgba=None):
    """Host render against the numpy reference: exact seg / rgb and depth to 1e-9 off silhouette edges; returns the edge fraction."""
    m, d, gpos, gmat, gsize, gtype = _oracle_scene(path, qpos)
    grgb = np.zeros((len(gtype), 3))
    col = np.asarray(Model(path).array("geom_rgba")).reshape(-1, 4) if rgba is None else None
    for i, g in enumerate(ids):
        grgb[g] = np.float32(rgba[i][:3] if rgba is not None else col[g][:3])
    rgb, depth, seg, _ = HR.render(path, qpos, cam, ids, W, H, rgba)
    args = (gpos, gmat, gsize, gtype, grgb, sorted(ids), cpos, cR, cam.fovy, W, H, cam.znear, cam.zfar)
    r_rgb, r_depth, r_seg = _reference(*args)
    edge = np.zeros((H, W), bool)
    for j in ((1e-6, 0), (-1e-6, 0), (0, 1e-6), (0, -1e-6)):
        j_rgb, _, j_seg = _reference(*args, jitter=j)
        edge |= (j_seg != r_seg) | np.any(j_rgb != r_rgb, -1)
    ok = ~edge
    assert np.array_equal(seg[ok], r_seg[ok])
    assert np.array_equal(rgb[ok], r_rgb[ok])
    assert np.abs(depth[ok] - r_depth[ok]).max() < 1e-9
    assert len(np.unique(r_seg)) >= 3, "the view shows too little of the scene to test anything"
    return edge.mean()


def _state(m, rng, xml):
    qp = m.key("down")[0].copy()
    qp[:6] += rng.uniform(-0.3, 0.3, 6)
    qp[6] = qp[10] = rng.uniform(0, 0.5)
    if xml == "main.xml":
        q = np.array([1.0, *rng.uniform(-0.4, 0.4, 3)])
        qp[17:21] = q / np.linalg.norm(q)
    return qp


@pytest.mark.parametrize("xml", ["main.xml", "ur3e_2f85.xml"])
def test_render_matches_numpy_reference_f64(assets, xml, capsys):
    path = assets + "/" + xml
    om = O.Model(path); model = Model(path); rng = np.random.default_rng(5)
    ids = default_geoms(model)
    rgba = rng.uniform(0.2, 1.0, (len(ids), 4)).astype(np.float32)   # distinct colours: the assets carry none
    tcp = model.name2id(_lib.OBJ_SITE, "tcp")
    fracs, wrist = [], 0
    for trial in range(3):
        qp = _state(om, rng, xml)
        # world camera (lookat form) over the arm
        cfg = dict(lookat=(0.25, 0.15, 0.15), distance=1.2, azimuth=90 + 30 * trial, elevation=-35.0, fovy=50.0)
        cam = make_camera(model, cfg)
        fracs.append(_compare(path, qp, cam, np.array(cam.pos[:]), _frame(cam.xyaxes[:]), ids, 48, 40, rgba))
        # wrist camera on tcp, looking along the site's +z (between the fingers) from 0.1 m back
        xyaxes = (0, 1, 0, 1, 0, 0)
        cam = _cam((0, 0, -0.1), xyaxes, fovy=70.0, objtype=_lib.OBJ_SITE, objid=tcp)
        _, d, *_ = _oracle_scene(path, qp)
        sp, sR = d.arr("site_xpos").reshape(-1, 3)[tcp], d.arr("site_xmat").reshape(-1, 3, 3)[tcp]
        try:
            fracs.append(_compare(path, qp, cam, sp + sR @ np.array([0, 0, -0.1]), sR @ _frame(xyaxes), ids, 40, 32, rgba))
            wrist += 1
        except AssertionError as e:   # a wrist view of one geom alone tests little; at least one of the three must show more
            if "too little" not in str(e):
                raise
    with capsys.disabled():
        print("\n%s: silhouette-edge pixel fractions %s" % (xml, ["%.4f" % f for f in fracs]))
    assert wrist >= 1 and max(fracs) < 0.05


def _pin_scene():
    model = Model(PINS)
    g = {n: model.name2id(_lib.OBJ_GEOM, n) for n in ("floor", "box", "lid", "hidden")}
    return model, g


def _down(h, fovy=45.0, **kw):
    # camera above the box's centre looking straight down: x right = world +x, y up = world +y
    return _cam((0.1, -0.05, h), (1, 0, 0, 0, 1, 0), fovy=fovy, **kw)


@pytest.mark.parametrize("fovy", [10.0, 45.0, 120.0])
def test_render_pins_top_down(fovy):
    model, g = _pin_scene()
    ids = default_geoms(model)
    assert g["hidden"] not in ids and sorted(ids) == sorted([g["floor"], g["box"], g["lid"]])
    h, W, H = 2.0, 33, 21
    rgb, depth, seg, _ = HR.render(PINS, np.zeros(1), _down(h, fovy), ids, W, H)
    assert not np.any(seg == g["lid"])                        # the lid faces down: its back side is towards the camera
    floor = seg == g["floor"]
    assert np.all(depth[floor] == h)                          # z-depth, not ray length: exactly h at any fovy
    # silhouette: the pixel centres whose ray meets the box top (z = 0.04) inside its rectangle, computed by hand
    ty = np.tan(np.radians(fovy) / 2); tx = ty * W / H
    px, py = np.meshgrid(np.arange(W), np.arange(H))
    x = (2 * (px + 0.5) / W - 1) * tx * (h - 0.04); y = (1 - 2 * (py + 0.5) / H) * ty * (h - 0.04)
    assert np.minimum(np.abs(np.abs(x) - 0.1), np.abs(np.abs(y) - 0.05)).min() > 1e-9    # no pixel centre on the boundary
    inside = (np.abs(x) <= 0.1) & (np.abs(y) <= 0.05)
    assert inside.any() or fovy == 120.0
    assert np.array_equal(seg == g["box"], inside)
    assert np.array_equal(floor, ~inside)
    assert np.abs(depth[inside] - (h - 0.04)).max() < 1e-12
    # head-on: the centre pixel's ray is the view axis, so red (1, 0, 0) shades to (255, 0, 0); the floor is blue (top default)
    if inside[H // 2, W // 2]:
        assert tuple(rgb[H // 2, W // 2]) == (255, 0, 0)
    assert np.all(rgb[floor][:, :2] == 0) and np.all(rgb[floor][:, 2] >= 255 * 0.3)
    # an rgba override, in the caller's geom order
    order = [g["lid"], g["box"], g["floor"]]
    rgba = [(0, 0, 0, 1), (0, 1, 0, 1), (1, 1, 1, 1)]
    rgb2, _, seg2, _ = HR.render(PINS, np.zeros(1), _down(h, fovy), order, W, H, rgba)
    assert np.array_equal(seg2, seg)
    if inside[H // 2, W // 2]:
        assert tuple(rgb2[H // 2, W // 2]) == (0, 255, 0)


def test_render_pins_front_plane_and_clipping():
    model, g = _pin_scene()
    ids = default_geoms(model)
    W, H = 25, 25
    # from below the lid looking up (+z): its front side, a 0.6 m square at distance 0.2; the rest misses
    up = _cam((0, 0, 0.3), (1, 0, 0, 0, -1, 0), fovy=90.0, zfar=7.0)
    rgb, depth, seg, _ = HR.render(PINS, np.zeros(1), up, ids, W, H)
    ty = 1.0
    c = (2 * (np.arange(W) + 0.5) / W - 1) * ty * 0.2
    inside = (np.abs(c)[None, :] <= 0.3) & (np.abs(c)[:, None] <= 0.3)
    assert np.array_equal(seg == g["lid"], inside) and np.all(seg[~inside] == -1)
    assert np.abs(depth[inside] - 0.2).max() < 1e-12 and np.all(depth[~inside] == 7.0) and np.all(rgb[~inside] == 0)
    # zfar: everything beyond it is background at depth zfar
    rgb, depth, seg, _ = HR.render(PINS, np.zeros(1), _down(2.0, zfar=1.5), ids, W, H)
    assert np.all(seg == -1) and np.all(depth == 1.5) and np.all(rgb == 0)
    # znear: the box top (1.96 m) is ignored, the floor (2 m) is not
    _, depth, seg, _ = HR.render(PINS, np.zeros(1), _down(2.0, znear=1.99), ids, W, H)
    assert np.all(seg == g["floor"]) and np.all(depth == 2.0)


def test_render_camera_forms():
    model = Model(PINS)
    ids = default_geoms(model)
    lookat, dist, az, el = np.array([0.1, -0.05, 0.0]), 1.5, 60.0, -50.0
    cam = make_camera(model, dict(lookat=lookat, distance=dist, azimuth=az, elevation=el))
    a, e = np.radians(az), np.radians(el)
    f = np.array([np.cos(e) * np.cos(a), np.cos(e) * np.sin(a), np.sin(e)])
    up = np.array([-np.sin(e) * np.cos(a), -np.sin(e) * np.sin(a), np.cos(e)])
    pos, xyaxes = lookat - dist * f, np.concatenate([np.cross(f, up), up])
    assert np.allclose(cam.pos[:], pos, atol=1e-15) and np.allclose(cam.xyaxes[:], xyaxes, atol=1e-15)
    assert (cam.fovy, cam.objtype) == (45.0, -1)
    assert np.allclose(_frame(cam.xyaxes[:])[:, 2], -f)          # the view (-z) is the forward direction
    explicit = _cam(pos, xyaxes)
    r1, r2 = HR.render(PINS, np.zeros(1), cam, ids, 30, 20), HR.render(PINS, np.zeros(1), explicit, ids, 30, 20)
    for x, y in zip(r1, r2):
        assert np.array_equal(x, y)
    assert np.any(r1[2] == model.name2id(_lib.OBJ_GEOM, "box"))


@pytest.mark.parametrize("kind", ["site", "body"])
def test_render_attached_camera_equals_world_camera(assets, kind):
    """An attached camera renders what a world camera at the anchor pose (from the kinematics query) renders."""
    path = assets + "/main.xml"
    model = Model(path); om = O.Model(path); rng = np.random.default_rng(2)
    ids = default_geoms(model)
    rgba = rng.uniform(0.2, 1.0, (len(ids), 4))
    qp = _state(om, rng, "main.xml")
    t, name = (_lib.OBJ_SITE, "tcp") if kind == "site" else (_lib.OBJ_XBODY, "wrist_3_link")
    i = model.name2id(_lib.OBJ_SITE if kind == "site" else _lib.OBJ_BODY, name)
    pos_l, xy_l = np.array([0.02, -0.01, -0.15]), np.array([0, 1, 0.1, 1, 0, 0])
    p, R, _ = HC.query(path, qp, np.zeros(om.nv), [t], [i])
    att = make_camera(model, {"pos": pos_l, "xyaxes": xy_l, kind: name, "fovy": 80.0})
    assert (att.objtype, att.objid) == (t, i)
    world = _cam(p[0] + R[0] @ pos_l, np.concatenate([R[0] @ xy_l[:3], R[0] @ xy_l[3:]]), fovy=80.0)
    a_rgb, a_depth, a_seg, _ = HR.render(path, qp, att, ids, 40, 30, rgba)
    w_rgb, w_depth, w_seg, _ = HR.render(path, qp, world, ids, 40, 30, rgba)
    same = a_seg == w_seg
    assert same.mean() > 0.98 and len(np.unique(a_seg)) >= 2
    assert np.abs(a_depth[same] - w_depth[same]).max() < 1e-9
    assert np.abs(a_rgb[same].astype(int) - w_rgb[same]).max() <= 1


def test_geom_rgba_loader(assets):
    m = Model(assets + "/main.xml")
    col = np.asarray(m.array("geom_rgba")).reshape(-1, 4)
    assert col.shape == (m.ngeom, 4) and np.all(col == [0.5, 0.5, 0.5, 1.0])          # MuJoCo's default: no rgba in the asset
    m = Model(PINS)
    col = np.asarray(m.array("geom_rgba")).reshape(-1, 4)
    want = dict(floor=(0, 0, 1, 1), box=(1, 0, 0, 1), lid=(0, 1, 0, 1), hidden=(1, 1, 1, 0))
    for n, c in want.items():
        assert tuple(col[m.name2id(_lib.OBJ_GEOM, n)]) == c, n                      # the lid inherits "green" through "thin"
    assert np.allclose(np.asarray(m.array("geom_size")).reshape(-1, 3)[m.name2id(_lib.OBJ_GEOM, "lid")], (0.3, 0.3, 0.01))


def test_render_argument_checks():
    model, g = _pin_scene()
    ok = _down(2.0)
    cases = [
        (None, [0], 8, 8, "null camera"),
        (_anchored((0, 0, 0), (1, 0, 0, 0, 1, 0), 45, 0.01, 10, 5, 0), [0], 8, 8, "objtype 5"),
        (_anchored((0, 0, 0), (1, 0, 0, 0, 1, 0), 45, 0.01, 10, _lib.OBJ_SITE, 9), [0], 8, 8, "id 9 is out of range"),
        (_anchored((0, 0, 0), (1, 0, 0, 0, 1, 0), 45, 0.01, 10, _lib.OBJ_XBODY, -1), [0], 8, 8, "id -1 is out of range"),
        (ok, [], 8, 8, "k=0"),
        (ok, [0] * 257, 8, 8, "k=257"),
        (ok, [0, 4], 8, 8, "id 4 is out of range"),
        (ok, [0], 0, 8, "image size"),
        (ok, [0], 8, 2049, "image size"),
        (_down(2.0, fovy=0.0), [0], 8, 8, "fovy"),
        (_down(2.0, fovy=180.0), [0], 8, 8, "fovy"),
        (_down(2.0, znear=0.0), [0], 8, 8, "znear"),
        (_down(2.0, znear=2.0, zfar=2.0), [0], 8, 8, "znear"),
        (_cam((0, 0, 1), (1, 0, 0, 2, 0, 0)), [0], 8, 8, "parallel"),
    ]
    for cam, ids, W, H, msg in cases:
        with pytest.raises(ValueError, match=msg):
            HR.render(PINS, np.zeros(1), cam, ids, W, H)
    # the call's checks
    assert HR.render_check(0, 1, True, 4, 4, False) == ""
    assert HR.render_check(0, 1, True, 2, 4, True) == ""
    for args, msg in [((1, 1, True, 4, 4, False), "unknown render id 1"), ((-1, 1, True, 4, 4, False), "unknown render id -1"),
                      ((0, 1, False, 4, 4, False), "all outputs are null"), ((0, 1, True, 0, 4, True), "m=0"),
                      ((0, 1, True, 3, 4, False), "not the batch size")]:
        assert msg in HR.render_check(*args)
