"""CPU suite: the narrow phase's box_box and plane_box (engine.cuh), compiled as plain C++ by tests/hostcheck in float64 and float32,
against an exact geometric reference that shares nothing with the kernel's rule: the penetration depth and the separating normal of two
boxes are the nearest facet of the convex hull of the 64 vertex differences (box 2 minus box 1), and a contact must sit on both
boxes' surfaces.  Closed-form pins (stacks, the 45-degree octagon, crossed edges, a box inside a box, the margin), properties over
random penetrating pairs, and a sweep of nearly parallel face-on-face stacks, where contacts used to be reported off both boxes."""
import os

import numpy as np
import pytest
from scipy.spatial import ConvexHull
from scipy.spatial.transform import Rotation

from tests.hostcheck import build as HC

PRECISIONS = [pytest.param(False, id="f64"), pytest.param(True, id="f32")]
SURF_TOL = {False: 1e-9, True: 1e-5}   # metres: how far a contact may sit from the surface it belongs to
CORNERS = np.array([[i, j, k] for k in (-1, 1) for j in (-1, 1) for i in (-1, 1)], dtype=np.float64)   # plane_box's corner order


def vertices(p, R, s):
    return CORNERS * s @ R.T + p


def reference(p1, R1, s1, p2, R2, s2):
    """(pen, normal from box 1 to box 2, gap) of two boxes: the Minkowski difference B2 - B1 is the hull of the 64 vertex differences;
    pen is its nearest facet's offset from the origin (> 0 when the boxes overlap), the normal minus that facet's outward normal,
    gap how much farther the nearest facet with another normal is (coplanar triangles of qhull merged)."""
    hull = ConvexHull((vertices(p2, R2, s2)[:, None, :] - vertices(p1, R1, s1)[None, :, :]).reshape(-1, 3))
    nrm, off = hull.equations[:, :3], -hull.equations[:, 3]
    i = int(np.argmin(off))
    other = np.linalg.norm(nrm - nrm[i], axis=1) > 1e-9
    return off[i], -nrm[i], off[other].min() - off[i]


def off_surface(x, p, R, s):
    """Distance from x to the surface of the box (p, R, s), in the box's own frame."""
    l = np.abs((x - p) @ R)
    return np.linalg.norm(np.maximum(l - s, 0)) if (l > s).any() else np.min(s - l)


def surface_error(c, boxes):
    """Largest distance of a manifold's points from the surfaces they belong to: pos - dist/2 n on box 1, pos + dist/2 n on box 2."""
    n, nrm, pos, dist = c
    (p1, R1, s1), (p2, R2, s2) = boxes
    return max([max(off_surface(pos[k] - dist[k] / 2 * nrm, p1, R1, s1), off_surface(pos[k] + dist[k] / 2 * nrm, p2, R2, s2)) for k in range(n)],
               default=0.0)


def same_set(a, b, tol):
    """Two point sets [n, 3] equal up to order."""
    return len(a) == len(b) and all(np.linalg.norm(b - x, axis=1).min() <= tol for x in a) and all(np.linalg.norm(a - x, axis=1).min() <= tol for x in b)


def rot(rng):
    return Rotation.random(random_state=rng).as_matrix()


def signed_permutation(rng):
    """A proper signed permutation P (det +1): R -> R P relabels a box's axes, its half-sizes become P^T s up to sign."""
    P = np.eye(3)[:, rng.permutation(3)] * rng.choice([-1.0, 1.0], 3)
    if np.linalg.det(P) < 0:
        P[:, 0] *= -1
    return P


def rot_z(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, -s, 0], [s, c, 0], [0, 0, 1.0]])


def rot_x(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[1.0, 0, 0], [0, c, -s], [0, s, c]])


def rot_y(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, 0, s], [0, 1.0, 0], [-s, 0, c]])


def in_world(W, t, p1, R1, p2, R2):
    """Both boxes moved by the same rigid motion (W, t)."""
    return W @ p1 + t, W @ R1, W @ p2 + t, W @ R2


# ---------------------------------------------------------------- closed-form pins
W0 = Rotation.from_rotvec([0.3, -0.7, 0.4]).as_matrix()   # a world frame with no axis along a coordinate axis
T0 = np.array([0.11, -0.23, 0.37])


def _stack(s1, s2, off, pen):
    """Box 2 on box 1's +z face, its centre at (off, top of box 1 + s2z - pen) in box 1's frame, both boxes axis-aligned there."""
    return np.zeros(3), np.eye(3), np.array([off[0], off[1], s1[2] + s2[2] - pen]), np.eye(3)


@pytest.mark.parametrize("use_float", PRECISIONS)
@pytest.mark.parametrize("off", [(0.0, 0.0), (0.04, -0.03)], ids=["aligned", "offset"])
def test_stack_face_on_face(use_float, off):
    """4 points at the corners of the overlap rectangle on box 1's top face, at mid-penetration, dist = -pen, normal = box 1's +z."""
    s1, s2, pen = np.array([0.05, 0.04, 0.02]), np.array([0.03, 0.02, 0.01]), 1e-3
    p1, R1, p2, R2 = _stack(s1, s2, off, pen)
    lo, hi = np.maximum(-s1[:2], np.array(off) - s2[:2]), np.minimum(s1[:2], np.array(off) + s2[:2])
    corners = np.array([[x, y, s1[2] - pen / 2] for x in (lo[0], hi[0]) for y in (lo[1], hi[1])])
    q1, M1, q2, M2 = in_world(W0, T0, p1, R1, p2, R2)
    n, nrm, pos, dist = HC.box_box(q1, M1, s1, q2, M2, s2, use_float=use_float)
    tol = 1e-12 if not use_float else 2e-7
    assert n == 4
    np.testing.assert_allclose(nrm, W0[:, 2], atol=tol)
    np.testing.assert_allclose(dist, -pen, atol=tol)
    assert same_set(pos, corners @ W0.T + T0, tol)


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_octagon_fills_the_stage(use_float):
    """Two equal squares, one turned 45 degrees about the stack axis: the overlap is a regular octagon, 8 points at its vertices, which
    is STAGE_PTS, the most a pair can emit."""
    a, h, pen = 0.05, 0.02, 1e-3
    s = np.array([a, a, h])
    p1, R1, p2, _ = _stack(s, s, (0, 0), pen)
    R2 = rot_z(np.pi / 4)
    b = a * (np.sqrt(2) - 1)
    octagon = np.array([[x, y, h - pen / 2] for x, y in ((a, b), (b, a), (-b, a), (-a, b), (-a, -b), (-b, -a), (b, -a), (a, -b))])
    q1, M1, q2, M2 = in_world(W0, T0, p1, R1, p2, R2)
    n, nrm, pos, dist = HC.box_box(q1, M1, s, q2, M2, s, use_float=use_float)
    tol = 1e-12 if not use_float else 2e-7
    assert n == 8
    np.testing.assert_allclose(nrm, W0[:, 2], atol=tol)
    np.testing.assert_allclose(dist, -pen, atol=tol)
    assert same_set(pos, octagon @ W0.T + T0, tol)


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_crossed_edges(use_float):
    """Box 1 on an edge along x, box 2 on an edge along y, pressed together: one point at the midpoint of the crossing, the exact
    depth, the normal along the common perpendicular of the two edges."""
    s1, s2, pen = np.array([0.04, 0.02, 0.02]), np.array([0.015, 0.03, 0.015]), 2e-3
    R1, R2 = rot_x(np.pi / 4), rot_y(np.pi / 4)
    top1, bottom2 = s1[1] * np.sqrt(2), s2[0] * np.sqrt(2)   # box 1's top edge and box 2's bottom edge, above / below their centres
    p1 = np.zeros(3)
    p2 = np.array([0.01, -0.005, top1 + bottom2 - pen])      # box 2's edge runs along y through x = 0.01
    q1, M1, q2, M2 = in_world(W0, T0, p1, R1, p2, R2)
    n, nrm, pos, dist = HC.box_box(q1, M1, s1, q2, M2, s2, use_float=use_float)
    tol = 1e-12 if not use_float else 2e-7
    assert n == 1
    np.testing.assert_allclose(nrm, W0[:, 2], atol=tol)
    np.testing.assert_allclose(dist, [-pen], atol=tol)
    np.testing.assert_allclose(pos[0], W0 @ np.array([0.01, 0, top1 - pen / 2]) + T0, atol=tol)
    assert reference(q1, M1, s1, q2, M2, s2)[0] == pytest.approx(pen, abs=1e-12)


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_box_inside_box(use_float):
    """A small box wholly inside a large one is pushed out through the nearest face: its 4 corners on that side, dist = -pen."""
    s1, s2, c = np.array([0.1, 0.1, 0.1]), np.array([0.01, 0.02, 0.005]), np.array([0.02, -0.03, 0.05])
    pen = s1[2] - (c[2] - s2[2])   # 0.055, less than the 0.09 needed along x or y
    q1, M1, q2, M2 = in_world(W0, T0, np.zeros(3), np.eye(3), c, np.eye(3))
    n, nrm, pos, dist = HC.box_box(q1, M1, s1, q2, M2, s2, use_float=use_float)
    tol = 1e-12 if not use_float else 2e-7
    assert n == 4
    np.testing.assert_allclose(nrm, W0[:, 2], atol=tol)
    np.testing.assert_allclose(dist, -pen, atol=tol)
    corners = np.array([[x, y, s1[2] - pen / 2] for x in (c[0] - s2[0], c[0] + s2[0]) for y in (c[1] - s2[1], c[1] + s2[1])])
    assert same_set(pos, corners @ W0.T + T0, tol)
    rp, rn, _ = reference(q1, M1, s1, q2, M2, s2)
    assert rp == pytest.approx(pen, abs=1e-12) and np.allclose(rn, W0[:, 2], atol=1e-12)


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_gap_around_margin(use_float):
    """Separated by a gap g: 4 points with dist = g just inside the margin, none just outside."""
    s1, s2, margin = np.array([0.05, 0.04, 0.02]), np.array([0.03, 0.02, 0.01]), 1e-3
    for g, want in ((margin * (1 - 1e-3), 4), (margin * (1 + 1e-3), 0)):
        q1, M1, q2, M2 = in_world(W0, T0, *_stack(s1, s2, (0.01, 0.005), -g))
        n, nrm, pos, dist = HC.box_box(q1, M1, s1, q2, M2, s2, margin=margin, use_float=use_float)
        assert n == want, g
        if want:
            tol = 1e-12 if not use_float else 2e-7
            np.testing.assert_allclose(dist, g, atol=tol)
            np.testing.assert_allclose(nrm, W0[:, 2], atol=tol)


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_plane_box(use_float):
    """Corners below the plane (or within the margin above it) whose offset from the box centre does not point up, the first 4 in
    corner order, each at the middle of its penetration: pos = corner - dist/2 n."""
    s = np.array([0.03, 0.02, 0.01])
    tol = 1e-12 if not use_float else 2e-7

    def check(P, Rb, c, margin, want_idx):
        pp, n_ = T0, P[:, 2]
        bpos = pp + P @ c
        bmat = P @ Rb
        n, nrm, pos, dist = HC.plane_box(pp, P, bpos, bmat, s, margin=margin, use_float=use_float)
        corners = vertices(bpos, bmat, s)[want_idx]
        d = (corners - pp) @ n_
        assert n == len(want_idx)
        if n:
            np.testing.assert_allclose(nrm, n_, atol=tol)
            np.testing.assert_allclose(dist, d, atol=tol)
            np.testing.assert_allclose(pos, corners - d[:, None] / 2 * n_, atol=tol)
        return d

    pen = 1e-3
    d = check(W0, np.eye(3), np.array([0.01, 0.02, s[2] - pen]), 0.0, [0, 1, 2, 3])   # resting: the 4 bottom corners
    np.testing.assert_allclose(d, -pen, atol=tol)
    th = 0.3                                                                          # tilted about y: the edge of corners 0, 2
    low = s[0] * np.sin(th) + s[2] * np.cos(th)
    d = check(W0, rot_y(-th), np.array([0, 0, low - pen]), 0.0, [0, 2])
    np.testing.assert_allclose(d, -pen, atol=tol)
    check(W0, np.eye(3), np.array([0, 0, s[2] + 4e-4]), 5e-4, [0, 1, 2, 3])          # within the margin above the plane
    check(W0, np.eye(3), np.array([0, 0, s[2] + 6e-4]), 5e-4, [])                    # beyond it
    # on an edge (45 degrees about x, half-sizes y = z, exact in both precisions): corners 0, 1 below, 2..5 level with the centre
    # and within the margin, 6, 7 above it: the first 4 in corner order
    se = np.array([0.03, 0.02, 0.02])
    s[:] = se
    R45 = np.array([[1, 0, 0], [0, np.sqrt(0.5), -np.sqrt(0.5)], [0, np.sqrt(0.5), np.sqrt(0.5)]])
    check(np.eye(3), R45, np.array([0, 0, 1e-3]), 2e-3, [0, 1, 2, 3])


# ---------------------------------------------------------------- properties over random penetrating pairs
def _random_pairs(seed, count):
    """count penetrating pairs (pen > 1e-6): sizes 5 mm - 10 cm, random orientations and offsets."""
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < count:
        s1, s2 = rng.uniform(0.005, 0.1, 3), rng.uniform(0.005, 0.1, 3)
        R1, R2, p1 = rot(rng), rot(rng), rng.uniform(-0.1, 0.1, 3)
        d = rng.normal(size=3)
        p2 = p1 + d / np.linalg.norm(d) * rng.uniform(0, 1) * (np.linalg.norm(s1) + np.linalg.norm(s2))
        pen, nref, gap = reference(p1, R1, s1, p2, R2, s2)
        if pen > 1e-6:
            out.append(((p1, R1, s1), (p2, R2, s2), pen, nref, gap))
    return out


PAIRS = None


def _pairs():
    global PAIRS
    if PAIRS is None:
        PAIRS = _random_pairs(7, 2000)
    return PAIRS


def clear(pen, gap):
    """The nearest facet is unique by a clear gap: no decision of the rule (face preference, edge slack, tie-breaks) can go either way."""
    return gap > 1e-3 * pen + 1e-6


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_random_pairs_manifold(use_float):
    """At least one contact, a unit normal equal to the exact separating direction where that is unique by a clear gap, no contact
    deeper than the penetration (up to the edge axes' slack), and every point on both surfaces."""
    tol = SURF_TOL[use_float]
    nclear = 0
    for i, (b1, b2, pen, nref, gap) in enumerate(_pairs()):
        c = HC.box_box(*b1, *b2, use_float=use_float)
        n, nrm, pos, dist = c
        assert n >= 1 and np.isfinite(pos).all() and np.isfinite(dist).all(), i
        assert abs(np.linalg.norm(nrm) - 1) < (1e-12 if not use_float else 1e-6), i
        assert dist.min() >= -pen * (1 + 1e-3) - 1e-9 - (0 if not use_float else 1e-6), (i, dist.min(), pen)
        assert surface_error(c, (b1, b2)) <= tol, i
        if clear(pen, gap):
            nclear += 1
            assert np.linalg.norm(nrm - nref) < (1e-9 if not use_float else 1e-5), (i, nrm, nref)
    assert nclear > 1800


def test_random_pairs_invariances():
    """float64: relabelling a box's axes, swapping the boxes (normal negated) and moving both boxes rigidly leave the manifold as a
    set; float32 gives the float64 set and is always finite.  Each away from the rule's decision boundaries."""
    rng = np.random.default_rng(11)
    for i, (b1, b2, pen, nref, gap) in enumerate(_pairs()):
        (p1, R1, s1), (p2, R2, s2) = b1, b2
        n, nrm, pos, dist = HC.box_box(*b1, *b2)
        f = HC.box_box(*b1, *b2, use_float=True)
        assert np.isfinite(f[2]).all() and np.isfinite(f[3]).all(), i
        if not clear(pen, gap):
            continue
        for which in (0, 1):
            P = signed_permutation(rng)
            args = [p1, R1 @ P, np.abs(P.T @ s1), p2, R2, s2] if which == 0 else [p1, R1, s1, p2, R2 @ P, np.abs(P.T @ s2)]
            m, mn, mp, md = HC.box_box(*args)
            assert m == n and np.allclose(mn, nrm, atol=1e-9) and same_set(mp, pos, 1e-9), (i, which)
        m, mn, mp, md = HC.box_box(*b2, *b1)
        assert m == n and np.allclose(mn, -nrm, atol=1e-9) and same_set(mp, pos, 1e-9), (i, "swap")
        W, t = rot(rng), rng.uniform(-1, 1, 3)
        q1, M1, q2, M2 = in_world(W, t, p1, R1, p2, R2)
        m, mn, mp, md = HC.box_box(q1, M1, s1, q2, M2, s2)
        assert m == n and np.allclose(mn, W @ nrm, atol=1e-9) and same_set(mp, pos @ W.T + t, 1e-9) and np.allclose(np.sort(md), np.sort(dist), atol=1e-9), (i, "motion")
        assert f[0] == n and np.allclose(f[1], nrm, atol=1e-5) and same_set(f[2], pos, 1e-5) and np.allclose(np.sort(f[3]), np.sort(dist), atol=1e-5), (i, "f32")


# ---------------------------------------------------------------- nearly parallel faces
TILTS = [0.0, 1e-9, 1e-8, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2]
PENS = [1e-6, 1e-5, 1e-4, 1e-3]


@pytest.mark.parametrize("use_float", PRECISIONS)
@pytest.mark.parametrize("tilt", TILTS)
def test_near_parallel_stacks_stay_on_surface(use_float, tilt):
    """Box 2 stacked face on face on box 1 at a small offset, turned by `tilt` about a random axis, the pair in a random world frame
    (so that tilt 0 is parallel only up to rounding), pressed in by 1 um - 1 mm: at least one contact, all on both surfaces."""
    rng = np.random.default_rng(int(tilt * 1e12) + 3 + (1 if use_float else 0))
    tol = SURF_TOL[use_float]
    for pen in PENS:
        for it in range(150):
            s1, s2 = rng.uniform(0.01, 0.05, 3), rng.uniform(0.01, 0.05, 3)
            W, ax = rot(rng), rng.normal(size=3)
            R2 = W @ Rotation.from_rotvec(ax / np.linalg.norm(ax) * tilt).as_matrix()
            off = rng.uniform(-1, 1, 2) * 0.5 * np.minimum(s1[:2], s2[:2])
            p1 = rng.uniform(-0.1, 0.1, 3)
            p2 = p1 + W @ np.array([off[0], off[1], s1[2] + s2[2] - pen])
            c = HC.box_box(p1, W, s1, p2, R2, s2, use_float=use_float)
            assert c[0] >= 1, (pen, it)
            err = surface_error(c, ((p1, W, s1), (p2, R2, s2)))
            assert err <= tol, (pen, it, c[0], err)


def _pressed_to(pen, p1, R1, s1, p2, R2, s2, axis):
    """p2 moved along -axis until the reference's penetration is pen (bisection over at most |p2 - p1|; box 2 starts clear of box 1)."""
    lo, hi = 0.0, float(np.linalg.norm(p2 - p1))
    for _ in range(80):
        mid = (lo + hi) / 2
        deeper = reference(p1, R1, s1, p2 - mid * axis, R2, s2)[0] < pen
        lo, hi = (mid, hi) if deeper else (lo, mid)
    return p2 - (lo + hi) / 2 * axis


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_tilted_stack_overhanging_the_rim_gets_one_edge_point(use_float):
    """Pinned behaviour: box 2 turned 0.4 rad about box 1's face normal and tilted 0.05 rad, hanging over box 1's rim and pressed in
    by 0.1 mm, so that box 2's low bottom edge crosses box 1's top rim edge.  The edge-edge axis, 0.05 rad from both face normals,
    beats them by more than the face preference, and the manifold is the one point where the two edges cross: on both surfaces, at
    the exact depth along the exact separating direction.  A slightly tilted face-on-face touch gets this single point rather than a
    clipped face polygon; changing that changes the contacts of every tilted touch."""
    s1, s2, pen = np.array([0.04, 0.03, 0.02]), np.array([0.03, 0.02, 0.01]), 1e-4
    R2 = rot_z(0.4) @ rot_y(0.05)
    p2 = _pressed_to(pen, np.zeros(3), np.eye(3), s1, np.array([0.05, 0.0, s1[2] + 2 * np.linalg.norm(s2)]), R2, s2, np.array([0, 0, 1.0]))
    q1, M1, q2, M2 = in_world(W0, T0, np.zeros(3), np.eye(3), p2, R2)
    c = HC.box_box(q1, M1, s1, q2, M2, s2, use_float=use_float)
    rp, rn, gap = reference(q1, M1, s1, q2, M2, s2)
    n, nrm, pos, dist = c
    assert rp == pytest.approx(pen, rel=1e-6)
    assert n == 1
    assert surface_error(c, ((q1, M1, s1), (q2, M2, s2))) <= SURF_TOL[use_float]
    assert abs(nrm @ W0[:, 2]) < 1 - 1e-4 and abs(nrm @ (W0 @ R2)[:, 2]) < 1 - 1e-4   # neither face normal
    np.testing.assert_allclose(nrm, rn, atol=1e-9 if not use_float else 1e-5)
    np.testing.assert_allclose(dist, [-rp], atol=1e-12 if not use_float else 1e-7)


# ---------------------------------------------------------------- the narrow phase inside the forward pass (tests/models/box_pair.xml)
BOX_PAIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "models", "box_pair.xml")
SIZE_A, SIZE_B = np.array([0.04, 0.035, 0.02]), np.array([0.038, 0.036, 0.015])   # box_pair.xml
GEOM_FLOOR, GEOM_A, GEOM_B = 0, 1, 2
MARGIN = {(GEOM_FLOOR, GEOM_A): 1e-3, (GEOM_FLOOR, GEOM_B): 1e-3, (GEOM_A, GEOM_B): 5e-4}
UP = np.array([0.0, 0.0, 0.6])   # box-box configurations sit this high: no plane contact


def _qpos(pa, Ra, pb, Rb):
    """box_pair.xml's qpos: the hinge, then each free joint's position and (w, x, y, z) quaternion."""
    qa, qb = (np.roll(Rotation.from_matrix(R).as_quat(), 1) for R in (Ra, Rb))
    return np.concatenate([[0.0], pa, qa, pb, qb])


def box_pair_states(seed):
    """[(name, qpos, clear)] for box_pair.xml, one configuration per environment: each family of the pins above with box_pair's own
    sizes, nearly parallel stacks, random penetrating pairs and plane-box contacts.  clear: away from the rule's decision boundaries,
    so that float32 must give float64's point set."""
    rng = np.random.default_rng(seed)
    sa, sb = SIZE_A, SIZE_B
    out = []

    def pair(name, pa, Ra, pb, Rb, clear=True):
        W = rot(rng)   # the whole configuration in a random world frame, lifted clear of the floor
        out.append((name, _qpos(W @ pa + UP, W @ Ra, W @ pb + UP, W @ Rb), clear))

    I = np.eye(3)
    pair("aligned stack", np.zeros(3), I, np.array([0, 0, sa[2] + sb[2] - 1e-3]), I)
    pair("offset stack", np.zeros(3), I, np.array([0.03, -0.02, sa[2] + sb[2] - 2e-4]), I)
    pair("gap inside the margin", np.zeros(3), I, np.array([0.01, 0.0, sa[2] + sb[2] + 4e-4]), I)
    pair("gap beyond the margin", np.zeros(3), I, np.array([0.01, 0.0, sa[2] + sb[2] + 6e-4]), I)
    # box b turned 45 degrees: each of its corners pokes out of one side of a's face and a's corners lie outside b, an octagon
    pair("octagon", np.zeros(3), I, np.array([0, 0, sa[2] + sb[2] - 1e-3]), rot_z(np.pi / 4))
    top, bottom = sa[1] * np.sqrt(2) / 2 + sa[2] * np.sqrt(2) / 2, sb[0] * np.sqrt(2) / 2 + sb[2] * np.sqrt(2) / 2
    pair("crossed edges", np.zeros(3), rot_x(np.pi / 4), np.array([0.01, -0.005, top + bottom - 1e-3]), rot_y(np.pi / 4))
    R2 = rot_z(0.4) @ rot_y(0.05)
    pair("tilted over the rim", np.zeros(3), I, _pressed_to(1e-4, np.zeros(3), I, sa, np.array([0.05, 0, 0.2]), R2, sb, np.array([0, 0, 1.0])), R2)
    for tilt in (0.0, 1e-9, 1e-6, 1e-4, 1e-2):
        for pen in (1e-6, 1e-4):
            ax = rng.normal(size=3)
            Rb = Rotation.from_rotvec(ax / np.linalg.norm(ax) * tilt).as_matrix()
            off = rng.uniform(-0.5, 0.5, 2) * np.minimum(sa[:2], sb[:2])
            pair("near-parallel %g / %g" % (tilt, pen), np.zeros(3), I, np.array([off[0], off[1], sa[2] + sb[2] - pen]), Rb, clear=tilt <= 1e-4)
    while len(out) < 40:
        Ra, Rb, d = rot(rng), rot(rng), rng.normal(size=3)
        pb = d / np.linalg.norm(d) * rng.uniform(0, 1) * (np.linalg.norm(sa) + np.linalg.norm(sb))
        p, _, gap = reference(np.zeros(3), Ra, sa, pb, Rb, sb)
        if p > 1e-5:
            pair("random", np.zeros(3), Ra, pb, Rb, clear=clear(p, gap))
    far = np.array([1.0, 1.0, 1.0])
    for name, R, z in (("resting on the floor", I, sa[2] - 1e-3), ("tilted on the floor", rot_y(0.3), sa[0] * np.sin(0.3) + sa[2] * np.cos(0.3) - 1e-3),
                       ("within the floor's margin", I, sa[2] + 5e-4)):
        out.append((name, _qpos(np.array([0.2, -0.1, z]), R, far, I), True))
    return out


def _pair_contacts(r, e, g1, g2):
    """(pos [k, 3], dist [k], normal [k, 3]) of environment e's contacts between g1 and g2 in a forward() result (numpy arrays)."""
    n = int(r["info"][e][0])
    sel = [c for c in range(n) if tuple(r["contact_geom"][e][c]) == (g1, g2)]
    return r["contact_pos"][e][sel], r["contact_dist"][e][sel], r["contact_frame"][e][sel][:, 0, :]


def narrow_phase_at(pos, mat, g1, g2, use_float=False):
    """What collision() keeps of the kernel's narrow phase for the pair (g1, g2) at the given geom poses: (pos, dist, normal [k, 3])."""
    margin = MARGIN[(g1, g2)]
    if g1 == GEOM_FLOOR:
        n, nrm, p, d = HC.plane_box(pos[g1], mat[g1], pos[g2], mat[g2], SIZE_A if g2 == GEOM_A else SIZE_B, margin=margin, use_float=use_float)
    else:
        n, nrm, p, d = HC.box_box(pos[g1], mat[g1], SIZE_A, pos[g2], mat[g2], SIZE_B, margin=margin, use_float=use_float)
    keep = d < margin
    return p[keep], d[keep], np.tile(nrm, (int(keep.sum()), 1))


def test_box_pair_model():
    """box_pair.xml: three explicit pairs with their margins, nq = 15 (the main.xml size class, whose generic kernel has room for 24
    contacts), and the configurations give the contact counts they are built for."""
    assert list(HC.model_array(BOX_PAIR, "pair_geom1")) == [GEOM_FLOOR, GEOM_FLOOR, GEOM_A]
    assert list(HC.model_array(BOX_PAIR, "pair_geom2")) == [GEOM_A, GEOM_B, GEOM_B]
    assert np.allclose(HC.model_array(BOX_PAIR, "pair_margin"), [MARGIN[k] for k in sorted(MARGIN)])
    assert np.allclose(HC.model_array(BOX_PAIR, "geom_size").reshape(3, 3)[1:], [SIZE_A, SIZE_B])
    assert list(HC.model_array(BOX_PAIR, "jnt_qposadr")) == [0, 1, 8]
    assert HC.max_contacts(BOX_PAIR) == 24


def test_box_pair_forward_contacts_are_the_narrow_phase():
    """The float64 forward pass (the kernel's source compiled for the CPU) reports, for every configuration of box_pair_states, exactly
    what box_box / plane_box give at its geom poses, in pair order; the octagon gives 8 points, a gap beyond the margin none."""
    counts = {}
    for name, qp, _ in box_pair_states(5):
        r = HC.forward(BOX_PAIR, qp, np.zeros(13), qacc=False, info=True, contact_geom=True, contact_dist=True, contact_pos=True, contact_frame=True)
        r = {k: v[None] for k, v in r.items()}
        pos, mat, _ = HC.query(BOX_PAIR, qp, np.zeros(13), [5] * 3, [0, 1, 2])
        mat = mat.reshape(3, 9)
        total = 0
        for g1, g2 in sorted(MARGIN):
            gp, gd, gn = _pair_contacts(r, 0, g1, g2)
            hp, hd, hn = narrow_phase_at(pos, mat, g1, g2)
            assert len(gd) == len(hd), (name, g1, g2)
            np.testing.assert_allclose(gp, hp, atol=1e-12, err_msg=name)
            np.testing.assert_allclose(gd, hd, atol=1e-12, err_msg=name)
            np.testing.assert_allclose(gn, hn, atol=1e-12, err_msg=name)
            total += len(gd)
        assert total == int(r["info"][0][0]), name
        counts[name] = total
    assert counts["octagon"] == 8 and counts["aligned stack"] == 4 and counts["crossed edges"] == 1 and counts["tilted over the rim"] == 1
    assert counts["gap inside the margin"] == 4 and counts["gap beyond the margin"] == 0
    assert counts["resting on the floor"] == 4 and counts["tilted on the floor"] == 2 and counts["within the floor's margin"] == 4
