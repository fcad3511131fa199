"""CPU suite: the geom-distance pass (distance.cuh), compiled as plain C++ by tests/hostcheck in float64 and float32, against the
reference in tests/distance_reference.py: closed forms, random disjoint pairs against BVLS, random overlapping pairs against the
oracle's box_box and the exact penetration, a sweep through contact, every candidate pair of main.xml at seeded states, and the accept /
reject matrix of compile_distance and distance_check."""
import os

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from oracle import oracle as O
from tests import distance_reference as R
from tests.hostcheck import distance as HD

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
MAIN = os.path.join(ROOT, "ur3e_b200", "assets", "main.xml")
BOX_PAIR = os.path.join(HERE, "models", "box_pair.xml")
PRECISIONS = [pytest.param(False, id="f64"), pytest.param(True, id="f32")]
TOL = {False: 1e-12, True: 1e-5}   # metres, for closed forms
I = np.eye(3)
SA, SB = np.array([0.04, 0.035, 0.02]), np.array([0.038, 0.036, 0.015])   # box_pair.xml
GEOM_FLOOR, GEOM_A, GEOM_B = 0, 1, 2


def box(p, Rm, s):
    return (np.asarray(p, dtype=np.float64), np.asarray(Rm, dtype=np.float64), np.asarray(s, dtype=np.float64), False)


def plane(p, Rm):
    return (np.asarray(p, dtype=np.float64), np.asarray(Rm, dtype=np.float64), np.zeros(3), True)


def rot(rng):
    return Rotation.random(random_state=rng).as_matrix()


def off_surface(x, p, Rm, s):
    """Distance of x from the surface of the box (p, Rm, s)."""
    l = np.abs((x - p) @ Rm)
    return np.linalg.norm(np.maximum(l - s, 0)) if (l > s).any() else np.min(s - l)


# ---------------------------------------------------------------- closed forms
@pytest.mark.parametrize("use_float", PRECISIONS)
def test_axis_aligned_gap(use_float):
    s1, s2 = np.array([0.1, 0.2, 0.3]), np.array([0.05, 0.1, 0.05])
    for g in (1e-4, 0.01, 0.3):
        d, ft = HD.pair(box([0, 0, 0], I, s1), box([0.02, 0.03, s1[2] + s2[2] + g], I, s2), use_float=use_float)
        assert abs(d - g) <= TOL[use_float]
        assert abs(np.linalg.norm(ft[3:] - ft[:3]) - g) <= TOL[use_float]
        assert abs(ft[2] - s1[2]) <= TOL[use_float] and abs(ft[5] - (s1[2] + g)) <= TOL[use_float]


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_corner_to_corner(use_float):
    s1, s2, off = np.array([0.1, 0.2, 0.3]), np.array([0.05, 0.1, 0.05]), np.array([0.03, 0.04, 0.12])
    d, ft = HD.pair(box([0, 0, 0], I, s1), box(s1 + s2 + off, I, s2), use_float=use_float)
    assert abs(d - np.linalg.norm(off)) <= TOL[use_float]
    assert np.abs(ft[:3] - s1).max() <= TOL[use_float] and np.abs(ft[3:] - (s1 + off)).max() <= TOL[use_float]


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_crossed_edges(use_float):
    """Two boxes turned 45 degrees about x and y: their top / bottom edges cross at right angles, gap g between the crossing points."""
    s1, s2, g = np.array([0.1, 0.05, 0.05]), np.array([0.04, 0.12, 0.04]), 0.02
    Rx = Rotation.from_euler("x", np.pi / 4).as_matrix()
    Ry = Rotation.from_euler("y", np.pi / 4).as_matrix()
    top, bottom = np.hypot(s1[1], s1[2]), np.hypot(s2[0], s2[2])
    c2 = np.array([0.01, -0.02, top + bottom + g])
    d, ft = HD.pair(box([0, 0, 0], Rx, s1), box(c2, Ry, s2), use_float=use_float)
    assert abs(d - g) <= TOL[use_float]
    assert np.abs(ft[:3] - [0.01, 0, top]).max() <= 10 * TOL[use_float]
    assert np.abs(ft[3:] - [0.01, -0.02 + 0.02, top + g]).max() <= 10 * TOL[use_float] or np.abs(ft[3:] - [0.01, 0, top + g]).max() <= 10 * TOL[use_float]


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_corner_aimed_at_face(use_float):
    """Box 2 turned so that one corner points straight down (its main diagonal along z) at box 1's top face."""
    s1, s2, g = np.array([0.2, 0.2, 0.05]), np.array([0.03, 0.03, 0.03]), 0.015
    R2 = Rotation.align_vectors([[0, 0, -1]], [[-1, -1, -1]])[0].as_matrix()
    c2 = np.array([0.02, -0.05, s1[2] + g + np.linalg.norm(s2)])
    d, ft = HD.pair(box([0, 0, 0], I, s1), box(c2, R2, s2), use_float=use_float)
    assert abs(d - g) <= TOL[use_float]
    assert np.abs(ft[:3] - [0.02, -0.05, s1[2]]).max() <= 10 * TOL[use_float]
    assert np.abs(ft[3:] - [0.02, -0.05, s1[2] + g]).max() <= 10 * TOL[use_float]


@pytest.mark.parametrize("use_float", PRECISIONS)
@pytest.mark.parametrize("plane_first", [True, False])
def test_tilted_box_over_plane(use_float, plane_first):
    s, a, h = np.array([0.05, 0.03, 0.02]), 0.3, 0.1
    Rb = Rotation.from_euler("y", a).as_matrix()
    v = R.vertices(np.array([0.1, 0.2, h]), Rb, s)
    low = v[np.argmin(v[:, 2])]
    pl, bx = plane([0, 0, 0], I), box([0.1, 0.2, h], Rb, s)
    d, ft = HD.pair(pl, bx, use_float=use_float) if plane_first else HD.pair(bx, pl, use_float=use_float)
    assert abs(d - low[2]) <= TOL[use_float]
    on_plane, vertex = (ft[:3], ft[3:]) if plane_first else (ft[3:], ft[:3])
    assert np.abs(vertex - low).max() <= TOL[use_float] and np.abs(on_plane - [low[0], low[1], 0]).max() <= TOL[use_float]
    # below the plane: the deepest vertex, signed
    d2, _ = HD.pair(plane([0, 0, h + 0.01], I), bx, use_float=use_float)
    assert abs(d2 - (low[2] - h - 0.01)) <= TOL[use_float]


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_distmax_cap(use_float):
    s = np.array([0.05, 0.05, 0.05])
    for g, dm in ((0.2, 0.1), (0.1, 0.1), (0.2, 0.0)):
        d, ft = HD.pair(box([0, 0, 0], I, s), box([0.1 + g, 0, 0], I, s), distmax=dm, use_float=use_float)
        assert d == np.float32(dm) if use_float else d == dm
        assert (ft == 0).all()
    d, ft = HD.pair(plane([0, 0, 0], I), box([0, 0, 0.5], I, s), distmax=0.2, use_float=use_float)
    assert abs(d - 0.2) <= TOL[use_float] and (ft == 0).all()
    d, _ = HD.pair(box([0, 0, 0], I, s), box([0.15, 0, 0], I, s), distmax=0.2, use_float=use_float)
    assert abs(d - 0.05) <= TOL[use_float]


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_swapped_order_swaps_fromto(use_float):
    rng = np.random.default_rng(3)
    s1, s2, off = np.array([0.1, 0.2, 0.3]), np.array([0.05, 0.1, 0.05]), np.array([0.03, 0.04, 0.12])
    for _ in range(20):
        W = rot(rng)
        b1, b2 = box([0, 0, 0], W, s1), box(W @ (s1 + s2 + off), W, s2)
        d, ft = HD.pair(b1, b2, use_float=use_float)
        e, fs = HD.pair(b2, b1, use_float=use_float)
        assert abs(d - e) <= TOL[use_float]
        assert np.abs(ft[:3] - fs[3:]).max() <= 10 * TOL[use_float] and np.abs(ft[3:] - fs[:3]).max() <= 10 * TOL[use_float]


def _random_pair(rng, sep):
    """Two random boxes whose centres are `sep` times the sum of their bounding radii apart, random directions and frames."""
    s1, s2 = rng.uniform(0.01, 0.2, 3), rng.uniform(0.01, 0.2, 3)
    u = rng.normal(size=3); u /= np.linalg.norm(u)
    c2 = u * sep * (np.linalg.norm(s1) + np.linalg.norm(s2))
    return (rng.normal(size=3) * 0.1, rot(rng), s1), (c2, rot(rng), s2)


def test_common_rigid_motion_keeps_dist():
    rng = np.random.default_rng(5)
    for _ in range(200):
        (p1, R1, s1), (p2, R2, s2) = _random_pair(rng, rng.uniform(0.3, 1.5))
        d, ft = HD.pair(box(p1, R1, s1), box(p2, R2, s2))
        W, t = rot(rng), rng.normal(size=3)
        e, fs = HD.pair(box(W @ p1 + t, W @ R1, s1), box(W @ p2 + t, W @ R2, s2))
        assert abs(d - e) <= 1e-12 + 1e-9 * abs(d)


# ---------------------------------------------------------------- random pairs
@pytest.mark.parametrize("use_float", PRECISIONS)
def test_random_disjoint_pairs_match_bvls(use_float):
    """2 000 random disjoint pairs: dist is BVLS's (1e-9 relative in float64, 1e-5 m in float32), |to - from| = dist and both points
    lie on their boxes' surfaces."""
    rng = np.random.default_rng(11)
    n = 0
    while n < 2000:
        (p1, R1, s1), (p2, R2, s2) = _random_pair(rng, rng.uniform(0.2, 1.3))
        if R.penetration(p1, R1, s1, p2, R2, s2) > -1e-9:
            continue
        ref, _, _ = R.box_box(p1, R1, s1, p2, R2, s2)
        d, ft = HD.pair(box(p1, R1, s1), box(p2, R2, s2), use_float=use_float)
        tol = 1e-5 if use_float else 1e-9 * ref + 1e-14
        assert abs(d - ref) <= tol, (n, d, ref)
        assert abs(np.linalg.norm(ft[3:] - ft[:3]) - d) <= (1e-5 if use_float else 1e-12)
        stol = 1e-5 if use_float else 1e-12
        assert off_surface(ft[:3], p1, R1, s1) <= stol and off_surface(ft[3:], p2, R2, s2) <= stol
        n += 1


def _box_pair_qpos(pa, Ra, pb, Rb):
    qa, qb = (np.roll(Rotation.from_matrix(Rm).as_quat(), 1) for Rm in (Ra, Rb))
    return np.concatenate([[0.0], pa, qa, pb, qb])


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_random_overlapping_pairs_are_the_collider(use_float):
    """Random overlapping pairs of box_pair.xml's two boxes: dist equals the oracle box_box's smallest contact dist (1e-12 in float64),
    and is not deeper than the exact penetration beyond the narrow phase's slack."""
    m = O.Model(BOX_PAIR)
    rng = np.random.default_rng(17)
    up = np.array([0.0, 0.0, 0.6])
    n = 0
    while n < 300:
        Ra, Rb, d = rot(rng), rot(rng), rng.normal(size=3)
        pb = d / np.linalg.norm(d) * rng.uniform(0, 1) * (np.linalg.norm(SA) + np.linalg.norm(SB))
        pen = R.penetration(np.zeros(3), Ra, SA, pb, Rb, SB)
        if pen < 1e-6:
            continue
        q = _box_pair_qpos(up, Ra, pb + up, Rb)
        ref = R.oracle_contact_dist(m, q, GEOM_A, GEOM_B)
        dist, ft = HD.distance(BOX_PAIR, [GEOM_A], [GEOM_B], q, use_float=use_float)
        if ref is None:   # the collider found no point: the exact path, near zero
            assert abs(dist[0]) <= 1e-6
        else:
            assert abs(dist[0] - ref) <= (1e-5 if use_float else 1e-12), (n, dist[0], ref)
        assert dist[0] >= -pen * (1 + 1e-3) - (1e-5 if use_float else 1e-12)
        assert abs(np.linalg.norm(ft[0, 3:] - ft[0, :3]) - abs(dist[0])) <= (1e-5 if use_float else 1e-12)
        n += 1


@pytest.mark.parametrize("use_float", PRECISIONS)
def test_sweep_through_contact(use_float):
    """box_pair.xml's box b lowered through box a's top from +1 cm to -1 cm (tilted, offset): dist is continuous and monotone, and the
    two regimes meet at zero within rounding."""
    Rb = Rotation.from_euler("xyz", [0.02, -0.03, 0.4]).as_matrix()
    up = np.array([0.0, 0.0, 0.6])
    probe = HD.distance(BOX_PAIR, [GEOM_A], [GEOM_B], _box_pair_qpos(up, I, up + [0.01, -0.005, 0.2], Rb))[0][0]
    z0 = 0.2 - probe   # about the centre height at first touch (the distance is not the vertical gap of the tilted box)
    zs = z0 + np.linspace(0.01, -0.01, 2001)
    ds = np.array([HD.distance(BOX_PAIR, [GEOM_A], [GEOM_B], _box_pair_qpos(up, I, up + [0.01, -0.005, z], Rb), use_float=use_float)[0][0] for z in zs])
    step = zs[0] - zs[1]
    tol = 1e-5 if use_float else 1e-12
    assert (np.diff(ds) <= tol).all()                     # monotone (non-increasing as b descends)
    assert (np.abs(np.diff(ds)) <= 1.01 * step + tol).all()   # continuous: Lipschitz 1 in the vertical offset for a descending box
    assert ds[0] > 0.009 and ds[-1] < -0.009
    i = int(np.argmax(ds <= 0))   # first sample at or past contact: the regimes meet there
    assert 0 < i and ds[i - 1] <= step + tol and -ds[i] <= step + tol


# ---------------------------------------------------------------- models
@pytest.mark.parametrize("use_float", PRECISIONS)
def test_main_candidate_pairs_at_seeded_states(use_float):
    """Every candidate pair of main.xml at the seeded states of the pick-and-place golden, against the reference on the oracle's own
    kinematics (BVLS, the oracle collider, vertex heights)."""
    m = O.Model(MAIN)
    g1 = np.array(m.py["pair_geom1"]).astype(np.int32)
    g2 = np.array(m.py["pair_geom2"]).astype(np.int32)
    gold = np.load(os.path.join(HERE, "golden", "env_v2_pick.npz"))
    for q in gold["seed_qpos"][::10]:
        dist, ft = HD.distance(MAIN, g1, g2, q, use_float=use_float)
        for j in range(len(g1)):
            ref, a, b = R.pair(m, q, int(g1[j]), int(g2[j]))
            if ref is None:
                continue
            tol = (2e-5 if use_float else 1e-9)
            assert abs(dist[j] - ref) <= tol + 1e-9 * abs(ref), (j, dist[j], ref)
            if a is not None and ref > 1e-6:
                assert abs(np.linalg.norm(ft[j, 3:] - ft[j, :3]) - dist[j]) <= tol


def test_distmax_and_outputs_of_the_whole_pass():
    """The per-state pass: distmax caps far pairs (the bounding early-out gives exactly distmax and zeros) and matches the uncapped
    values below it; the float32 pass is within 1e-5 m of float64."""
    m = O.Model(MAIN)
    g1 = np.array(m.py["pair_geom1"]).astype(np.int32)
    g2 = np.array(m.py["pair_geom2"]).astype(np.int32)
    q = np.load(os.path.join(HERE, "golden", "env_v2_pick.npz"))["seed_qpos"][0]
    d, ft = HD.distance(MAIN, g1, g2, q)
    dc, fc = HD.distance(MAIN, g1, g2, q, distmax=0.05)
    far = d >= 0.05
    assert far.any() and (~far).any()
    assert (dc[far] == 0.05).all() and (fc[far] == 0).all()
    assert (dc[~far] == d[~far]).all() and (fc[~far] == ft[~far]).all()
    df, ff = HD.distance(MAIN, g1, g2, q, use_float=True)
    assert np.abs(df - d).max() <= 1e-5


# ---------------------------------------------------------------- accept / reject
def test_compile_accepts_and_rejects():
    m = O.Model(MAIN)
    gt = np.array(m.py["geom_type"]).reshape(-1)
    planes = [int(i) for i in np.flatnonzero(gt == 0)]
    boxes = [int(i) for i in np.flatnonzero(gt == 6)]
    others = [int(i) for i in np.flatnonzero((gt != 0) & (gt != 6))]
    assert HD.compile_check(MAIN, [boxes[0], planes[0]], [boxes[1], boxes[2]]) == ""
    assert HD.compile_check(MAIN, [boxes[0]] * 256, [boxes[1]] * 256) == ""
    assert "outside [1, 256]" in HD.compile_check(MAIN, [boxes[0]] * 257, [boxes[1]] * 257)
    assert "outside [1, 256]" in HD.compile_check(MAIN, [boxes[0]], [boxes[1]], k=0)
    assert "null geom list" in HD.compile_check(MAIN, [], [])
    assert "out of range" in HD.compile_check(MAIN, [m.ngeom], [boxes[0]])
    assert "out of range" in HD.compile_check(MAIN, [boxes[0]], [-1])
    assert "itself" in HD.compile_check(MAIN, [boxes[0]], [boxes[0]])
    assert "two planes" in HD.compile_check(MAIN, [planes[0]], [planes[1]])
    if others:
        assert "only box and plane" in HD.compile_check(MAIN, [others[0]], [boxes[0]])


def test_check_accepts_and_rejects():
    assert HD.check(0, 1, 10, 10, False, False, True) == ""
    assert HD.check(0, 1, 3, 10, True, False, True) == ""
    assert HD.check(0, 1, 3, 10, False, True, True) == ""
    assert "unknown distance id" in HD.check(1, 1, 10, 10, False, False, True)
    assert "unknown distance id" in HD.check(-1, 1, 10, 10, False, False, True)
    assert "m=0" in HD.check(0, 1, 0, 10, True, False, True)
    assert "not both" in HD.check(0, 1, 3, 10, True, True, True)
    assert "m must equal n" in HD.check(0, 1, 3, 10, False, False, True)
    assert "all outputs are null" in HD.check(0, 1, 10, 10, False, False, False)
    assert "NaN" in HD.check(0, 1, 10, 10, False, False, True, distmax=np.nan)


def test_staging_rows():
    """The overlapping path's rows laid over the queries' arena: 13 for main.xml's size class in both precisions."""
    assert HD.rows(MAIN) == 13 and HD.rows(MAIN, True) == 13
