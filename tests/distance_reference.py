"""TEST-ONLY reference for the geom-distance pass (ur3e_b200/csrc/distance.cuh), sharing no code or idea with its feature enumeration:

    box-box, disjoint     a bounded linear least-squares problem: minimise |c1 + R1 u - c2 - R2 v| over |u| <= s1, |v| <= s2, solved
                          exactly by scipy's bounded-variable least squares (BVLS, an active-set method)
    box-box, overlapping  the exact penetration depth from the nearest facet of the convex hull of the 64 vertex differences (the
                          Minkowski difference), and the collider's own value from the float64 oracle's box_box through its forward pass
    plane-box             the signed heights of the 8 vertices over the plane
    geom poses            the oracle's own kinematics (d.geom_xpos / d.geom_xmat after set_state + forward)"""
import numpy as np
from scipy.optimize import lsq_linear
from scipy.spatial import ConvexHull

from oracle import oracle as O

CORNERS = np.array([[i, j, k] for k in (-1, 1) for j in (-1, 1) for i in (-1, 1)], dtype=np.float64)


def vertices(p, R, s):
    return CORNERS * s @ R.T + p


def box_box(p1, R1, s1, p2, R2, s2):
    """(dist, from [3], to [3]) of two disjoint boxes by BVLS; dist 0 when they touch or overlap."""
    A = np.hstack([R1, -R2])
    b = p2 - p1
    s = np.concatenate([s1, s2])
    r = lsq_linear(A, b, bounds=(-s, s), method="bvls", tol=1e-15, lsmr_tol=None)
    x, y = p1 + R1 @ r.x[:3], p2 + R2 @ r.x[3:]
    return float(np.linalg.norm(x - y)), x, y


def penetration(p1, R1, s1, p2, R2, s2):
    """Exact penetration depth (> 0 when the boxes overlap): the nearest facet of the Minkowski difference B2 - B1."""
    hull = ConvexHull((vertices(p2, R2, s2)[:, None, :] - vertices(p1, R1, s1)[None, :, :]).reshape(-1, 3))
    return float(np.min(-hull.equations[:, 3]))


def plane_box(pp, pR, bp, bR, s):
    """(dist, point on the plane, vertex) for the plane (pp, pR: z axis = normal) and a box: the lowest vertex's signed height."""
    n = pR[:, 2]
    v = vertices(bp, bR, s)
    h = (v - pp) @ n
    i = int(np.argmin(h))
    return float(h[i]), v[i] - h[i] * n, v[i]


def geom_poses(m, qpos):
    """(geom_xpos [ngeom, 3], geom_xmat [ngeom, 3, 3]) of the oracle model m at qpos."""
    d = O.Data(m)
    d.set_state(np.asarray(qpos, dtype=np.float64), np.zeros(m.nv))
    d.forward()
    return np.array(d.geom_xpos).reshape(-1, 3).copy(), np.array(d.geom_xmat).reshape(-1, 3, 3).copy()


def oracle_contact_dist(m, qpos, g1, g2):
    """Smallest dist of the oracle collider's contacts between geoms g1 and g2 at qpos (the pair must be on the candidate list, and
    the geoms overlap so that its margin plays no part); None without such a contact."""
    d = O.Data(m)
    d.set_state(np.asarray(qpos, dtype=np.float64), np.zeros(m.nv))
    d.forward()
    ds = [c.dist for c in d.contacts() if (c.geom1, c.geom2) == (g1, g2)]
    return min(ds) if ds else None


def pair(m, qpos, g1, g2):
    """Reference (dist, from, to) of a candidate-list pair (g1, g2) of the oracle model m at qpos: BVLS for disjoint boxes, the oracle
    collider's smallest contact dist for overlapping ones (points None), vertex heights for a plane."""
    pos, mat = geom_poses(m, qpos)
    size = np.array(m.py["geom_size"]).reshape(-1, 3)
    gt = np.array(m.py["geom_type"]).reshape(-1)
    if gt[g1] == 0:
        return plane_box(pos[g1], mat[g1], pos[g2], mat[g2], size[g2])
    if gt[g2] == 0:
        dd, a, b = plane_box(pos[g2], mat[g2], pos[g1], mat[g1], size[g1])
        return dd, b, a
    boxes = (pos[g1], mat[g1], size[g1], pos[g2], mat[g2], size[g2])
    if penetration(*boxes) > 0:
        return oracle_contact_dist(m, qpos, g1, g2), None, None
    return box_box(*boxes)
