"""CPU suite: the kinematics-query source (query.cuh + query_model.h), compiled as plain C++ by tests/hostcheck, against the oracle.

Every body (inertial and body frame), geom and site of each scene is queried at random states in float64 and compared with the
oracle's forward() arrays, with mj_objectVelocity, and with central differences of the queried poses themselves."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.hostcheck import query as HQ

XMLS = ["ur3e_raw.xml", "ur3e_2f85.xml", "main.xml"]
BODY, XBODY, GEOM, SITE = 1, 2, 5, 6


def _state(m, rng, xml):
    qp = m.key("down")[0].copy() if m.nkey else np.zeros(m.nq)
    qp[:6] += rng.uniform(-0.3, 0.3, 6)
    if m.nq >= 14:
        qp[6] = qp[10] = rng.uniform(0, 0.5)
    if xml == "main.xml":
        qp[16] -= rng.uniform(0, 0.001)
        q = np.array([1.0, *rng.uniform(-0.4, 0.4, 3)])
        qp[17:21] = q / np.linalg.norm(q)      # a tilted mug, so that the free joint's rotation is exercised
    return qp, rng.uniform(-1, 1, m.nv)


def _all_objects(m):
    objs = [(t, i) for t in (BODY, XBODY) for i in range(m.nbody)] + [(GEOM, i) for i in range(m.ngeom)] + [(SITE, i) for i in range(m.nsite)]
    return np.array([o[0] for o in objs]), np.array([o[1] for o in objs])


def _reference(m, d, types, ids):
    """Poses from forward()'s arrays and mj_objectVelocity restated from cvel and subtree_com: (pos, mat, vel world, vel local)."""
    nb = m.nbody
    arr = lambda n, w: d.arr(n).reshape(-1, w)
    frames = {BODY: (arr("xipos", 3), arr("ximat", 9)), XBODY: (arr("xpos", 3), arr("xmat", 9)),
              GEOM: (arr("geom_xpos", 3), arr("geom_xmat", 9)), SITE: (arr("site_xpos", 3), arr("site_xmat", 9))}
    owner = {BODY: np.arange(nb), XBODY: np.arange(nb), GEOM: np.asarray(m.py["geom_bodyid"]), SITE: np.asarray(m.py["site_bodyid"])}
    cvel = arr("cvel", 6); com = arr("subtree_com", 3); root = np.asarray(m.py["body_rootid"])
    pos, mat, vw, vl = [], [], [], []
    for t, i in zip(types, ids):
        p, R = frames[t][0][i], frames[t][1][i].reshape(3, 3)
        b = owner[t][i]; cv = cvel[b]
        w, v = cv[:3], cv[3:] + np.cross(cv[:3], p - com[root[b]])
        pos.append(p); mat.append(R); vw.append(np.hstack([w, v])); vl.append(np.hstack([R.T @ w, R.T @ v]))
    return np.array(pos), np.array(mat), np.array(vw), np.array(vl)


def _integrate(m, qp, qv, eps, xml):
    """qpos advanced by eps * qvel; the mug's quaternion by its local angular velocity (MuJoCo's free-joint convention)."""
    q = qp.copy()
    if xml != "main.xml":
        return q + eps * qv
    q[:14] += eps * qv[:14]
    q[14:17] += eps * qv[14:17]
    w = qv[17:20]; a = np.linalg.norm(w) * eps
    dq = np.array([np.cos(a / 2), *(np.sin(a / 2) * w / np.linalg.norm(w))])
    q0 = qp[17:21]
    q[17:21] = [q0[0] * dq[0] - q0[1:] @ dq[1:], *(q0[0] * dq[1:] + dq[0] * q0[1:] + np.cross(q0[1:], dq[1:]))]
    return q


@pytest.mark.parametrize("xml", XMLS)
def test_query_matches_oracle_f64(assets, xml):
    path = assets + "/" + xml
    m = O.Model(path); d = O.Data(m); rng = np.random.default_rng(11)
    types, ids = _all_objects(m)
    for _ in range(4):
        qp, qv = _state(m, rng, xml)
        d.reset(); d.set_state(qp, qv); d.forward()
        rp, rm, rvw, rvl = _reference(m, d, types, ids)
        pos, mat, vw = HQ.query(path, qp, qv, types, ids, local=0)
        _, _, vl = HQ.query(path, qp, qv, types, ids, local=1)
        assert np.abs(pos - rp).max() <= 1e-12
        assert np.abs(mat - rm).max() <= 1e-12
        assert np.abs(vw - rvw).max() <= 1e-12
        assert np.abs(vl - rvl).max() <= 1e-12
        sites = types == SITE
        for local, v in ((0, vw), (1, vl)) if sites.any() else ():
            ref = np.array([d.site_velocity(int(i), local) for i in ids[sites]])
            assert np.abs(v[sites] - ref).max() <= 1e-12


@pytest.mark.parametrize("xml", XMLS)
def test_query_velocity_is_derivative_of_pose(assets, xml):
    """Second source for the velocities: central differences of the queried poses along qvel."""
    path = assets + "/" + xml
    m = O.Model(path); rng = np.random.default_rng(12)
    types, ids = _all_objects(m)
    eps = 1e-5
    for _ in range(4):
        qp, qv = _state(m, rng, xml)
        _, R, v = HQ.query(path, qp, qv, types, ids)
        pp, Rp, _ = HQ.query(path, _integrate(m, qp, qv, eps, xml), qv, types, ids)
        pm, Rm, _ = HQ.query(path, _integrate(m, qp, qv, -eps, xml), qv, types, ids)
        assert np.abs((pp - pm) / (2 * eps) - v[:, 3:]).max() < 1e-6
        w = v[:, :3]
        W = np.zeros((len(w), 3, 3))
        W[:, 0, 1], W[:, 0, 2], W[:, 1, 2] = -w[:, 2], w[:, 1], -w[:, 0]
        W -= W.transpose(0, 2, 1)
        assert np.abs((Rp - Rm) / (2 * eps) - W @ R).max() < 1e-6


def test_tcp_at_keyframe_down_matches_reference_record(assets):
    """The reference records the tcp position at keyframe "down" as 0.29799994 0.13349916 0.1682003 (its assets/main.xml:415)."""
    path = assets + "/main.xml"
    m = O.Model(path)
    qp, qv = m.key("down")
    pos, _, _ = HQ.query(path, qp, qv, [SITE], [m.id("site", "tcp")])
    assert np.abs(pos[0] - [0.29799994, 0.13349916, 0.1682003]).max() <= 5e-8


def test_query_rejects_bad_objects(assets):
    path = assets + "/main.xml"
    m = O.Model(path)
    qp, qv = m.key("down")
    for t, i in (([3], [0]), ([BODY], [m.nbody]), ([GEOM], [-1]), ([SITE], [m.nsite])):
        with pytest.raises(ValueError):
            HQ.query(path, qp, qv, t, i)
    for k in (0, 257):
        with pytest.raises(ValueError):
            HQ.query(path, qp, qv, [SITE] * k, [0] * k)
    HQ.query(path, qp, qv, [SITE] * 256, [0] * 256)
