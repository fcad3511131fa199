"""CPU suite: the Jacobian / mass-matrix query (query.cuh query_jac_env), compiled as plain C++ by tests/hostcheck, in
float64.

Every body (inertial and body frame), geom and site of each scene is queried at random states and its jacp / jacr compared with
the oracle's mj_jac at the object's point; M and qfrc_bias with the oracle's forward().  Second sources: the kinematics query's
mj_objectVelocity, central differences of the queried poses, and the closed-form double pendulum."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.hostcheck import build as HC
from tests.test_query_cpu import BODY, GEOM, SITE, XBODY, XMLS, _all_objects, _integrate, _reference, _state

HERE = os.path.dirname(os.path.abspath(__file__))


def _owner(m, types, ids):
    """The loaded model's body each object is attached to (what mj_jacSite / mj_jacGeom / mj_jacBody* pass to mj_jac)."""
    gb, sb = np.asarray(m.py["geom_bodyid"]), np.asarray(m.py["site_bodyid"])
    return np.array([i if t in (BODY, XBODY) else (gb[i] if t == GEOM else sb[i]) for t, i in zip(types, ids)])


@pytest.mark.parametrize("xml", XMLS)
def test_query_jac_matches_oracle_f64(assets, xml):
    path = assets + "/" + xml
    m = O.Model(path); d = O.Data(m); rng = np.random.default_rng(21)
    types, ids = _all_objects(m)
    owner = _owner(m, types, ids)
    for _ in range(4):
        qp, qv = _state(m, rng, xml)
        d.reset(); d.set_state(qp, qv); d.forward()
        points = _reference(m, d, types, ids)[0]
        jacp, jacr, M, bias = HC.query_jac(path, qp, qv, types, ids)
        for j in range(len(types)):
            rp, rr = d.jac(points[j], int(owner[j]))
            assert np.abs(jacp[j] - rp).max() <= 1e-12, (types[j], ids[j])
            assert np.abs(jacr[j] - rr).max() <= 1e-12, (types[j], ids[j])
        rM = d.fullM()
        assert np.abs(M - rM).max() <= 1e-12 * np.abs(rM).max()
        assert np.array_equal(M, M.T)
        assert np.abs(bias - np.asarray(d.qfrc_bias)).max() <= 1e-10


@pytest.mark.parametrize("xml", XMLS)
def test_query_jac_times_qvel_is_object_velocity(assets, xml):
    """mj_objectVelocity (world frame) = [jacr; jacp] qvel, against the kinematics query of the same objects."""
    path = assets + "/" + xml
    m = O.Model(path); rng = np.random.default_rng(22)
    types, ids = _all_objects(m)
    for _ in range(4):
        qp, qv = _state(m, rng, xml)
        jacp, jacr, _, _ = HC.query_jac(path, qp, qv, types, ids, M=False, qfrc_bias=False)
        _, _, vel = HC.query(path, qp, qv, types, ids, local=0)
        assert np.abs(jacr @ qv - vel[:, :3]).max() <= 1e-12
        assert np.abs(jacp @ qv - vel[:, 3:]).max() <= 1e-12


@pytest.mark.parametrize("xml", XMLS)
def test_query_jac_is_derivative_of_pose(assets, xml):
    """Central differences of the queried poses along v: (p(q+) - p(q-)) / 2 eps = jacp v and (R(q+) - R(q-)) / 2 eps = [jacr v]x R,
    with q+- integrated from the same v (the mug's quaternion by its local angular velocity)."""
    path = assets + "/" + xml
    m = O.Model(path); rng = np.random.default_rng(23)
    types, ids = _all_objects(m)
    eps = 1e-5
    for _ in range(4):
        qp, v = _state(m, rng, xml)
        jacp, jacr, _, _ = HC.query_jac(path, qp, v, types, ids, M=False, qfrc_bias=False)
        _, R, _ = HC.query(path, qp, v, types, ids)
        pp, Rp, _ = HC.query(path, _integrate(m, qp, v, eps, xml), v, types, ids)
        pm, Rm, _ = HC.query(path, _integrate(m, qp, v, -eps, xml), v, types, ids)
        assert np.abs((pp - pm) / (2 * eps) - jacp @ v).max() < 1e-6
        w = jacr @ v
        W = np.zeros((len(w), 3, 3))
        W[:, 0, 1], W[:, 0, 2], W[:, 1, 2] = -w[:, 2], w[:, 1], -w[:, 0]
        W -= W.transpose(0, 2, 1)
        assert np.abs((Rp - Rm) / (2 * eps) - W @ R).max() < 1e-6


def test_query_mass_matrix_and_bias_double_pendulum_textbook():
    """M and qfrc_bias without objects (query_id = -1) against the closed-form double pendulum of
    test_analytic_pins.py::test_double_pendulum_mass_matrix_and_bias_textbook: M11 = I1 + I2 + m1 lc1^2 + m2 (l1^2 + lc2^2 + 2 l1 lc2 c2),
    M12 = I2 + m2 (lc2^2 + l1 lc2 c2), M22 = I2 + m2 lc2^2; bias = Coriolis / centrifugal (h = -m2 l1 lc2 s2) + gravity."""
    path = os.path.join(HERE, "models", "double_pendulum.xml")
    m1, m2, l1, lc1, lc2, I1, I2, G = 2.0, 1.5, 0.5, 0.3, 0.25, 0.04, 0.02, 9.81
    rng = np.random.default_rng(24)
    for _ in range(6):
        q = rng.uniform(-2.5, 2.5, 2); v = rng.uniform(-3, 3, 2)
        c2, s2 = np.cos(q[1]), np.sin(q[1])
        M = np.array([[I1 + I2 + m1 * lc1 ** 2 + m2 * (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * c2), I2 + m2 * (lc2 ** 2 + l1 * lc2 * c2)],
                      [I2 + m2 * (lc2 ** 2 + l1 * lc2 * c2), I2 + m2 * lc2 ** 2]])
        h = -m2 * l1 * lc2 * s2
        grav = np.array([m1 * G * lc1 * np.sin(q[0]) + m2 * G * (l1 * np.sin(q[0]) + lc2 * np.sin(q[0] + q[1])), m2 * G * lc2 * np.sin(q[0] + q[1])])
        bias = np.array([h * (2 * v[0] * v[1] + v[1] ** 2), -h * v[0] ** 2]) + grav
        jp, jr, gotM, gotb = HC.query_jac(path, q, v, jacp=False, jacr=False)
        assert jp is None and jr is None
        assert np.abs(gotM - M).max() < 1e-12 and np.abs(gotb - bias).max() < 1e-11, (gotM, M, gotb, bias)
        # each output alone is the same value
        assert np.array_equal(HC.query_jac(path, q, v, jacp=False, jacr=False, qfrc_bias=False)[2], gotM)
        assert np.array_equal(HC.query_jac(path, q, v, jacp=False, jacr=False, M=False)[3], gotb)


def test_query_jac_outputs_are_independent(assets):
    """Asking for fewer outputs changes none of the others (the Jacobians without dynamics, M without the Jacobians)."""
    path = assets + "/main.xml"
    m = O.Model(path)
    qp, qv = _state(m, np.random.default_rng(25), "main.xml")
    types, ids = _all_objects(m)
    full = HC.query_jac(path, qp, qv, types, ids)
    assert np.array_equal(HC.query_jac(path, qp, qv, types, ids, jacr=False, M=False, qfrc_bias=False)[0], full[0])
    assert np.array_equal(HC.query_jac(path, qp, qv, types, ids, jacp=False, M=False, qfrc_bias=False)[1], full[1])
    assert np.array_equal(HC.query_jac(path, qp, qv, types, ids, jacp=False, jacr=False)[2], full[2])


def test_query_jac_rejections(assets):
    path = assets + "/main.xml"
    m = O.Model(path)
    qp, qv = m.key("down")
    tcp = m.id("site", "tcp")
    with pytest.raises(ValueError):    # unknown query id
        HC.query_jac(path, qp, qv, [SITE], [tcp], query_id=1)
    with pytest.raises(ValueError):
        HC.query_jac(path, qp, qv, [SITE], [tcp], query_id=-2)
    with pytest.raises(ValueError):    # no query compiled: id 0 is unknown too
        HC.query_jac(path, qp, qv, query_id=0, jacp=False, jacr=False)
    for jp, jr in ((True, False), (False, True)):   # jacp / jacr without objects
        with pytest.raises(ValueError):
            HC.query_jac(path, qp, qv, [SITE], [tcp], query_id=-1, jacp=jp, jacr=jr, M=True)
    with pytest.raises(ValueError):    # all outputs null
        HC.query_jac(path, qp, qv, [SITE], [tcp], jacp=False, jacr=False, M=False, qfrc_bias=False)
    with pytest.raises(ValueError):
        HC.query_jac(path, qp, qv, jacp=False, jacr=False, M=False, qfrc_bias=False)
    # the same objects with query_id = -1 are fine for M / qfrc_bias alone
    HC.query_jac(path, qp, qv, [SITE], [tcp], query_id=-1, jacp=False, jacr=False)
