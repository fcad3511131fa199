"""CPU suite: the inverse-kinematics solve (ik.cuh ik_env), compiled as plain C++ by tests/hostcheck, in float64, against the numpy
restatement of dm_control's qpos_from_site_pose in tests/ik_reference.py on the oracle; closed-form pins on a two-link planar arm; the
accept / reject matrix of compile_ik and ik_check."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests import ik_reference as R
from tests.hostcheck import ik as HI

HERE = os.path.dirname(os.path.abspath(__file__))
PLANAR = os.path.join(HERE, "models", "ik_planar.xml")
ARM = list(range(6))   # the six arm joints, ids 0 .. 5 in all three models
L1, L2 = 0.5, 0.3      # ik_planar.xml


def _object(m):
    """The tcp site where the model has one; ur3e_raw.xml has no sites: the last body's frame."""
    if "tcp" in m.names["site"]:
        return R.SITE, m.names["site"].index("tcp")
    return R.XBODY, m.nbody - 1


def _problems(m, n, seed):
    """n (start qpos, target pos, target quat): targets from the kinematics of random in-limit arm configurations, starts at those
    configurations perturbed by up to 0.3 rad."""
    rng = np.random.default_rng(seed)
    ot, oid = _object(m)
    q0 = np.array(m.arr("qpos0")).copy()
    d = O.Data(m); d.reset()
    out = []
    for _ in range(n):
        qt = q0.copy(); qt[:6] = rng.uniform(-2.5, 2.5, 6)
        d.set_state(qt, np.zeros(m.nv)); d.forward()
        p, Rm, _, _ = R.frame(m, d, ot, oid)
        qs = qt.copy(); qs[:6] += rng.uniform(-0.3, 0.3, 6)
        out.append((qs, p, R.mat2quat(Rm)))
    return out


TARGETS = {"pos": (True, False), "quat": (False, True), "both": (True, True)}


@pytest.mark.parametrize("which", list(TARGETS))
@pytest.mark.parametrize("scene", ["main.xml", "ur3e_2f85.xml", "ur3e_raw.xml"])
def test_host_matches_reference(assets, scene, which):
    """The first 1, 2 and 3 updates agree to 1e-10; full runs end with the same status and steps and qpos within 1e-8.  Position
    only on the arm is the r < nj branch (the push-through system J J^T)."""
    path = os.path.join(assets, scene)
    m = O.Model(path)
    ot, oid = _object(m)
    wp, wq = TARGETS[which]
    for qs, p, q in _problems(m, 4, 11):
        kw = dict(target_pos=p if wp else None, target_quat=q if wq else None)
        for ms in (1, 2, 3):
            h = HI.ik(path, ot, oid, ARM, qs, max_steps=ms, **kw)
            r = R.solve(m, ot, oid, ARM, qs, max_steps=ms, **kw)
            assert np.abs(h[0] - r[0]).max() <= 1e-10 and h[2:] == r[2:]
            assert abs(h[1] - r[1]) <= 1e-10
        h = HI.ik(path, ot, oid, ARM, qs, **kw)
        r = R.solve(m, ot, oid, ARM, qs, **kw)
        assert h[2:] == r[2:] and h[3] == R.CONVERGED
        assert np.abs(h[0] - r[0]).max() <= 1e-8
        assert np.array_equal(h[0][6:], qs[6:])   # only the selected joints move


def test_other_object_kinds(assets):
    """A geom, a body frame and an inertial frame as the object, with the default options (the call's NULL) and with a rotation
    weight: host and reference agree."""
    path = os.path.join(assets, "main.xml")
    m = O.Model(path)
    (qs, _, _), = _problems(m, 1, 5)
    d = O.Data(m); d.reset()
    qt = qs.copy(); qt[:6] += 0.2
    d.set_state(qt, np.zeros(m.nv)); d.forward()
    wrist = m.names["body"].index("wrist_3_link")
    geom = next(g for g in range(m.ngeom) if m.py["geom_bodyid"][g] == wrist)
    for ot, oid in ((R.GEOM, geom), (R.XBODY, wrist), (R.BODY, wrist)):
        p, Rm, _, _ = R.frame(m, d, ot, oid)
        for opt in ({}, dict(rot_weight=0.3, max_steps=50)):
            h = HI.ik(path, ot, oid, ARM, qs, p, R.mat2quat(Rm), **opt)
            r = R.solve(m, ot, oid, ARM, qs, p, R.mat2quat(Rm), **opt)
            assert h[2:] == r[2:] and h[3] == R.CONVERGED
            assert np.abs(h[0] - r[0]).max() <= 1e-8


def _planar_tip(a, r):
    return np.array([r * np.cos(a), r * np.sin(a), 0.0])


def test_planar_reachable_is_analytic():
    """A reachable target converges to the closed-form elbow solution (q2 > 0) from a start on that side; position only on two
    joints is the r > nj branch (J^T J)."""
    t = _planar_tip(0.4, 0.6)
    c2 = (t @ t - L1 * L1 - L2 * L2) / (2 * L1 * L2)
    q2 = np.arccos(c2); q1 = np.arctan2(t[1], t[0]) - np.arctan2(L2 * np.sin(q2), L1 + L2 * np.cos(q2))
    q, err, steps, status = HI.ik(PLANAR, HI.OBJ_SITE, 0, [0, 1], [0.3, 1.0], target_pos=t)
    assert status == R.CONVERGED and err < 1e-14 and 0 < steps < 100
    assert np.abs(q - [q1, q2]).max() <= 1e-10
    r = R.solve(O.Model(PLANAR), R.SITE, 0, [0, 1], [0.3, 1.0], target_pos=t)
    assert r[2:] == (steps, status) and np.abs(r[0] - q).max() <= 1e-10


def test_planar_unreachable_ends_stretched():
    """A target beyond reach (1.2 > l1 + l2) ends with the arm stretched towards it: q2 on its lower limit 0, q1 near the target's
    angle, err_norm near the distance left; no convergence."""
    q, err, steps, status = HI.ik(PLANAR, HI.OBJ_SITE, 0, [0, 1], [0.3, 1.0], target_pos=_planar_tip(0.5, 1.2))
    assert status == R.NO_PROGRESS
    assert q[1] == 0.0 and abs(q[0] - 0.5) < 5e-3
    assert abs(err - 0.4) < 1e-4


def test_planar_limit():
    """A target whose exact solutions both need q1 > 1 ends on that limit, unconverged, as the reference does."""
    t = _planar_tip(2.0, 0.6)
    q, err, steps, status = HI.ik(PLANAR, HI.OBJ_SITE, 0, [0, 1], [0.3, 1.0], target_pos=t)
    assert q[0] == 1.0 and status != R.CONVERGED and err > 0.1
    r = R.solve(O.Model(PLANAR), R.SITE, 0, [0, 1], [0.3, 1.0], target_pos=t)
    assert r[2:] == (steps, status) and np.abs(r[0] - q).max() <= 1e-10


def test_planar_orientation_and_zero_quaternion():
    """Orientation only: the tip's frame turns by q1 + q2 about z.  A zero quaternion is the identity (mju_normalize4), so the target
    is q1 + q2 = 0; a scaled quaternion is normalised first."""
    half = 0.35
    _, err, _, status = HI.ik(PLANAR, HI.OBJ_SITE, 0, [0, 1], [0.3, 1.0], target_quat=[3 * np.cos(half), 0, 0, 3 * np.sin(half)])
    q, _, _, _ = HI.ik(PLANAR, HI.OBJ_SITE, 0, [0, 1], [0.3, 1.0], target_quat=[np.cos(half), 0, 0, np.sin(half)])
    assert status == R.CONVERGED and abs(q.sum() - 2 * half) < 1e-12
    q, _, _, status = HI.ik(PLANAR, HI.OBJ_SITE, 0, [0, 1], [0.3, 1.0], target_quat=[0, 0, 0, 0])
    assert status == R.CONVERGED and abs(q.sum()) < 1e-12


def test_compile_accept_reject(assets):
    path = os.path.join(assets, "main.xml")
    m = O.Model(path)
    tcp = m.names["site"].index("tcp")
    assert HI.compile_check(path, HI.OBJ_SITE, tcp, ARM) == ""
    assert HI.compile_check(path, HI.OBJ_XBODY, 3, [0]) == ""
    assert HI.compile_check(path, HI.OBJ_GEOM, 0, [0, 1, 2]) == ""
    assert HI.compile_check(path, HI.OBJ_BODY, 5, list(range(m.nv - 6))) == ""   # every hinge: nv - 6 of the mug's free joint
    free = next(j for j in range(m.py["njnt"]) if m.py["jnt_type"][j] == 0)
    cases = [((3, tcp, ARM), "objtype"), ((HI.OBJ_SITE, m.nsite, ARM), "out of range"), ((HI.OBJ_GEOM, -1, ARM), "out of range"),
             ((HI.OBJ_SITE, tcp, [0, 1, 0]), "listed twice"),
             ((HI.OBJ_SITE, tcp, [0, m.py["njnt"]]), "out of range"), ((HI.OBJ_SITE, tcp, [-1]), "out of range"),
             ((HI.OBJ_SITE, tcp, [free]), "not a hinge or slide")]
    for args, why in cases:
        err = HI.compile_check(path, *args)
        assert why in err, (args, err)
    assert "outside [1, nv" in HI.compile_check(path, HI.OBJ_SITE, tcp, [0], nj=0)
    assert "outside [1, nv" in HI.compile_check(path, HI.OBJ_SITE, tcp, list(range(m.nv)) + [0], nj=m.nv + 1)
    assert "null joint list" in HI.compile_check(path, HI.OBJ_SITE, tcp, [], nj=1)
    with pytest.raises(ValueError, match="listed twice"):
        HI.ik(path, HI.OBJ_SITE, tcp, [1, 1], np.zeros(m.nq), target_pos=[0.3, 0, 0.3])


def test_call_accept_reject():
    ok = dict(id_=0, nik=1, m=8, n=8, env_ids=False, qpos0=False, pos=True, quat=False, out=True, any_=True)
    assert HI.check(**ok) == ""
    assert HI.check(**dict(ok, env_ids=True, m=3)) == "" and HI.check(**dict(ok, qpos0=True, m=1)) == ""
    assert HI.check(**dict(ok, quat=True)) == "" and HI.check(**dict(ok, pos=False, quat=True)) == ""
    assert HI.check(**dict(ok, m=2 ** 31 - 1, env_ids=True)) == ""
    assert HI.check(**ok, opt={}) == "" and HI.check(**ok, opt=dict(tol=0, rot_weight=0, regularization_threshold=0, regularization_strength=0)) == ""
    assert HI.check(**ok, opt=dict(max_steps=1)) == "" and HI.check(**ok, opt=dict(max_steps=10000)) == ""
    bad = [(dict(id_=1), "unknown ik id"), (dict(id_=-1), "unknown ik id"), (dict(m=0, env_ids=True), "m=0"),
           (dict(m=2 ** 31, env_ids=True), "m=2147483648"), (dict(env_ids=True, qpos0=True), "not both"), (dict(m=7), "m must equal n"),
           (dict(pos=False), "no target"), (dict(out=False, any_=False), "out is null"), (dict(any_=False), "all outputs are null")]
    for kw, why in bad:
        assert why in HI.check(**dict(ok, **kw)), kw
    nan = float("nan")
    for k, v, why in [("tol", -1e-9, "tol"), ("tol", nan, "tol"), ("rot_weight", -1, "rot_weight"), ("regularization_threshold", -0.1, "regularization_threshold"),
                      ("regularization_strength", -1e-3, "regularization_strength"), ("max_update_norm", 0, "max_update_norm"),
                      ("max_update_norm", nan, "max_update_norm"), ("progress_thresh", 0, "progress_thresh"), ("progress_thresh", -1, "progress_thresh"),
                      ("max_steps", 0, "max_steps"), ("max_steps", 10001, "max_steps")]:
        assert why in HI.check(**ok, opt={k: v}), (k, v)
