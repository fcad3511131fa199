"""CPU suite: the inverse-dynamics query (query_inv.cuh inverse_query_env), compiled as plain C++ by tests/hostcheck, in float64, against
the mj_inverse restatement of tests/inverse_reference.py on the oracle (both exact at a given acceleration, so they agree to rounding);
that restatement against the oracle's own forward pass and step; closed-form pins; the argument check."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests import inverse_reference as R
from tests.hostcheck import inverse as HI
from tests.test_analytic_pins import G, M_BOX, model_path, rest_penetration
from tests.test_forward_query_cpu import _closing, _folded, _pressed

HERE = os.path.dirname(os.path.abspath(__file__))
PENDULUM = os.path.join(HERE, "models", "double_pendulum.xml")
HINGES = os.path.join(HERE, "models", "hinge_pins.xml")


def rel(a, b, floor):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor))) if a.size else 0.0


def _states(m, path, kind):
    if kind == "pressed":
        return _pressed(m, np.random.default_rng(41))
    if kind == "closing":
        return _closing(m, 255.0, 450, 90) if "main" in path else _closing(m, 255.0, 600, 150)
    if kind == "folded":
        return _folded(m)
    rng = np.random.default_rng(43)   # random states of a model
    qp0 = np.array(m.arr("qpos0")).copy()
    out = []
    for _ in range(5):
        qp = qp0.copy(); qp[:6] += rng.uniform(-1, 1, 6)
        out.append((qp, rng.uniform(-1, 1, m.nv), np.zeros(m.nv), rng.uniform(-5, 5, m.nu)))
    return out


def _forward_qacc(m, qp, qv, ws, u):
    d = O.Data(m); d.reset(); d.set_state(qp, qv); d.arr("qacc_warmstart")[:] = ws; d.ctrl[:] = u; d.forward()
    return d


CASES = [("main.xml", "pressed"), ("main.xml", "closing"), ("main.xml", "folded"), ("ur3e_2f85.xml", "closing"), ("ur3e_2f85.xml", "random"),
         ("ur3e_raw.xml", "random")]


@pytest.mark.parametrize("discrete", [False, True], ids=["continuous", "discrete"])
@pytest.mark.parametrize("scene,kind", CASES)
def test_host_matches_reference(assets, scene, kind, discrete):
    """ncon, nefc, the contact order, qfrc_inverse, qfrc_constraint and the contact forces at random accelerations and at the oracle's
    forward qacc, to rounding (both sides are exact at a given acceleration)."""
    path = os.path.join(assets, scene)
    m = O.Model(path)
    rng = np.random.default_rng(47)
    Cn = HI.max_contacts(path)
    seen = 0
    for qp, qv, ws, u in _states(m, path, kind):
        for qacc in (rng.uniform(-5, 5, m.nv), _forward_qacc(m, qp, qv, ws, u).qacc.copy()):
            r = R.inverse(m, qp, qv, qacc, discrete)
            h = HI.inverse(path, qp, qv, qacc, discrete)
            n = r["ncon"]
            assert list(h["info"]) == [n, r["nefc"], 0]
            scale = np.abs(r["qfrc_inverse"]).max() + 1.0
            assert np.abs(h["qfrc_inverse"] - r["qfrc_inverse"]).max() <= 1e-9 * scale
            assert np.abs(h["qfrc_constraint"] - r["qfrc_constraint"]).max() <= 1e-9 * scale
            if Cn:
                assert np.array_equal(h["contact_geom"][:n], r["contact_geom"]) and (h["contact_geom"][n:] == -1).all()
                fs = np.abs(r["contact_force"]).max(initial=0) + 1.0
                assert np.abs(h["contact_force"][:n] - r["contact_force"]).max(initial=0) <= 1e-9 * fs
                assert not h["contact_force"][n:].any() and not h["contact_force"][:, 3:].any()
            seen += n > 0
    if kind in ("pressed", "closing", "folded"):
        assert seen >= 2


@pytest.mark.parametrize("scene", ["main.xml", "ur3e_2f85.xml", "ur3e_raw.xml"])
def test_reference_inverts_oracle_forward(assets, scene):
    """inverse(forward(ctrl).qacc) returns qfrc_actuator and forward's qfrc_constraint, within the float64 solver's tolerance."""
    path = os.path.join(assets, scene)
    m = O.Model(path)
    for qp, qv, ws, u in _states(m, path, "pressed" if scene == "main.xml" else "random"):
        d = _forward_qacc(m, qp, qv, ws, u)
        r = R.inverse(m, qp, qv, d.qacc.copy())
        assert rel(r["qfrc_inverse"], d.qfrc_actuator, 1e-1) < 1e-6
        assert rel(r["qfrc_constraint"], d.qfrc_constraint, 1e-1) < 1e-6


@pytest.mark.parametrize("scene", ["main.xml", "ur3e_raw.xml"])
def test_reference_inverts_oracle_step(assets, scene):
    """After one step, the discrete convention at the pre-step state and (qvel' - qvel) / h returns the step's qfrc_actuator; the
    continuous one does not on the damped main.xml (the arm joints' damping 1.0 at h = 0.001)."""
    path = os.path.join(assets, scene)
    m = O.Model(path)
    damped = bool((np.asarray(m.arr("dof_damping")) > 0).any())
    for qp, qv, ws, u in _states(m, path, "pressed" if scene == "main.xml" else "random"):
        d = O.Data(m); d.reset(); d.set_state(qp, qv); d.arr("qacc_warmstart")[:] = ws; d.ctrl[:] = u
        d.step(1)
        acc = (d.qvel - qv) / m.timestep
        fa = d.qfrc_actuator.copy()   # the step's pre-integration value
        disc = R.inverse(m, qp, qv, acc, discrete=True)["qfrc_inverse"]
        cont = R.inverse(m, qp, qv, acc, discrete=False)["qfrc_inverse"]
        assert rel(disc, fa, 1e-1) < 1e-6
        if damped:
            assert np.abs(cont - fa).max() > 1e3 * np.abs(disc - fa).max() + 1e-6
        else:
            assert np.array_equal(cont, disc)


SOURCES = ["reference", "kernel-source"]


def _inv(source, path, qp, qv, qacc, discrete=False):
    if source == "reference":
        r = R.inverse(O.Model(path), qp, qv, qacc, discrete)
        return r["qfrc_inverse"], r["qfrc_constraint"]
    h = HI.inverse(path, qp, qv, qacc, discrete, contact_geom=False, contact_force=False)
    return h["qfrc_inverse"], h["qfrc_constraint"]


@pytest.mark.parametrize("source", SOURCES)
def test_box_at_rest_pin(tmp_path, source):
    """The box of box_on_plane.xml at its rest penetration with qvel = qacc = 0: the contacts carry the weight, nothing else acts."""
    p = model_path(tmp_path)
    m = O.Model(p)
    qp = np.array(m.arr("qpos0")).copy(); qp[3] = 0.01 - rest_penetration(G)
    fi, fc = _inv(source, p, qp, np.zeros(m.nv), np.zeros(m.nv))
    assert np.abs(fi).max() < 1e-9 * M_BOX * G
    assert abs(fc[3] - M_BOX * G) < 1e-9 * M_BOX * G and np.abs(np.delete(fc, 3)).max() < 1e-12


@pytest.mark.parametrize("source", SOURCES)
def test_box_in_free_fall_pin(tmp_path, source):
    """The same box off the plane: holding it still takes its weight on z; free fall takes nothing."""
    p = model_path(tmp_path, z0=0.5)
    m = O.Model(p)
    qp = np.array(m.arr("qpos0")).copy()
    fi, fc = _inv(source, p, qp, np.zeros(m.nv), np.zeros(m.nv))
    want = np.zeros(m.nv); want[3] = M_BOX * G
    assert np.abs(fi - want).max() < 1e-12 and not fc.any()
    acc = np.zeros(m.nv); acc[3] = -G
    fi, _ = _inv(source, p, qp, np.zeros(m.nv), acc)
    assert np.abs(fi).max() < 1e-12


@pytest.mark.parametrize("source", SOURCES)
def test_double_pendulum_textbook(source):
    """qfrc_inverse = M(q) qacc + C(q, qdot) + G(q) with test_analytic_pins.py's closed forms, at random (q, qdot, qddot)."""
    m1, m2, l1, lc1, lc2, I1, I2 = 2.0, 1.5, 0.5, 0.3, 0.25, 0.04, 0.02
    rng = np.random.default_rng(5)
    for _ in range(6):
        q = rng.uniform(-2.5, 2.5, 2); v = rng.uniform(-3, 3, 2); a = rng.uniform(-10, 10, 2)
        c2, s2 = np.cos(q[1]), np.sin(q[1])
        M = np.array([[I1 + I2 + m1 * lc1 ** 2 + m2 * (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * c2), I2 + m2 * (lc2 ** 2 + l1 * lc2 * c2)],
                      [I2 + m2 * (lc2 ** 2 + l1 * lc2 * c2), I2 + m2 * lc2 ** 2]])
        h = -m2 * l1 * lc2 * s2
        grav = np.array([m1 * G * lc1 * np.sin(q[0]) + m2 * G * (l1 * np.sin(q[0]) + lc2 * np.sin(q[0] + q[1])), m2 * G * lc2 * np.sin(q[0] + q[1])])
        want = M @ a + np.array([h * (2 * v[0] * v[1] + v[1] ** 2), -h * v[0] ** 2]) + grav
        for discrete in (False, True):   # no damping: the two conventions coincide
            fi, fc = _inv(source, PENDULUM, q, v, a, discrete)
            assert np.abs(fi - want).max() < 1e-11 and not fc.any()


@pytest.mark.parametrize("source", SOURCES)
def test_damped_hinge_pin(source):
    """The damped servo hinge of hinge_pins.xml (damping B = 2, no gravity, no limit): (I + h B) a + B qdot with the discrete
    convention, I a + B qdot without; I includes the armature."""
    m = O.Model(HINGES)
    k = m.id("joint", "servo")
    I = 0.5 + float(np.asarray(m.arr("dof_armature"))[k]); B, h = 2.0, m.timestep
    rng = np.random.default_rng(7)
    for _ in range(4):
        qp = rng.uniform(-0.3, 0.3, m.nq); qv = rng.uniform(-2, 2, m.nv); a = rng.uniform(-20, 20, m.nv)
        fd, _ = _inv(source, HINGES, qp, qv, a, True)
        fcn, _ = _inv(source, HINGES, qp, qv, a, False)
        assert abs(fd[k] - ((I + h * B) * a[k] + B * qv[k])) < 1e-12
        assert abs(fcn[k] - (I * a[k] + B * qv[k])) < 1e-12


def test_inverse_check_matrix():
    """Every rejected combination of ur3e_batch_inverse's arguments, and the accepted ones."""
    ok = dict(qpos=True, qvel=True, m=5, n=3, qacc=True, out=True, con=True, any_=True, ncmax=24)
    assert HI.inverse_check(**ok) == ""
    assert HI.inverse_check(**dict(ok, qpos=False, qvel=False, m=3)) == ""            # the stored state, m = n
    assert HI.inverse_check(**dict(ok, m=1)) == "" and HI.inverse_check(**dict(ok, m=2 ** 31 - 1)) == ""
    assert HI.inverse_check(**dict(ok, con=False, ncmax=0)) == ""
    bad = [(dict(qvel=False), "without qvel"), (dict(qpos=False), "without qpos"), (dict(m=0), "states"), (dict(m=-1), "states"),
           (dict(m=2 ** 31), "states"), (dict(qpos=False, qvel=False, m=4), "stored state"), (dict(qacc=False), "qacc is null"),
           (dict(out=False), "out is null"), (dict(any_=False, con=False), "all outputs"), (dict(ncmax=0), "contact outputs")]
    for kw, why in bad:
        msg = HI.inverse_check(**dict(ok, **kw))
        assert why in msg, (kw, msg)

