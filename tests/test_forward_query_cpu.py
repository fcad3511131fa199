"""CPU suite: the forward-dynamics query (query_fwd.cuh forward_query_env), compiled as plain C++ by tests/hostcheck, in
float64, against the oracle's forward() at the same (qpos, qvel, warm start, ctrl): the contact list, the contact forces, qacc,
qfrc_constraint and the sensor record; the box-at-rest pin on the query's own contact forces; the contacts-only pass against the full
one; the argument check."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.hostcheck import build as HC
from tests.test_analytic_pins import G, M_BOX, model_path

HERE = os.path.dirname(os.path.abspath(__file__))
ALL = dict(qacc=True, qfrc_constraint=True, info=True, contact_geom=True, contact_dist=True, contact_pos=True, contact_frame=True,
           contact_force=True, flags=True, sensordata=True)
GEOMETRY = ("contact_geom", "contact_dist", "contact_pos", "contact_frame")


def rel(a, b, floor):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor))) if a.size else 0.0


def _pressed(m, rng, n=6):
    """test_gpu_parity.py's _random_states: random arm and finger poses at keyframe 'down', the mug pressed into the table."""
    qp0, _ = m.key("down")
    out = []
    for _ in range(n):
        qp = qp0.copy(); qp[:6] += rng.uniform(-0.3, 0.3, 6); qp[6] = qp[10] = rng.uniform(0, 0.6); qp[16] -= rng.uniform(0, 0.002)
        out.append((qp, rng.uniform(-0.5, 0.5, m.nv), np.zeros(m.nv), rng.uniform(-5, 5, m.nu)))
    return out


def _closing(m, u6, steps, every):
    """Oracle trajectory from keyframe 'down' with the gripper commanded shut (u[6] = u6): states with the pads on the mug (main.xml)
    or on each other (ur3e_2f85.xml), with the oracle's warm start at each sampled state."""
    d = O.Data(m); qp, qv = m.key("down"); d.reset(); d.set_state(qp, qv)
    u = np.zeros(m.nu); u[6] = u6
    out = []
    for k in range(steps):
        d.ctrl[:] = u; d.step(1)
        if k % every == every - 1:
            out.append((d.qpos.copy(), d.qvel.copy(), np.asarray(d.qacc_warmstart).copy(), u.copy()))
    return out


def _folded(m):
    g = np.load(os.path.join(HERE, "golden", "collision.npz"))
    return [(q, g["qvel"], np.zeros(m.nv), np.zeros(m.nu)) for q in g["v2_qpos"]]


def _oracle(m, qp, qv, ws, u):
    d = O.Data(m); d.reset(); d.set_state(qp, qv); d.arr("qacc_warmstart")[:] = ws; d.ctrl[:] = u; d.forward()
    return d


def _check(path, m, states, need_contacts):
    seen = 0
    for qp, qv, ws, u in states:
        d = _oracle(m, qp, qv, ws, u)
        r = HC.forward(path, qp, qv, ws, u, **ALL)
        ncon, nefc, _, ovf = r["info"]
        assert (ncon, nefc, ovf) == (d.ncon, d.nefc, 0)
        seen += ncon > 0
        # the contacts, matched after sorting by (geom1, geom2, pos); the query's order also equals the oracle's (pair-list order,
        # then the narrow phase's point order), checked as it is
        oc = d.contacts()
        og = np.array([[c.geom1, c.geom2] for c in oc], dtype=np.int64).reshape(-1, 2)
        assert np.array_equal(r["contact_geom"][:ncon], og)
        def key(g, p):   # positions rounded to 1e-9 m, so that a last-bit difference in one coordinate cannot reorder the rest
            p = np.round(p, 9)
            return np.lexsort((p[:, 2], p[:, 1], p[:, 0], g[:, 1], g[:, 0]))
        op = np.array([c.pos[:] for c in oc]).reshape(-1, 3)
        i, j = key(r["contact_geom"][:ncon], r["contact_pos"][:ncon]), key(og, op)
        assert np.array_equal(r["contact_geom"][:ncon][i], og[j])
        assert np.abs(r["contact_dist"][:ncon][i] - np.array([c.dist for c in oc])[j]).max(initial=0) <= 1e-12
        assert np.abs(r["contact_pos"][:ncon][i] - op[j]).max(initial=0) <= 1e-12
        ofr = np.array([c.frame[:] for c in oc]).reshape(-1, 3, 3)
        assert np.abs(r["contact_frame"][:ncon][i] - ofr[j]).max(initial=0) <= 1e-12
        f = np.asarray(d.efc_force)
        of = np.array([f[c.efc_address:c.efc_address + 3] for c in oc]).reshape(-1, 3)
        assert rel(r["contact_force"][:ncon][i, :3], of[j], 1e-1) < 1e-6 and not r["contact_force"][:ncon, 3:].any()
        # padding past ncon: geom -1 and zeros
        assert (r["contact_geom"][ncon:] == -1).all()
        for k in ("contact_dist", "contact_pos", "contact_frame", "contact_force"):
            assert not r[k][ncon:].any(), k
        # the solver-tolerance bound of test_gpu_parity.py::test_main_forward_internals_via_queries_f64
        assert rel(r["qacc"], d.qacc, 1e-1) < 1e-6
        assert rel(r["qfrc_constraint"], d.qfrc_constraint, 1e-1) < 1e-6
        s = r["sensordata"]
        o = d.sensors()
        assert rel(s[:7], o[:7], 1e-1) < 1e-6
        if "handle_site" in m.names["site"]:   # the step's record evaluates the two touch sensors only with all four tracked sites
            assert rel(s[7:9], o[7:9], 1e-1) < 1e-6
        assert np.array_equal(s[21:21 + m.nu], u)
        if m.names["site"] and "tcp" in m.names["site"]:
            t = m.id("site", "tcp")
            assert np.abs(s[9:12] - d.site_xpos.reshape(-1, 3)[t]).max() <= 1e-12
            assert np.abs(s[12:21] - d.site_xmat.reshape(-1, 9)[t]).max() <= 1e-12
        if "sensor_torque_site" in m.py and len(m.py["sensor_torque_site"]):
            assert rel(s[28:46], d.torque_sensors().ravel(), 1e-1) < 1e-6
    assert seen >= need_contacts


def test_forward_matches_oracle_pressed_mug(assets):
    """Random main.xml states with the mug pressed into the table, random nonzero ctrl."""
    path = assets + "/main.xml"
    m = O.Model(path)
    _check(path, m, _pressed(m, np.random.default_rng(31)), 6)


def test_forward_matches_oracle_closing_on_mug(assets):
    """States of a scripted close on the mug: pads, hull and mug in contact, the oracle's warm start."""
    path = assets + "/main.xml"
    m = O.Model(path)
    states = _closing(m, 255.0, 450, 90)
    _check(path, m, states, 5)
    r = HC.forward(path, *states[-1], flags=True)
    assert r["flags"] & 3 == 3      # both pads on the mug


def test_forward_matches_oracle_folded_arm(assets):
    """The folded-arm and table poses of tests/golden/collision.npz (self-collision, pads and gripper base on the table)."""
    path = assets + "/main.xml"
    m = O.Model(path)
    _check(path, m, _folded(m), 4)


def test_forward_matches_oracle_pads_closed_2f85(assets):
    """ur3e_2f85.xml with the pads closed on each other."""
    path = assets + "/ur3e_2f85.xml"
    m = O.Model(path)
    _check(path, m, _closing(m, 255.0, 600, 150), 2)


def test_forward_raw_arm(assets):
    """ur3e_raw.xml: no contact pairs (C = 0); qacc, the sensor record and info against the oracle."""
    path = assets + "/ur3e_raw.xml"
    m = O.Model(path)
    assert HC.max_contacts(path) == 0
    rng = np.random.default_rng(33)
    for _ in range(3):
        qp = rng.uniform(-1, 1, m.nq); qv = rng.uniform(-1, 1, m.nv); u = rng.uniform(-5, 5, m.nu)
        d = _oracle(m, qp, qv, np.zeros(m.nv), u)
        r = HC.forward(path, qp, qv, ctrl=u, qfrc_constraint=True, info=True, flags=True, sensordata=True)
        assert list(r["info"]) == [0, d.nefc, r["info"][2], 0] and r["flags"] == 0
        assert rel(r["qacc"], d.qacc, 1e-1) < 1e-6 and rel(r["qfrc_constraint"], d.qfrc_constraint, 1e-1) < 1e-6
        assert rel(r["sensordata"][:7], d.sensors()[:7], 1e-1) < 1e-9


def test_folded_arm_flags_match_reference_fixture(assets):
    """At the five poses of tests/golden/collision.npz the flags and ncon equal what the reference's own gym_utils returned."""
    path = assets + "/main.xml"
    g = np.load(os.path.join(HERE, "golden", "collision.npz"))
    for kind in ("v2", "v0"):
        for e, q in enumerate(g[kind + "_qpos"]):
            r = HC.forward(path, q, g["qvel"], qacc=False, info=True, flags=True)
            assert r["info"][0] == g[kind + "_ncon"][e]
            assert bool(r["flags"] & 8) == bool(g[kind + "_self_collision"][e]) and bool(r["flags"] & 4) == bool(g[kind + "_table_collision"][e])


def test_box_at_rest_contact_forces_from_query():
    """tests/models/box_on_plane.xml after 3 000 steps of the kernel's own source: read through the query, the four corner normal forces
    are m g / 4 (1e-9 relative) and the tangential forces vanish (< 1e-12) -- the pin test_analytic_pins.py checks on the oracle's
    efc_force."""
    import tempfile
    import pathlib
    with tempfile.TemporaryDirectory() as tmp:
        p = model_path(pathlib.Path(tmp))
        m = O.Model(p)
        r = HC.run(p, np.array(m.arr("qpos0")).copy(), np.zeros(m.nv), np.zeros(m.nu), np.zeros(m.nv), 3000)
        assert r["warn"] == 0 and r["overflow"] == 0
        q = HC.forward(p, r["qpos"], r["qvel"], r["qacc"], info=True, contact_force=True)
    n = q["info"][0]
    assert n == 4
    f = q["contact_force"][:n]
    assert np.abs(f[:, 0] / (M_BOX * G / 4) - 1).max() < 1e-9
    assert np.abs(f[:, 1:]).max() < 1e-12


@pytest.mark.parametrize("states", ["pressed", "closing"])
def test_contacts_only_pass_equals_full_pass(assets, states):
    """Asking only for contact geometry, info and flags runs kinematics and collision alone; the geometry, flags, contact count and the
    contact overflow bit are identical to the full pass's."""
    path = assets + "/main.xml"
    m = O.Model(path)
    S = _pressed(m, np.random.default_rng(35)) if states == "pressed" else _closing(m, 255.0, 450, 90)
    for qp, qv, ws, u in S:
        full = HC.forward(path, qp, qv, ws, u, **ALL)
        geo = HC.forward(path, qp, qv, ws, u, qacc=False, info=True, flags=True, **{k: True for k in GEOMETRY})
        for k in GEOMETRY:
            assert np.array_equal(geo[k], full[k]), k
        assert geo["flags"] == full["flags"]
        assert geo["info"][0] == full["info"][0] and geo["info"][3] == full["info"][3] & 1
        assert geo["info"][1] == 0 and geo["info"][2] == 0


def test_forward_outputs_are_independent(assets):
    """Each output alone is the same value as with every output requested (info alone runs the contacts-only pass: its ncon is the
    same, nefc and the iteration count are 0 there)."""
    path = assets + "/main.xml"
    m = O.Model(path)
    qp, qv, ws, u = _closing(m, 255.0, 360, 360)[0]
    full = HC.forward(path, qp, qv, ws, u, **ALL)
    for k in ALL:
        one = HC.forward(path, qp, qv, ws, u, **{j: j == k for j in ALL})
        if k == "info":
            assert one[k][0] == full[k][0] and one[k][1] == one[k][2] == 0
        else:
            assert np.array_equal(one[k], full[k]), k


def test_forward_zero_ctrl_is_default(assets):
    path = assets + "/main.xml"
    m = O.Model(path)
    qp, qv, ws, _ = _pressed(m, np.random.default_rng(36), 1)[0]
    a = HC.forward(path, qp, qv, ws, None, qacc=True, sensordata=True)
    b = HC.forward(path, qp, qv, ws, np.zeros(m.nu), qacc=True, sensordata=True)
    assert np.array_equal(a["qacc"], b["qacc"]) and np.array_equal(a["sensordata"], b["sensordata"])


def test_forward_rejections(assets):
    # the argument check itself: out null, nothing requested, a contact output without contacts
    for out in (0, 1):
        for con in (0, 1):
            for any_ in (0, 1):
                for C in (0, 12, 24):
                    ok = HC.forward_check(out, con, any_, C)
                    assert ok == (bool(out) and bool(any_) and not (con and C == 0)), (out, con, any_, C)
    # through the host-compiled entry point
    main, raw = assets + "/main.xml", assets + "/ur3e_raw.xml"
    qp, qv = O.Model(main).key("down")
    with pytest.raises(ValueError):
        HC.forward(main, qp, qv, qacc=False)
    mr = O.Model(raw)
    for k in GEOMETRY + ("contact_force",):
        with pytest.raises(ValueError):
            HC.forward(raw, np.zeros(mr.nq), np.zeros(mr.nv), **{k: True})
    HC.forward(raw, np.zeros(mr.nq), np.zeros(mr.nv), qacc=False, flags=True)   # flags need no contact storage
