"""GPU suite for the forward-dynamics queries (ur3e_batch_forward, SimBatch.forward, the contact accessors of ur3e_b200/utils.py): the
compiled sm_100a kernel against the float64 oracle at the batch's stored state, against the reference's recorded collision predicates,
against the step's own forward pass, float32 against float64, and non-interference with the step path."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as O
import ur3e_b200._lib as lib
from ur3e_b200 import utils as U
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.envs import UR3eVecEnv
from ur3e_b200.model import Model
from tests.test_gpu_query import _move_j, _run, _v2

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
IDS = {"v2": "gymnasium_env/ur3e-v2", "v0": "gymnasium_env/ur3e-v0"}
ALL = dict(qacc=True, qfrc_constraint=True, info=True, contact_geom=True, contact_dist=True, contact_pos=True, contact_frame=True,
           contact_force=True, flags=True, sensordata=True)
NO_CONTACT = dict(qacc=True, qfrc_constraint=True, info=True, flags=True, sensordata=True)


def rel(a, b, floor):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor))) if a.size else 0.0


def _np(r):
    return {k: (v.double().cpu().numpy() if v.is_floating_point() else v.cpu().numpy()) for k, v in r._asdict().items() if v is not None}


def _batch_for(assets, scene, n, dtype):
    if scene == "main.xml":
        return _v2(assets, n, dtype, auto_reset=1)
    return _move_j(assets, scene, n, dtype)


def _random_main_states(m, rng, n):
    """test_gpu_parity.py's _random_states: keyframe 'down', random arm and fingers, the mug pressed into the table."""
    qp0, _ = m.key("down")
    qp = np.tile(qp0, (n, 1)); qv = rng.uniform(-0.5, 0.5, (n, m.nv))
    qp[:, :6] += rng.uniform(-0.3, 0.3, (n, 6))
    qp[:, 6] = qp[:, 10] = rng.uniform(0, 0.6, n)
    qp[:, 16] -= rng.uniform(0, 0.002, n)
    return qp, qv


def _check_against_oracle(b, r, envs, ctrl=None):
    om = O.Model(b.model.path)
    qp, qv, ws = (x.double().cpu().numpy() for x in b.get_state())
    nc = 0
    for e in envs:
        d = O.Data(om); d.reset(); d.set_state(qp[e], qv[e]); d.arr("qacc_warmstart")[:] = ws[e]
        d.ctrl[:] = 0 if ctrl is None else ctrl[e]
        d.forward()
        ncon, nefc, _, ovf = r["info"][e]
        assert (ncon, nefc, ovf) == (d.ncon, d.nefc, 0), e
        nc += ncon
        if "contact_geom" in r:
            oc = d.contacts()
            assert np.array_equal(r["contact_geom"][e, :ncon], np.array([[c.geom1, c.geom2] for c in oc]).reshape(-1, 2)), e   # the oracle's order
            for k, f in (("contact_dist", lambda c: [c.dist]), ("contact_pos", lambda c: c.pos[:]), ("contact_frame", lambda c: c.frame[:])):
                ref = np.array([f(c) for c in oc]).reshape(r[k][e, :ncon].shape)
                assert np.abs(r[k][e, :ncon] - ref).max(initial=0) <= 1e-10, (e, k)
            fo = np.asarray(d.efc_force)
            ref = np.array([fo[c.efc_address:c.efc_address + 3] for c in oc]).reshape(-1, 3)
            assert rel(r["contact_force"][e, :ncon, :3], ref, 1e-1) < 1e-6, e
            assert (r["contact_geom"][e, ncon:] == -1).all() and not r["contact_force"][e, ncon:].any() and not r["contact_pos"][e, ncon:].any()
        assert rel(r["qacc"][e], d.qacc, 1e-1) < 1e-6, e
        assert rel(r["qfrc_constraint"][e], d.qfrc_constraint, 1e-1) < 1e-6, e
        assert rel(r["sensordata"][e, :7], d.sensors()[:7], 1e-1) < 1e-6, e
    return nc


@pytest.mark.parametrize("scene", ["main.xml", "ur3e_2f85.xml", "ur3e_raw.xml"])
def test_forward_matches_oracle_f64(assets, scene):
    """After 300 seeded random steps, 16 sampled environments: ncon, nefc, the contact list in the oracle's order (geometry within
    1e-10), the contact forces, qacc, qfrc_constraint (solver tolerance: 1e-6 relative) and the actuator forces of the sensor record
    against the oracle seeded with get_state(), warm start included."""
    b, lo, hi = _batch_for(assets, scene, 256, torch.float64)
    _run(b, lo, hi, 300, seed=3)
    r = _np(b.forward(**(ALL if b.max_contacts else NO_CONTACT)))
    envs = np.random.default_rng(0).choice(b.n, 16, replace=False)
    nc = _check_against_oracle(b, r, envs)
    if scene == "main.xml":
        assert nc > 0


def test_forward_matches_oracle_with_ctrl_f64(assets):
    """Random main.xml states with the mug in contact and a random ctrl per environment."""
    n = 64
    b, _, _ = _v2(assets, n, torch.float64)
    om = O.Model(b.model.path); rng = np.random.default_rng(41)
    qp, qv = _random_main_states(om, rng, n)
    b.reset(); b.set_state(torch.tensor(qp, device="cuda"), torch.tensor(qv, device="cuda"))
    u = rng.uniform(-5, 5, (n, om.nu))
    r = _np(b.forward(ctrl=torch.tensor(u, device="cuda"), **ALL))
    assert _check_against_oracle(b, r, range(0, n, 4), u) > 0


@pytest.mark.parametrize("kind", ["v2", "v0"])
def test_collision_accessors_vs_reference_fixture(kind):
    """tests/golden/collision.npz: after set_state at the five poses, get_self_collision, get_table_collision and get_ncon equal what the
    reference's own gym_utils returned at those states."""
    g = np.load(GOLD + "/collision.npz")
    n = len(g[kind + "_qpos"])
    env = UR3eVecEnv(IDS[kind], n, dtype=torch.float64, auto_reset=False, reset_noise=lib.NOISE_NONE)
    env.reset()
    env.set_state(torch.tensor(g[kind + "_qpos"], device="cuda"), torch.tensor(np.tile(g["qvel"], (n, 1)), device="cuda"))
    cache = U.init_collision_cache(None)
    assert U.get_self_collision(None, env, cache).cpu().tolist() == [bool(x) for x in g[kind + "_self_collision"]]
    assert U.get_table_collision(None, env, cache).cpu().tolist() == [bool(x) for x in g[kind + "_table_collision"]]
    assert U.get_ncon(None, env).cpu().tolist() == [int(x) for x in g[kind + "_ncon"]]


def test_self_collision_flag_agrees_with_termination():
    """At the folded-arm poses the query's self-collision flag is set exactly where the step then terminates for a collision."""
    g = np.load(GOLD + "/collision.npz")
    n = len(g["v2_qpos"])
    env = UR3eVecEnv(IDS["v2"], n, dtype=torch.float64, auto_reset=False, reset_noise=lib.NOISE_NONE)
    env.reset()
    env.set_state(torch.tensor(g["v2_qpos"], device="cuda"), torch.tensor(np.tile(g["qvel"], (n, 1)), device="cuda"))
    flag = U.get_self_collision(None, env).cpu().numpy()
    _, _, term, _, _ = env.step(torch.tensor(g["v2_action"], device="cuda"))
    assert flag.tolist() == term.cpu().numpy().tolist() == [False, True, True, False, False]
    assert env.episode_stats()["term_collision"] == 2


def test_forward_is_the_steps_forward_pass():
    """float64 main.xml, CTRL_RAW, frame_skip 1, sensors on: forward(ctrl=a) then step(a).  The step's sensor record equals sensordata and
    the record's new warm start (get_state()[2], the step's qacc) equals qacc, to 1e-12 relative; whether they are bitwise equal is
    printed.  This is the step's own forward pass evaluated off the step path."""
    m = Model(os.path.join(os.path.dirname(lib.__file__), "assets", "main.xml"))
    n = 128
    cfg = env_config(ctrl_mode=lib.CTRL_RAW, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=m.nu, frame_skip=1)   # OBS_STATE holds at most 32 values
    b = SimBatch(m, cfg, n, 0, torch.float64)
    b.enable_sensors()
    om = O.Model(m.path); rng = np.random.default_rng(43)
    qp, qv = _random_main_states(om, rng, n)
    b.reset(); b.set_state(torch.tensor(qp, device="cuda"), torch.tensor(qv, device="cuda"))
    bitwise = True
    for k in range(20):
        a = torch.tensor(rng.uniform(-3, 3, (n, m.nu)), device="cuda")
        a[:, 6] = 255.0 * (k % 2)
        r = b.forward(ctrl=a, qacc=True, sensordata=True)
        qacc, sens = r.qacc.clone(), r.sensordata.clone()
        b.step(a)
        ws = b.get_state()[2]
        assert rel(sens.cpu().numpy(), b.sensors.cpu().numpy(), 1e-3) <= 1e-12, k
        assert rel(qacc.cpu().numpy(), ws.cpu().numpy(), 1e-3) <= 1e-12, k
        bitwise &= bool(torch.equal(sens, b.sensors)) and bool(torch.equal(qacc, ws))
    assert b.forward(qacc=False, info=True).info[:, 0].sum().item() > 0
    print("forward query vs step: bitwise equal =", bitwise)


def test_forward_f32_against_f64(assets):
    """A float32 and a float64 batch given the same 512 float32-rounded states (main.xml, mug pressed into the table).  The contact
    geometry is a short chain of float32 products from qpos (~1e-6 relative per level, ten levels, lever arms under 1 m): positions
    and distances within 2e-5, frames within 1e-4 (a normal is a difference of such positions divided by a length of order 1).  The
    float32 solver stops at 8 Newton iterations or tolerance 1e-7 instead of converging to 1e-15, and from a stiff state (random
    velocities with the mug pressed up to 2 mm into the table) and a zero warm start the capped solve can end far from the float64
    one (measured: 17.6 N of a 24 N constraint force).  Against the dual reference (tests/test_solver_dual_cpu.py::
    test_host_f32_cold_start_is_capped_not_wrong) that is the iteration cap, not a different row set: the row sets are equal and the
    same float32 solve given 50 iterations converges in 10-13 to the reference.  So the dynamics are compared over the environments whose float32 solve stopped before the cap, per
    environment relative to its largest entry (floor 1): qacc and qfrc_constraint within 1e-3 in every such environment (measured
    on a B200: at most 1.2e-4, 453 of 512 environments).  The split of the load among the corner contacts is poorly conditioned, so per-contact forces enter only through
    their sum J^T f = qfrc_constraint."""
    n = 512
    b64, _, _ = _v2(assets, n, torch.float64)
    b32, _, _ = _v2(assets, n, torch.float32)
    om = O.Model(b64.model.path)
    qp, qv = _random_main_states(om, np.random.default_rng(45), n)
    qp, qv = qp.astype(np.float32), qv.astype(np.float32)
    for b in (b64, b32):
        b.reset(); b.set_state(torch.tensor(qp, dtype=b.dtype, device="cuda"), torch.tensor(qv, dtype=b.dtype, device="cuda"))
    r64, r32 = _np(b64.forward(**ALL)), _np(b32.forward(**ALL))
    same = [e for e in range(n) if np.array_equal(r64["contact_geom"][e], r32["contact_geom"][e])]
    assert len(same) >= 0.95 * n
    for e in same:
        c = r64["info"][e, 0]
        assert np.abs(r32["contact_pos"][e, :c] - r64["contact_pos"][e, :c]).max(initial=0) < 2e-5, e
        assert np.abs(r32["contact_dist"][e, :c] - r64["contact_dist"][e, :c]).max(initial=0) < 2e-5, e
        assert np.abs(r32["contact_frame"][e, :c] - r64["contact_frame"][e, :c]).max(initial=0) < 1e-4, e
    conv = [e for e in same if r32["info"][e, 2] < 8]
    assert len(conv) >= n // 2
    for k in ("qacc", "qfrc_constraint"):
        err = np.array([np.abs(r32[k][e] - r64[k][e]).max() / max(1.0, np.abs(r64[k][e]).max()) for e in conv])
        print("f32 vs f64 %s over %d converged envs: median %.2e, p95 %.2e, max %.2e" % (k, len(conv), np.median(err), np.percentile(err, 95), err.max()))
        assert err.max() < 1e-3, k
    assert (r32["flags"] == r64["flags"]).mean() >= 0.95


def test_forward_is_read_only():
    """Two float32 ur3e-v2 batches with every tier in use; one calls forward (all outputs, with ctrl) after every step.  The stored states
    and the observations stay bit-identical, and each call adds exactly one launch."""
    n = 2048
    ea = UR3eVecEnv(IDS["v2"], n, dtype=torch.float32)
    eb = UR3eVecEnv(IDS["v2"], n, dtype=torch.float32)
    ea.reset(seed=5); eb.reset(seed=5)
    rng = np.random.default_rng(47)
    lo, hi = ea.single_action_space.low, ea.single_action_space.high
    u = torch.zeros(n, ea.batch.model.nu, device="cuda")
    for _ in range(60):
        a = torch.tensor(lo + (hi - lo) * rng.random((n, len(lo))), dtype=torch.float32, device="cuda")
        oa = ea.step(a)[0].clone(); ob = eb.step(a)[0].clone()
        c0 = eb.batch.launch_count
        eb.batch.forward(ctrl=u, **ALL)
        assert eb.batch.launch_count == c0 + 1
        assert torch.equal(oa, ob)
    for x, y in zip(ea.batch.get_state(), eb.batch.get_state()):
        assert torch.equal(x, y)
    info = eb.batch.kernel_info()["lite"]
    assert info["lite_tier_steps"] > 0


@pytest.mark.parametrize("n", [1, 13])
def test_forward_launch_shapes_and_streams(assets, n):
    """A single environment and a partial block (13 environments, not a multiple of the block's warps), on the default stream and
    on a side stream: the same values, against the oracle; entries past ncon are geom -1 and zeros."""
    b, _, _ = _v2(assets, n, torch.float64)
    om = O.Model(b.model.path)
    qp, qv = _random_main_states(om, np.random.default_rng(49 + n), n)
    b.reset(); b.set_state(torch.tensor(qp, device="cuda"), torch.tensor(qv, device="cuda"))
    r = _np(b.forward(**ALL))
    _check_against_oracle(b, r, range(n))
    side = torch.cuda.Stream()
    outs = {k: torch.full_like(v, -3) for k, v in b.forward(**ALL)._asdict().items()}
    side.wait_stream(torch.cuda.current_stream())   # the fills above run on the default stream
    with torch.cuda.stream(side):
        s = b.forward(**outs)
    side.synchronize()
    for k, v in s._asdict().items():
        assert v.data_ptr() == outs[k].data_ptr()
        assert np.array_equal(v.double().cpu().numpy() if v.is_floating_point() else v.cpu().numpy(), r[k]), k
    for e in range(n):
        c = r["info"][e, 0]
        assert c < b.max_contacts
        assert (r["contact_geom"][e, c:] == -1).all()
        for k in ("contact_dist", "contact_pos", "contact_frame", "contact_force"):
            assert not r[k][e, c:].any(), k


def test_max_contacts(assets):
    assert [_batch_for(assets, s, 4, torch.float32)[0].max_contacts for s in ("main.xml", "ur3e_2f85.xml", "ur3e_raw.xml")] == [24, 12, 0]


def test_forward_error_paths(assets):
    b, _, _ = _v2(assets, 8, torch.float32)
    nv, Cn = b.model.nv, b.max_contacts
    with pytest.raises(ValueError):
        b.forward(qacc=False)                                                              # nothing requested
    with pytest.raises(ValueError):
        b.forward(qacc=torch.zeros(8, nv + 1, device="cuda"))                              # shape
    with pytest.raises(ValueError):
        b.forward(qacc=torch.zeros(8, nv, dtype=torch.float64, device="cuda"))             # dtype
    with pytest.raises(ValueError):
        b.forward(qacc=torch.zeros(8, nv))                                                 # device
    with pytest.raises(ValueError):
        b.forward(info=torch.zeros(8, 4, device="cuda"))                                   # integer output given as float
    with pytest.raises(ValueError):
        b.forward(contact_frame=torch.zeros(8, Cn, 9, device="cuda"))                      # [n, C, 3, 3]
    with pytest.raises(ValueError):
        b.forward(ctrl=torch.zeros(8, b.model.nu + 1, device="cuda"))                      # ctrl shape
    with pytest.raises(ValueError):
        b.forward(ctrl=torch.zeros(8, b.model.nu, dtype=torch.float64, device="cuda"))     # ctrl dtype
    raw, _, _ = _move_j(assets, "ur3e_raw.xml", 4, torch.float32)
    with pytest.raises(ValueError):
        raw.forward(contact_geom=True)
    raw.forward(flags=True)
    # the C ABI itself
    L = b._L
    st = lib.ForwardOut()
    assert L.ur3e_batch_forward(b.ptr, None, None, None) != 0 and "out" in lib.last_error()
    assert L.ur3e_batch_forward(b.ptr, None, C.byref(st), None) != 0 and "null" in lib.last_error()
    t = torch.zeros(4, 12, 2, dtype=torch.int32, device="cuda")
    st2 = lib.ForwardOut(); st2.contact_geom = t.data_ptr()
    assert raw._L.ur3e_batch_forward(raw.ptr, None, C.byref(st2), None) != 0 and "contact" in lib.last_error()
    assert L.ur3e_batch_forward(None, None, C.byref(st), None) != 0
    assert L.ur3e_batch_max_contacts(None) < 0
    torch.cuda.synchronize()


def test_contact_accessors(assets):
    """How the utils accessors are wired to SimBatch.forward and the kinematics query (the same kernels: their values are checked
    independently by the oracle tests and the collision.npz fixture test above), and one launch per accessor call, after a scripted
    close on the mug."""
    n = 64
    env = UR3eVecEnv(IDS["v0"], n, dtype=torch.float64, auto_reset=False, reset_noise=lib.NOISE_NONE)
    o = env.reset()[0]
    tcp = o[0, :3].cpu().numpy()
    for k in range(120):   # descend onto the mug, then close
        a = np.hstack([tcp - np.array([0, 0, 0.002 * min(k, 40)]), 1.0 if k >= 60 else -1.0])
        env.step(torch.tensor(np.tile(a, (n, 1)), device="cuda"))
    b = env.batch
    r = b.forward(qacc=False, info=True, flags=True)
    f = r.flags.cpu().numpy()
    assert np.array_equal(U.get_ncon(None, env).cpu().numpy(), r.info[:, 0].cpu().numpy())
    assert np.array_equal(U.get_self_collision(None, env).cpu().numpy(), (f & 8) != 0)
    assert np.array_equal(U.get_table_collision(None, env).cpu().numpy(), (f & 4) != 0)
    g = U.get_block_grasp_state(None, env).cpu().numpy()
    assert np.array_equal(g, (f & 1) + ((f >> 1) & 1))
    tcp, mug = U.get_site_xpos(None, env, "tcp").cpu().numpy(), U.get_site_xpos(None, env, "handle_site").cpu().numpy()
    e = np.abs(tcp - mug)
    want = (g == 2) & (e[:, 0] < 0.01) & (e[:, 1] < 0.005) & (e[:, 2] < 0.05)
    c0 = b.launch_count
    assert np.array_equal(U.get_robust_block_grasp_state(None, env).cpu().numpy(), want)
    assert b.launch_count == c0 + 2
    c0 = b.launch_count
    U.get_ncon(None, env); U.get_self_collision(None, env); U.get_block_grasp_state(None, env)
    assert b.launch_count == c0 + 3


@pytest.mark.parametrize("scene", ["main.xml", "ur3e_raw.xml"])
def test_forward_ctrl_from_sensor_record(assets, scene):
    """forward(ctrl=utils.get_ctrl(b)) after steps with sensors on: get_ctrl is a strided [n, 7] view into the sensor record (and has
    7 columns also for ur3e_raw.xml's nu = 6).  The result equals that of an explicit contiguous [n, nu] copy of the same ctrl, and
    the query's own sensor record carries that ctrl."""
    b, lo, hi = _batch_for(assets, scene, 64, torch.float32)
    nu = b.model.nu
    b.enable_sensors()
    _run(b, lo, hi, 20, seed=11)
    u = U.get_ctrl(b)
    assert not u.is_contiguous() and u.shape == (b.n, 7)
    explicit = u[:, :nu].clone().contiguous()
    assert explicit.abs().max().item() > 0
    a = [x.clone() for x in b.forward(ctrl=u, qacc=True, sensordata=True)[::9]]
    e = [x.clone() for x in b.forward(ctrl=explicit, qacc=True, sensordata=True)[::9]]
    z = b.forward(ctrl=None, qacc=True)[0].clone()
    assert torch.equal(a[0], e[0]) and torch.equal(a[1], e[1])
    assert torch.equal(a[1][:, 21:21 + nu], explicit)
    assert not torch.equal(a[0], z)   # the ctrl reached the dynamics
