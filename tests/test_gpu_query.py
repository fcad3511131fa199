"""GPU suite for the kinematics queries (ur3e_batch_query, SimBatch.query, ur3e_b200/utils.py accessors): the compiled sm_100a
kernel against the float64 oracle at the batch's stored state, against the in-kernel observation, float32 against float64, and
non-interference with the step path."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import envs as OE
from oracle import oracle as O
import ur3e_b200._lib as lib
from ur3e_b200 import presets
from ur3e_b200 import utils as U
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.model import Model
from tests.test_query_cpu import BODY, GEOM, SITE, XBODY, _all_objects, _reference

KIND = {BODY: "body", XBODY: "xbody", GEOM: "geom", SITE: "site"}


def _v2(assets, n, dtype, **over):
    m = Model(assets + "/main.xml")
    _, kw, lo, hi = presets.ENV_SPECS["gymnasium_env/ur3e-v2"]
    return SimBatch(m, presets.make_config(m, kw, **over), n, 0, dtype), np.asarray(lo), np.asarray(hi)


def _move_j(assets, xml, n, dtype):
    m = Model(assets + "/" + xml)
    na = 6 if m.nu <= 6 else 7
    cfg = env_config(ctrl_mode=lib.CTRL_PD_JOINT, obs_kind=lib.OBS_STATE, obs_dim=m.nq + m.nv, act_dim=na, gains=OE.GAINS_J)
    lo = np.full(na, -0.6); hi = np.full(na, 0.6)
    if na == 7:
        lo[6], hi[6] = 0.0, 255.0
    return SimBatch(m, cfg, n, 0, dtype), lo, hi


def _run(b, lo, hi, steps, seed):
    rng = np.random.default_rng(seed)
    b.reset(seed=seed)
    for _ in range(steps):
        a = lo + (hi - lo) * rng.random((b.n, len(lo)))
        b.step(torch.tensor(a, dtype=b.dtype, device=b.device))


def _whole_model_query(b):
    om = O.Model(b.model.path)
    types, ids = _all_objects(om)
    return om, types, ids, b.query([(KIND[t], int(i)) for t, i in zip(types, ids)])


def _check_against_oracle(b, om, types, ids, q, envs, tol_pose, tol_mat, tol_vel):
    pos, mat, vw = (x.double().cpu().numpy() for x in q(pos=True, mat=True, vel=True, local=False))
    vl = q(pos=False, vel=True, local=True)[2].double().cpu().numpy()
    qp, qv, _ = (x.double().cpu().numpy() for x in b.get_state())
    d = O.Data(om)
    for e in envs:
        d.reset(); d.set_state(qp[e], qv[e]); d.forward()
        rp, rm, rvw, rvl = _reference(om, d, types, ids)
        assert np.abs(pos[e] - rp).max() <= tol_pose, e
        assert np.abs(mat[e] - rm).max() <= tol_mat, e
        assert np.abs(vw[e] - rvw).max() <= tol_vel, e
        assert np.abs(vl[e] - rvl).max() <= tol_vel, e


@pytest.mark.parametrize("scene", ["main.xml", "ur3e_2f85.xml", "ur3e_raw.xml"])
def test_whole_model_query_matches_oracle_f64(assets, scene):
    """After 300 seeded random steps (main.xml: ur3e-v2 with auto-reset, so some envs have reset and some touch the mug or the
    table; the other scenes under joint-space PD), 16 sampled envs: poses <= 1e-12, velocities <= 1e-10, both flg_local values."""
    if scene == "main.xml":
        b, lo, hi = _v2(assets, 256, torch.float64, auto_reset=1)
    else:
        b, lo, hi = _move_j(assets, scene, 256, torch.float64)
    _run(b, lo, hi, 300, seed=3)
    if scene == "main.xml":
        st = b.stats_dict(reset=False)
        assert st["episodes"] > 0 and st["ncon_sum"] > 0
    om, types, ids, q = _whole_model_query(b)
    envs = np.random.default_rng(0).choice(b.n, 16, replace=False)
    _check_against_oracle(b, om, types, ids, q, envs, 1e-12, 1e-12, 1e-10)


def test_accessors_agree_with_observation_at_reset(assets):
    """Right after reset both the observation and the query see fresh kinematics of the stored state."""
    b, _, _ = _v2(assets, 64, torch.float64)
    obs = b.reset(seed=5).clone()
    tol = 1e-12
    assert (U.get_site_xpos(None, b, "tcp") - obs[:, 0:3]).abs().max() <= tol
    assert (U.get_site_xpos(None, b, "handle_site") - obs[:, 3:6]).abs().max() <= tol
    assert (U.get_ghost_xpos(None, b) - obs[:, 6:9]).abs().max() <= tol
    assert (U.get_site_vel(None, b, "tcp")[:, 3:] - obs[:, 15:18]).abs().max() <= tol
    qp, qv, _ = b.get_state()
    assert torch.equal(U.get_finger_jnt_disp(None, b), qp[:, 6]) and torch.equal(U.get_finger_jnt_vel(None, b), qv[:, 6])
    # the remaining accessors against the oracle for env 0
    om = O.Model(b.model.path); d = O.Data(om)
    d.reset(); d.set_state(qp[0].cpu().numpy(), qv[0].cpu().numpy()); d.forward()
    tcp, mug = om.id("site", "tcp"), om.id("body", "fish")
    R = d.site_xmat.reshape(-1, 3, 3)[tcp]
    assert np.abs(U.get_site_R(None, b, "tcp")[0].cpu().numpy() - R).max() <= tol
    assert np.abs(U.get_site_xmat(None, b, "tcp")[0].cpu().numpy() - R.ravel()).max() <= tol
    from scipy.spatial.transform import Rotation
    assert np.abs(U.get_site_xrotvec(None, b, "tcp")[0].cpu().numpy() - Rotation.from_matrix(R).as_rotvec()).max() <= 1e-9
    assert np.abs(U.get_body_xpos(None, b, "fish")[0].cpu().numpy() - d.xpos.reshape(-1, 3)[mug]).max() <= tol
    assert np.abs(U.get_body_xmat(None, b, "fish")[0].cpu().numpy() - d.xmat.reshape(-1, 9)[mug]).max() <= tol
    g = om.names["geom"].index("ghost")
    assert np.abs(U.get_geom_xpos(None, b, "ghost")[0].cpu().numpy() - d.geom_xpos.reshape(-1, 3)[g]).max() <= tol
    assert np.abs(U.get_geom_xmat(None, b, "ghost")[0].cpu().numpy() - d.geom_xmat.reshape(-1, 9)[g]).max() <= tol


def test_accessor_golden_tcp_and_cached_query(assets):
    """The reference's recorded tcp position at keyframe "down" (its assets/main.xml:415); a repeated accessor is one launch."""
    b, _, _ = _v2(assets, 4, torch.float64, reset_noise=lib.NOISE_NONE)
    b.reset(seed=0)
    p = U.get_site_xpos(None, b, "tcp")
    assert (p - torch.tensor([0.29799994, 0.13349916, 0.1682003], dtype=torch.float64, device="cuda")).abs().max() <= 5e-8
    n0 = b.launch_count
    p2 = U.get_site_xpos(None, b, "tcp")
    assert b.launch_count == n0 + 1 and p2.data_ptr() == p.data_ptr()


def test_f32_query_against_f64_oracle(assets):
    """float32 production batch, 4096 envs after 200 random steps; 256 sampled envs against the float64 oracle at the same stored
    state.  Bounds from float32 rounding through a 10-level kinematic chain, not measured: poses 1e-5 m, matrices 1e-5,
    velocities 1e-4 absolute."""
    b, lo, hi = _v2(assets, 4096, torch.float32, auto_reset=1)
    _run(b, lo, hi, 200, seed=4)
    om, types, ids, q = _whole_model_query(b)
    envs = np.random.default_rng(1).choice(b.n, 256, replace=False)
    _check_against_oracle(b, om, types, ids, q, envs, 1e-5, 1e-5, 1e-4)


def test_query_does_not_disturb_the_step_path(assets):
    """Two identical float32 batches with every tier in use (lite cap lowered to 4 contacts; the grasp schedule of
    test_gpu_parity.py::test_tier_choice_is_deterministic_and_shard_invariant, so that a part of the batch is in grasp); one runs the
    whole-model query after every step on the same stream.  Outputs, final state and statistics agree bit for bit; launch counts
    differ by exactly the number of queries."""
    n, steps = 192, 260
    cfg = dict(ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2, reset_key=1,
               term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500, reset_noise=lib.NOISE_LOW, auto_reset=1, lite_max_contacts=4)
    m = Model(assets + "/main.xml")
    a_b, b_b = SimBatch(m, env_config(**cfg), n, 0, torch.float32), SimBatch(m, env_config(**cfg), n, 0, torch.float32)
    _, _, _, q = _whole_model_query(b_b)
    oa = a_b.reset(seed=9).clone(); ob = b_b.reset(seed=9).clone()
    assert torch.equal(oa, ob)
    mug0 = oa[:, 3:6].clone()
    c0a, c0b = a_b.launch_count, b_b.launch_count
    full_seen = 0
    for k in range(steps):
        a = torch.empty(n, 4, device="cuda")
        a[:, 0:2] = a_b.obs[:, 3:5]
        a[:, 2] = mug0[:, 2] + 0.02 + max(0.0, 0.1 - 0.002 * k)
        a[:, 3] = 1.0 if k > 90 else 0.0
        a[::3, 3] = 0.0                                               # a third of the batch never closes: mixed tiers
        a = a.contiguous()
        ra = [x.clone() for x in a_b.step(a)]
        rb = [x.clone() for x in b_b.step(a)]
        q(pos=True, mat=True, vel=True)
        for x, y in zip(ra, rb):
            assert torch.equal(x, y), k
        if k % 20 == 0:
            torch.cuda.synchronize()
            full_seen = max(full_seen, a_b.kernel_info()["lite"]["last_overflow_envs"])
    assert full_seen > 0
    for x, y in zip(a_b.get_state(), b_b.get_state()):
        assert torch.equal(x, y)
    assert a_b.stats_dict() == b_b.stats_dict()
    assert (b_b.launch_count - c0b) - (a_b.launch_count - c0a) == steps


@pytest.mark.parametrize("n", [1, 17])
def test_small_and_partial_blocks(assets, n):
    """n = 1, and n = 17: one full block of 16 warps plus one env in float32, 9 + 8 warps in float64."""
    for dtype, tol in ((torch.float64, 1e-12), (torch.float32, 1e-5)):
        b, lo, hi = _v2(assets, n, dtype, auto_reset=1)
        _run(b, lo, hi, 20, seed=6)
        om, types, ids, q = _whole_model_query(b)
        _check_against_oracle(b, om, types, ids, q, range(n), tol, tol, 100 * tol)


def test_query_on_a_side_stream_after_a_step(assets):
    b, lo, hi = _v2(assets, 64, torch.float64)
    b.reset(seed=2)
    om, types, ids, q = _whole_model_query(b)
    s = torch.cuda.Stream()
    a = torch.tensor(np.tile((lo + hi) / 2, (b.n, 1)), dtype=b.dtype, device=b.device)
    with torch.cuda.stream(s):
        for _ in range(5):
            b.step(a)
        pos = q(pos=True)[0].clone()
        qp, qv, _ = b.get_state()
    s.synchronize()
    d = O.Data(om)
    for e in (0, 63):
        d.reset(); d.set_state(qp[e].cpu().numpy(), qv[e].cpu().numpy()); d.forward()
        assert np.abs(pos[e].cpu().numpy() - _reference(om, d, types, ids)[0]).max() <= 1e-12


def test_query_errors(assets):
    b, _, _ = _v2(assets, 4, torch.float64)
    b.reset()
    with pytest.raises(ValueError):
        b.query([("joint", "elbow_joint")])
    with pytest.raises(KeyError):
        b.query([("site", "no_such_site")])
    with pytest.raises(ValueError):
        b.query([("body", b.model.nbody)])
    with pytest.raises(ValueError):
        b.query([])
    with pytest.raises(ValueError):
        b.query([("site", "tcp")] * 257)
    q = b.query([("site", "tcp")] * 256)
    assert q(pos=True)[0].shape == (4, 256, 3)
    with pytest.raises(ValueError):
        q(pos=False)
    for bad in (torch.empty(4, 256, 2, dtype=torch.float64, device="cuda"), torch.empty(4, 256, 3, dtype=torch.float32, device="cuda"),
                torch.empty(4, 256, 3, dtype=torch.float64)):
        with pytest.raises(ValueError):
            q(pos=bad)
    # the C ABI itself
    L = lib.load()
    t = (C.c_int32 * 1)(lib.OBJ_SITE); i = (C.c_int32 * 1)(0)
    assert L.ur3e_batch_query_create(b.ptr, t, i, 0) < 0 and L.ur3e_batch_query_create(b.ptr, t, i, 257) < 0
    t[0] = lib.OBJ_JOINT
    assert L.ur3e_batch_query_create(b.ptr, t, i, 1) < 0
    t[0] = lib.OBJ_GEOM; i[0] = b.model.ngeom
    assert L.ur3e_batch_query_create(b.ptr, t, i, 1) < 0
    out = torch.empty(4, 256, 3, dtype=torch.float64, device="cuda")
    assert L.ur3e_batch_query(b.ptr, q.id, None, None, None, 0, None) != 0
    assert L.ur3e_batch_query(b.ptr, 1000, C.c_void_p(out.data_ptr()), None, None, 0, None) != 0
