"""GPU suite for the Jacobian / mass-matrix queries (ur3e_batch_query_jac, Query.jac, SimBatch.mass_matrix, the mj_jac* accessors of
ur3e_b200/utils.py): the compiled sm_100a kernel against the float64 oracle and the debug forward pass at the batch's stored
state, float32 against float64, a user-side pid_task_ctrl against the fused controller, and non-interference with the step path."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import envs as OE
from oracle import oracle as O
import ur3e_b200._lib as lib
from ur3e_b200 import utils as U
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.model import Model
from tests.test_gpu_query import _move_j, _run, _v2, _whole_model_query
from tests.test_query_jac_cpu import _owner
from tests.test_query_cpu import _reference


def _batch_for(assets, scene, n, dtype, **over):
    if scene == "main.xml":
        return _v2(assets, n, dtype, auto_reset=1, **over)
    return _move_j(assets, scene, n, dtype)


def _all_jac(q):
    return [x.double().cpu().numpy() for x in q.jac(jacp=True, jacr=True, M=True, qfrc_bias=True)]


def _check_jac_against_oracle(b, om, types, ids, q, envs, tol):
    jacp, jacr, M, bias = _all_jac(q)
    qp, qv, _ = (x.double().cpu().numpy() for x in b.get_state())
    owner = _owner(om, types, ids)
    d = O.Data(om)
    for e in envs:
        d.reset(); d.set_state(qp[e], qv[e]); d.forward()
        points = _reference(om, d, types, ids)[0]
        for j in range(len(types)):
            rp, rr = d.jac(points[j], int(owner[j]))
            assert np.abs(jacp[e, j] - rp).max() <= tol and np.abs(jacr[e, j] - rr).max() <= tol, (e, types[j], ids[j])
        assert np.abs(M[e] - d.fullM()).max() <= tol, e
        assert np.abs(bias[e] - np.asarray(d.qfrc_bias)).max() <= tol, e


@pytest.mark.parametrize("scene", ["main.xml", "ur3e_2f85.xml", "ur3e_raw.xml"])
def test_query_jac_matches_oracle_f64(assets, scene):
    """After 300 seeded random steps (the recipe of test_gpu_query.py::test_whole_model_query_matches_oracle_f64), 16 sampled envs:
    jacp / jacr of every object, M and qfrc_bias within 1e-10 of the oracle at get_state(); M and qfrc_bias within 1e-12 of
    debug_forward, which runs the step's own forward pass."""
    b, lo, hi = _batch_for(assets, scene, 256, torch.float64)
    _run(b, lo, hi, 300, seed=3)
    if scene == "main.xml":
        st = b.stats_dict(reset=False)
        assert st["episodes"] > 0 and st["ncon_sum"] > 0
    om, types, ids, q = _whole_model_query(b)
    envs = np.random.default_rng(0).choice(b.n, 16, replace=False)
    _check_jac_against_oracle(b, om, types, ids, q, envs, 1e-10)
    M, bias = (x.cpu().numpy() for x in b.mass_matrix(M=True, qfrc_bias=True))
    for e in envs[:4]:
        dbg = b.debug_forward(int(e))
        assert np.abs(M[e] - dbg["M"]).max() <= 1e-12 and np.abs(bias[e] - dbg["qfrc_bias"]).max() <= 1e-12, e


def test_query_jac_f32_against_f64(assets):
    """A float32 and a float64 batch given the same 1024 states by set_state (main.xml, mug tilted and in contact).  float32 rounds at
    6e-8; a Jacobian column is a unit axis or a lever arm under 1 m composed through at most ten levels of 3x3 products (the float32
    build also uses ~1-ulp sin/cos and approximate division), so 1e-5 absolute leaves ten times the error that chain can build up.
    M (entries below 1, smallest eigenvalue ~4e-5) and qfrc_bias (gravity-dominated, ~12 N) are sums of the same products:
    1e-5 relative to each environment's largest entry."""
    n = 1024
    b64, _, _ = _v2(assets, n, torch.float64)
    b32, _, _ = _v2(assets, n, torch.float32)
    om = O.Model(b64.model.path)
    qp, qv = _random_main_states(om, np.random.default_rng(7), n)
    # both batches get the float32-rounded state, so that only the arithmetic differs
    qp, qv = qp.astype(np.float32), qv.astype(np.float32)
    for b in (b64, b32):
        b.reset()
        b.set_state(torch.tensor(qp, device="cuda").to(b.dtype), torch.tensor(qv, device="cuda").to(b.dtype))
    r64 = _all_jac(_whole_model_query(b64)[3])
    r32 = _all_jac(_whole_model_query(b32)[3])
    assert np.abs(r32[0] - r64[0]).max() <= 1e-5 and np.abs(r32[1] - r64[1]).max() <= 1e-5
    for k in (2, 3):
        scale = np.abs(r64[k]).reshape(n, -1).max(1)
        err = np.abs(r32[k] - r64[k]).reshape(n, -1).max(1)
        assert (err <= 1e-5 * scale).all(), (k, float((err / scale).max()))


def _random_main_states(om, rng, n):
    qp0, _ = om.key("down")
    qp = np.tile(qp0, (n, 1)); qv = rng.uniform(-1, 1, (n, om.nv))
    qp[:, :6] += rng.uniform(-0.3, 0.3, (n, 6))
    qp[:, 6] = qp[:, 10] = rng.uniform(0, 0.5, n)
    qp[:, 16] -= rng.uniform(0, 0.001, n)
    quat = np.hstack([np.ones((n, 1)), rng.uniform(-0.4, 0.4, (n, 3))])
    qp[:, 17:21] = quat / np.linalg.norm(quat, axis=1, keepdims=True)
    return qp, qv


def _rotvec_to_mat(rv):
    th = rv.norm(dim=1, keepdim=True)
    k = rv / th
    K = torch.zeros(rv.shape[0], 3, 3, dtype=rv.dtype, device=rv.device)
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -k[:, 2], k[:, 1], -k[:, 0]
    K = K - K.transpose(1, 2)
    s, c = torch.sin(th)[:, :, None], torch.cos(th)[:, :, None]
    return torch.eye(3, dtype=rv.dtype, device=rv.device) + s * K + (1 - c) * K @ K


def test_user_side_pid_task_ctrl_equals_fused_controller(assets):
    """pid_task_ctrl (controller_func.py:87-104) restated in torch from Query.jac's tcp jacp / jacr (arm columns :6), the query's tcp
    pose, qvel and qfrc_bias[:6], at the state set_state left: tau = J^T (Kp e - Kd J qvel) + qfrc_bias, grip = traj[6] * ctrlrange.
    One UR3E_CTRL_PID_TASK step from that state records the fused controller's d.ctrl in the sensor record [21:28); the two agree
    within 1e-10 in float64, so the query's outputs are all a user-side controller needs."""
    n = 64
    m = Model(assets + "/main.xml")
    gains = OE.GAINS_MUG
    b = SimBatch(m, env_config(ctrl_mode=lib.CTRL_PID_TASK, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=7, frame_skip=1, gains=gains), n, 0, torch.float64)
    b.reset()
    om = O.Model(b.model.path); rng = np.random.default_rng(8)
    qp, qv = _random_main_states(om, rng, n)
    b.set_state(torch.tensor(qp, device="cuda"), torch.tensor(qv, device="cuda"))
    q = b.query([("site", "tcp")])
    jacp, jacr, _, bias = q.jac(jacp=True, jacr=True, qfrc_bias=True)
    pos, mat, _ = q(pos=True, mat=True)
    _, qvel, _ = b.get_state()
    tcp, R = pos[:, 0].clone(), mat[:, 0].clone()
    J = torch.cat([jacp[:, 0, :, :6], jacr[:, 0, :, :6]], 1)                     # [n, 6, 6]: rows px py pz rx ry rz
    traj = torch.empty(n, 7, dtype=torch.float64, device="cuda")
    traj[:, :3] = tcp + torch.tensor(rng.uniform(-0.05, 0.05, (n, 3)), device="cuda")
    traj[:, 3:6] = torch.tensor(OE.TOOL_ROTVEC + rng.uniform(-0.3, 0.3, (n, 3)), device="cuda")
    traj[:, 6] = torch.tensor(rng.uniform(0, 1, n), device="cuda")
    g = torch.tensor(gains, dtype=torch.float64, device="cuda")
    e = torch.cat([traj[:, :3] - tcp, U._rotvec(_rotvec_to_mat(traj[:, 3:6]) @ R.transpose(1, 2))], 1)
    Jv = (J @ qvel[:, :6, None])[:, :, 0]
    kp, kd = torch.cat([g[0:3], g[6:9]]), torch.cat([g[3:6], g[9:12]])
    F = kp * e - kd * Jv
    u_arm = (J.transpose(1, 2) @ F[:, :, None])[:, :, 0] + bias[:, :6]
    u_grip = traj[:, 6] * float(m.actuator_ctrlrange[-1][1])
    sens = b.enable_sensors()
    b.step(traj.contiguous())
    fused = sens[:, 21:28]
    assert (fused[:, :6] - u_arm).abs().max().item() <= 1e-10
    assert (fused[:, 6] - u_grip).abs().max().item() <= 1e-10
    assert u_arm.abs().max().item() > 1.0          # a controller that does act


def test_query_jac_does_not_disturb_the_step_path(assets):
    """Two identically seeded float32 ur3e-v2 batches with auto-reset; one also calls Query.jac (every output) and mass_matrix
    after each of 200 steps.  Outputs, final state and statistics agree bit for bit; every call is exactly one launch."""
    n, steps = 192, 200
    a_b, lo, hi = _v2(assets, n, torch.float32, auto_reset=1)
    b_b, _, _ = _v2(assets, n, torch.float32, auto_reset=1)
    _, _, _, q = _whole_model_query(b_b)
    assert torch.equal(a_b.reset(seed=9), b_b.reset(seed=9))
    rng = np.random.default_rng(9)
    for k in range(steps):
        a = torch.tensor(lo + (hi - lo) * rng.random((n, len(lo))), dtype=torch.float32, device="cuda")
        ra = [x.clone() for x in a_b.step(a)]
        rb = [x.clone() for x in b_b.step(a)]
        c0 = b_b.launch_count
        q.jac(jacp=True, jacr=True, M=True, qfrc_bias=True)
        assert b_b.launch_count == c0 + 1
        b_b.mass_matrix(M=True, qfrc_bias=True)
        assert b_b.launch_count == c0 + 2
        for x, y in zip(ra, rb):
            assert torch.equal(x, y), k
    for x, y in zip(a_b.get_state(), b_b.get_state()):
        assert torch.equal(x, y)
    assert a_b.stats_dict() == b_b.stats_dict()


@pytest.mark.parametrize("n", [1, 17])
def test_query_jac_small_and_partial_blocks(assets, n):
    """n = 1, and n = 17 (16 + 1 warps in float32, 9 + 8 in float64): every environment against the oracle."""
    for dtype, tol in ((torch.float64, 1e-10), (torch.float32, 1e-4)):
        b, lo, hi = _v2(assets, n, dtype, auto_reset=1)
        _run(b, lo, hi, 20, seed=6)
        om, types, ids, q = _whole_model_query(b)
        _check_jac_against_oracle(b, om, types, ids, q, range(n), tol)


def test_query_jac_side_stream_and_positive_definite_M(assets):
    """A launch on a side stream gives the default stream's results bit for bit; M is symmetric and Cholesky succeeds for every
    environment of a 4096-environment batch after 200 random steps, in both dtypes."""
    for dtype in (torch.float64, torch.float32):
        b, lo, hi = _v2(assets, 4096, dtype, auto_reset=1)
        _run(b, lo, hi, 200, seed=10)
        q = b.query([("site", "tcp"), ("body", "fish"), ("xbody", "wrist_3_link"), ("geom", "ghost")])
        ref = [x.clone() for x in q.jac(jacp=True, jacr=True, M=True, qfrc_bias=True)]
        refm = [x.clone() for x in b.mass_matrix(M=True, qfrc_bias=True)]
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            got = [x.clone() for x in q.jac(jacp=True, jacr=True, M=True, qfrc_bias=True)]
            gotm = [x.clone() for x in b.mass_matrix(M=True, qfrc_bias=True)]
        s.synchronize()
        for x, y in zip(ref + refm, got + gotm):
            assert torch.equal(x, y)
        assert torch.equal(ref[2], refm[0]) and torch.equal(ref[3], refm[1])
        M = refm[0]
        assert torch.equal(M, M.transpose(1, 2))
        _, info = torch.linalg.cholesky_ex(M)
        assert (info == 0).all()


def test_query_jac_errors(assets):
    b, _, _ = _v2(assets, 4, torch.float64)
    b.reset()
    nv = b.model.nv
    q = b.query([("site", "tcp"), ("geom", "ghost")])
    with pytest.raises(ValueError):
        q.jac(jacp=False)
    with pytest.raises(ValueError):
        b.mass_matrix(M=False)
    for bad in (torch.empty(4, 2, 3, nv - 1, dtype=torch.float64, device="cuda"), torch.empty(4, 1, 3, nv, dtype=torch.float64, device="cuda"),
                torch.empty(4, 2, 3, nv, dtype=torch.float32, device="cuda"), torch.empty(4, 2, 3, nv, dtype=torch.float64)):
        with pytest.raises(ValueError):
            q.jac(jacp=bad)
        with pytest.raises(ValueError):
            q.jac(jacp=False, jacr=bad)
    for bad in (torch.empty(4, nv, nv + 1, dtype=torch.float64, device="cuda"), torch.empty(4, nv, nv, dtype=torch.float32, device="cuda"),
                torch.empty(4, nv, nv, dtype=torch.float64)):
        with pytest.raises(ValueError):
            b.mass_matrix(M=bad)
    with pytest.raises(ValueError):
        b.mass_matrix(M=False, qfrc_bias=torch.empty(4, nv + 1, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        U.mj_jacSite(None, b, torch.empty(4, 3, nv, dtype=torch.float32, device="cuda"), None, "tcp")
    # caller tensors of the right kind are written in place
    jp = torch.full((4, 2, 3, nv), float("nan"), dtype=torch.float64, device="cuda")
    assert q.jac(jacp=jp)[0] is jp and torch.isfinite(jp).all()
    # the C ABI itself
    L = lib.load()
    out = torch.empty(4, 2, 3, nv, dtype=torch.float64, device="cuda"); M = torch.empty(4, nv, nv, dtype=torch.float64, device="cuda")
    p, pm = C.c_void_p(out.data_ptr()), C.c_void_p(M.data_ptr())
    c0 = b.launch_count
    assert L.ur3e_batch_query_jac(b.ptr, 1000, p, None, None, None, None) != 0        # unknown id
    assert L.ur3e_batch_query_jac(b.ptr, -2, None, None, pm, None, None) != 0         # unknown id
    assert L.ur3e_batch_query_jac(b.ptr, -1, p, None, pm, None, None) != 0            # jacp without objects
    assert L.ur3e_batch_query_jac(b.ptr, -1, None, p, None, None, None) != 0          # jacr without objects
    assert L.ur3e_batch_query_jac(b.ptr, q.id, None, None, None, None, None) != 0     # all outputs null
    assert L.ur3e_batch_query_jac(None, q.id, p, None, None, None, None) != 0         # null batch
    assert b.launch_count == c0                                                       # a rejected call launches nothing
    assert L.ur3e_batch_query_jac(b.ptr, -1, None, None, pm, None, None) == 0
    assert L.ur3e_batch_query_jac(b.ptr, q.id, p, None, None, None, None) == 0
    assert b.launch_count == c0 + 2


def test_utils_accessors_equal_query_jac(assets):
    """mj_jacSite / mj_jacBody / mj_jacBodyCom / mj_jacGeom(m, d, jacp, jacr, obj) with ids or names write what Query.jac returns;
    get_full_M / get_qfrc_bias equal mass_matrix."""
    b, lo, hi = _v2(assets, 32, torch.float64, auto_reset=1)
    _run(b, lo, hi, 50, seed=11)
    om = O.Model(b.model.path)
    nv = b.model.nv
    objs = (("site", "tcp", U.mj_jacSite), ("xbody", "wrist_3_link", U.mj_jacBody), ("body", "fish", U.mj_jacBodyCom), ("geom", "ghost", U.mj_jacGeom))
    for kind, name, fn in objs:
        ref_p, ref_r, _, _ = (x.clone() if x is not None else None for x in b.query([(kind, name)]).jac(jacp=True, jacr=True))
        oid = om.id("body" if kind in ("xbody", "body") else kind, name)
        for obj in (name, oid):
            jp = torch.zeros(b.n, 3, nv, dtype=torch.float64, device="cuda"); jr = torch.zeros_like(jp)
            assert fn(None, b, jp, jr, obj) is None
            assert torch.equal(jp, ref_p[:, 0]) and torch.equal(jr, ref_r[:, 0]), (kind, obj)
        jr2 = torch.zeros_like(jr)
        fn(None, b, None, jr2, name)
        assert torch.equal(jr2, ref_r[:, 0])
    c0 = b.launch_count
    U.mj_jacSite(None, b, None, None, "tcp")       # nothing asked: nothing launched (MuJoCo computes nothing either)
    assert b.launch_count == c0
    M, bias = (x.clone() for x in b.mass_matrix(M=True, qfrc_bias=True))
    assert torch.equal(U.get_full_M(None, b), M) and torch.equal(U.get_qfrc_bias(None, b), bias)
    assert U.get_full_M(None, b).shape == (b.n, nv, nv) and U.get_qfrc_bias(None, b).shape == (b.n, nv)
