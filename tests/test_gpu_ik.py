"""GPU suite for inverse kinematics (ur3e_batch_ik, SimBatch.ik): the compiled sm_100a kernel against dm_control's loop restated in
tests/ik_reference.py and against the host build, round trips through forward kinematics on main.xml in both precisions (checked
through set_state + Query, not the solve's own err_norm), the start sources, untouched records, streams, float32 against float64, every
rejected call, and the trajectory conversion of INTEGRATION.md."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as O
import ur3e_b200._lib as lib
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.controller import build_traj as BT
from ur3e_b200.model import Model
from tests import ik_reference as R
from tests.hostcheck import ik as HI


def _batch(assets, xml, n, dtype):
    m = Model(assets + "/" + xml)
    obs = dict(obs_kind=lib.OBS_V2, obs_dim=24) if xml == "main.xml" else dict(obs_kind=lib.OBS_STATE, obs_dim=m.nq + m.nv)
    return SimBatch(m, env_config(ctrl_mode=lib.CTRL_RAW, act_dim=m.nu, frame_skip=1, **obs), n, 0, dtype)


def _t(x, b, dtype=None):
    return torch.tensor(np.ascontiguousarray(x), dtype=dtype or b.dtype, device=b.device)


def _quat(mat):
    """[m, 4] quaternions of [m, 3, 3] rotations (mju_mat2Quat)."""
    return np.array([R.mat2quat(r) for r in np.asarray(mat, dtype=np.float64)])


def _targets(b, n, seed, spread=0.3):
    """(true qpos, start qpos, tcp pos, tcp quat) [n, ...] in float64: the tcp pose of random in-limit arm configurations, from the
    batch's own query after set_state; starts perturbed by up to `spread` rad."""
    rng = np.random.default_rng(seed)
    q0 = np.asarray(b.model.array("qpos0"), dtype=np.float64)
    qt = np.tile(q0, (n, 1)); qt[:, :6] = rng.uniform(-2.5, 2.5, (n, 6))
    qs = qt.copy(); qs[:, :6] += rng.uniform(-spread, spread, (n, 6))
    pos, mat = _pose(b, qt)
    return qt, qs, pos, _quat(mat)


def _pose(b, qpos):
    """tcp pos [n, 3] and mat [n, 3, 3] (float64) of the batch's environments set to qpos [n, nq] (n = the batch's size)."""
    qp = qpos.contiguous() if isinstance(qpos, torch.Tensor) else _t(qpos, b)
    b.set_state(qp, torch.zeros(b.n, b.model.nv, dtype=b.dtype, device=b.device))
    q = b.__dict__.setdefault("_tcp_query", b.query([("site", "tcp")]))
    pos, mat, _ = q(pos=True, mat=True)
    return pos[:, 0].double().cpu().numpy(), mat[:, 0].double().cpu().numpy()


def _pose_err(b, qpos, pos, quat):
    """|p* - p| + |rotvec(q* q^-1)| of the returned configurations, through set_state + Query."""
    p, mat = _pose(b, qpos)
    cur = _quat(mat)
    rot = np.array([np.linalg.norm(R.quat2vel(R.mulquat(R.normalize4(t), c * np.array([1, -1, -1, -1])))) for t, c in zip(quat, cur)])
    return np.linalg.norm(pos - p, axis=1) + rot


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_round_trip_main(assets, dtype):
    """Targets from forward kinematics, starts perturbed by up to 0.3 rad: float64 converges everywhere, float32 in >= 99 % of the
    problems at its default tol; every converged configuration's pose, checked through set_state + Query, is within its err_norm
    (plus the float32 query's own rounding)."""
    n = 512
    b = _batch(assets, "main.xml", n, dtype)
    _, qs, pos, quat = _targets(b, n, 3)
    ik = b.ik(("site", "tcp"))
    r = ik(_t(pos, b), _t(quat, b), qpos=_t(qs, b))
    info = r.info.cpu().numpy(); err = r.err_norm.double().cpu().numpy(); q = r.qpos.double().cpu().numpy()
    ok = info[:, 1] == 0
    if dtype == torch.float64:
        assert ok.all(), np.unique(info[:, 1], return_counts=True)
        assert (err < 1e-14).all()
    else:
        assert ok.mean() >= 0.99, np.unique(info[:, 1], return_counts=True)
        assert (err[ok] < 1e-5).all()
    check = _pose_err(b, r.qpos.clone(), pos, quat)
    slack = 1e-12 if dtype == torch.float64 else 2e-5
    assert (check[ok] <= err[ok] + slack).all(), (check[ok] - err[ok]).max()
    assert np.array_equal(q[:, 6:], np.asarray(_t(qs, b).double().cpu())[:, 6:])   # only the arm joints move
    lo, hi = np.asarray(b.model.array("jnt_range")).reshape(-1, 2)[:6].T
    assert (q[:, :6] >= lo).all() and (q[:, :6] <= hi).all()


@pytest.mark.parametrize("which", ["pos", "quat", "both"])
@pytest.mark.parametrize("scene", ["main.xml", "ur3e_2f85.xml", "ur3e_raw.xml"])
def test_f64_matches_reference_and_host(assets, scene, which):
    """float64: the kernel's qpos, err_norm, steps and status against the host build (to rounding, same steps and status) and the
    numpy reference (1e-8), with a few updates and full runs."""
    n = 8
    b = _batch(assets, scene, n, torch.float64)
    om = O.Model(b.model.path)
    if "tcp" in om.names["site"]:
        obj, ot, oid = ("site", "tcp"), R.SITE, om.names["site"].index("tcp")
    else:
        obj, ot, oid = ("xbody", om.nbody - 1), R.XBODY, om.nbody - 1
    rng = np.random.default_rng(7)
    q0 = np.asarray(b.model.array("qpos0"), dtype=np.float64)
    qt = np.tile(q0, (n, 1)); qt[:, :6] = rng.uniform(-2.5, 2.5, (n, 6))
    qs = qt.copy(); qs[:, :6] += rng.uniform(-0.3, 0.3, (n, 6))
    d = O.Data(om); d.reset()
    pos, quat = [], []
    for e in range(n):
        d.set_state(qt[e], np.zeros(om.nv)); d.forward()
        p, Rm, _, _ = R.frame(om, d, ot, oid); pos.append(p); quat.append(R.mat2quat(Rm))
    kw = dict(target_pos=_t(pos, b) if which != "quat" else None, target_quat=_t(quat, b) if which != "pos" else None)
    ik = b.ik(obj)
    for ms in (2, 100):
        r = ik(qpos=_t(qs, b), max_steps=ms, **kw)
        q, err, info = r.qpos.cpu().numpy(), r.err_norm.cpu().numpy(), r.info.cpu().numpy()
        for e in range(n):
            tk = dict(target_pos=pos[e] if which != "quat" else None, target_quat=quat[e] if which != "pos" else None)
            h = HI.ik(b.model.path, ot, oid, list(range(6)), qs[e], max_steps=ms, **tk)
            ref = R.solve(om, ot, oid, list(range(6)), qs[e], max_steps=ms, **tk)
            assert tuple(info[e]) == h[2:] == ref[2:]
            assert np.abs(q[e] - h[0]).max() <= 1e-12 and abs(err[e] - h[1]) <= 1e-12
            assert np.abs(q[e] - ref[0]).max() <= 1e-8


def test_sources_records_ids_streams(assets):
    """env_ids with repeats and out-of-range ids (NaN, status 3); the stored-state source (no ids) and the qpos0 source agree bit for
    bit with env_ids at the same configurations; the records are unchanged; a side stream ordered after the default stream gives
    the same result."""
    n = 64
    b = _batch(assets, "main.xml", n, torch.float64)
    qt, qs, pos, quat = _targets(b, n, 9)
    b.set_state(_t(qs, b), torch.zeros(n, b.model.nv, dtype=b.dtype, device=b.device))
    before = [x.clone() for x in b.get_state()]
    ik = b.ik(("site", "tcp"))
    tp, tq = _t(pos, b), _t(quat, b)
    r_all = ik(tp, tq)
    q_all, e_all, i_all = r_all.qpos.clone(), r_all.err_norm.clone(), r_all.info.clone()
    qst = before[0]   # the stored qpos (set_state may normalise the mug's quaternion)
    r_q = ik(tp, tq, qpos=qst)
    assert torch.equal(r_q.qpos, q_all) and torch.equal(r_q.err_norm, e_all) and torch.equal(r_q.info, i_all)
    ids = torch.tensor([5, 5, -1, 63, n, 0, 2 ** 31 - 1], dtype=torch.int32, device=b.device)
    valid = [0, 1, 3, 5]
    src = [5, 5, 63, 0]
    r_i = ik(tp[[5, 5, 0, 63, 0, 0, 0]].contiguous(), tq[[5, 5, 0, 63, 0, 0, 0]].contiguous(), env_ids=ids)
    for k, e in zip(valid, src):
        tgt = 5 if k < 2 else (63 if k == 3 else 0)
        ref = ik(tp[[tgt]].contiguous(), tq[[tgt]].contiguous(), qpos=qst[[e]].contiguous())
        assert torch.equal(r_i.qpos[k], ref.qpos[0]) and torch.equal(r_i.info[k], ref.info[0])
    for k in (2, 4, 6):
        assert torch.isnan(r_i.qpos[k]).all() and torch.isnan(r_i.err_norm[k]) and r_i.info[k].tolist() == [0, 3]
    after = b.get_state()
    assert all(torch.equal(x, y) for x, y in zip(before, after))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        out = torch.empty_like(q_all)
        ik(tp, tq, qpos=qst, qpos_out=out, err_norm=False, info=False)
    torch.cuda.current_stream().wait_stream(s)
    assert torch.equal(out, q_all)


def test_f32_against_f64(assets):
    """Where both precisions converge, their solutions' tcp poses agree (the joint angles themselves may differ by float32 rounding
    amplified by the conditioning)."""
    n = 256
    b64, b32 = _batch(assets, "main.xml", n, torch.float64), _batch(assets, "main.xml", n, torch.float32)
    _, qs, pos, quat = _targets(b64, n, 21)
    r64 = b64.ik(("site", "tcp"))(_t(pos, b64), _t(quat, b64), qpos=_t(qs, b64))
    r32 = b32.ik(("site", "tcp"))(_t(pos, b32), _t(quat, b32), qpos=_t(qs, b32))
    ok = (r64.info[:, 1] == 0).cpu().numpy() & (r32.info[:, 1] == 0).cpu().numpy()
    assert ok.mean() >= 0.99
    e32 = _pose_err(b64, r32.qpos.double().contiguous(), pos, quat)
    assert e32[ok].max() < 2e-5
    q64, q32 = r64.qpos.cpu().numpy(), r32.qpos.double().cpu().numpy()
    assert np.median(np.abs(q64 - q32).max(axis=1)[ok]) < 1e-3


def test_rejected_calls(assets):
    b = _batch(assets, "main.xml", 4, torch.float32)
    tp = torch.zeros(4, 3, device=b.device); tq = torch.zeros(4, 4, device=b.device)
    with pytest.raises(ValueError, match="not one of"):
        b.ik(("joint", 0))
    with pytest.raises(KeyError):
        b.ik(("site", "nope"))
    with pytest.raises(KeyError):
        b.ik(("site", "tcp"), joints=["nope"])
    with pytest.raises(ValueError, match="listed twice"):
        b.ik(("site", "tcp"), joints=[0, 0])
    with pytest.raises(ValueError, match="not a hinge"):
        b.ik(("site", "tcp"), joints=[b.model.njnt - 1])   # the mug's free joint
    with pytest.raises(ValueError, match="out of range"):
        b.ik(("geom", 10 ** 6))
    ik = b.ik(("site", "tcp"))
    assert ik.joints == list(range(6))
    for kw, exc, why in [(dict(), ValueError, "target"), (dict(target_pos=tp, env_ids=torch.zeros(4, dtype=torch.int32, device=b.device), qpos=torch.zeros(4, b.model.nq, device=b.device)), ValueError, "not both"),
                         (dict(target_pos=tp[:3].contiguous()), ValueError, "shape"), (dict(target_pos=tp.double()), ValueError, "float"),
                         (dict(target_pos=tp, qpos_out=False, err_norm=False, info=False), ValueError, "at least one"),
                         (dict(target_quat=tq, tol=-1.0), RuntimeError, "tol"), (dict(target_quat=tq, max_steps=0), RuntimeError, "max_steps"),
                         (dict(target_quat=tq, max_steps=10001), RuntimeError, "max_steps"), (dict(target_quat=tq, max_update_norm=0.0), RuntimeError, "max_update_norm"),
                         (dict(target_quat=tq, progress_thresh=float("nan")), RuntimeError, "progress_thresh"),
                         (dict(target_quat=tq, rot_weight=-1.0), RuntimeError, "rot_weight"),
                         (dict(target_quat=tq, regularization_strength=-1.0), RuntimeError, "regularization_strength"),
                         (dict(target_quat=tq, regularization_threshold=-1.0), RuntimeError, "regularization_threshold")]:
        with pytest.raises(exc, match=why):
            ik(**kw)
    # the C entry point's own checks: unknown id, m != n without a source, m < 1, NULL out
    L, s = b._L, b._stream()
    assert L.ur3e_batch_ik(b.ptr, 7, None, None, 4, tp.data_ptr(), None, None, lib.IKOut(None, tp.data_ptr(), None), s) != 0
    assert "unknown ik id" in lib.last_error()
    assert L.ur3e_batch_ik(b.ptr, ik.id, None, None, 3, tp.data_ptr(), None, None, lib.IKOut(None, tp.data_ptr(), None), s) != 0
    assert "m must equal n" in lib.last_error()
    assert L.ur3e_batch_ik(b.ptr, ik.id, None, tp.data_ptr(), 0, tp.data_ptr(), None, None, lib.IKOut(None, tp.data_ptr(), None), s) != 0
    assert "m=0" in lib.last_error()
    assert L.ur3e_batch_ik(b.ptr, ik.id, None, None, 4, tp.data_ptr(), None, None, None, s) != 0
    assert "out is null" in lib.last_error()
    assert L.ur3e_batch_ik(b.ptr, ik.id, None, None, 4, tp.data_ptr(), None, None, lib.IKOut(None, tp.data_ptr(), None), s) == 0   # NULL options


def test_trajectory_conversion(assets):
    """INTEGRATION.md's conversion of a build_traj_l line [T, N, 7] (pos, rotvec, grip) into joint waypoints for move_j.run: T calls,
    each seeded from the previous solution; every waypoint's tcp pose, through set_state + Query, matches its target.  The orientation line
    interpolates rotation vectors near the start's, as build_traj_l does; tol 1e-10 rather than the float64 default 1e-14, which sits
    at the rounding floor of err_norm."""
    N, T = 16, 10
    b = _batch(assets, "main.xml", N, torch.float64)
    key = b.model.keyframe("down").qpos
    q = torch.tensor(np.tile(key, (N, 1)), dtype=b.dtype, device=b.device)
    p0, m0 = _pose(b, q)
    rng = np.random.default_rng(4)
    from scipy.spatial.transform import Rotation
    rv0 = Rotation.from_matrix(m0).as_rotvec()
    start = np.hstack([p0, rv0, np.zeros((N, 1))])
    stop = start.copy(); stop[:, :3] += rng.uniform(-0.08, 0.08, (N, 3)); stop[:, 3:6] = rv0 + rng.uniform(-0.2, 0.2, (N, 3))
    traj = BT.build_traj_l_point_custom(start, stop, hold=1, num_points=T, device=b.device)   # [T, N, 7]
    ik = b.ik(("site", "tcp"))
    joint_traj = torch.empty(T, N, 7, dtype=b.dtype, device=b.device)
    for t in range(T):
        rv = traj[t, :, 3:6]
        ang = rv.norm(dim=1, keepdim=True)
        axis = torch.where(ang > 0, rv / ang.clamp_min(1e-300), torch.zeros_like(rv))
        quat = torch.cat([torch.cos(ang / 2), axis * torch.sin(ang / 2)], dim=1)
        r = ik(traj[t, :, :3].contiguous(), quat.contiguous(), qpos=q, tol=1e-10)
        q = r.qpos.clone()
        joint_traj[t, :, :6] = q[:, :6]; joint_traj[t, :, 6] = traj[t, :, 6]
        assert (r.info[:, 1] == 0).all()
        err = _pose_err(b, q, traj[t, :, :3].cpu().numpy(), quat.cpu().numpy())
        assert err.max() < 1e-9
