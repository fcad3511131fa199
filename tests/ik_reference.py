"""TEST-ONLY reference for the inverse-kinematics solve: dm_control.utils.inverse_kinematics.qpos_from_site_pose restated in numpy on the
float64 oracle, with the batch's documented differences (ur3e_b200/csrc/ik.cuh).

    kinematics        the oracle's set_state + forward (the object's frame from d.site_xpos / d.xpos / d.xipos / d.geom_xpos and
                      their xmat); the Jacobian from mj_jacSite, or mj_jac at the object's point for the other kinds
    rotation error    mju_mat2Quat -> mju_mulQuat(target, mju_negQuat(current)) -> mju_quat2Vel, as dm_control computes it
    the step          dm_control's nullspace_method: the nj x nj normal equations, np.linalg.solve with regularisation, np.linalg.lstsq
                      without (numpy's default cut-off: the minimum-norm step; dm_control's rcond=-1 keeps rounding-noise singular
                      values of the rank-deficient J^T J when r < nj)
    differences       the clamp of limited joints to jnt_range; err_norm and steps describe the returned qpos (the error is evaluated
                      after the last update too, and converged means that configuration is within tol)

This is a different route from the kernel's: quaternions instead of rot_err's matrix -> rotation vector, the oracle's Jacobians
instead of jac_col() on cdof, and the nj x nj normal equations instead of the push-through form J^T (J J^T + lambda I)^-1 e."""
import numpy as np

from oracle import oracle as O

BODY, XBODY, GEOM, SITE = 1, 2, 5, 6   # UR3E_OBJ_*
CONVERGED, MAX_STEPS, NO_PROGRESS = 0, 1, 2
DEFAULTS = dict(tol=1e-14, rot_weight=1.0, regularization_threshold=0.1, regularization_strength=3e-2, max_update_norm=2.0, progress_thresh=20.0,
                max_steps=100)


def mat2quat(R):
    """mju_mat2Quat of a row-major 3 x 3 rotation."""
    m = np.asarray(R, dtype=np.float64).reshape(9)
    q = np.zeros(4)
    if m[0] + m[4] + m[8] > 0:
        q[0] = 0.5 * np.sqrt(1 + m[0] + m[4] + m[8])
        q[1:] = 0.25 * np.array([m[7] - m[5], m[2] - m[6], m[3] - m[1]]) / q[0]
    elif m[0] > m[4] and m[0] > m[8]:
        q[1] = 0.5 * np.sqrt(1 + m[0] - m[4] - m[8])
        q[0], q[2], q[3] = 0.25 * np.array([m[7] - m[5], m[1] + m[3], m[2] + m[6]]) / q[1]
    elif m[4] > m[8]:
        q[2] = 0.5 * np.sqrt(1 - m[0] + m[4] - m[8])
        q[0], q[1], q[3] = 0.25 * np.array([m[2] - m[6], m[1] + m[3], m[5] + m[7]]) / q[2]
    else:
        q[3] = 0.5 * np.sqrt(1 - m[0] - m[4] + m[8])
        q[0], q[1], q[2] = 0.25 * np.array([m[3] - m[1], m[2] + m[6], m[5] + m[7]]) / q[3]
    return normalize4(q)


def normalize4(q):
    """mju_normalize4: a quaternion of norm < 1e-15 becomes the identity."""
    q = np.asarray(q, dtype=np.float64)
    n = np.linalg.norm(q)
    return np.array([1.0, 0, 0, 0]) if n < 1e-15 else q / n


def mulquat(a, b):
    """mju_mulQuat"""
    return np.array([a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                     a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]])


def quat2vel(q):
    """mju_quat2Vel(q, dt = 1): axis times angle, the angle wrapped into (-pi, pi]."""
    axis = np.asarray(q[1:], dtype=np.float64)
    s = np.linalg.norm(axis)
    axis = axis / s if s >= 1e-15 else np.array([1.0, 0, 0])
    a = 2 * np.arctan2(s, q[0])
    if a > np.pi:
        a -= 2 * np.pi
    return axis * a


def frame(m, d, objtype, objid):
    """(world point [3], rotation [3, 3], jacp [3, nv], jacr [3, nv]) of the object after d.forward()."""
    pos, mat = {BODY: ("xipos", "ximat"), XBODY: ("xpos", "xmat"), GEOM: ("geom_xpos", "geom_xmat"), SITE: ("site_xpos", "site_xmat")}[objtype]
    p = d.arr(pos).reshape(-1, 3)[objid].copy(); R = d.arr(mat).reshape(-1, 3, 3)[objid].copy()
    if objtype == SITE:
        jp, jr = d.jac_site(objid)
    else:
        body = objid if objtype in (BODY, XBODY) else m.py["geom_bodyid"][objid]
        jp, jr = d.jac(p, body)
    return p, R, jp, jr


def solve(m, objtype, objid, joints, qpos, target_pos=None, target_quat=None, **opt):
    """(qpos [nq], err_norm, steps, status) of one problem on the oracle model m; opt overrides dm_control's float64 defaults."""
    o = dict(DEFAULTS); o.update(opt)
    jt, jd, jq = m.py["jnt_type"], m.py["jnt_dofadr"], m.py["jnt_qposadr"]
    lim, rng = np.asarray(m.py["jnt_limited"]), np.asarray(m.py["jnt_range"], dtype=np.float64).reshape(-1, 2)
    joints = [int(j) for j in joints]
    assert all(jt[j] in (2, 3) for j in joints)   # hinge or slide
    dofs = [jd[j] for j in joints]
    tq = None if target_quat is None else normalize4(target_quat)
    q = np.array(qpos, dtype=np.float64)
    d = O.Data(m); d.reset()
    steps, status = 0, MAX_STEPS
    while True:
        d.set_state(q, np.zeros(m.nv)); d.forward()
        p, R, jp, jr = frame(m, d, objtype, objid)
        err, rows, err_norm = [], [], 0.0
        if target_pos is not None:
            e = np.asarray(target_pos, dtype=np.float64) - p
            err.append(e); rows.append(jp); err_norm += np.linalg.norm(e)
        if tq is not None:
            cur = mat2quat(R)
            e = quat2vel(mulquat(tq, cur * np.array([1, -1, -1, -1])))
            err.append(e); rows.append(jr); err_norm += o["rot_weight"] * np.linalg.norm(e)
        if err_norm < o["tol"]:
            status = CONVERGED
            break
        if steps == o["max_steps"]:
            break
        J = np.vstack(rows)[:, dofs]; e = np.concatenate(err)
        H, g = J.T @ J, J.T @ e
        if err_norm > o["regularization_threshold"]:
            dq = np.linalg.solve(H + o["regularization_strength"] * np.eye(len(dofs)), g)
        else:
            dq = np.linalg.lstsq(H, g, rcond=None)[0]
        dn = np.linalg.norm(dq)
        with np.errstate(divide="ignore"):
            if err_norm / dn > o["progress_thresh"]:
                status = NO_PROGRESS
                break
        if dn > o["max_update_norm"]:
            dq *= o["max_update_norm"] / dn
        for j, v in zip(joints, dq):
            a = jq[j]
            q[a] += v
            if lim[j]:
                q[a] = min(max(q[a], rng[j, 0]), rng[j, 1])
        steps += 1
    return q, err_norm, steps, status
