"""Batched counterparts of the reference's state readers (utils/utils.py, controller/controller_func.py): same names, the
`d` argument is a SimBatch (or a UR3eVecEnv) instead of an MjData, and every value gains a leading environment axis.

    env = UR3eVecEnv("gymnasium_env/ur3e-v2", 4096); env.batch.enable_sensors(); env.reset(); env.step(a)
    get_jnt_torques(env)              # [N, 7]   utils/utils.py:201-211 (the seven actuatorfrc sensors)
    get_grasp_contact(env)            # ([N], [N])  utils/utils.py:243-245 (left, right touch sensor)
    get_boolean_grasp_contact(env)    # [N] bool    utils/utils.py:238-240
    get_task_space_state(env)         # [N, 7]   controller_func.py:191-200: tcp xpos, tcp rotvec, grasp flag
    get_joint_space_state(env)        # [N, 7]   controller_func.py:203-211: qpos[:6], grasp flag
    get_ctrl(env)                     # [N, 7]   d.ctrl as the fused controller set it (the `u` of pid_task_ctrl / move_j.ctrl)
    get_torque_sensors(env)           # [N, 6, 3]  the <torque> site sensors of assets/main.xml:384-391 (shoulder_pan .. wrist_3)

The sensors are the ones of the step's last mj_step (MuJoCo fills d.sensordata in the forward pass, before integrating),
so a call after `step` returns what the reference's loops log after `mj_step`.  Environments that were auto-reset in that
step report the sensors of their terminal step.

Poses and velocities of named objects (utils/utils.py:129-189, utils/gym_utils.py:20-39,207-219) take the reference's (m, d, name)
signature; `m` is accepted for drop-in use and may be None.  They run a kinematics query (SimBatch.query) at the stored state:

    get_site_xpos(m, d, "tcp")        # [N, 3]     d.site("tcp").xpos
    get_site_xmat / get_site_R        # [N, 9] / [N, 3, 3]
    get_site_xrotvec                  # [N, 3]     scipy Rotation.from_matrix(site_xmat).as_rotvec()
    get_site_vel(m, d, "tcp")         # [N, 6]     mj_objectVelocity(mjOBJ_SITE, flg_local=0): [rot(3), lin(3)]
    get_body_xpos / get_body_xmat     # [N, 3] / [N, 9]  d.body(name).xpos / .xmat (body frame)
    get_geom_xpos / get_geom_xmat     # [N, 3] / [N, 9]
    get_ghost_xpos(m, d)              # [N, 3]     body "ghost" (the v2 observation's target)
    get_finger_jnt_disp / _vel(m, d)  # [N]        qpos[6] / qvel[6]

These are MuJoCo's values after reset / set_state + mj_forward.  After a step MuJoCo's d.xpos etc. still hold the last substep's
pre-integration kinematics (SURVEY F9) while these are one substep newer; the stale tcp pose is get_task_space_state's.  Every
accessor reuses one cached query per (batch, kind, name): one kernel launch per call, and the returned tensor is overwritten by
the next call of the same accessor.

Jacobians, the mass matrix and the bias forces (controller_func.py:87-104, move_l.py:46-47,69-70) run Query.jac /
SimBatch.mass_matrix at the same stored state, one launch per call:

    mj_jacSite(m, d, jacp, jacr, site)    # writes jacp, jacr: caller tensors [N, 3, nv] or None; site an id or a name
    mj_jacBody / mj_jacBodyCom / mj_jacGeom(m, d, jacp, jacr, obj)   # body frame / centre of mass / geom
    get_full_M(m, d)                      # [N, nv, nv]  mj_fullM(m, M, d.qM)
    get_qfrc_bias(m, d)                   # [N, nv]      d.qfrc_bias

After a step MuJoCo's d.qfrc_bias and the Jacobian it would compute belong to the last substep's pre-integration state (SURVEY F9);
these are one substep newer, the same state as the pose accessors above.

The contact predicates (utils/gym_utils.py:98-201) read the contact list of SimBatch.forward at the same stored state; they need no
ctrl, so they run its contacts-only pass (kinematics and collision), one launch per call:

    get_ncon(m, d)                                   # [N] int32    d.ncon
    get_self_collision(m, d, collision_cache=None)   # [N] bool     two robot_base bodies not both in the gripper subtree touch
    get_table_collision(m, d, collision_cache=None)  # [N] bool     the gripper subtree touches the table
    get_block_grasp_state(m, d)                      # [N] int32    distinct pads touching the mug (the v0 observation's o[9])
    get_robust_block_grasp_state(m, d)               # [N] bool     both pads, and the tcp within the mug-handle thresholds

After a step MuJoCo's d.contact still holds the contacts of the last substep before integration (SURVEY F9); these are one substep
newer, the same state as the pose accessors above.
"""
import math

import torch


def _batch(d):
    return getattr(d, "batch", d)


def _sensors(d):
    b = _batch(d)
    if getattr(b, "sensors", None) is None:
        raise RuntimeError("sensor output is off: call batch.enable_sensors() before stepping")
    return b.sensors


def get_jnt_torques(d):
    return _sensors(d)[:, :7]


get_joint_torques = get_jnt_torques   # the name controller/move_*.py import (SURVEY F5)


def get_ctrl(d):
    """d.ctrl of the step's last mj_step, before MuJoCo's ctrlrange clamp (what the reference's loops store in `ctrls[t]`)."""
    return _sensors(d)[:, 21:28]


def get_torque_sensors(d):
    """d.sensor("<joint>_torque").data for the six arm joints: interaction torque between each link and its parent at the joint's
    force-torque site, in the site frame."""
    return _sensors(d)[:, 28:46].reshape(-1, 6, 3)


def get_grasp_contact(d):
    s = _sensors(d)
    return s[:, 8], s[:, 7]           # (left_pad1_contact, right_pad1_contact), the reference's order


def get_boolean_grasp_contact(d, contact_threshold=0.1):
    # the reference compares the TUPLE (left, right) > (thr, thr): lexicographic, i.e. left > thr, or left == thr and right > thr
    left, right = get_grasp_contact(d)
    return (left > contact_threshold) | ((left == contact_threshold) & (right > contact_threshold))


def _rotvec(R):
    """scipy Rotation.from_matrix(R).as_rotvec() for a batch of rotation matrices [N, 3, 3] (angle in [0, pi])."""
    t = R[:, 0, 0] + R[:, 1, 1] + R[:, 2, 2]
    # quaternion (w, x, y, z) by the largest-component rule, then canonical w >= 0
    q = torch.empty(R.shape[0], 4, dtype=R.dtype, device=R.device)
    c = torch.stack([t, R[:, 0, 0], R[:, 1, 1], R[:, 2, 2]], 1).argmax(1)
    for k in range(4):
        m = c == k
        if not m.any():
            continue
        r = R[m]
        if k == 0:
            w = 1 + r[:, 0, 0] + r[:, 1, 1] + r[:, 2, 2]
            qq = torch.stack([w, r[:, 2, 1] - r[:, 1, 2], r[:, 0, 2] - r[:, 2, 0], r[:, 1, 0] - r[:, 0, 1]], 1)
        else:
            i = k - 1; j = (i + 1) % 3; l = (i + 2) % 3
            v = [None] * 4
            v[1 + i] = 1 + r[:, i, i] - r[:, j, j] - r[:, l, l]
            v[1 + j] = r[:, j, i] + r[:, i, j]
            v[1 + l] = r[:, l, i] + r[:, i, l]
            v[0] = r[:, l, j] - r[:, j, l]
            qq = torch.stack(v, 1)
        q[m] = qq / qq.norm(dim=1, keepdim=True)
    q = torch.where(q[:, :1] < 0, -q, q)
    sn = q[:, 1:].norm(dim=1)
    ang = 2 * torch.atan2(sn, q[:, 0])
    k = torch.where(sn < 1e-12, torch.full_like(sn, 2.0), ang / sn.clamp_min(1e-300))
    return q[:, 1:] * k[:, None]


def get_task_space_state(d):
    """[tcp xpos (3), tcp rotvec (3), grasp flag] per environment (controller_func.py:191-200).  The tcp pose is the one of the
    step's last forward pass, i.e. the pose the next controller call will read (SURVEY F9)."""
    s = _sensors(d)
    pos, mat = s[:, 9:12], s[:, 12:21].reshape(-1, 3, 3)
    g = get_boolean_grasp_contact(d).to(pos.dtype)
    return torch.cat([pos, _rotvec(mat), g[:, None]], 1)


def get_joint_space_state(d):
    """[qpos[:6], grasp flag] per environment (controller_func.py:203-211)."""
    b = _batch(d)
    qpos, _, _ = b.get_state()
    return torch.cat([qpos[:, :6], get_boolean_grasp_contact(d).to(qpos.dtype)[:, None]], 1)


def _query(d, kind, name):
    b = _batch(d)
    cache = b.__dict__.setdefault("_accessor_queries", {})
    q = cache.get((kind, name))
    if q is None:
        q = cache[(kind, name)] = b.query([(kind, name)])
    return q


def _pos(d, kind, name):
    return _query(d, kind, name)(pos=True)[0][:, 0]


def _mat(d, kind, name):
    return _query(d, kind, name)(pos=False, mat=True)[1][:, 0]


def get_site_xpos(m, d, name):
    return _pos(d, "site", name)


def get_site_R(m, d, name):
    return _mat(d, "site", name)


def get_site_xmat(m, d, name):
    return get_site_R(m, d, name).reshape(-1, 9)


def get_site_xrotvec(m, d, name):
    return _rotvec(get_site_R(m, d, name))


def get_site_vel(m, d, name):
    """mj_objectVelocity(mjOBJ_SITE, flg_local=0): [angular (3), linear (3)] in world axes."""
    return _query(d, "site", name)(pos=False, vel=True)[2][:, 0]


def get_body_xpos(m, d, name):
    return _pos(d, "xbody", name)


def get_body_xmat(m, d, name):
    return _mat(d, "xbody", name).reshape(-1, 9)


def get_geom_xpos(m, d, name):
    return _pos(d, "geom", name)


def get_geom_xmat(m, d, name):
    return _mat(d, "geom", name).reshape(-1, 9)


def get_ghost_xpos(m, d):
    return get_body_xpos(m, d, "ghost")


def get_finger_jnt_disp(m, d):
    return _batch(d).get_state()[0][:, 6]


def get_finger_jnt_vel(m, d):
    return _batch(d).get_state()[1][:, 6]


def _jac(d, kind, obj, jacp, jacr):
    """MuJoCo's mj_jac* calling convention: writes into jacp / jacr ([N, 3, nv] tensors, either may be None), returns nothing."""
    if jacp is None and jacr is None:
        return
    b = _batch(d)
    nv = b.model.nv
    outs = []
    for t in (jacp, jacr):
        if t is None:
            outs.append(False)
        else:
            b._chk(t, (b.n, 3, nv))
            outs.append(t.view(b.n, 1, 3, nv))   # the query's [N, k = 1, 3, nv] layout, same memory
    _query(d, kind, obj).jac(jacp=outs[0], jacr=outs[1])


def mj_jacSite(m, d, jacp, jacr, site):
    _jac(d, "site", site, jacp, jacr)


def mj_jacBody(m, d, jacp, jacr, body):
    """Jacobian of the body frame's origin (d.xpos[body])."""
    _jac(d, "xbody", body, jacp, jacr)


def mj_jacBodyCom(m, d, jacp, jacr, body):
    """Jacobian of the body's centre of mass (d.xipos[body])."""
    _jac(d, "body", body, jacp, jacr)


def mj_jacGeom(m, d, jacp, jacr, geom):
    _jac(d, "geom", geom, jacp, jacr)


def get_full_M(m, d):
    return _batch(d).mass_matrix(M=True)[0]


def get_qfrc_bias(m, d):
    return _batch(d).mass_matrix(M=False, qfrc_bias=True)[1]


def _contact_flags(d):
    """contact_bits of every environment (1 mug - left pad, 2 mug - right pad, 4 gripper - table, 8 self-collision), one launch."""
    return _batch(d).forward(qacc=False, flags=True).flags


def init_collision_cache(m):
    """Accepted for drop-in use: the batch classifies the collidable geoms once, when it is created.  Returns an opaque value that
    the collision accessors ignore."""
    return None


def get_ncon(m, d):
    return _batch(d).forward(qacc=False, info=True).info[:, 0]


def get_self_collision(m, d, collision_cache=None):
    return (_contact_flags(d) & 8) != 0


def get_table_collision(m, d, collision_cache=None):
    return (_contact_flags(d) & 4) != 0


def get_block_grasp_state(m, d):
    """Number of distinct gripper pads (left_pad, right_pad bodies) in contact with the mug: 0, 1 or 2 (gym_utils.py:108-128, the v0
    observation's o[9]).  The reference's exact signature is not recorded in this repository; (m, d) follows its other accessors."""
    f = _contact_flags(d)
    return (f & 1) + ((f >> 1) & 1)


def get_robust_block_grasp_state(m, d):
    """Both pads touch the mug and the tcp is within (0.01, 0.005, 0.05) of the handle_site per axis (gym_utils.py:98-106, the v2
    observation's o[23]).  Two launches: the contact flags and one kinematics query of the two sites.  The reference's exact
    signature is not recorded in this repository; (m, d) follows its other accessors."""
    both = (_contact_flags(d) & 3) == 3
    p = _query_pair(d, (("site", "tcp"), ("site", "handle_site")))(pos=True)[0]
    e = (p[:, 0] - p[:, 1]).abs()
    return both & (e[:, 0] < 0.01) & (e[:, 1] < 0.005) & (e[:, 2] < 0.05)


def _query_pair(d, objects):
    b = _batch(d)
    cache = b.__dict__.setdefault("_accessor_queries", {})
    q = cache.get(objects)
    if q is None:
        q = cache[objects] = b.query(list(objects))
    return q
