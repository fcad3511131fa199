"""TEST-ONLY reference for the inverse-dynamics query: MuJoCo 3.3.3's mj_inverse (soft constraints, Euler, no sensors) restated from
its definition on top of the float64 oracle's position and velocity stages.

    fwd_position + fwd_velocity   the oracle's forward() at (qpos, qvel), ctrl 0 (it leaves kinematics, cinert, cdof, cdof_dot, cvel,
                                  qM, qfrc_bias, qfrc_passive, the contacts and the rows with efc_J, efc_D and efc_aref)
    mj_discreteAcc                a = qM^-1 (qM + h diag(damping)) qacc through the dense qM's Cholesky factor (discrete only)
    mj_invConstraint              efc_force = the constraint law at jar = J a - aref (mj_constraintUpdate: equality, friction loss,
                                  limits, elliptic cones), qfrc_constraint = J^T efc_force
    qfrc_inverse                  rne(flg_acc = 1) + armature a - qfrc_passive - qfrc_constraint

The M a of the kernel (a product with the packed M) is not this route: here the body accelerations are propagated down the tree and the
inertial wrenches summed back up (mj_rne with the acceleration term), with the armature added per dof."""
import numpy as np
import scipy.linalg

from oracle import oracle as O

EQUALITY, FRICTION, LIMIT, ELLIPTIC = 0, 1, 3, 7   # the oracle's efc_type values (mjCNSTR_*)


def _mul_inert(i, v):
    """cinert (10: I00 I11 I22 I01 I02 I12, m c, m) times a motion vector [rot, lin] about the tree's reference point."""
    I = np.array([[i[0], i[3], i[4]], [i[3], i[1], i[5]], [i[4], i[5], i[2]]]); h = i[6:9]; mass = i[9]
    return np.hstack([I @ v[:3] + np.cross(h, v[3:]), mass * v[3:] - np.cross(h, v[:3])])


def rne_acc(m, d, qacc):
    """mj_rne(flg_acc = 1): M qacc + qfrc_bias without the armature, by the recursive Newton-Euler pass over the oracle's cinert, cvel,
    cdof and cdof_dot."""
    nb, nv = m.nbody, m.nv
    par, dofbody = m.py["body_parentid"], m.py["dof_bodyid"]
    cin = d.arr("cinert").reshape(nb, 10); cvel = d.arr("cvel").reshape(nb, 6)
    cdof = d.arr("cdof").reshape(nv, 6); cdd = d.arr("cdof_dot").reshape(nv, 6); qvel = d.arr("qvel")
    cacc = np.zeros((nb, 6)); cacc[0, 3:] = -np.asarray(m.py["opt"]["gravity"], dtype=float)
    cfrc = np.zeros((nb, 6))
    for b in range(1, nb):
        cacc[b] = cacc[par[b]]
        for k in range(nv):
            if dofbody[k] == b:
                cacc[b] = cacc[b] + cdd[k] * qvel[k] + cdof[k] * qacc[k]
        Iv = _mul_inert(cin[b], cvel[b])
        cfrc[b] = _mul_inert(cin[b], cacc[b]) + np.hstack([np.cross(cvel[b, :3], Iv[:3]) + np.cross(cvel[b, 3:], Iv[3:]), np.cross(cvel[b, :3], Iv[3:])])
    for b in range(nb - 1, 0, -1):
        if par[b] > 0:
            cfrc[par[b]] += cfrc[b]
    return np.array([cdof[k] @ cfrc[dofbody[k]] for k in range(nv)])


def constraint_force(m, d, jar):
    """mj_constraintUpdate's efc_force at jar (no cone Hessian), row by row on the oracle's rows."""
    nefc = d.nefc
    t, Dr, fl = d.arr("efc_type")[:nefc], d.arr("efc_D")[:nefc], d.arr("efc_frictionloss")[:nefc]
    f = np.zeros(nefc)
    for r in range(nefc):
        if t[r] == EQUALITY:
            f[r] = -Dr[r] * jar[r]
        elif t[r] == FRICTION:
            rf = fl[r] / Dr[r]
            f[r] = fl[r] if jar[r] <= -rf else (-fl[r] if jar[r] >= rf else -Dr[r] * jar[r])
        elif t[r] == LIMIT:
            f[r] = -Dr[r] * jar[r] if jar[r] < 0 else 0.0
    for c in d.contacts():
        a = c.efc_address
        if a < 0:
            continue
        mu, fr = c.mu, np.array(c.friction[:2])
        U = np.hstack([jar[a] * mu, jar[a + 1:a + 3] * fr])
        N, T = U[0], float(np.hypot(U[1], U[2]))
        if N >= mu * T or (T <= 0 and N >= 0):
            f[a:a + 3] = 0.0
        elif mu * N + T <= 0 or (T <= 0 and N < 0):
            f[a:a + 3] = -Dr[a:a + 3] * jar[a:a + 3]
        else:
            Dm = Dr[a] / (mu * mu * (1 + mu * mu))
            f0 = -Dm * (N - mu * T) * mu
            f[a] = f0; f[a + 1:a + 3] = -f0 / T * U[1:] * fr
    return f


def inverse(m, qpos, qvel, qacc, discrete=False):
    """mj_inverse at (qpos, qvel, qacc) of the oracle model m: dict with qfrc_inverse, qfrc_constraint, ncon, nefc, contact_geom [ncon, 2]
    and contact_force [ncon, 6] (0 for a contact without rows), plus the continuous acceleration a it used and the oracle Data."""
    d = O.Data(m); d.reset(); d.set_state(qpos, qvel); d.forward()
    nv, h = m.nv, m.timestep
    qacc = np.asarray(qacc, dtype=np.float64)
    damping = np.asarray(m.arr("dof_damping"), dtype=np.float64)
    a = qacc.copy()
    if discrete and (damping > 0).any():
        M = d.fullM()
        a = scipy.linalg.cho_solve(scipy.linalg.cho_factor(M, lower=True), M @ qacc + h * damping * qacc)
    nefc = d.nefc
    J = d.arr("efc_J")[:nefc * nv].reshape(nefc, nv)
    f = constraint_force(m, d, J @ a - d.arr("efc_aref")[:nefc])
    qfrc_constraint = J.T @ f
    qfrc_inverse = rne_acc(m, d, a) + np.asarray(m.arr("dof_armature")) * a - d.arr("qfrc_passive") - qfrc_constraint
    con = d.contacts()
    cf = np.zeros((len(con), 6))
    for k, c in enumerate(con):
        if c.efc_address >= 0:
            cf[k, :3] = f[c.efc_address:c.efc_address + 3]
    return dict(qfrc_inverse=qfrc_inverse, qfrc_constraint=qfrc_constraint, ncon=d.ncon, nefc=nefc, a=a, data=d,
                contact_geom=np.array([[c.geom1, c.geom2] for c in con], dtype=np.int64).reshape(-1, 2), contact_force=cf)
