"""TEST-ONLY helper: compile the kernel source (engine.cuh) and the query sources (query.cuh, query_fwd.cuh) as plain C++ (see
host_check.cpp) and bind them."""
import ctypes as C
import atexit
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SRCS = [os.path.join(HERE, "host_check.cpp"), os.path.join(ROOT, "ur3e_b200", "csrc", "mjcf.cpp")]
NSENSOR = 46
FLOAT_OUTS = ("qacc", "qfrc_constraint", "contact_dist", "contact_pos", "contact_frame", "contact_force", "sensordata")
INT_OUTS = ("info", "contact_geom", "flags")
_L = None


def lib():
    """Compiled once per process into a temporary directory (the tree may be read-only)."""
    global _L
    if _L is None:
        tmp = tempfile.mkdtemp(prefix="ur3e_hostcheck_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostcheck.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unused", "-ffp-contract=off", "-o", so] + SRCS)
        _L = C.CDLL(so)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        _L.hc_query.argtypes = [C.c_char_p, dp, dp, ip, ip, C.c_int, C.c_int, dp, dp, dp]
        _L.hc_query_jac.argtypes = [C.c_char_p, dp, dp, ip, ip, C.c_int, C.c_int, dp, dp, dp, dp]
        _L.hc_forward.argtypes = [C.c_char_p, dp, dp, dp, dp, C.POINTER(dp), C.POINTER(ip)]
        _L.hc_max_contacts.argtypes = [C.c_char_p]
        _L.hc_forward_check.argtypes = [C.c_int] * 4
        _L.hc_box_box.argtypes = [C.c_int, dp, dp, dp, dp, dp, dp, C.c_double, dp]
        _L.hc_plane_box.argtypes = [C.c_int, dp, dp, dp, dp, dp, C.c_double, dp]
    return _L


def _p(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def run(xml, qpos, qvel, ctrl, ws, nsteps, use_float=0, max_iter=50, tol=1e-15):
    L = lib()
    dims = np.zeros(11, dtype=np.int32)
    assert L.hc_model_dims(xml.encode(), dims.ctypes.data_as(C.POINTER(C.c_int))) == 0
    nq, nv = int(dims[0]), int(dims[1])
    oq = np.zeros(nq); ov = np.zeros(nv); oa = np.zeros(nv); oM = np.zeros((nv, nv)); ob = np.zeros(nv); ofc = np.zeros(nv); info = np.zeros(8, dtype=np.int32)
    a = [np.ascontiguousarray(x, dtype=np.float64) for x in (qpos, qvel, ctrl, ws)]
    rc = L.hc_run(xml.encode(), use_float, _p(a[0]), _p(a[1]), _p(a[2]), _p(a[3]), nsteps, max_iter, C.c_double(tol), _p(oq), _p(ov), _p(oa), _p(oM), _p(ob), _p(ofc),
                  info.ctypes.data_as(C.POINTER(C.c_int)))
    assert rc == 0
    return dict(qpos=oq, qvel=ov, qacc=oa, M=oM, bias=ob, fc=ofc, ncon=int(info[0]), nefc=int(info[1]), iters=int(info[2]), warn=int(info[3]), overflow=int(info[4]), arena=int(info[5]))


def sensors(xml, qpos, qvel, ctrl):
    """The step kernel's logging record (include/ur3e_b200.h UR3E_NSENSOR) after a forward pass at the given state."""
    out = np.zeros(NSENSOR)
    a = [np.ascontiguousarray(x, dtype=np.float64) for x in (qpos, qvel, ctrl)]
    assert lib().hc_sensors(xml.encode(), _p(a[0]), _p(a[1]), _p(a[2]), _p(out)) == 0
    return out


def model_array(xml, name, cap=8192):
    out = np.zeros(cap)
    k = lib().hc_model_array(xml.encode(), name.encode(), _p(out), cap)
    assert k >= 0, name
    return out[:k]


def query(xml, qpos, qvel, objtype, objid, local=0):
    """(pos [k, 3], mat [k, 3, 3], vel [k, 6]) of the objects at (qpos, qvel), float64."""
    k = len(objtype)
    pos = np.zeros((k, 3)); mat = np.zeros((k, 9)); vel = np.zeros((k, 6))
    qp, qv = (np.ascontiguousarray(x, dtype=np.float64) for x in (qpos, qvel))
    t, i = (np.ascontiguousarray(x, dtype=np.int32) for x in (objtype, objid))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    rc = lib().hc_query(xml.encode(), _p(qp), _p(qv), ip(t), ip(i), k, int(local), _p(pos), _p(mat), _p(vel))
    if rc != 0:
        raise ValueError("hc_query rejected the query (%d)" % rc)
    return pos, mat.reshape(k, 3, 3), vel


def query_jac(xml, qpos, qvel, objtype=(), objid=(), jacp=True, jacr=True, M=True, qfrc_bias=True, query_id=None):
    """(jacp [k, 3, nv], jacr [k, 3, nv], M [nv, nv], qfrc_bias [nv]) at (qpos, qvel), float64, None for an output not asked for.
    The objects are compiled as the batch's query 0 (none when empty); query_id defaults to 0 with objects, -1 without."""
    k, nv = len(objtype), len(qvel)
    if query_id is None:
        query_id = 0 if k else -1
    outs = [np.zeros(s) if want else None for want, s in ((jacp, (k, 3, nv)), (jacr, (k, 3, nv)), (M, (nv, nv)), (qfrc_bias, (nv,)))]
    qp, qv = (np.ascontiguousarray(x, dtype=np.float64) for x in (qpos, qvel))
    t, i = (np.ascontiguousarray(x, dtype=np.int32).reshape(-1) for x in (objtype, objid))
    dp = lambda a: _p(a) if a is not None else None
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    rc = lib().hc_query_jac(xml.encode(), _p(qp), _p(qv), ip(t), ip(i), k, int(query_id), *[dp(o) for o in outs])
    if rc != 0:
        raise ValueError("hc_query_jac rejected the call (%d)" % rc)
    return tuple(outs)


STAGE_W = 3 + 4 * 8   # engine.cuh: normal, then STAGE_PTS x (pos, dist)


def _stage(n, row):
    """(n, normal [3], pos [n, 3], dist [n]) of a staging row.  Past the n points the row holds box_box's frames and clip
    polygon, which collision() never reads."""
    pts = row[3:3 + 4 * n].reshape(n, 4)
    return n, row[:3].copy(), pts[:, :3].copy(), pts[:, 3].copy()


def box_box(p1, R1, s1, p2, R2, s2, margin=0.0, use_float=False):
    """The kernel's box_box<float / double> on boxes (centre, world frame [3, 3], half-sizes): (n, normal from box 1 to box 2,
    pos [n, 3], dist [n]).  The normal is meaningless when n = 0."""
    a = [np.ascontiguousarray(x, dtype=np.float64).reshape(-1) for x in (p1, R1, s1, p2, R2, s2)]
    row = np.zeros(STAGE_W)
    n = lib().hc_box_box(int(bool(use_float)), *[_p(x) for x in a], C.c_double(margin), _p(row))
    return _stage(n, row)


def plane_box(ppos, pmat, bpos, bmat, size, margin=0.0, use_float=False):
    """The kernel's plane_box<float / double>: (n, plane normal, pos [n, 3], dist [n]), at most 4 corners in corner order."""
    a = [np.ascontiguousarray(x, dtype=np.float64).reshape(-1) for x in (ppos, pmat, bpos, bmat, size)]
    row = np.zeros(STAGE_W)
    n = lib().hc_plane_box(int(bool(use_float)), *[_p(x) for x in a], C.c_double(margin), _p(row))
    return _stage(n, row)


def forward_check(out, con, any_, ncmax):
    """forward_query_check: True when ur3e_batch_forward accepts the combination."""
    return lib().hc_forward_check(int(out), int(con), int(any_), int(ncmax)) == 0


def max_contacts(xml):
    return lib().hc_max_contacts(xml.encode())


def forward(xml, qpos, qvel, ws=None, ctrl=None, qacc=True, qfrc_constraint=False, info=False, contact_geom=False, contact_dist=False,
            contact_pos=False, contact_frame=False, contact_force=False, flags=False, sensordata=False):
    """dict of the requested outputs of one mj_forward at (qpos, qvel, warm start ws = 0 by default) with ctrl (None = zero), float64;
    shapes as SimBatch.forward's without the environment axis (contact_frame [C, 3, 3]).  Outputs are pre-filled with NaN / a sentinel,
    so that an entry the query leaves unwritten shows.  Raises ValueError when the call is rejected."""
    nv, Cn = len(qvel), max_contacts(xml)
    want = dict(qacc=qacc, qfrc_constraint=qfrc_constraint, info=info, contact_geom=contact_geom, contact_dist=contact_dist,
                contact_pos=contact_pos, contact_frame=contact_frame, contact_force=contact_force, flags=flags, sensordata=sensordata)
    shape = dict(qacc=(nv,), qfrc_constraint=(nv,), info=(4,), contact_geom=(Cn, 2), contact_dist=(Cn,), contact_pos=(Cn, 3),
                 contact_frame=(Cn, 3, 3), contact_force=(Cn, 6), flags=(1,), sensordata=(NSENSOR,))
    out = {}
    for k, w in want.items():
        if w:
            out[k] = np.full(shape[k], -7, dtype=np.int32) if k in INT_OUTS else np.full(shape[k], np.nan)
            if out[k].size == 0:   # a zero-length output still counts as asked for (the call then rejects it)
                out[k] = np.full(1, np.nan)
    dp = C.POINTER(C.c_double); ip = C.POINTER(C.c_int32)
    fo = (dp * len(FLOAT_OUTS))(*[out[k].ctypes.data_as(dp) if k in out else dp() for k in FLOAT_OUTS])
    io = (ip * len(INT_OUTS))(*[out[k].ctypes.data_as(ip) if k in out else ip() for k in INT_OUTS])
    qp, qv = (np.ascontiguousarray(x, dtype=np.float64) for x in (qpos, qvel))
    w = np.zeros(nv) if ws is None else np.ascontiguousarray(ws, dtype=np.float64)
    u = None if ctrl is None else np.ascontiguousarray(ctrl, dtype=np.float64)
    rc = lib().hc_forward(xml.encode(), _p(qp), _p(qv), _p(w), _p(u) if u is not None else None, fo, io)
    if rc != 0:
        raise ValueError("hc_forward rejected the call (%d)" % rc)
    if "flags" in out:
        out["flags"] = int(out["flags"][0])
    return out
