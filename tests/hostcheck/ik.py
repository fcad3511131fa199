"""TEST-ONLY helper: compile the inverse-kinematics solve (ik.cuh, see host_ik.cpp) as plain C++ and bind it."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SRCS = [os.path.join(HERE, "host_ik.cpp"), os.path.join(ROOT, "ur3e_b200", "csrc", "mjcf.cpp")]
OBJ_BODY, OBJ_XBODY, OBJ_GEOM, OBJ_SITE = 1, 2, 5, 6
_L = None


class Options(C.Structure):
    """ur3e_ik_options"""
    _fields_ = [(k, C.c_double) for k in ("tol", "rot_weight", "regularization_threshold", "regularization_strength", "max_update_norm",
                                          "progress_thresh")] + [("max_steps", C.c_int32), ("reserved_", C.c_int32)]


DEFAULTS = dict(tol=1e-14, rot_weight=1.0, regularization_threshold=0.1, regularization_strength=3e-2, max_update_norm=2.0, progress_thresh=20.0,
                max_steps=100)


def options(**kw):
    """Options with dm_control's float64 defaults, overridden by kw."""
    o = dict(DEFAULTS); o.update(kw)
    return Options(**o)


def lib():
    """Compiled once per process into a temporary directory (the tree may be read-only); the flags of tests/hostcheck/build.py."""
    global _L
    if _L is None:
        tmp = tempfile.mkdtemp(prefix="ur3e_hostik_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostik.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unused", "-ffp-contract=off", "-o", so] + SRCS)
        _L = C.CDLL(so)
        dp, ip, op = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(Options)
        _L.hi_ik.argtypes = [C.c_char_p, C.c_int, C.c_int, ip, C.c_int, dp, dp, dp, op, dp, dp, ip]
        _L.hi_ik_compile.argtypes = [C.c_char_p, C.c_int, C.c_int, ip, C.c_int]
        _L.hi_ik_check.argtypes = [C.c_int, C.c_int, C.c_longlong, C.c_longlong] + [C.c_int] * 6 + [op]
        _L.hi_error.restype = C.c_char_p
    return _L


def _ids(joints):
    j = np.ascontiguousarray(joints, dtype=np.int32).reshape(-1)
    return j, j.ctypes.data_as(C.POINTER(C.c_int32))


def ik(xml, objtype, objid, joints, qpos, target_pos=None, target_quat=None, **opt):
    """(qpos [nq], err_norm, steps, status) of one problem, float64, as the batch solves it; opt overrides dm_control's defaults
    (none given = the call's NULL options).  Raises ValueError with the reason when the family or the call is rejected."""
    dp = C.POINTER(C.c_double)
    j, jp = _ids(joints)
    q = np.ascontiguousarray(qpos, dtype=np.float64)
    tp = None if target_pos is None else np.ascontiguousarray(target_pos, dtype=np.float64)
    tq = None if target_quat is None else np.ascontiguousarray(target_quat, dtype=np.float64)
    qo, eo, info = np.full(q.size, np.nan), np.full(1, np.nan), np.full(2, -7, np.int32)
    o = C.byref(options(**opt)) if opt else None
    rc = lib().hi_ik(xml.encode(), int(objtype), int(objid), jp, len(j), q.ctypes.data_as(dp), tp.ctypes.data_as(dp) if tp is not None else None,
                     tq.ctypes.data_as(dp) if tq is not None else None, o, qo.ctypes.data_as(dp), eo.ctypes.data_as(dp),
                     info.ctypes.data_as(C.POINTER(C.c_int32)))
    if rc != 0:
        raise ValueError("hi_ik rejected the call (%d): %s" % (rc, lib().hi_error().decode()))
    return qo, float(eo[0]), int(info[0]), int(info[1])


def compile_check(xml, objtype, objid, joints, nj=None):
    """compile_ik: "" when ur3e_batch_ik_create accepts the family, else the reason."""
    j, jp = _ids(joints)
    L = lib()
    return "" if L.hi_ik_compile(xml.encode(), int(objtype), int(objid), jp if j.size else None, len(j) if nj is None else nj) == 0 else L.hi_error().decode()


def check(id_, nik, m, n, env_ids, qpos0, pos, quat, out, any_, opt=None):
    """ik_check: "" when ur3e_batch_ik accepts the combination, else the reason; opt a dict of overrides or None (NULL)."""
    L = lib()
    o = C.byref(options(**opt)) if opt is not None else None
    rc = L.hi_ik_check(id_, nik, m, n, int(env_ids), int(qpos0), int(pos), int(quat), int(out), int(any_), o)
    return "" if rc == 0 else L.hi_error().decode()
