"""TEST-ONLY helper: compile the kinematics-query source (ur3e_b200/csrc/query.cuh) as plain C++ (see host_query.cpp) and bind it."""
import ctypes as C
import atexit
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "ur3e_b200", "csrc")
SRCS = [os.path.join(HERE, "host_query.cpp"), os.path.join(CSRC, "mjcf.cpp")]
DEPS = SRCS + [os.path.join(CSRC, f) for f in ("query.cuh", "query_model.h", "engine.cuh", "warp_model.cuh", "dev_model.h", "compile_model.h",
                                                "host_model.h", "xml_mini.h", "merge_bodies.h")] + [os.path.join(ROOT, "include", "ur3e_b200.h")]
_L = None


def lib():
    """Compiled once per process into a temporary directory (the tree may be read-only)."""
    global _L
    if _L is None:
        tmp = tempfile.mkdtemp(prefix="ur3e_hostquery_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostquery.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unused", "-ffp-contract=off", "-o", so] + SRCS)
        _L = C.CDLL(so)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        _L.hc_query.argtypes = [C.c_char_p, dp, dp, ip, ip, C.c_int, C.c_int, dp, dp, dp]
    return _L


def query(xml, qpos, qvel, objtype, objid, local=0):
    """(pos [k, 3], mat [k, 3, 3], vel [k, 6]) of the objects at (qpos, qvel), float64."""
    k = len(objtype)
    pos = np.zeros((k, 3)); mat = np.zeros((k, 9)); vel = np.zeros((k, 6))
    qp, qv = (np.ascontiguousarray(x, dtype=np.float64) for x in (qpos, qvel))
    t, i = (np.ascontiguousarray(x, dtype=np.int32) for x in (objtype, objid))
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    rc = lib().hc_query(xml.encode(), dp(qp), dp(qv), ip(t), ip(i), k, int(local), dp(pos), dp(mat), dp(vel))
    if rc != 0:
        raise ValueError("hc_query rejected the query (%d)" % rc)
    return pos, mat.reshape(k, 3, 3), vel
