"""TEST-ONLY helper: compile the Jacobian / mass-matrix query source (ur3e_b200/csrc/query.cuh query_jac_env) as plain C++ (see
host_query_jac.cpp) and bind it."""
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
SRCS = [os.path.join(HERE, "host_query_jac.cpp"), os.path.join(CSRC, "mjcf.cpp")]
_L = None


def lib():
    """Compiled once per process into a temporary directory (the tree may be read-only)."""
    global _L
    if _L is None:
        tmp = tempfile.mkdtemp(prefix="ur3e_hostqueryjac_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostqueryjac.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unused", "-ffp-contract=off", "-o", so] + SRCS)
        _L = C.CDLL(so)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        _L.hc_query_jac.argtypes = [C.c_char_p, dp, dp, ip, ip, C.c_int, C.c_int, dp, dp, dp, dp]
    return _L


def query_jac(xml, qpos, qvel, objtype=(), objid=(), jacp=True, jacr=True, M=True, qfrc_bias=True, query_id=None):
    """(jacp [k, 3, nv], jacr [k, 3, nv], M [nv, nv], qfrc_bias [nv]) at (qpos, qvel), float64, None for an output not asked for.
    The objects are compiled as the batch's query 0 (none when empty); query_id defaults to 0 with objects, -1 without."""
    k, nv = len(objtype), len(qvel)
    if query_id is None:
        query_id = 0 if k else -1
    outs = [np.zeros(s) if want else None for want, s in ((jacp, (k, 3, nv)), (jacr, (k, 3, nv)), (M, (nv, nv)), (qfrc_bias, (nv,)))]
    qp, qv = (np.ascontiguousarray(x, dtype=np.float64) for x in (qpos, qvel))
    t, i = (np.ascontiguousarray(x, dtype=np.int32).reshape(-1) for x in (objtype, objid))
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    rc = lib().hc_query_jac(xml.encode(), dp(qp), dp(qv), ip(t), ip(i), k, int(query_id), *[dp(o) for o in outs])
    if rc != 0:
        raise ValueError("hc_query_jac rejected the call (%d)" % rc)
    return tuple(outs)
