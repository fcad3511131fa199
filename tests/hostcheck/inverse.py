"""TEST-ONLY helper: compile the inverse-dynamics query's source (query_inv.cuh, see host_inverse.cpp) as plain C++ and bind it."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SRCS = [os.path.join(HERE, "host_inverse.cpp"), os.path.join(ROOT, "ur3e_b200", "csrc", "mjcf.cpp")]
_L = None


def lib():
    """Compiled once per process into a temporary directory (the tree may be read-only); the flags of tests/hostcheck/build.py."""
    global _L
    if _L is None:
        tmp = tempfile.mkdtemp(prefix="ur3e_hostinverse_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostinverse.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unused", "-ffp-contract=off", "-o", so] + SRCS)
        _L = C.CDLL(so)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        _L.hi_inverse.argtypes = [C.c_char_p, dp, dp, dp, C.c_int, dp, dp, ip, ip, dp]
        _L.hi_inverse_check.argtypes = [C.c_int, C.c_int, C.c_longlong, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        _L.hi_max_contacts.argtypes = [C.c_char_p]
        _L.hi_error.restype = C.c_char_p
    return _L


def max_contacts(xml):
    return lib().hi_max_contacts(xml.encode())


def inverse(xml, qpos, qvel, qacc, discrete=False, qfrc_inverse=True, qfrc_constraint=True, info=True, contact_geom=True, contact_force=True):
    """dict of the requested outputs of mj_inverse at (qpos, qvel, qacc), float64, as the batch computes them; shapes as SimBatch.inverse's
    without the state axis.  Outputs are pre-filled with NaN / a sentinel, so that an entry the pass leaves unwritten shows.  Contact
    outputs are skipped for a model without contact pairs.  Raises ValueError with the reason when the call is rejected."""
    nv, Cn = len(qvel), max_contacts(xml)
    want = dict(qfrc_inverse=(qfrc_inverse, (nv,), np.float64), qfrc_constraint=(qfrc_constraint, (nv,), np.float64),
                info=(info, (3,), np.int32), contact_geom=(contact_geom and Cn > 0, (Cn, 2), np.int32),
                contact_force=(contact_force and Cn > 0, (Cn, 6), np.float64))
    out = {k: (np.full(s, np.nan) if t is np.float64 else np.full(s, -7, np.int32)) for k, (w, s, t) in want.items() if w}
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    ptr = lambda k, t: out[k].ctypes.data_as(t) if k in out else None
    qp, qv, qa = (np.ascontiguousarray(x, dtype=np.float64) for x in (qpos, qvel, qacc))
    rc = lib().hi_inverse(xml.encode(), qp.ctypes.data_as(dp), qv.ctypes.data_as(dp), qa.ctypes.data_as(dp), int(bool(discrete)),
                          ptr("qfrc_inverse", dp), ptr("qfrc_constraint", dp), ptr("info", ip), ptr("contact_geom", ip), ptr("contact_force", dp))
    if rc != 0:
        raise ValueError("hi_inverse rejected the call (%d): %s" % (rc, lib().hi_error().decode()))
    return out


def inverse_check(qpos, qvel, m, n, qacc, out, con, any_, ncmax):
    """inverse_query_check: "" when ur3e_batch_inverse accepts the combination, else the reason."""
    L = lib()
    return "" if L.hi_inverse_check(int(qpos), int(qvel), m, n, int(qacc), int(out), int(con), int(any_), int(ncmax)) == 0 else L.hi_error().decode()
