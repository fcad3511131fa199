"""TEST-ONLY helper: compile the forward-dynamics query source (ur3e_b200/csrc/query_fwd.cuh forward_query_env) as plain C++ (see
host_forward.cpp) and bind it."""
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
SRCS = [os.path.join(HERE, "host_forward.cpp"), os.path.join(CSRC, "mjcf.cpp")]
NSENSOR = 46
FLOAT_OUTS = ("qacc", "qfrc_constraint", "contact_dist", "contact_pos", "contact_frame", "contact_force", "sensordata")
INT_OUTS = ("info", "contact_geom", "flags")
_L = None


def lib():
    """Compiled once per process into a temporary directory (the tree may be read-only)."""
    global _L
    if _L is None:
        tmp = tempfile.mkdtemp(prefix="ur3e_hostforward_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostforward.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unused", "-ffp-contract=off", "-o", so] + SRCS)
        _L = C.CDLL(so)
        dp = C.POINTER(C.c_double)
        _L.hc_forward.argtypes = [C.c_char_p, dp, dp, dp, dp, C.POINTER(dp), C.POINTER(C.POINTER(C.c_int32))]
        _L.hc_max_contacts.argtypes = [C.c_char_p]
        _L.hc_forward_check.argtypes = [C.c_int] * 4
    return _L


def check(out, con, any_, ncmax):
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
    rc = lib().hc_forward(xml.encode(), qp.ctypes.data_as(dp), qv.ctypes.data_as(dp), w.ctypes.data_as(dp), u.ctypes.data_as(dp) if u is not None else None, fo, io)
    if rc != 0:
        raise ValueError("hc_forward rejected the call (%d)" % rc)
    if "flags" in out:
        out["flags"] = int(out["flags"][0])
    return out
