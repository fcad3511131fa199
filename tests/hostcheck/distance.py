"""TEST-ONLY helper: compile the geom-distance pass (distance.cuh, see host_distance.cpp) as plain C++ and bind it."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SRCS = [os.path.join(HERE, "host_distance.cpp"), os.path.join(ROOT, "ur3e_b200", "csrc", "mjcf.cpp")]
_L = None


def lib():
    """Compiled once per process into a temporary directory (the tree may be read-only); the flags of tests/hostcheck/build.py."""
    global _L
    if _L is None:
        tmp = tempfile.mkdtemp(prefix="ur3e_hostdist_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostdist.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unused", "-ffp-contract=off", "-o", so] + SRCS)
        _L = C.CDLL(so)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        _L.hd_pair.argtypes = [C.c_int, C.c_int, dp, dp, dp, C.c_int, dp, dp, dp, C.c_double, dp]
        _L.hd_pair.restype = None
        _L.hd_distance.argtypes = [C.c_char_p, C.c_int, ip, ip, C.c_int, dp, C.c_double, dp, dp]
        _L.hd_compile.argtypes = [C.c_char_p, ip, ip, C.c_int]
        _L.hd_check.argtypes = [C.c_int, C.c_int, C.c_longlong, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_double]
        _L.hd_rows.argtypes = [C.c_char_p, C.c_int]
        _L.hd_error.restype = C.c_char_p
    return _L


def _d(a):
    a = np.ascontiguousarray(a, dtype=np.float64).reshape(-1)
    return a, a.ctypes.data_as(C.POINTER(C.c_double))


def _i(a):
    a = np.ascontiguousarray(a, dtype=np.int32).reshape(-1)
    return a, a.ctypes.data_as(C.POINTER(C.c_int32))


def pair(g1, g2, distmax=np.inf, use_float=False):
    """geom_distance of one pair at given world poses: g = (p [3], R [3, 3], size [3], is_plane).  Returns (dist, fromto [6])."""
    keep, args = [], []
    for p, R, s, pl in (g1, g2):
        args.append(int(bool(pl)))
        for x in (p, R, s):
            a, ptr = _d(x); keep.append(a); args.append(ptr)
    out = np.full(7, np.nan)
    lib().hd_pair(int(bool(use_float)), *args, C.c_double(distmax), out.ctypes.data_as(C.POINTER(C.c_double)))
    return float(out[0]), out[1:].copy()


def distance(xml, geom1, geom2, qpos, distmax=np.inf, use_float=False):
    """(dist [k], fromto [k, 6]) of the pairs at qpos, as one warp of ur3e_batch_distance computes them.  Raises ValueError with the
    reason when the pair set is rejected."""
    a, ap = _i(geom1)
    b, bp = _i(geom2)
    q, qp = _d(qpos)
    k = a.size
    dist, fromto = np.full(k, np.nan), np.full((k, 6), np.nan)
    rc = lib().hd_distance(xml.encode(), int(bool(use_float)), ap, bp, k, qp, C.c_double(distmax), dist.ctypes.data_as(C.POINTER(C.c_double)),
                           fromto.ctypes.data_as(C.POINTER(C.c_double)))
    if rc != 0:
        raise ValueError("hd_distance rejected the pair set (%d): %s" % (rc, lib().hd_error().decode()))
    return dist, fromto


def compile_check(xml, geom1, geom2, k=None):
    """compile_distance: "" when ur3e_batch_distance_create accepts the pair set, else the reason."""
    a, ap = _i(geom1)
    b, bp = _i(geom2)
    L = lib()
    return "" if L.hd_compile(xml.encode(), ap if a.size else None, bp if b.size else None, a.size if k is None else k) == 0 else L.hd_error().decode()


def check(id_, ndist, m, n, env_ids, qpos, any_, distmax=np.inf):
    """distance_check: "" when ur3e_batch_distance accepts the combination, else the reason."""
    L = lib()
    return "" if L.hd_check(id_, ndist, m, n, int(env_ids), int(qpos), int(any_), C.c_double(distmax)) == 0 else L.hd_error().decode()


def rows(xml, use_float=False):
    """Staging rows per warp of the overlapping path for the model's size class."""
    return lib().hd_rows(xml.encode(), int(bool(use_float)))
