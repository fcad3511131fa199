"""TEST-ONLY helper: compile the renderer's source (render.cuh, see host_render.cpp) as plain C++ and bind it."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from ur3e_b200._lib import Camera

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SRCS = [os.path.join(HERE, "host_render.cpp"), os.path.join(ROOT, "ur3e_b200", "csrc", "mjcf.cpp")]
_L = None


def lib():
    """Compiled once per process into a temporary directory (the tree may be read-only); the flags of tests/hostcheck/build.py."""
    global _L
    if _L is None:
        tmp = tempfile.mkdtemp(prefix="ur3e_hostrender_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostrender.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unused", "-ffp-contract=off", "-o", so] + SRCS)
        _L = C.CDLL(so)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        _L.hr_render.argtypes = [C.c_char_p, dp, C.POINTER(Camera), ip, C.c_int, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_void_p, dp, ip, dp]
        _L.hr_render_check.argtypes = [C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_longlong, C.c_int]
        _L.hr_error.restype = C.c_char_p
    return _L


def _p(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def render(xml, qpos, cam, geom_ids, width, height, rgba=None):
    """One environment at qpos rendered by the host-compiled render.cuh, float64: (rgb [H, W, 3] uint8, depth [H, W], seg [H, W]
    int32, pose [k + 1, 12]).  cam: a ur3e_b200._lib.Camera, or None (a null camera).  Raises ValueError with the reason when the
    renderer is rejected."""
    k = len(geom_ids)
    rgb = np.zeros((height, width, 3), np.uint8); depth = np.full((height, width), np.nan); seg = np.full((height, width), -7, np.int32)
    pose = np.full((k + 1, 12), np.nan)
    ids = np.ascontiguousarray(geom_ids, dtype=np.int32)
    col = None if rgba is None else np.ascontiguousarray(rgba, dtype=np.float32)
    qp = np.ascontiguousarray(qpos, dtype=np.float64)
    camp = C.byref(cam) if cam is not None else C.cast(None, C.POINTER(Camera))
    rc = lib().hr_render(xml.encode(), _p(qp), camp, ids.ctypes.data_as(C.POINTER(C.c_int32)), k,
                         col.ctypes.data_as(C.POINTER(C.c_float)) if col is not None else None, width, height, rgb.ctypes.data, _p(depth),
                         seg.ctypes.data_as(C.POINTER(C.c_int32)), _p(pose))
    if rc != 0:
        raise ValueError("hr_render rejected the renderer (%d): %s" % (rc, lib().hr_error().decode()))
    return rgb, depth, seg, pose


def render_check(render_id, nrender, any_, m, n, env_ids):
    """render_check: "" when ur3e_batch_render accepts the combination, else the reason."""
    L = lib()
    return "" if L.hr_render_check(render_id, nrender, int(any_), m, n, int(env_ids)) == 0 else L.hr_error().decode()
