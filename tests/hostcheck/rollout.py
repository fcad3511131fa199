"""TEST-ONLY helper: compile the rollout's argument check (rollout.h, see host_rollout.cpp) as plain C++ and bind it."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
_L = None


def lib():
    """Compiled once per process into a temporary directory (the tree may be read-only)."""
    global _L
    if _L is None:
        tmp = tempfile.mkdtemp(prefix="ur3e_hostrollout_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostrollout.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, os.path.join(HERE, "host_rollout.cpp")])
        _L = C.CDLL(so)
        _L.hro_rollout_check.argtypes = [C.c_longlong, C.c_longlong] + [C.c_int] * 7
        _L.hro_error.restype = C.c_char_p
    return _L


def rollout_check(m, T, actions=True, src_ids=True, qpos0=False, qvel0=False, ws0=False, out=True, any_=True):
    """rollout_check: "" when ur3e_batch_rollout accepts the combination, else the reason."""
    L = lib()
    rc = L.hro_rollout_check(m, T, int(actions), int(src_ids), int(qpos0), int(qvel0), int(ws0), int(out), int(any_))
    return "" if rc == 0 else L.hro_error().decode()
