"""ctypes binding of libur3e_b200.so (include/ur3e_b200.h).  There is no CPU fallback: if the CUDA
library is missing or no GPU is present, constructing a batch raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("UR3E_B200_LIB") or os.path.join(_HERE, "libur3e_b200.so")   # the override selects a variant build (tools/canary_check.sh)

F32, F64 = 0, 1
OBJ_BODY, OBJ_JOINT, OBJ_GEOM, OBJ_SITE, OBJ_TENDON, OBJ_ACTUATOR, OBJ_KEY = 1, 3, 5, 6, 18, 19, 23
OBJ_XBODY = 2   # body frame (mjOBJ_XBODY), kinematics queries only
CTRL_RAW, CTRL_PD_JOINT, CTRL_PID_TASK, CTRL_PID_TASK_ENV, CTRL_PINV = 0, 1, 2, 3, 4
OBS_STATE, OBS_V2, OBS_V0, OBS_DIRECT = 0, 1, 2, 3
REW_NONE, REW_V2, REW_V0, REW_MINUS1 = 0, 1, 2, 3
TERM_NONE, TERM_V2, TERM_V0 = 0, 1, 2
NOISE_NONE, NOISE_LOW, NOISE_MED, NOISE_HIGH = 0, 1, 2, 3
STAT_NAMES = ["episodes", "return_sum", "length_sum", "successes", "term_reach", "term_toppled", "term_collision", "truncations",
              "unstable_resets", "nefc_sum", "ncon_sum", "solver_iter_sum", "substeps", "overflow_steps", "pad_contact_steps", "steps"]
NSENSOR = 46
SENSOR_NCTRL = 7   # d.ctrl columns of the sensor record, [21, 28), zero past nu (utils.get_ctrl)


class ModelDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("nq", "nv", "nu", "nbody", "njnt", "ngeom", "nsite", "neq", "ntendon", "npair", "nkey")] + [("timestep", C.c_double)]


class EnvConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("ctrl_mode", "obs_kind", "reward_kind", "term_kind", "frame_skip", "act_dim", "obs_dim", "max_steps",
                                          "reset_key", "reset_noise", "auto_reset", "solver_iterations")] + [
        ("solver_tolerance", C.c_double), ("gains", C.c_double * 24), ("tool_rotvec", C.c_double * 3), ("env_id_base", C.c_int64),
        ("single_tier", C.c_int32), ("lite_max_contacts", C.c_int32), ("lite_max_rows", C.c_int32), ("reserved_", C.c_int32)]


# ur3e_forward_out: the ten device pointers of ur3e_batch_forward, in this order (FORWARD_OUTPUTS)
FORWARD_OUTPUTS = ("qacc", "qfrc_constraint", "info", "contact_geom", "contact_dist", "contact_pos", "contact_frame", "contact_force", "flags", "sensordata")


class ForwardOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in FORWARD_OUTPUTS]


# ur3e_rollout_out: the eight device pointers of ur3e_batch_rollout, in this order (ROLLOUT_OUTPUTS)
ROLLOUT_OUTPUTS = ("qpos", "qvel", "obs", "reward", "terminated", "truncated", "sensordata", "info")


class RolloutOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ROLLOUT_OUTPUTS]


class Camera(C.Structure):
    """ur3e_camera: anchor (objtype -1 = world, OBJ_XBODY or OBJ_SITE; objid), pos / xyaxes in the anchor frame, fovy (degrees), znear, zfar."""
    _fields_ = [("objtype", C.c_int32), ("objid", C.c_int32), ("pos", C.c_double * 3), ("xyaxes", C.c_double * 6), ("fovy", C.c_double),
                ("znear", C.c_double), ("zfar", C.c_double)]


EXPORTS = ["ur3e_last_error", "ur3e_model_load", "ur3e_model_destroy", "ur3e_model_info", "ur3e_model_name2id", "ur3e_model_id2name",
           "ur3e_model_array", "ur3e_model_num_warnings", "ur3e_model_warning", "ur3e_batch_create", "ur3e_batch_destroy", "ur3e_batch_reset",
           "ur3e_batch_step", "ur3e_batch_step_host", "ur3e_batch_get_state", "ur3e_batch_set_state", "ur3e_batch_stats", "ur3e_batch_set_sensor_buffer",
           "ur3e_batch_launch_count", "ur3e_batch_kernel_info", "ur3e_batch_state_bytes", "ur3e_batch_tier_info", "ur3e_batch_kernel_timing", "ur3e_batch_kernel_times", "ur3e_batch_mid_tier_info",
           "ur3e_batch_query_create", "ur3e_batch_query", "ur3e_batch_query_jac", "ur3e_batch_max_contacts", "ur3e_batch_forward",
           "ur3e_batch_render_create", "ur3e_batch_render", "ur3e_batch_rollout"]

_lib = None


def load():
    """Load the shared library and declare the prototypes of every symbol in include/ur3e_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (ur3e_b200 has no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, cp, i64, u8p, dp = C.c_void_p, C.c_char_p, C.c_int64, C.c_void_p, C.POINTER(C.c_double)
    L.ur3e_last_error.restype = cp; L.ur3e_last_error.argtypes = []
    L.ur3e_model_load.restype = vp; L.ur3e_model_load.argtypes = [cp]
    L.ur3e_model_destroy.restype = None; L.ur3e_model_destroy.argtypes = [vp]
    L.ur3e_model_info.argtypes = [vp, C.POINTER(ModelDims)]
    L.ur3e_model_name2id.argtypes = [vp, C.c_int, cp]
    L.ur3e_model_id2name.restype = cp; L.ur3e_model_id2name.argtypes = [vp, C.c_int, C.c_int]
    L.ur3e_model_array.argtypes = [vp, cp, C.POINTER(vp), C.POINTER(i64), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.ur3e_model_num_warnings.argtypes = [vp]
    L.ur3e_model_warning.restype = cp; L.ur3e_model_warning.argtypes = [vp, C.c_int]
    L.ur3e_batch_create.restype = vp; L.ur3e_batch_create.argtypes = [vp, C.POINTER(EnvConfig), i64, C.c_int, C.c_int]
    L.ur3e_batch_destroy.restype = None; L.ur3e_batch_destroy.argtypes = [vp]
    L.ur3e_batch_reset.argtypes = [vp, u8p, C.c_uint64, vp, vp]
    L.ur3e_batch_step.argtypes = [vp, vp, vp, vp, u8p, u8p, vp, vp]
    L.ur3e_batch_step_host.argtypes = [vp, vp, vp, vp, u8p, u8p]
    L.ur3e_batch_get_state.argtypes = [vp, vp, vp, vp, vp]
    L.ur3e_batch_set_state.argtypes = [vp, vp, vp, vp, vp]
    L.ur3e_batch_stats.argtypes = [vp, vp, C.c_int, vp]
    L.ur3e_batch_set_sensor_buffer.argtypes = [vp, vp]
    L.ur3e_batch_launch_count.restype = i64; L.ur3e_batch_launch_count.argtypes = [vp]
    L.ur3e_batch_kernel_info.argtypes = [vp] + [C.POINTER(C.c_int32)] * 4
    L.ur3e_batch_state_bytes.argtypes = [vp]
    L.ur3e_batch_tier_info.argtypes = [vp, C.POINTER(C.c_int64)]
    L.ur3e_batch_mid_tier_info.argtypes = [vp] + [C.POINTER(C.c_int32)] * 3
    L.ur3e_batch_kernel_timing.argtypes = [vp, C.c_int]
    L.ur3e_batch_kernel_times.argtypes = [vp, dp]
    L.ur3e_batch_query_create.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int32]
    L.ur3e_batch_query.argtypes = [vp, C.c_int, vp, vp, vp, C.c_int, vp]
    L.ur3e_batch_query_jac.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp]
    L.ur3e_batch_max_contacts.argtypes = [vp]
    L.ur3e_batch_forward.argtypes = [vp, vp, C.POINTER(ForwardOut), vp]
    L.ur3e_batch_render_create.argtypes = [vp, C.POINTER(Camera), C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_float), C.c_int32, C.c_int32]
    L.ur3e_batch_render.argtypes = [vp, C.c_int, vp, i64, vp, vp, vp, vp]
    L.ur3e_batch_rollout.argtypes = [vp, vp, vp, vp, vp, i64, C.c_int32, vp, C.POINTER(RolloutOut), vp]
    _lib = L
    return L


def last_error():
    return load().ur3e_last_error().decode()


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (what, rc, last_error()))
