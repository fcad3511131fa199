"""SimBatch: N environments resident on one B200, stepped by one fused kernel launch.

Thin torch front-end over the C ABI (include/ur3e_b200.h): tensors are passed by `data_ptr()`, zero-copy;
torch supplies device memory and streams only.  dtype float32 = production, float64 = validation build.
"""
import ctypes as C
from collections import namedtuple

import numpy as np
import torch

from . import _lib
from .model import Model


def env_config(**kw):
    c = _lib.EnvConfig()
    c.frame_skip = 1; c.reset_key = -1; c.auto_reset = 0
    gains = kw.pop("gains", None)
    rotvec = kw.pop("tool_rotvec", (-1.209, -1.209, 1.209))   # reference ur3e_env2.py:74
    for k, v in kw.items():
        if not hasattr(c, k):
            raise TypeError("unknown env_config field %r" % k)
        setattr(c, k, v)
    if gains is not None:
        g = list(np.asarray(gains, dtype=np.float64).ravel())
        if len(g) > 24:
            raise ValueError("at most 24 gains")
        for i, v in enumerate(g):
            c.gains[i] = v
    for i in range(3):
        c.tool_rotvec[i] = rotvec[i]
    return c


ForwardResult = namedtuple("ForwardResult", _lib.FORWARD_OUTPUTS)


class SimBatch:
    def __init__(self, model, cfg, n_envs, device=0, dtype=torch.float32):
        if not torch.cuda.is_available():
            raise RuntimeError("ur3e_b200 needs a CUDA device (there is no CPU fallback)")
        self._L = _lib.load()
        self.model = model if isinstance(model, Model) else Model(model)
        self.cfg = cfg
        self.n = int(n_envs)
        self.device = torch.device("cuda", device)
        self.dtype = dtype
        code = {torch.float32: _lib.F32, torch.float64: _lib.F64}[dtype]
        self.ptr = self._L.ur3e_batch_create(self.model.ptr, C.byref(cfg), self.n, device, code)
        if not self.ptr:
            raise RuntimeError("ur3e_batch_create: " + _lib.last_error())
        self.obs_dim, self.act_dim = cfg.obs_dim, cfg.act_dim
        kw = dict(device=self.device)
        self.obs = torch.zeros(self.n, self.obs_dim, dtype=dtype, **kw)
        self.final_obs = torch.zeros(self.n, self.obs_dim, dtype=dtype, **kw)
        self.reward = torch.zeros(self.n, dtype=dtype, **kw)
        self.terminated = torch.zeros(self.n, dtype=torch.uint8, **kw)
        self.truncated = torch.zeros(self.n, dtype=torch.uint8, **kw)
        self._stats = torch.zeros(16, dtype=torch.float64, **kw)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _chk(self, t, shape, dtype=None):
        dtype = dtype or self.dtype
        if not (t.is_cuda and t.device == self.device and t.dtype == dtype and t.is_contiguous() and tuple(t.shape) == tuple(shape)):
            raise ValueError("expected a contiguous %s tensor of shape %s on %s, got %s %s on %s" % (dtype, tuple(shape), self.device, t.dtype, tuple(t.shape), t.device))
        return C.c_void_p(t.data_ptr())

    def reset(self, seed=0, mask=None):
        mp = None
        if mask is not None:
            mask = mask.to(torch.uint8).contiguous()
            mp = self._chk(mask, (self.n,), torch.uint8)
        _lib.check(self._L.ur3e_batch_reset(self.ptr, mp, seed, C.c_void_p(self.obs.data_ptr()), self._stream()), "ur3e_batch_reset")
        return self.obs

    def step(self, actions, want_final_obs=True):
        """One env-step for every environment (one kernel launch).  Returns views of the batch-owned output tensors."""
        a = self._chk(actions, (self.n, self.act_dim))
        fo = C.c_void_p(self.final_obs.data_ptr()) if want_final_obs else None
        _lib.check(self._L.ur3e_batch_step(self.ptr, a, C.c_void_p(self.obs.data_ptr()), C.c_void_p(self.reward.data_ptr()),
                                           C.c_void_p(self.terminated.data_ptr()), C.c_void_p(self.truncated.data_ptr()), fo, self._stream()), "ur3e_batch_step")
        return self.obs, self.reward, self.terminated, self.truncated

    def step_host(self, actions, obs, reward, terminated, truncated):
        """Host-buffer entry point (numpy arrays or pinned CPU tensors): H2D, step, D2H, synchronise."""
        def p(x):
            return C.c_void_p(x.data_ptr() if isinstance(x, torch.Tensor) else x.ctypes.data)
        _lib.check(self._L.ur3e_batch_step_host(self.ptr, p(actions), p(obs), p(reward), p(terminated), p(truncated)), "ur3e_batch_step_host")

    def get_state(self):
        qpos = torch.empty(self.n, self.model.nq, dtype=self.dtype, device=self.device)
        qvel = torch.empty(self.n, self.model.nv, dtype=self.dtype, device=self.device)
        ws = torch.empty(self.n, self.model.nv, dtype=self.dtype, device=self.device)
        _lib.check(self._L.ur3e_batch_get_state(self.ptr, C.c_void_p(qpos.data_ptr()), C.c_void_p(qvel.data_ptr()), C.c_void_p(ws.data_ptr()), self._stream()), "ur3e_batch_get_state")
        return qpos, qvel, ws

    def set_state(self, qpos, qvel, qacc_warmstart=None):
        """MujocoEnv.set_state: write qpos/qvel for every env and run the forward pass (fresh kinematics cache)."""
        qp = self._chk(qpos, (self.n, self.model.nq)); qv = self._chk(qvel, (self.n, self.model.nv))
        ws = self._chk(qacc_warmstart, (self.n, self.model.nv)) if qacc_warmstart is not None else None
        _lib.check(self._L.ur3e_batch_set_state(self.ptr, qp, qv, ws, self._stream()), "ur3e_batch_set_state")

    def enable_sensors(self, on=True):
        """Attach (or detach) the [n, 21] logging output: after every step `self.sensors` holds, from the step's last mj_step,
        7 x actuatorfrc, the two touch sensors (reference assets/main.xml:392-408) and the tcp site pose; see ur3e_b200/utils.py."""
        self.sensors = torch.zeros(self.n, _lib.NSENSOR, dtype=self.dtype, device=self.device) if on else None
        _lib.check(self._L.ur3e_batch_set_sensor_buffer(self.ptr, C.c_void_p(self.sensors.data_ptr()) if on else None), "ur3e_batch_set_sensor_buffer")
        return self.sensors

    def stats(self, reset=True):
        _lib.check(self._L.ur3e_batch_stats(self.ptr, C.c_void_p(self._stats.data_ptr()), int(reset), self._stream()), "ur3e_batch_stats")
        return self._stats

    def stats_dict(self, reset=True):
        v = self.stats(reset).cpu().numpy()
        return {k: float(v[i]) for i, k in enumerate(_lib.STAT_NAMES)}

    def query(self, objects):
        """A kinematics query over a fixed list of objects: [(kind, name_or_id), ...] with kind "body" (inertial frame, d.xipos /
        d.ximat), "xbody" (body frame, d.xpos / d.xmat, what d.body(name).xpos returns), "geom" or "site".  See Query."""
        return Query(self, objects)

    def mass_matrix(self, M=True, qfrc_bias=False):
        """mj_fullM and d.qfrc_bias of every environment at the stored state: (M [n, nv, nv], qfrc_bias [n, nv]), None for an
        output not asked for.  One launch on the current torch stream; the output convention and the semantics are Query.jac's
        (this is Query.jac without objects)."""
        nv = self.model.nv
        outs = _outs(self, self.__dict__.setdefault("_mass_own", {}), "mass_matrix",
                     dict(M=(M, (self.n, nv, nv), None), qfrc_bias=(qfrc_bias, (self.n, nv), None)))
        _lib.check(self._L.ur3e_batch_query_jac(self.ptr, -1, None, None, *map(_ptr, outs.values()), self._stream()), "ur3e_batch_query_jac")
        return tuple(outs.values())

    @property
    def max_contacts(self):
        """C: contacts stored per environment by the step's largest size class and by forward() (24 for main.xml, 12 for
        ur3e_2f85.xml, 0 for a model without contact pairs)."""
        return int(self._L.ur3e_batch_max_contacts(self.ptr))

    def forward(self, ctrl=None, qacc=True, qfrc_constraint=False, info=False, contact_geom=False, contact_dist=False, contact_pos=False,
                contact_frame=False, contact_force=False, flags=False, sensordata=False):
        """One mj_forward per environment at the stored state (ur3e_batch_forward): one launch on the current torch stream,
        returning a ForwardResult named tuple with None for every output not asked for.  Each output argument is False, True (a
        tensor owned by the batch, overwritten by the next call) or a tensor of its shape to write into; the integer outputs are
        int32, the others in the batch's dtype.  C = max_contacts.

            qacc, qfrc_constraint [n, nv]      d.qacc, d.qfrc_constraint
            info [n, 4] int32                  ncon, nefc, solver iterations, overflow bits (1 contacts, 2 constraint rows)
            contact_geom [n, C, 2] int32       d.contact[k].geom1 / geom2 (ids of the loaded model), -1 past ncon
            contact_dist [n, C], contact_pos [n, C, 3], contact_frame [n, C, 3, 3]   d.contact[k].dist / pos / frame (row 0: the
                                               normal, from geom1 to geom2)
            contact_force [n, C, 6]            mj_contactForce: [fn, ft1, ft2, 0, 0, 0] in the contact frame
            flags [n] int32                    1 mug - left pad, 2 mug - right pad, 4 gripper - table, 8 self-collision, over
                                               all ncon contacts (on a row overflow the step's bits see only those with rows)
            sensordata [n, 46]                 the layout of the step's sensor record (enable_sensors)

        Entries past ncon are geom -1 and zeros.  Contacts are in pair-list order, then in the narrow phase's point order within a pair.
        ctrl [n, nu] (batch dtype, any strides: a strided tensor is copied) is the actuation the dynamics see; None means zero.  The
        [n, 7] d.ctrl block of the sensor record is accepted as it is (its columns past nu are zero), so passing
        ur3e_b200.utils.get_ctrl(self) (with sensors enabled) applies the actuation of the last step.  When only contact geometry, info or flags are asked for, the
        kernel runs kinematics and collision alone: info then reports nefc = 0 and 0 iterations.

        The values are mj_forward's at the stored state (qpos, qvel and the solver's warm start), i.e. MuJoCo's d.contact,
        d.efc_force, d.qacc and d.sensordata after reset or set_state.  After a step MuJoCo's d.contact still holds the contacts of
        the last substep before integration (SURVEY F9); these are one substep newer, the state query() sees.
        """
        n, nv, Cn = self.n, self.model.nv, self.max_contacts
        i32 = torch.int32
        table = dict(qacc=(qacc, (n, nv), None), qfrc_constraint=(qfrc_constraint, (n, nv), None), info=(info, (n, 4), i32),
                     contact_geom=(contact_geom, (n, Cn, 2), i32), contact_dist=(contact_dist, (n, Cn), None),
                     contact_pos=(contact_pos, (n, Cn, 3), None), contact_frame=(contact_frame, (n, Cn, 3, 3), None),
                     contact_force=(contact_force, (n, Cn, 6), None), flags=(flags, (n,), i32), sensordata=(sensordata, (n, _lib.NSENSOR), None))
        if Cn == 0:
            asked = [k for k, (a, _, _) in table.items() if k.startswith("contact_") and a is not False and a is not None]
            if asked:
                raise ValueError("%s: the model has no contact pairs (max_contacts = 0)" % ", ".join(asked))
        outs = ForwardResult(**_outs(self, self.__dict__.setdefault("_forward_own", {}), "forward", table))
        u = None
        if ctrl is not None:
            nu = self.model.nu
            if tuple(ctrl.shape) == (n, _lib.SENSOR_NCTRL) and nu < _lib.SENSOR_NCTRL:
                ctrl = ctrl[:, :nu]   # utils.get_ctrl's width: the record pads d.ctrl with zeros past nu
            # the kernel reads ctrl + e * nu: a strided view (get_ctrl's rows are NSENSOR apart) is copied, on the current stream
            ctrl = ctrl.contiguous()
            u = self._chk(ctrl, (n, nu))
        st = _lib.ForwardOut(*[o.data_ptr() if o is not None else None for o in outs])
        _lib.check(self._L.ur3e_batch_forward(self.ptr, u, C.byref(st), self._stream()), "ur3e_batch_forward")
        return outs

    @property
    def launch_count(self):
        return int(self._L.ur3e_batch_launch_count(self.ptr))

    def kernel_info(self):
        v = [C.c_int32() for _ in range(4)]
        _lib.check(self._L.ur3e_batch_kernel_info(self.ptr, *[C.byref(x) for x in v]), "ur3e_batch_kernel_info")
        t = (C.c_int64 * 8)()
        _lib.check(self._L.ur3e_batch_tier_info(self.ptr, t), "ur3e_batch_tier_info")
        d = dict(arena_bytes=v[0].value, warps_per_block=v[1].value, blocks_per_sm=v[2].value, regs_per_thread=v[3].value,
                 state_bytes=int(self._L.ur3e_batch_state_bytes(self.ptr)))
        if t[0]:
            d["lite"] = dict(arena_bytes=int(t[0]), warps_per_block=int(t[1]), blocks_per_sm=int(t[2]), regs_per_thread=int(t[3]),
                             lite_tier_steps=int(t[4]), full_only_steps=int(t[5]), last_overflow_envs=int(t[6]))
            mv = [C.c_int32() for _ in range(3)]
            _lib.check(self._L.ur3e_batch_mid_tier_info(self.ptr, *[C.byref(x) for x in mv]), "ur3e_batch_mid_tier_info")
            if mv[0].value:
                d["grasp_tier"] = dict(arena_bytes=mv[0].value, warps_per_block=mv[1].value, regs_per_thread=mv[2].value)
        return d

    def kernel_timing(self, enable=True):
        """Bracket every step-kernel launch with CUDA events on the launching stream (measurement aid, see kernel_times)."""
        _lib.check(self._L.ur3e_batch_kernel_timing(self.ptr, int(enable)), "ur3e_batch_kernel_timing")

    def kernel_times(self):
        """{tier: (total ms, launches)} of the step kernels since kernel_timing(True); synchronises."""
        v = (C.c_double * 6)()
        _lib.check(self._L.ur3e_batch_kernel_times(self.ptr, v), "ur3e_batch_kernel_times")
        return {"lite": (v[0], int(v[1])), "full": (v[2], int(v[3])), "side": (v[4], int(v[5]))}

    def close(self):
        if getattr(self, "ptr", None):
            self._L.ur3e_batch_destroy(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Query:
    """Poses and velocities of k objects in every environment of a batch (ur3e_batch_query_create / ur3e_batch_query).

    Calling it launches one kernel on the current torch stream and returns (pos [n, k, 3], mat [n, k, 3, 3], vel [n, k, 6]), None
    for an output not asked for.  vel is mj_objectVelocity's [rot(3), lin(3)], in the object's frame when local=True.  Each output
    argument is False, True (a tensor owned by the query, overwritten by its next call, like step's outputs) or a tensor of that
    shape and the batch's dtype on its device to write into.

    The values are evaluated at the stored state: what MuJoCo's d.xpos / d.site_xpos / ... hold after reset or set_state +
    mj_forward.  After a step MuJoCo's arrays still hold the last substep's pre-integration kinematics (SURVEY F9); the query's
    values are one substep newer than those.
    """
    KINDS = {"body": _lib.OBJ_BODY, "xbody": _lib.OBJ_XBODY, "geom": _lib.OBJ_GEOM, "site": _lib.OBJ_SITE}

    def __init__(self, batch, objects):
        self.batch = batch
        types, ids = [], []
        for kind, obj in objects:
            if kind not in self.KINDS:
                raise ValueError("object kind %r is not one of %s" % (kind, sorted(self.KINDS)))
            if isinstance(obj, str):
                i = batch.model.name2id(_lib.OBJ_BODY if kind == "xbody" else self.KINDS[kind], obj)
                if i < 0:
                    raise KeyError("%s %r is not in the model" % (kind, obj))
                obj = i
            types.append(self.KINDS[kind]); ids.append(int(obj))
        self.k = len(types)
        t = (C.c_int32 * max(self.k, 1))(*types); i = (C.c_int32 * max(self.k, 1))(*ids)
        qid = batch._L.ur3e_batch_query_create(batch.ptr, t, i, self.k)
        if qid < 0:
            raise ValueError("ur3e_batch_query_create: " + _lib.last_error())
        self.id = qid
        self._own = {}

    def __call__(self, pos=True, mat=False, vel=False, local=False):
        n, k = self.batch.n, self.k
        outs = _outs(self.batch, self._own, "a query", dict(pos=(pos, (n, k, 3), None), mat=(mat, (n, k, 3, 3), None), vel=(vel, (n, k, 6), None)))
        _lib.check(self.batch._L.ur3e_batch_query(self.batch.ptr, self.id, *map(_ptr, outs.values()), int(bool(local)), self.batch._stream()), "ur3e_batch_query")
        return tuple(outs.values())

    def jac(self, jacp=True, jacr=False, M=False, qfrc_bias=False):
        """Jacobians of the k objects, with the mass matrix and the bias forces (ur3e_batch_query_jac): one launch on the current
        torch stream, returning (jacp [n, k, 3, nv], jacr [n, k, 3, nv], M [n, nv, nv], qfrc_bias [n, nv]), None for an output not
        asked for.  Outputs follow __call__'s convention (False, True or a caller tensor).

        jacp / jacr are MuJoCo's (3, nv) translational / rotational Jacobians per object, at the object's world point: mj_jacSite
        for a "site", mj_jacBody for an "xbody" (the body frame's origin), mj_jacBodyCom for a "body" (its centre of mass),
        mj_jacGeom for a "geom".  M is mj_fullM (dense, symmetric, armature included); qfrc_bias is d.qfrc_bias (Coriolis,
        centrifugal and gravity forces).

        The values are evaluated at the stored state: what MuJoCo holds after reset or set_state + mj_forward.  After a step
        MuJoCo's d.qfrc_bias and the Jacobian it would compute are the last substep's pre-integration values (SURVEY F9), as is the
        cache the fused task-space controllers read; these are one substep newer, the same state __call__ sees.
        """
        n, k, nv = self.batch.n, self.k, self.batch.model.nv
        outs = _outs(self.batch, self._own, "Query.jac", dict(jacp=(jacp, (n, k, 3, nv), None), jacr=(jacr, (n, k, 3, nv), None),
                                                              M=(M, (n, nv, nv), None), qfrc_bias=(qfrc_bias, (n, nv), None)))
        _lib.check(self.batch._L.ur3e_batch_query_jac(self.batch.ptr, self.id, *map(_ptr, outs.values()), self.batch._stream()), "ur3e_batch_query_jac")
        return tuple(outs.values())


def _outs(batch, own, what, table):
    """Output arguments {name: (arg, shape, dtype)}: each is False / None (not wanted), True (a tensor kept in `own` under its
    name, overwritten by the next call) or a caller tensor, checked; dtype None is the batch's.  Returns {name: tensor or None} in
    the table's order; raises ValueError when no output is wanted."""
    outs = {}
    for name, (arg, shape, dtype) in table.items():
        if arg is False or arg is None:
            outs[name] = None
        elif arg is True:
            if name not in own:
                own[name] = torch.empty(shape, dtype=dtype or batch.dtype, device=batch.device)
            outs[name] = own[name]
        else:
            batch._chk(arg, shape, dtype)
            outs[name] = arg
    if all(o is None for o in outs.values()):
        raise ValueError("%s needs at least one of %s" % (what, ", ".join(table)))
    return outs


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None
