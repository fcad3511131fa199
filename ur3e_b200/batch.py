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
RolloutResult = namedtuple("RolloutResult", _lib.ROLLOUT_OUTPUTS)


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

    def renderer(self, width, height, camera, geoms=None, rgba=None):
        """An offscreen renderer of this batch (ur3e_batch_render_create): width x height images of `geoms` (names or ids of box /
        plane geoms; None = every geom whose geom_rgba alpha is > 0) seen from `camera` (a dict, see make_camera).  rgba [k, 4]
        overrides the model's geom_rgba per geom.  See Renderer."""
        return Renderer(self, width, height, camera, geoms, rgba)

    def rollout(self, actions, env_ids=None, state=None, qpos=False, qvel=False, obs=True, reward=True, terminated=True, truncated=True,
                sensordata=False, info=False):
        """mujoco.rollout for this batch (ur3e_batch_rollout): m copies of environments stepped T env-steps with `actions`, leaving
        the batch untouched.  Returns a RolloutResult named tuple with None for every output not asked for; outputs follow
        forward()'s convention (False, True = a tensor owned by the batch, reallocated when (T, m) changes, or a caller tensor).

            actions [T, m, act_dim]            contiguous, the batch's dtype; step t's actions are actions[t]
            env_ids int32 [m] (CUDA)           rollout j starts from a copy of environment env_ids[j]'s whole record, so it is
                                               bit-identical to stepping that environment with the same actions up to its first
                                               done; ids may repeat and m may exceed n.  An id outside [0, n) starts from a bad
                                               state that the step resets to qpos0 (info[j, 0] >= 1)
            state (qpos [m, nq], qvel [m, nv][, qacc_warmstart [m, nv]])   or rollouts start as set_state leaves a fresh record
            neither                            every environment branched once (m = n)

            qpos [T, m, nq], qvel [T, m, nv]   the state after each env-step
            obs [T, m, obs_dim], reward [T, m], terminated, truncated uint8 [T, m]   what step returns
            sensordata [T, m, 46]              the step's sensor record (enable_sensors) from each env-step's last mj_step
            info int32 [m, 2]                  env-steps with a bad-state reset, env-steps with a contact / row overflow

        There is no auto-reset: after a done the rollout keeps stepping and the flags are what the environment computes; mask the
        steps after the first done.  Time-major: .transpose(0, 1) gives mujoco.rollout's [nroll, nstep, ...].  The call runs the
        step kernels T times on the current torch stream; the batch's records, statistics and sensor buffer are not modified.  A
        batch's rollouts share one workspace: calls on different streams must be ordered.
        """
        if env_ids is not None and state is not None:
            raise ValueError("rollout: give env_ids or state, not both")
        if actions.dim() != 3:
            raise ValueError("rollout: actions must be [T, m, act_dim], got shape %s" % (tuple(actions.shape),))
        T = int(actions.shape[0])
        ids = qp = qv = ws = None
        if state is not None:
            if len(state) not in (2, 3):
                raise ValueError("rollout: state is (qpos, qvel) or (qpos, qvel, qacc_warmstart)")
            m = int(state[0].shape[0])
            qp = self._chk(state[0], (m, self.model.nq)); qv = self._chk(state[1], (m, self.model.nv))
            ws = self._chk(state[2], (m, self.model.nv)) if len(state) == 3 and state[2] is not None else None
        else:
            if env_ids is None:
                if getattr(self, "_all_ids", None) is None:
                    self._all_ids = torch.arange(self.n, dtype=torch.int32, device=self.device)
                env_ids = self._all_ids
            m = int(env_ids.numel())
            ids = self._chk(env_ids, (m,), torch.int32)
        a = self._chk(actions, (T, m, self.act_dim))
        if getattr(self, "_rollout_tm", None) != (T, m):
            self._rollout_own, self._rollout_tm = {}, (T, m)   # owned outputs follow the latest call's (T, m)
        u8, i32 = torch.uint8, torch.int32
        table = dict(qpos=(qpos, (T, m, self.model.nq), None), qvel=(qvel, (T, m, self.model.nv), None), obs=(obs, (T, m, self.obs_dim), None),
                     reward=(reward, (T, m), None), terminated=(terminated, (T, m), u8), truncated=(truncated, (T, m), u8),
                     sensordata=(sensordata, (T, m, _lib.NSENSOR), None), info=(info, (m, 2), i32))
        outs = RolloutResult(**_outs(self, self._rollout_own, "rollout", table))
        st = _lib.RolloutOut(*[o.data_ptr() if o is not None else None for o in outs])
        _lib.check(self._L.ur3e_batch_rollout(self.ptr, ids, qp, qv, ws, m, T, a, C.byref(st), self._stream()), "ur3e_batch_rollout")
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


def make_camera(model, camera):
    """ur3e_camera from a dict, in one of two forms, both with fovy (vertical, degrees; 45), znear (0.01) and zfar (50.0) in metres:

        {"pos": (3,), "xyaxes": (6,)} with optionally "body": name or id (the body frame) or "site": name or id -- MJCF <camera
            pos xyaxes> in that anchor's frame (the world's without one): x right, y up, the view along -z;
        {"lookat": (3,), "distance": d, "azimuth": az, "elevation": el} (degrees) -- gymnasium's default_camera_config keys, a world
            camera in MuJoCo's free-camera parametrisation: forward f = (cos el cos az, cos el sin az, sin el), position
            lookat - d f, up (-sin el cos az, -sin el sin az, cos el), right f x up.
    """
    cam = dict(camera)
    c = _lib.Camera()
    c.fovy = float(cam.pop("fovy", 45.0)); c.znear = float(cam.pop("znear", 0.01)); c.zfar = float(cam.pop("zfar", 50.0))
    c.objtype, c.objid = -1, 0
    if "lookat" in cam:
        lookat = np.asarray(cam.pop("lookat"), dtype=np.float64)
        dist = float(cam.pop("distance")); az = np.radians(float(cam.pop("azimuth"))); el = np.radians(float(cam.pop("elevation")))
        f = np.array([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el)])
        up = np.array([-np.sin(el) * np.cos(az), -np.sin(el) * np.sin(az), np.cos(el)])
        pos, xyaxes = lookat - dist * f, np.concatenate([np.cross(f, up), up])
    else:
        pos = np.asarray(cam.pop("pos"), dtype=np.float64); xyaxes = np.asarray(cam.pop("xyaxes"), dtype=np.float64)
        for kind, t in (("body", _lib.OBJ_XBODY), ("site", _lib.OBJ_SITE)):
            if kind in cam:
                obj = cam.pop(kind)
                i = model.name2id(_lib.OBJ_BODY if kind == "body" else t, obj) if isinstance(obj, str) else int(obj)
                if i < 0:
                    raise KeyError("%s %r is not in the model" % (kind, obj))
                c.objtype, c.objid = t, i
    if cam:
        raise ValueError("unknown camera keys %s" % sorted(cam))
    if pos.shape != (3,) or xyaxes.shape != (6,):
        raise ValueError("camera pos needs 3 numbers and xyaxes 6")
    for i in range(3):
        c.pos[i] = pos[i]
    for i in range(6):
        c.xyaxes[i] = xyaxes[i]
    return c


def default_geoms(model):
    """Ids of the geoms a renderer draws by default: every geom whose geom_rgba alpha is > 0."""
    return [int(i) for i in np.nonzero(np.asarray(model.array("geom_rgba")).reshape(-1, 4)[:, 3] > 0)[0]]


class Renderer:
    """Offscreen RGB, depth and geom-segmentation images of selected environments (ur3e_batch_render).

    Calling it launches two kernels on the current torch stream and returns (rgb [m, H, W, 3] uint8, depth [m, H, W] in the batch's
    dtype, seg [m, H, W] int32), None for an output not asked for; each output argument is False, True (a tensor owned by the
    renderer, overwritten by its next call) or a caller tensor of that shape to write into.  env_ids is an int32 CUDA tensor [m]
    (None = every environment); an id outside [0, n) renders as background.  Row 0 is the top of the image.

    depth is the z-depth in metres along the camera's view axis (gymnasium's linearised depth_array, not the ray length); a miss or
    a hit beyond zfar reports zfar and hits nearer than znear are ignored.  seg is the hit geom's id in the model, -1 for background.
    Geoms are opaque boxes and planes (a plane is seen only from its front side) under a headlight, rgb * (0.3 + 0.7 max(0, -n.d)),
    on black; no shadows, textures or anti-aliasing.

    The images are of the stored state: what MuJoCo's d.geom_xpos / d.geom_xmat hold after reset or set_state + mj_forward.  After a
    step MuJoCo's arrays still hold the last substep's pre-integration kinematics (SURVEY F9); the images are one substep newer than
    those, the state query() sees.  A batch's renderers share one pose scratch: calls on different streams must be ordered.
    """

    def __init__(self, batch, width, height, camera, geoms=None, rgba=None):
        self.batch, self.width, self.height = batch, int(width), int(height)
        ids = default_geoms(batch.model) if geoms is None else []
        for g in (geoms if geoms is not None else []):
            i = batch.model.name2id(_lib.OBJ_GEOM, g) if isinstance(g, str) else int(g)
            if i < 0:
                raise KeyError("geom %r is not in the model" % (g,))
            ids.append(i)
        self.geoms, self.k = ids, len(ids)
        self.camera = make_camera(batch.model, camera)
        col = None
        if rgba is not None:
            col = np.ascontiguousarray(rgba, dtype=np.float32)
            if col.shape != (self.k, 4):
                raise ValueError("rgba must be [k, 4] = [%d, 4], got %s" % (self.k, col.shape))
        g = (C.c_int32 * max(self.k, 1))(*ids)
        rid = batch._L.ur3e_batch_render_create(batch.ptr, C.byref(self.camera), g, self.k,
                                                col.ctypes.data_as(C.POINTER(C.c_float)) if col is not None else None, self.width, self.height)
        if rid < 0:
            raise ValueError("ur3e_batch_render_create: " + _lib.last_error())
        self.id = rid
        self._own = {}

    def __call__(self, env_ids=None, rgb=True, depth=False, seg=False):
        b = self.batch
        if env_ids is None:
            m, ep = b.n, None
        else:
            m = int(env_ids.numel())
            ep = b._chk(env_ids, (m,), torch.int32)
        H, W = self.height, self.width
        for name in [k for k, t in self._own.items() if t.shape[0] != m]:
            del self._own[name]   # owned outputs follow the latest call's m
        outs = _outs(b, self._own, "Renderer", dict(rgb=(rgb, (m, H, W, 3), torch.uint8), depth=(depth, (m, H, W), None), seg=(seg, (m, H, W), torch.int32)))
        _lib.check(b._L.ur3e_batch_render(b.ptr, self.id, ep, m, *map(_ptr, outs.values()), b._stream()), "ur3e_batch_render")
        return tuple(outs.values())
