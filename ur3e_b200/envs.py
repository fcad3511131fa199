"""Vectorised drop-in environments with the reference's Gymnasium ids and spaces.

    env = UR3eVecEnv("gymnasium_env/ur3e-v2", num_envs=65536)      # torch tensors in/out, zero-copy
    obs, info = env.reset(seed=0)
    obs, reward, terminated, truncated, info = env.step(actions)   # actions: cuda tensor [N, act_dim]

replaces N copies of the reference's env classes behind SB3's SubprocVecEnv
(reference gymnasium_src/scripts/regular_rl/rl/train_rl.py:38-44; env classes gymnasium_env/envs/*.py;
registration gymnasium_env/envs/register_envs.py:4-25).  Auto-reset follows the SB3 VecEnv convention: a finished
environment returns its reset observation and the terminal one is available as `final_obs` / infos[i]["terminal_observation"].
gymnasium and stable_baselines3 are optional imports (neither is present in the build container): when they import, `UR3eVecEnv`
derives from `gymnasium.vector.VectorEnv`, `UR3eEnv` from `gymnasium.Env` and `SB3VecEnv` from SB3's `VecEnv`, so `isinstance`
checks in the trainers (SB3's `_wrap_env`, `VecNormalize`) accept them as they are.
"""
import pickle
import time

import numpy as np
import torch

from . import _lib, presets
from .batch import SimBatch

# UR3eEnv's camera when no default_camera_config is given: a constant world camera that frames the arm (base at the origin, ~0.5 m
# reach) and the mug's reset region (x 0.3 .. 0.45, y 0.13 .. 0.38 on the table), looking along +y and 45 degrees down.  It is not
# derived from MuJoCo's model statistics (stat.center / stat.extent), so it does not match MuJoCo's default free camera.
DEFAULT_CAMERA_CONFIG = {"lookat": (0.25, 0.2, 0.15), "distance": 1.4, "azimuth": 90.0, "elevation": -45.0, "fovy": 45.0}
from .model import Model, asset

ENV_IDS = tuple(presets.ENV_SPECS.keys())


class Box:
    """Minimal stand-in for gymnasium.spaces.Box (used when gymnasium is not installed)."""

    def __init__(self, low, high, shape=None, dtype=np.float64):
        self.dtype = np.dtype(dtype)
        self.low = np.broadcast_to(np.asarray(low, dtype=dtype), shape).copy() if shape is not None else np.asarray(low, dtype=dtype)
        self.high = np.broadcast_to(np.asarray(high, dtype=dtype), shape).copy() if shape is not None else np.asarray(high, dtype=dtype)
        self.shape = self.low.shape

    def sample(self, rng=None):
        rng = rng or np.random.default_rng()
        lo = np.where(np.isfinite(self.low), self.low, -1.0); hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return rng.uniform(lo, hi).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))


def _box(low, high, shape=None, dtype=np.float64):
    try:
        from gymnasium import spaces
        return spaces.Box(low=low, high=high, shape=shape, dtype=dtype)
    except Exception:
        return Box(low, high, shape, dtype)


def _optional_base(module, attr):
    """`module.attr` when it imports (so that isinstance checks of the trainers pass), else `object`."""
    try:
        mod = __import__(module, fromlist=[attr])
        return getattr(mod, attr)
    except Exception:
        return object


_VectorEnvBase = _optional_base("gymnasium.vector", "VectorEnv")
_EnvBase = _optional_base("gymnasium", "Env")
_SB3VecEnvBase = _optional_base("stable_baselines3.common.vec_env", "VecEnv")


class UR3eVecEnv(_VectorEnvBase):
    """N environments of one of the reference's four ids on one GPU (torch API; a gymnasium.vector.VectorEnv when gymnasium imports)."""

    metadata = {"render_modes": ["rgb_array", "depth_array"], "autoreset_mode": "same_step"}

    def __init__(self, env_id="gymnasium_env/ur3e-v2", num_envs=1, device=0, dtype=torch.float32, auto_reset=True, env_id_base=0, render_mode=None,
                 width=480, height=480, default_camera_config=None, camera_id=None, camera_name=None, **config_overrides):
        if env_id not in presets.ENV_SPECS:
            raise ValueError("unknown env id %r (known: %s)" % (env_id, ", ".join(ENV_IDS)))
        if camera_id is not None or camera_name is not None:
            raise ValueError("camera_id / camera_name: the model's <camera> elements are not loaded; use default_camera_config")
        xml, kw, _, _ = presets.ENV_SPECS[env_id]
        self.env_id, self.num_envs = env_id, int(num_envs)
        self.render_mode = render_mode      # "rgb_array" / "depth_array" render (render()); None and "human" (train_rl.py:41) render nothing
        self.width, self.height = int(width), int(height)
        self.default_camera_config = dict(DEFAULT_CAMERA_CONFIG if default_camera_config is None else default_camera_config)
        self._renderer = None
        self.model = Model(asset(xml))
        self.cfg = presets.make_config(self.model, kw, auto_reset=int(bool(auto_reset)), env_id_base=env_id_base, **config_overrides)
        self.batch = SimBatch(self.model, self.cfg, self.num_envs, device, dtype)
        lo, hi = presets.action_bounds(self.model, env_id)
        self.single_action_space = _box(lo, hi, dtype=np.float64)
        self.single_observation_space = _box(-np.inf, np.inf, (self.cfg.obs_dim,), np.float64)     # ur3e_env2.py:44-48
        self.action_space = _box(np.tile(lo, (self.num_envs, 1)), np.tile(hi, (self.num_envs, 1)), dtype=np.float64)
        self.observation_space = _box(-np.inf, np.inf, (self.num_envs, self.cfg.obs_dim), np.float64)
        self.frame_skip = self.cfg.frame_skip
        self.dt = self.model.opt.timestep * self.frame_skip
        self.metadata = dict(self.metadata, render_fps=int(round(1.0 / self.dt)))                  # ur3e_env2.py:19-28
        self.device, self.dtype = self.batch.device, dtype
        self._seed = 0

    # ---- gymnasium.vector-style API (torch tensors)
    def reset(self, *, seed=None, options=None):
        if seed is not None:
            self._seed = int(seed)
        return self.batch.reset(self._seed), {}

    def step(self, actions):
        if not isinstance(actions, torch.Tensor):
            actions = torch.as_tensor(np.asarray(actions), dtype=self.dtype, device=self.device)
        if actions.dtype != self.dtype or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=self.dtype).contiguous()
        if tuple(actions.shape) != (self.num_envs, self.cfg.act_dim):
            raise ValueError("Action dimension mismatch: expected %s, got %s" % ((self.num_envs, self.cfg.act_dim), tuple(actions.shape)))   # MujocoEnv.do_simulation
        obs, rew, term, trunc = self.batch.step(actions)
        return obs, rew, term.bool(), trunc.bool(), {"final_obs": self.batch.final_obs}

    def render(self, env_ids=None):
        """Images of the stored state (see ur3e_b200.batch.Renderer) on the device: render_mode "rgb_array" gives uint8 [m, H, W, 3],
        "depth_array" the z-depth [m, H, W] in metres; env_ids (int32 CUDA tensor [m]) selects environments, None = all.  The
        camera is default_camera_config (UR3eVecEnv.DEFAULT_CAMERA_CONFIG when none was given).  Any other render_mode returns None.
        The returned tensor is owned by the env and overwritten by the next call."""
        if self.render_mode not in ("rgb_array", "depth_array"):
            return None
        if self._renderer is None:
            self._renderer = self.batch.renderer(self.width, self.height, self.default_camera_config)
        rgb = self.render_mode == "rgb_array"
        out = self._renderer(env_ids, rgb=rgb, depth=not rgb)
        return out[0] if rgb else out[1]

    def set_state(self, qpos, qvel):
        """MujocoEnv.set_state for every env (qpos [N,nq], qvel [N,nv])."""
        self.batch.set_state(qpos, qvel)

    def get_state(self):
        return self.batch.get_state()

    def episode_stats(self, reset=True):
        return self.batch.stats_dict(reset)

    def close(self, **kwargs):
        self.batch.close()


class UR3eEnv(_EnvBase):
    """Single-environment view with the reference classes' gymnasium.Env contract (`gym.make(id)`): float64 numpy in and out,
    `reset(seed=, options=) -> (obs, info)`, `step(a) -> (obs, reward, terminated, truncated, {})`, no auto-reset
    (reference gymnasium_env/envs/ur3e_env2.py:72-109).  One environment per launch is a debugging / evaluation convenience;
    training wants UR3eVecEnv."""

    metadata = {"render_modes": ["human", "rgb_array", "depth_array"]}

    def __init__(self, env_id="gymnasium_env/ur3e-v2", render_mode=None, device=0, dtype=torch.float64, width=480, height=480, default_camera_config=None,
                 camera_id=None, camera_name=None, **config_overrides):
        self.venv = UR3eVecEnv(env_id, 1, device, dtype, auto_reset=False, render_mode=render_mode, width=width, height=height,
                               default_camera_config=default_camera_config, camera_id=camera_id, camera_name=camera_name, **config_overrides)
        self.observation_space, self.action_space = self.venv.single_observation_space, self.venv.single_action_space
        self.render_mode = render_mode
        self.metadata = dict(self.metadata, render_fps=self.venv.metadata["render_fps"])
        self.frame_skip, self.dt, self.model = self.venv.frame_skip, self.venv.dt, self.venv.model

    def reset(self, *, seed=None, options=None):
        # reset noise: Philox stream keyed by (seed, env id, episode counter), so consecutive resets draw different mug positions
        # (the reference draws from numpy's global stream on every reset, gym_utils.py:58-59)
        obs, info = self.venv.reset(seed=seed)
        return obs[0].double().cpu().numpy(), {}

    def step(self, action):
        a = np.asarray(action, dtype=np.float64).reshape(1, -1)
        obs, rew, term, trunc, _ = self.venv.step(a)
        return obs[0].double().cpu().numpy(), float(rew[0].item()), bool(term[0].item()), bool(trunc[0].item()), {}

    def render(self):
        """gymnasium MujocoEnv.render: render_mode "rgb_array" gives a (height, width, 3) uint8 numpy image, "depth_array" a
        (height, width) float64 z-depth in metres, of the stored state (ur3e_b200.batch.Renderer); None and "human" (no viewer)
        give None.  width / height (480) and default_camera_config are constructor arguments as in MujocoEnv; without a
        default_camera_config the camera is the constant DEFAULT_CAMERA_CONFIG, not MuJoCo's model-statistics free camera."""
        img = self.venv.render()
        if img is None:
            return None
        return img[0].cpu().numpy() if self.render_mode == "rgb_array" else img[0].double().cpu().numpy()

    def close(self):
        self.venv.close()


class SB3VecEnv(_SB3VecEnvBase):
    """stable_baselines3 VecEnv over the batched simulator (numpy at the boundary, as SB3 expects); a real
    `stable_baselines3.common.vec_env.VecEnv` subclass when SB3 imports.

    Provides what `make_vec_env(..., vec_env_cls=SubprocVecEnv)` + `Monitor` give the reference's trainers
    (train_rl.py:38-57): step_async/step_wait, auto-reset with infos[i]["terminal_observation"],
    infos[i]["TimeLimit.truncated"], infos[i]["episode"] = {"r", "l", "t"}, per-index get_attr/set_attr/env_method, seed, close.
    `venv` may be any object with UR3eVecEnv's torch API (tests pass a CPU stand-in)."""

    def __init__(self, env_id="gymnasium_env/ur3e-v2", n_envs=1, device=0, dtype=torch.float32, venv=None, **kw):
        self.venv = venv if venv is not None else UR3eVecEnv(env_id, n_envs, device, dtype, auto_reset=True, **kw)
        n_envs = self.venv.num_envs
        if _SB3VecEnvBase is not object:
            super().__init__(n_envs, self.venv.single_observation_space, self.venv.single_action_space)
        self.num_envs = n_envs
        self.observation_space = self.venv.single_observation_space
        self.action_space = self.venv.single_action_space
        self.render_mode = getattr(self.venv, "render_mode", None)
        self._actions = None
        self._ret = np.zeros(n_envs); self._len = np.zeros(n_envs, dtype=np.int64)
        self._seed = 0
        self._t0 = time.time()
        self._attrs = [dict() for _ in range(n_envs)]      # per-environment attribute overlay (set_attr with indices)

    def _indices(self, indices):
        if indices is None:
            return list(range(self.num_envs))
        return [int(i) for i in np.atleast_1d(indices)]

    def seed(self, seed=None):
        self._seed = 0 if seed is None else int(seed)
        return [self._seed + i for i in range(self.num_envs)]

    def reset(self):
        obs, _ = self.venv.reset(seed=self._seed)
        self._ret[:] = 0; self._len[:] = 0
        return obs.double().cpu().numpy()

    def step_async(self, actions):
        self._actions = np.asarray(actions)

    def step_wait(self):
        obs, rew, term, trunc, info = self.venv.step(self._actions)
        obs_n = obs.double().cpu().numpy(); rew_n = rew.double().cpu().numpy()
        term_n = term.cpu().numpy().astype(bool); trunc_n = trunc.cpu().numpy().astype(bool); done = term_n | trunc_n
        self._ret += rew_n; self._len += 1
        infos = [{} for _ in range(self.num_envs)]
        if done.any():
            fo = info["final_obs"].double().cpu().numpy()
            now = round(time.time() - self._t0, 6)
            for i in np.nonzero(done)[0]:
                infos[i]["terminal_observation"] = fo[i]
                infos[i]["TimeLimit.truncated"] = bool(trunc_n[i] and not term_n[i])
                infos[i]["episode"] = {"r": round(float(self._ret[i]), 6), "l": int(self._len[i]), "t": now}     # Monitor's record
                self._ret[i] = 0; self._len[i] = 0
        return obs_n, rew_n, done, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def get_attr(self, attr_name, indices=None):
        return [self._attrs[i][attr_name] if attr_name in self._attrs[i] else getattr(self.venv, attr_name) for i in self._indices(indices)]

    def set_attr(self, attr_name, value, indices=None):
        for i in self._indices(indices):
            self._attrs[i][attr_name] = value

    def env_method(self, method_name, *method_args, indices=None, **method_kwargs):
        return [getattr(self.venv, method_name)(*method_args, **method_kwargs) for _ in self._indices(indices)]

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False for _ in self._indices(indices)]

    def get_images(self):
        """One (H, W, 3) uint8 numpy image per environment when the wrapped env's render_mode is "rgb_array" (SB3's
        VecEnv.render("rgb_array") and VecVideoRecorder ask for every environment's image: all N are rendered and copied to the
        host), else [None] * n."""
        if self.render_mode != "rgb_array":
            return [None] * self.num_envs
        return list(self.venv.render().cpu().numpy())

    def close(self):
        self.venv.close()


class RunningMeanStd:
    """Running mean / variance over batches (Chan et al. parallel update), on whatever device the tensors live on: the
    statistics SB3's VecNormalize keeps per observation feature and for the discounted return."""

    def __init__(self, shape=(), epsilon=1e-4, device=None, dtype=torch.float64):
        self.mean = torch.zeros(shape, dtype=dtype, device=device)
        self.var = torch.ones(shape, dtype=dtype, device=device)
        self.count = float(epsilon)

    def update(self, x):
        x = x.to(self.mean.dtype)
        bm, bv, bc = x.mean(dim=0), x.var(dim=0, unbiased=False), x.shape[0]
        delta = bm - self.mean
        tot = self.count + bc
        m2 = self.var * self.count + bv * bc + delta * delta * (self.count * bc / tot)
        self.mean = self.mean + delta * (bc / tot); self.var = m2 / tot; self.count = tot


class VecNormalizeGPU:
    """Device-side equivalent of `stable_baselines3.common.vec_env.VecNormalize` around a UR3eVecEnv (torch tensors stay on the GPU):
    running observation statistics, optional return-based reward scaling, clipping, `training` switch, `save` / `load`
    (reference train_rl.py:46-57, 89-90: `VecNormalize(venv, norm_obs=True, norm_reward=False, clip_obs=...)`,
    `VecNormalize.load(path, venv)`, `venv.save(path)`)."""

    def __init__(self, venv, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99, epsilon=1e-8):
        self.venv, self.training, self.norm_obs, self.norm_reward = venv, training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = float(clip_obs), float(clip_reward), float(gamma), float(epsilon)
        self.num_envs = venv.num_envs
        dev = getattr(venv, "device", None)
        self.obs_rms = RunningMeanStd((venv.single_observation_space.shape[0],), device=dev)
        self.ret_rms = RunningMeanStd((), device=dev)
        self.returns = torch.zeros(self.num_envs, dtype=torch.float64, device=dev)
        self.old_obs = self.old_reward = None
        for k in ("single_observation_space", "single_action_space", "observation_space", "action_space", "metadata"):
            setattr(self, k, getattr(venv, k, None))

    def normalize_obs(self, obs):
        if not self.norm_obs:
            return obs
        o = (obs.to(torch.float64) - self.obs_rms.mean) / torch.sqrt(self.obs_rms.var + self.epsilon)
        return o.clamp(-self.clip_obs, self.clip_obs).to(obs.dtype)

    def normalize_reward(self, reward):
        if not self.norm_reward:
            return reward
        r = reward.to(torch.float64) / torch.sqrt(self.ret_rms.var + self.epsilon)
        return r.clamp(-self.clip_reward, self.clip_reward).to(reward.dtype)

    def unnormalize_obs(self, obs):
        return (obs.to(torch.float64) * torch.sqrt(self.obs_rms.var + self.epsilon) + self.obs_rms.mean).to(obs.dtype) if self.norm_obs else obs

    def get_original_obs(self):
        return self.old_obs

    def get_original_reward(self):
        return self.old_reward

    def reset(self, **kw):
        obs, info = self.venv.reset(**kw)
        self.old_obs = obs.clone()
        self.returns.zero_()
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs), info

    def step(self, actions):
        obs, rew, term, trunc, info = self.venv.step(actions)
        self.old_obs, self.old_reward = obs.clone(), rew.clone()
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        if self.training and self.norm_reward:
            self.returns = self.returns * self.gamma + rew.to(torch.float64)
            self.ret_rms.update(self.returns)
        done = term | trunc
        if "final_obs" in info:
            info = dict(info, final_obs=self.normalize_obs(info["final_obs"]))
        self.returns = torch.where(done, torch.zeros_like(self.returns), self.returns)
        return self.normalize_obs(obs), self.normalize_reward(rew), term, trunc, info

    def state_dict(self):
        return dict(obs_mean=self.obs_rms.mean.cpu(), obs_var=self.obs_rms.var.cpu(), obs_count=self.obs_rms.count, ret_mean=self.ret_rms.mean.cpu(),
                    ret_var=self.ret_rms.var.cpu(), ret_count=self.ret_rms.count, clip_obs=self.clip_obs, clip_reward=self.clip_reward, gamma=self.gamma,
                    epsilon=self.epsilon, norm_obs=self.norm_obs, norm_reward=self.norm_reward, training=self.training)

    def save(self, path):
        with open(path, "wb") as f:
            pickle.dump(self.state_dict(), f)

    @classmethod
    def load(cls, path, venv):
        with open(path, "rb") as f:
            sd = pickle.load(f)
        self = cls(venv, sd["training"], sd["norm_obs"], sd["norm_reward"], sd["clip_obs"], sd["clip_reward"], sd["gamma"], sd["epsilon"])
        dev = self.obs_rms.mean.device
        self.obs_rms.mean, self.obs_rms.var, self.obs_rms.count = sd["obs_mean"].to(dev), sd["obs_var"].to(dev), sd["obs_count"]
        self.ret_rms.mean, self.ret_rms.var, self.ret_rms.count = sd["ret_mean"].to(dev), sd["ret_var"].to(dev), sd["ret_count"]
        return self

    def __getattr__(self, name):          # everything else (episode_stats, set_state, close ...) goes to the wrapped env
        return getattr(self.__dict__["venv"], name)


def register_envs():
    """Register the reference's four ids (gymnasium_env/envs/register_envs.py:4-25) with gymnasium: `entry_point` = the single-env
    view, `vector_entry_point` = the batched env (`gym.make_vec(id, num_envs=...)`).  Returns False when gymnasium is not installed."""
    try:
        import gymnasium
    except ImportError:
        return False
    for env_id in ENV_IDS:
        def make_one(_id=env_id, **kw):
            return UR3eEnv(_id, **kw)

        def make_vec(num_envs=1, _id=env_id, **kw):
            return UR3eVecEnv(_id, num_envs, **kw)
        gymnasium.register(id=env_id, entry_point=make_one, vector_entry_point=make_vec)
    return True
