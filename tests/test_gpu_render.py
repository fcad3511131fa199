"""GPU suite for offscreen rendering (ur3e_batch_render, SimBatch.renderer, the env adapters' render / get_images): the compiled
sm_100a kernels against the host-compiled float64 render of the same stored states, float32 against float64, environment
selection, non-interference with the step path and the adapters."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import envs as OE
import ur3e_b200._lib as lib
from ur3e_b200.batch import SimBatch, default_geoms, env_config
from ur3e_b200.envs import SB3VecEnv, UR3eEnv, UR3eVecEnv
from ur3e_b200.model import Model
from tests.hostcheck import render as HR
from tests.test_gpu_query import _run, _v2

WORLD = dict(lookat=(0.25, 0.2, 0.15), distance=1.3, azimuth=110.0, elevation=-35.0, fovy=50.0)
WRIST = dict(pos=(0, 0, -0.1), xyaxes=(0, 1, 0, 1, 0, 0), site="tcp", fovy=70.0)


def _colours(k):
    return np.random.default_rng(3).uniform(0.2, 1.0, (k, 4)).astype(np.float32)


def _host(b, r, qp, rgba):
    return HR.render(b.model.path, qp, r.camera, r.geoms, r.width, r.height, rgba)


@pytest.mark.parametrize("camera", ["world", "wrist"])
def test_f64_render_equals_host_render(assets, camera):
    """After 300 random steps, the GPU images equal the host-compiled float64 render of the stored states: seg / rgb exactly,
    depth to 1e-12."""
    b, lo, hi = _v2(assets, 24, torch.float64, auto_reset=1)
    _run(b, lo, hi, 300, seed=8)
    k = len(default_geoms(b.model)); rgba = _colours(k)
    r = b.renderer(40, 32, WORLD if camera == "world" else WRIST, rgba=rgba)
    rgb, depth, seg = (x.cpu().numpy() for x in r(rgb=True, depth=True, seg=True))
    qp = b.get_state()[0].cpu().numpy()
    for e in range(b.n):
        h_rgb, h_depth, h_seg, _ = _host(b, r, qp[e], rgba)
        assert np.array_equal(seg[e], h_seg), e
        assert np.array_equal(rgb[e], h_rgb), e
        assert np.abs(depth[e] - h_depth).max() <= 1e-12, e
    assert len(np.unique(seg)) >= 4


def test_f32_render_against_f64(assets, capsys):
    """The float32 batch at the float64 batch's stored states: seg / rgb agree except on silhouette-edge pixels (counted and
    bounded), depth to 1e-5 relative where seg agrees."""
    b64, lo, hi = _v2(assets, 256, torch.float64, auto_reset=1)
    _run(b64, lo, hi, 200, seed=4)
    qp, qv, _ = b64.get_state()
    b32, _, _ = _v2(assets, 256, torch.float32, auto_reset=1)
    b32.set_state(qp.float().contiguous(), qv.float().contiguous())
    k = len(default_geoms(b64.model)); rgba = _colours(k)
    out = {}
    for name, b in (("f64", b64), ("f32", b32)):
        r = b.renderer(64, 64, WORLD, rgba=rgba)
        out[name] = [x.double().cpu().numpy() for x in r(rgb=True, depth=True, seg=True)]
    (rgb64, d64, s64), (rgb32, d32, s32) = out["f64"], out["f32"]
    same = s64 == s32
    frac = 1 - same.mean()
    with capsys.disabled():
        print("\nfloat32 vs float64: %d of %d pixels differ in seg (%.5f)" % ((~same).sum(), same.size, frac))
    assert frac < 2e-3
    assert (np.abs(d32 - d64)[same] / d64[same]).max() < 1e-5
    shade = same & (np.abs(rgb32 - rgb64).max(-1) > 2)   # the same geom but another face: box edges
    assert shade.mean() < 2e-3


def test_env_selection(assets):
    b, lo, hi = _v2(assets, 40, torch.float32, auto_reset=1)
    _run(b, lo, hi, 30, seed=2)
    r = b.renderer(37, 23, WORLD)
    full = [x.clone() for x in r(rgb=True, depth=True, seg=True)]
    ids = torch.tensor([5, 0, 39, 5, 17, 5], dtype=torch.int32, device="cuda")
    sub = r(ids, rgb=True, depth=True, seg=True)
    for x, y in zip(sub, full):
        assert torch.equal(x, y[ids.long()])
    # out-of-range ids give background and -1; the step's outputs afterwards are those of an unrendered twin
    twin, _, _ = _v2(assets, 40, torch.float32, auto_reset=1)
    _run(twin, lo, hi, 30, seed=2)
    bad = torch.tensor([-1, 40, 3, 1 << 30], dtype=torch.int32, device="cuda")
    rgb, depth, seg = r(bad, rgb=True, depth=True, seg=True)
    for i in (0, 1, 3):
        assert torch.all(rgb[i] == 0) and torch.all(seg[i] == -1) and torch.all(depth[i] == 50.0)
    assert torch.equal(seg[2], full[2][3])
    a = torch.tensor(np.tile((lo + hi) / 2, (40, 1)), dtype=torch.float32, device="cuda")
    for x, y in zip(b.step(a), twin.step(a)):
        assert torch.equal(x, y)
    # one environment, a 1 x 1 image
    one, _, _ = _v2(assets, 1, torch.float64)
    one.reset(seed=0)
    r1 = one.renderer(1, 1, WORLD)
    rgb, depth, seg = r1(rgb=True, depth=True, seg=True)
    h_rgb, h_depth, h_seg, _ = _host(one, r1, one.get_state()[0][0].cpu().numpy(), None)
    assert rgb.shape == (1, 1, 1, 3) and np.array_equal(rgb[0].cpu().numpy(), h_rgb) and int(seg[0, 0, 0]) == int(h_seg[0, 0])
    assert abs(float(depth[0, 0, 0]) - float(h_depth[0, 0])) <= 1e-12


def test_render_does_not_disturb_the_step_path(assets):
    """Two identical float32 batches, one rendering after every step on the same stream: outputs and final state agree bit for
    bit, and each render call adds exactly two launches."""
    n, steps = 96, 120
    m = Model(assets + "/main.xml")
    cfg = dict(ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2, reset_key=1,
               term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500, reset_noise=lib.NOISE_LOW, auto_reset=1)
    a_b, b_b = SimBatch(m, env_config(**cfg), n, 0, torch.float32), SimBatch(m, env_config(**cfg), n, 0, torch.float32)
    r = b_b.renderer(32, 32, WRIST)
    oa = a_b.reset(seed=9).clone(); b_b.reset(seed=9)
    mug0 = oa[:, 3:6].clone()
    c0a, c0b = a_b.launch_count, b_b.launch_count
    for k in range(steps):
        a = torch.empty(n, 4, device="cuda")
        a[:, 0:2] = a_b.obs[:, 3:5]
        a[:, 2] = mug0[:, 2] + 0.02 + max(0.0, 0.1 - 0.002 * k)
        a[:, 3] = 1.0 if k > 60 else 0.0
        a = a.contiguous()
        ra = [x.clone() for x in a_b.step(a)]
        rb = [x.clone() for x in b_b.step(a)]
        r(rgb=True, depth=True, seg=True)
        for x, y in zip(ra, rb):
            assert torch.equal(x, y), k
    for x, y in zip(a_b.get_state(), b_b.get_state()):
        assert torch.equal(x, y)
    assert (b_b.launch_count - c0b) - (a_b.launch_count - c0a) == 2 * steps


def test_render_on_a_side_stream(assets):
    b, lo, hi = _v2(assets, 16, torch.float32, auto_reset=1)
    _run(b, lo, hi, 10, seed=1)
    r = b.renderer(48, 48, WORLD)
    ref = [x.clone() for x in r(rgb=True, depth=True, seg=True)]
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = [x.clone() for x in r(rgb=torch.empty(16, 48, 48, 3, dtype=torch.uint8, device="cuda"),
                                    depth=torch.empty(16, 48, 48, device="cuda"), seg=torch.empty(16, 48, 48, dtype=torch.int32, device="cuda"))]
    s.synchronize()
    for x, y in zip(got, ref):
        assert torch.equal(x, y)


def test_render_errors(assets):
    b, _, _ = _v2(assets, 4, torch.float32)
    L = lib.load()
    with pytest.raises(ValueError, match="fovy"):
        b.renderer(8, 8, dict(WORLD, fovy=180.0))
    with pytest.raises(KeyError):
        b.renderer(8, 8, WORLD, geoms=["no_such_geom"])
    r = b.renderer(8, 8, WORLD, geoms=["table", "fish"])
    assert r.k == 2
    with pytest.raises(ValueError, match="at least one"):
        r(rgb=False)
    with pytest.raises(ValueError):
        r(torch.zeros(2, dtype=torch.int64, device="cuda"))
    assert L.ur3e_batch_render(b.ptr, 7, None, 4, C.c_void_p(1), None, None, None) != 0 and "unknown render id" in lib.last_error()
    assert L.ur3e_batch_render(b.ptr, r.id, None, 3, C.c_void_p(1), None, None, None) != 0 and "batch size" in lib.last_error()


def test_adapters_render(assets):
    env = UR3eEnv(render_mode="rgb_array")
    env.reset(seed=0)
    img = env.render()
    assert isinstance(img, np.ndarray) and img.shape == (480, 480, 3) and img.dtype == np.uint8 and img.max() > 0
    env.close()
    env = UR3eEnv(render_mode="depth_array", width=64, height=48)
    env.reset(seed=0)
    d = env.render()
    assert d.shape == (48, 64) and d.dtype == np.float64 and 0 < d.min() < d.max() <= 50.0
    env.close()
    env = UR3eEnv(render_mode=None)
    assert env.render() is None
    env.close()
    with pytest.raises(ValueError):
        UR3eEnv(render_mode="rgb_array", camera_name="top")
    venv = UR3eVecEnv(num_envs=6, render_mode="rgb_array", width=40, height=30)
    assert venv.metadata["render_modes"] == ["rgb_array", "depth_array"]
    venv.reset(seed=0)
    imgs = venv.render()
    assert imgs.is_cuda and tuple(imgs.shape) == (6, 30, 40, 3)
    sb3 = SB3VecEnv(venv=venv)
    got = sb3.get_images()
    assert len(got) == 6 and all(g.shape == (30, 40, 3) for g in got)
    assert all(g is None for g in SB3VecEnv(venv=UR3eVecEnv(num_envs=2)).get_images())
