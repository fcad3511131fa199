"""GPU suite for rollouts (ur3e_batch_rollout, SimBatch.rollout): a branch is bit-identical to the live environment's future (float32
on the tiered batch and float64, every model family), repeated / permuted / out-of-range source ids, explicit states against
set_state + step, the float64 oracle, no auto-reset after a done, and the batch left untouched."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import envs as OE
import ur3e_b200._lib as lib
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.model import Model, asset
from tests.test_gpu_parity import make, rel

# the tiered main.xml configuration of test_tier_choice_is_deterministic_and_shard_invariant: lower lite caps, so that all three tiers run
V2 = dict(ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2, reset_key=1,
          term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500, reset_noise=lib.NOISE_LOW, auto_reset=1, lite_max_contacts=4)
ASSETS = os.path.dirname(asset("main.xml"))
OUTS = ("obs", "reward", "terminated", "truncated", "sensordata")


def _scripted(b, mug, k, z0=None):
    """The scripted approach and grasp of the tier test at step k: hover over the mug (xy of `mug`, height over z0 = the mug's initial
    height, default mug's own), descend, close from step 90; a third never closes."""
    a = torch.empty(b.n, 4, device="cuda", dtype=b.dtype)
    a[:, 0:2] = mug[:, 0:2]
    a[:, 2] = (mug[:, 2] if z0 is None else z0) + 0.02 + max(0.0, 0.1 - 0.002 * k)
    a[:, 3] = 1.0 if k > 90 else 0.0
    a[::3, 3] = 0.0
    return a


def _v2_settled(n, dtype, settle=100, track_from=None, **over):
    """A v2 batch after `settle` scripted steps; with track_from, also the most environments the full tier stepped in one step from
    that step on."""
    b = make(ASSETS, "main.xml", n, dtype, **dict(V2, **over))
    z0 = b.reset(seed=9)[:, 5].clone()
    full = 0
    for k in range(settle):
        b.step(_scripted(b, b.obs[:, 3:6], k, z0).contiguous())
        if track_from is not None and k >= track_from:
            torch.cuda.synchronize()
            full = max(full, b.kernel_info()["lite"]["last_overflow_envs"])
    b.z0 = z0
    return (b, full) if track_from is not None else b


def _live_vs_branch(b, acts, tiered=False):
    """Roll out every environment once with acts [T, n, act_dim] and every output, then step the live batch (sensors enabled) with
    the same actions; assert bitwise equality up to and including each environment's first done.  Returns (most environments the
    full tier stepped in one live step of the window, first-done index per environment)."""
    T, n = acts.shape[0], b.n
    r = {k: v.clone() for k, v in b.rollout(acts, qpos=True, qvel=True, sensordata=True, info=True)._asdict().items()}
    live = {k: [] for k in OUTS + ("qpos", "qvel")}
    full = 0
    for t in range(T):
        o, rw, te, tr = b.step(acts[t])
        done = (te | tr).bool()
        live["obs"].append(torch.where(done[:, None], b.final_obs, o).clone())   # the live batch auto-resets: compare the terminal obs
        live["reward"].append(rw.clone()); live["terminated"].append(te.clone()); live["truncated"].append(tr.clone())
        live["sensordata"].append(b.sensors.clone())
        qp, qv, _ = b.get_state()
        live["qpos"].append(qp); live["qvel"].append(qv)
        if tiered:
            torch.cuda.synchronize()
            full = max(full, b.kernel_info()["lite"]["last_overflow_envs"])
    live = {k: torch.stack(v) for k, v in live.items()}
    done = (live["terminated"] | live["truncated"]).bool()
    first = torch.where(done.any(0), done.int().argmax(0), torch.full((n,), T, device=done.device))
    t_idx = torch.arange(T, device=done.device)[:, None]
    upto, before = t_idx <= first[None], t_idx < first[None]   # the state after a done step is the live batch's reset state
    for k in OUTS:
        assert torch.equal(r[k][upto], live[k][upto]), k
    for k in ("qpos", "qvel"):
        assert torch.equal(r[k][before], live[k][before]), k
    assert int(upto.sum()) > T * n // 2
    return full, first


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_branch_equals_live_future_main(dtype):
    """main.xml v2 with the tier test's scripted grasp: a rollout from arange(n) equals the live batch stepped with the same actions,
    bitwise, up to each environment's first done; in float32 environments are on the full tier around and in the window."""
    tiered = dtype == torch.float32
    b, full = _v2_settled(96, dtype, settle=200, track_from=100 if tiered else None) if tiered else (_v2_settled(96, dtype, settle=200), 0)
    b.enable_sensors()
    mug = b.obs[:, 3:6].clone()
    acts = torch.stack([_scripted(b, mug, 200 + k, b.z0) for k in range(60)]).contiguous()
    full = max(full, _live_vs_branch(b, acts, tiered=tiered)[0])
    if tiered:
        assert full > 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_branch_equals_live_future_single_class(dtype):
    """ur3e_2f85.xml (task-space controller, truncation at 40 steps) and ur3e_raw.xml (joint PD): the same property."""
    rng = np.random.default_rng(3)
    g = make(ASSETS, "ur3e_2f85.xml", 24, dtype, ctrl_mode=lib.CTRL_PID_TASK, obs_kind=lib.OBS_STATE, obs_dim=28, act_dim=7,
             gains=OE.GAINS_TASK, reset_key=1, max_steps=40, auto_reset=1, frame_skip=3)
    g.reset()
    g.enable_sensors()
    tcp = g.query([("site", "tcp")])(pos=True)[0][:, 0].double().cpu().numpy()
    T = 60
    a = np.zeros((T, g.n, 7))
    a[:, :, :3] = tcp[None] + rng.uniform(-0.04, 0.04, (1, g.n, 3))
    a[:, :, 3:6] = OE.TOOL_ROTVEC
    a[:, :, 6] = rng.uniform(0, 1, (T, g.n))
    _, first = _live_vs_branch(g, torch.tensor(a, dtype=dtype, device="cuda"))
    assert int(first.max()) == 40   # truncated when t = 40 before the step's increment

    m = Model(ASSETS + "/ur3e_raw.xml")
    r = SimBatch(m, env_config(ctrl_mode=lib.CTRL_PD_JOINT, obs_kind=lib.OBS_STATE, obs_dim=12, act_dim=6, gains=OE.GAINS_J), 24, 0, dtype)
    r.reset()
    r.enable_sensors()
    a = np.cumsum(rng.uniform(-0.05, 0.05, (T, r.n, 6)), axis=0)
    _live_vs_branch(r, torch.tensor(a, dtype=dtype, device="cuda"))


def test_repeated_and_permuted_ids():
    """Copies of one source with equal actions are bitwise equal to each other and to that source at another position and another
    m, including m > n."""
    b = _v2_settled(16, torch.float32, settle=95)
    T, n = 24, b.n
    mug = b.obs[:, 3:6].clone()
    per_src = torch.stack([_scripted(b, mug, 95 + k) for k in range(T)])   # [T, n, 4]: the actions of a rollout follow its source
    outs = dict(qpos=True, qvel=True, obs=True, reward=True, terminated=True, truncated=True, info=True)
    ref = {k: v.clone() for k, v in b.rollout(per_src.contiguous(), **outs)._asdict().items() if v is not None}
    g = torch.Generator(device="cpu"); g.manual_seed(0)
    for ids in ([3, 3, 7, 0, 3, 15], torch.randint(0, n, (3 * n + 5,), generator=g).tolist() + [3, 3]):
        idt = torch.tensor(ids, dtype=torch.int32, device="cuda")
        got = b.rollout(per_src[:, idt.long()].contiguous(), env_ids=idt, **outs)
        for k, v in ref.items():
            w = getattr(got, k)
            assert torch.equal(w, v[idt.long()] if k == "info" else v[:, idt.long()]), (len(ids), k)


def test_batch_untouched():
    """Two identical batches, one of which runs rollouts (both source kinds, every output) between its steps: records, statistics,
    the sensor buffer, the tier step counts and the later step outputs stay bitwise equal."""
    A, B = _v2_settled(48, torch.float32, settle=0), _v2_settled(48, torch.float32, settle=0)
    for x in (A, B):
        x.enable_sensors()
    mug = A.obs[:, 3:6].clone()
    qp0, qv0, ws0 = (t[:10].contiguous() for t in A.get_state())
    ids = torch.tensor([5, 5, 0, 47, 12, 3, 60, -2], dtype=torch.int32, device="cuda")
    outs = dict(qpos=True, qvel=True, obs=True, reward=True, terminated=True, truncated=True, sensordata=True, info=True)
    launches = B.launch_count
    for k in range(130):
        a = _scripted(A, mug, k).contiguous()
        if k % 10 == 0:
            A.rollout(a[None].repeat(5, 1, 1).contiguous(), **outs)
            A.rollout(a[ids.long().clamp(0, A.n - 1)][None].repeat(3, 1, 1).contiguous(), env_ids=ids, **outs)
            A.rollout(a[:10][None].repeat(4, 1, 1).contiguous(), state=(qp0, qv0), **outs)
            A.rollout(a[:10][None].repeat(4, 1, 1).contiguous(), state=(qp0, qv0, ws0), **outs)
        oa, ob = A.step(a), B.step(a)
        for x, y in zip(oa, ob):
            assert torch.equal(x, y), k
        assert torch.equal(A.final_obs, B.final_obs) and torch.equal(A.sensors, B.sensors), k
    for x, y in zip(A.get_state(), B.get_state()):
        assert torch.equal(x, y)
    assert A.stats_dict() == B.stats_dict()
    la, lb = A.kernel_info()["lite"], B.kernel_info()["lite"]
    assert (la["lite_tier_steps"], la["full_only_steps"]) == (lb["lite_tier_steps"], lb["full_only_steps"]) == (130, 0)
    assert A.launch_count > B.launch_count > launches


@pytest.mark.parametrize("warm", [False, True])
def test_explicit_states_equal_set_state_then_step(warm):
    """A rollout from explicit states S on a batch of n != m equals a fresh auto_reset=0 batch of m that resets, set_state(S) and steps."""
    src = _v2_settled(12, torch.float32, settle=110)
    qp, qv, ws = src.get_state()
    state = (qp, qv, ws) if warm else (qp, qv)
    mug = src.obs[:, 3:6].clone()
    T = 40
    acts = torch.stack([_scripted(src, mug, 110 + k) for k in range(T)]).contiguous()
    b = make(ASSETS, "main.xml", 20, torch.float32, **V2)
    b.reset(seed=1)
    r = b.rollout(acts, state=state, qpos=True, qvel=True)
    f = make(ASSETS, "main.xml", 12, torch.float32, **dict(V2, auto_reset=0))
    f.reset(seed=4)
    f.set_state(*state)
    for t in range(T):
        o, rw, te, tr = f.step(acts[t])
        fq, fv, _ = f.get_state()
        for x, y in ((r.obs[t], o), (r.reward[t], rw), (r.terminated[t], te), (r.truncated[t], tr), (r.qpos[t], fq), (r.qvel[t], fv)):
            assert torch.equal(x, y), t


def test_oracle_task_space_f64():
    """float64 explicit-state rollout on ur3e_2f85.xml, pid_task_ctrl every mj_step, 1500 steps against the oracle's control loop:
    qpos and qvel within 1e-9 relative on every step, no re-seeding (the setting of test_gripper_task_space_f64)."""
    xml = ASSETS + "/ur3e_2f85.xml"
    loop = OE.OracleCtrlLoop(xml, "pid_task", OE.GAINS_TASK)
    b = make(ASSETS, "ur3e_2f85.xml", 3, torch.float64, ctrl_mode=lib.CTRL_PID_TASK, obs_kind=lib.OBS_STATE, obs_dim=28, act_dim=7,
             gains=OE.GAINS_TASK, reset_key=1)
    b.reset()
    qp, qv = loop.m.key("down"); loop.set_state(qp, qv)
    loop.d.forward()
    tcp0 = loop.d.site_xpos.reshape(-1, 3)[loop.tcp].copy()
    T = 1500
    tgt = np.stack([np.hstack([tcp0 + [0.05, -0.03, 0.04], OE.TOOL_ROTVEC, 0.5 if k > 700 else 0.0]) for k in range(T)])
    st = tuple(torch.tensor(x[None], dtype=torch.float64, device="cuda") for x in (qp, qv))
    r = b.rollout(torch.tensor(tgt[:, None], dtype=torch.float64, device="cuda"), state=st, qpos=True, qvel=True, obs=False, info=True)
    rq, rv = r.qpos[:, 0].cpu().numpy(), r.qvel[:, 0].cpu().numpy()
    worst = 0.0
    for k in range(T):
        q, v = loop.step(tgt[k])
        worst = max(worst, rel(rq[k], q), rel(rv[k], v))
    assert worst < 1e-9, worst
    assert r.info.abs().sum().item() == 0


def test_no_reset_after_done():
    """v2 with max_steps 5 from a reset, T = 10: truncated from step 4 on, the rollout keeps stepping (bitwise the trajectory of an
    auto_reset=0 batch; no jump back to the keyframe) and info is zero."""
    b = make(ASSETS, "main.xml", 8, torch.float32, **dict(V2, max_steps=5))
    o0 = b.reset(seed=2).clone()
    T = 10
    a = torch.zeros(T, b.n, 4, device="cuda")
    a[:, :, :3] = o0[None, :, :3] + torch.tensor([0.08, -0.05, 0.06], device="cuda")
    a = a.contiguous()
    r = b.rollout(a, qpos=True, info=True)
    assert bool((r.truncated[4:] == 1).all()) and not bool(r.truncated[:4].any())
    assert r.info.abs().sum().item() == 0
    f = make(ASSETS, "main.xml", 8, torch.float32, **dict(V2, max_steps=5, auto_reset=0))
    f.reset(seed=2)
    for t in range(T):
        o = f.step(a[t])[0]
        assert torch.equal(r.obs[t], o), t
    assert (r.obs[T - 1, :, :3] - o0[:, :3]).norm(dim=1).min().item() > 1e-3   # the tcp moved on, away from the reset pose


def test_invalid_ids():
    """Ids -1 and n among valid ones: finite outputs, info[:, 0] >= 1 for those two, and the valid rollouts are bitwise equal to a
    call without them."""
    b = _v2_settled(16, torch.float32, settle=20)
    n, T = b.n, 12
    a = torch.stack([_scripted(b, b.obs[:, 3:6], 20 + k) for k in range(T)])   # [T, n, 4]
    ids = [0, -1, 5, n, 2]
    valid = [0, 2, 4]
    idt = torch.tensor(ids, dtype=torch.int32, device="cuda")
    acts = a[:, idt.long().clamp(0, n - 1)].contiguous()
    outs = dict(qpos=True, qvel=True, obs=True, reward=True, terminated=True, truncated=True, sensordata=True, info=True)
    r = {k: v.clone() for k, v in b.rollout(acts, env_ids=idt, **outs)._asdict().items()}
    for k in ("qpos", "qvel", "obs", "reward", "sensordata"):
        assert bool(torch.isfinite(r[k]).all()), k
    assert r["info"][1, 0].item() >= 1 and r["info"][3, 0].item() >= 1
    sub = torch.tensor([ids[j] for j in valid], dtype=torch.int32, device="cuda")
    s = b.rollout(acts[:, valid].contiguous(), env_ids=sub, **outs)
    for k, v in s._asdict().items():
        assert torch.equal(v, r[k][valid] if k == "info" else r[k][:, valid]), k


def test_side_stream_and_rejected_calls():
    b = _v2_settled(16, torch.float32, settle=20)
    T, n = 6, b.n
    a = b.obs[:, :4].clone()
    a[:, 3] = 0.5
    acts = a[None].repeat(T, 1, 1).contiguous()
    ref = [x.clone() for x in b.rollout(acts, obs=True, reward=True)[2:4]]
    s = torch.cuda.Stream()
    # the caller orders the side stream after the default one: acts, the batch's rollout workspace and the owned outputs (which
    # ref's clones read) were last used there (ur3e_batch_rollout: calls on different streams must be ordered by the caller)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = [x.clone() for x in b.rollout(acts, obs=True, reward=True)[2:4]]
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    assert all(torch.equal(x, y) for x, y in zip(ref, got))

    ids = torch.arange(n, dtype=torch.int32, device="cuda")
    st = tuple(t.contiguous() for t in b.get_state()[:2])
    with pytest.raises(ValueError):
        b.rollout(acts, env_ids=ids, state=st)
    with pytest.raises(ValueError):
        b.rollout(acts, obs=False, reward=False, terminated=False, truncated=False)
    with pytest.raises(ValueError):
        b.rollout(acts.double())
    with pytest.raises(ValueError):
        b.rollout(acts[0])
    with pytest.raises(ValueError):
        b.rollout(acts, env_ids=ids.long())
    with pytest.raises(RuntimeError, match="T=0"):
        b.rollout(acts[:0].contiguous())

    L = b._L
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    rew = torch.empty(T, n, device="cuda")
    out = lib.RolloutOut(reward=rew.data_ptr())
    none = lib.RolloutOut()
    qp, qv = st
    cases = [  # (src, qpos0, qvel0, ws0, m, T, actions, out) -> message
        ((ids, None, None, None, n, T, acts, out), None),
        ((ids, qp, qv, None, n, T, acts, out), "both sources"),
        ((None, None, None, None, n, T, acts, out), "no source"),
        ((None, qp, None, None, n, T, acts, out), "without qvel0"),
        ((None, None, qv, None, n, T, acts, out), "without qpos0"),
        ((ids, None, None, None, n, T, None, out), "actions is null"),
        ((ids, None, None, None, 0, T, acts, out), "m=0"),
        ((ids, None, None, None, 2 ** 31, T, acts, out), "2^31"),
        ((ids, None, None, None, n, 0, acts, out), "T=0"),
        ((ids, None, None, None, n, T, acts, None), "out is null"),
        ((ids, None, None, None, n, T, acts, none), "all outputs are null"),
    ]
    for (src, q0, v0, w0, m, t, act, o), msg in cases:
        rc = L.ur3e_batch_rollout(b.ptr, vp(src), vp(q0), vp(v0), vp(w0), m, t, vp(act), C.byref(o) if o is not None else None, b._stream())
        if msg is None:
            assert rc == 0, lib.last_error()
        else:
            assert rc < 0 and msg in lib.last_error(), (msg, lib.last_error())
    torch.cuda.synchronize()
    assert torch.equal(rew, ref[1])
