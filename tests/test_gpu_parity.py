"""GPU parity: the CUDA path (through the C ABI) against the float64 oracle on identical states and actions.

Tolerances (BASELINE.json north_star): float64 build <= 1e-9 relative per step on contact-free trajectories,
<= 1e-4 relative per step (re-seeded from the oracle state) on contact-rich ones; float32 drift bounds stated per test.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import envs as OE
from oracle import oracle as O
import ur3e_b200._lib as lib
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.model import Model


def rel(a, b, floor=1e-3):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor)))


def make(assets, xml, n, dtype, **cfg):
    m = Model(assets + "/" + xml)
    c = env_config(**cfg)
    return SimBatch(m, c, n, 0, dtype)


def test_raw_move_j_f64(assets):
    """config 1: ur3e_raw.xml, pd_joint_ctrl on a joint-space trajectory, no re-seeding, 1e-9 relative per step."""
    xml = assets + "/ur3e_raw.xml"
    loop = OE.OracleCtrlLoop(xml, "pd_joint", OE.GAINS_J)
    b = make(assets, "ur3e_raw.xml", 2, torch.float64, ctrl_mode=lib.CTRL_PD_JOINT, obs_kind=lib.OBS_STATE, obs_dim=12, act_dim=6, gains=OE.GAINS_J)
    b.reset()
    loop.set_state(np.zeros(6), np.zeros(6))
    rng = np.random.default_rng(42)
    way = np.cumsum(rng.uniform(-0.02, 0.02, (40, 6)), axis=0)
    worst = 0.0
    for k in range(4000):
        tgt = way[k // 100]
        qp, qv = loop.step(tgt)
        a = torch.tensor(np.tile(tgt, (2, 1)), dtype=torch.float64, device="cuda")
        obs, *_ = b.step(a)
        o = obs[0].cpu().numpy()
        worst = max(worst, rel(o[:6], qp), rel(o[6:], qv))
    assert worst < 1e-9, worst
    assert torch.equal(obs[0], obs[1])


def test_config1_build_traj_j_stream_f64(assets):
    """BASELINE.md section 4 gate 1 / SURVEY 8d config 1 on the stated stream: ur3e_raw.xml (dt 1e-4), pd_joint_ctrl through
    move_j.get_joint_delta with config_j.yml gains, q0 = qvel0 = 0, targets = build_traj_j(zeros(7), hold=120) (np.random.seed(42):
    500 waypoints x 120 = 60 000 rows, first six columns), no re-seeding: qpos and qvel within 1e-9 relative on every step."""
    from ur3e_b200.controller import build_traj as BT
    traj = BT.build_traj_j(np.zeros(7), hold=120)           # [60000, 7]; pinned to the reference's own output by tests/test_build_traj_cpu.py
    tj = traj.to(torch.float64).cpu().numpy()
    assert tj.shape == (60000, 7)
    xml = assets + "/ur3e_raw.xml"
    loop = OE.OracleCtrlLoop(xml, "pd_joint", OE.GAINS_J)
    b = make(assets, "ur3e_raw.xml", 1, torch.float64, ctrl_mode=lib.CTRL_PD_JOINT, obs_kind=lib.OBS_STATE, obs_dim=12, act_dim=6, gains=OE.GAINS_J)
    b.reset()
    loop.set_state(np.zeros(6), np.zeros(6))
    acts = traj[:, :6].to(device="cuda", dtype=torch.float64).contiguous()
    T = tj.shape[0]
    rec = torch.empty(T, 12, dtype=torch.float64, device="cuda")
    for k in range(T):
        obs, *_ = b.step(acts[k:k + 1])
        rec[k] = obs[0]
    got = rec.cpu().numpy()
    worst = 0.0
    for k in range(T):
        qp, qv = loop.step(tj[k, :6])
        worst = max(worst, rel(got[k, :6], qp), rel(got[k, 6:], qv))
    assert worst < 1e-9, worst
    assert np.abs(got[:, :6]).max() > 0.3      # the arm does move along the stream


def test_gripper_task_space_f64(assets):
    """config 2 semantics: ur3e_2f85.xml, pid_task_ctrl every mj_step, contact-free, 1e-9 relative per step (no re-seeding)."""
    xml = assets + "/ur3e_2f85.xml"
    loop = OE.OracleCtrlLoop(xml, "pid_task", OE.GAINS_TASK)
    b = make(assets, "ur3e_2f85.xml", 1, torch.float64, ctrl_mode=lib.CTRL_PID_TASK, obs_kind=lib.OBS_STATE, obs_dim=28, act_dim=7, gains=OE.GAINS_TASK, reset_key=1)
    b.reset()
    qp, qv = loop.m.key("down"); loop.set_state(qp, qv)
    loop.d.forward()
    tcp0 = loop.d.site_xpos.reshape(-1, 3)[loop.tcp].copy()
    worst = 0.0
    for k in range(1500):
        tgt = np.hstack([tcp0 + [0.05, -0.03, 0.04], OE.TOOL_ROTVEC, 0.5 if k > 700 else 0.0])
        qp, qv = loop.step(tgt)
        obs, *_ = b.step(torch.tensor(tgt[None], dtype=torch.float64, device="cuda"))
        o = obs[0].cpu().numpy()
        worst = max(worst, rel(o[:14], qp), rel(o[14:], qv))
    assert worst < 1e-9, worst


def _random_states(m, rng, n, lift=False):
    qp0, _ = m.key("down")
    qp = np.tile(qp0, (n, 1)); qv = rng.uniform(-0.5, 0.5, (n, m.nv))
    qp[:, :6] += rng.uniform(-0.3, 0.3, (n, 6))
    qp[:, 6] = qp[:, 10] = rng.uniform(0, 0.6, n)
    qp[:, 16] -= rng.uniform(0, 0.002, n)  # mug pressed into the table: contacts active
    return qp, qv


def test_main_forward_internals_via_queries_f64(assets):
    """mj_forward quantities (M, qfrc_bias, qacc, ncon, nefc, the tcp Jacobian) on random main.xml states with mug-table contacts,
    read for every environment through forward(), mass_matrix() and Query.jac."""
    m = O.Model(assets + "/main.xml"); d = O.Data(m)
    rng = np.random.default_rng(3)
    n = 8
    qp, qv = _random_states(m, rng, n)
    b = make(assets, "main.xml", n, torch.float64, ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2, reset_key=1, term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500)
    b.reset()
    b.set_state(torch.tensor(qp, device="cuda"), torch.tensor(qv, device="cuda"))
    fwd = b.forward(qacc=True, info=True)
    qacc, info = fwd.qacc.cpu().numpy(), fwd.info.cpu().numpy()
    M, bias = (x.cpu().numpy() for x in b.mass_matrix(M=True, qfrc_bias=True))
    jacp, jacr = (x.cpu().numpy() for x in b.query([("site", "tcp")]).jac(jacp=True, jacr=True)[:2])
    for e in range(n):
        d.reset(); d.set_state(qp[e], qv[e]); d.forward()
        assert info[e, 0] == d.ncon and info[e, 1] == d.nefc
        assert rel(M[e], d.fullM(), 1e-6) < 1e-9
        assert rel(bias[e], d.qfrc_bias) < 1e-9
        assert rel(qacc[e], d.qacc, 1e-1) < 1e-6
        jp, jr = d.jac_site(m.id("site", "tcp"))
        assert rel(np.vstack([jacp[e, 0, :, :6], jacr[e, 0, :, :6]]), np.vstack([jp[:, :6], jr[:, :6]]), 1e-3) < 1e-9


@pytest.mark.parametrize("kind", ["v2", "v0", "indirect"])
def test_env_step_reseeded_f64(assets, kind):
    """Env.step parity (obs, reward, done) with per-step re-seeding from the oracle state: <= 1e-4 relative per step."""
    xml = assets + "/main.xml"
    env = OE.OracleEnv(xml, kind)
    cfgs = dict(
        v2=dict(obs_kind=lib.OBS_V2, obs_dim=24, frame_skip=2, term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500, gains=OE.GAINS_MUG),
        v0=dict(obs_kind=lib.OBS_V0, obs_dim=13, frame_skip=2, term_kind=lib.TERM_V0, reward_kind=lib.REW_V0, max_steps=500, gains=OE.GAINS_V0),
        indirect=dict(obs_kind=lib.OBS_V2, obs_dim=24, frame_skip=1, term_kind=lib.TERM_NONE, reward_kind=lib.REW_MINUS1, max_steps=2500, gains=OE.GAINS_MUG))
    b = make(assets, "main.xml", 1, torch.float64, ctrl_mode=lib.CTRL_PID_TASK_ENV, act_dim=4, reset_key=1, **cfgs[kind])
    b.reset()
    o0 = env.reset()
    assert rel(b.obs[0].cpu().numpy(), o0) < 1e-9
    rng = np.random.default_rng(7)
    mug = o0[3:6].copy()
    worst = 0.0
    for k in range(300):
        # scripted approach + grasp so that pad-mug contacts occur
        tgt = mug + [0, 0, 0.02 + max(0.0, 0.1 - 0.001 * k)]
        a = np.hstack([tgt + rng.normal(0, 0.002, 3), 1.0 if k > 150 else 0.0])
        # re-seed the GPU state from the oracle's (qpos, qvel, warmstart) and replay its stale cache by stepping from the same state
        qp, qv, ws = env.d.qpos.copy(), env.d.qvel.copy(), env.d.qacc_warmstart.copy()
        if k % 25 == 0:
            env.set_state(qp, qv); env.t = k
            b.set_state(torch.tensor(qp[None], device="cuda"), torch.tensor(qv[None], device="cuda"))
        o, r, te, tr = env.step(a)
        obs, rew, term, trunc = b.step(torch.tensor(a[None], dtype=torch.float64, device="cuda"))
        worst = max(worst, rel(obs[0].cpu().numpy(), o), rel(rew[0].item(), r, 1.0))
        assert bool(term[0].item()) == te and bool(trunc[0].item()) == tr, (k, term, te, trunc, tr)
        if te or tr:
            break
    assert worst < 1e-4, worst


def test_f32_drift_main(assets):
    """float32 production build vs the float64 build on the v2 env: stated drift bound over 200 env-steps of a resting scene
    (obs abs error <= 2e-3; the scripted motion is slow so the chaos of contact switching is not excited)."""
    cfg = dict(ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2, reset_key=1,
               term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500)
    b32 = make(assets, "main.xml", 4, torch.float32, **cfg); b64 = make(assets, "main.xml", 4, torch.float64, **cfg)
    o32 = b32.reset().clone(); o64 = b64.reset().clone()
    assert torch.allclose(o32.double(), o64, atol=1e-5)
    a = o64[:, 0:3].clone(); a[:, 2] += 0.02
    a = torch.cat([a, torch.zeros(4, 1, dtype=torch.float64, device="cuda")], 1)
    for k in range(200):
        o64, *_ = b64.step(a); o32, *_ = b32.step(a.float())
    assert torch.isfinite(o32).all()
    assert (o32.double() - o64).abs().max().item() < 2e-3


def test_auto_reset_and_stats(assets):
    """In-kernel auto-reset: truncation after max_steps resets t, returns the reset obs and keeps the terminal obs; counters add up."""
    n = 64
    b = make(assets, "main.xml", n, torch.float32, ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2,
             reset_key=1, term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=5, auto_reset=1, reset_noise=lib.NOISE_HIGH)
    o0 = b.reset(seed=123).clone()
    assert o0[:, 3].std() > 0 and o0[:, 4].std() > 0            # mug x,y noise differs per env
    assert (o0[:, 3] >= 0.29799994 - 1e-6).all() and (o0[:, 3] <= 0.31799994 + 1e-6).all()
    a = torch.cat([o0[:, 0:3], torch.zeros(n, 1, device="cuda")], 1).contiguous()
    ndone, lens, tlen = 0, torch.zeros(n, device="cuda"), 0.0
    for k in range(10):
        obs, rew, term, trunc = b.step(a)
        done = (term | trunc).bool()
        lens += 1
        ndone += int(done.sum().item()); tlen += float(lens[done].sum().item()); lens[done] = 0
        assert (lens <= 5).all()                                 # nobody outlives max_steps
        # a finished env returns its reset observation (tcp back at the keyframe) and keeps the terminal one in final_obs
        if done.any():
            assert (obs[done][:, 0:3] - o0[done][:, 0:3]).abs().max() < 1e-5
    assert ndone >= n                                            # every env was truncated at least once in 10 steps
    st = b.stats_dict()
    assert st["episodes"] == ndone and st["substeps"] == n * 10 * 2
    assert st["length_sum"] == tlen


@pytest.mark.parametrize("noise,ylo,yhi", [(lib.NOISE_LOW, -0.1, 0.01), (lib.NOISE_MED, -0.2, 0.1), (lib.NOISE_HIGH, -0.25, 0.2)])
def test_reset_noise_ranges(assets, noise, ylo, yhi):
    """gym_utils.py:48-60: mug x in [0, 0.02], y in the level's range, added to keyframe 'down' (main.xml:416-419); both fill their range."""
    n = 4096
    b = make(assets, "main.xml", n, torch.float32, ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2,
             reset_key=1, term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500, reset_noise=noise)
    o = b.reset(seed=77).double().cpu().numpy()
    dx, dy = o[:, 3] - 0.29799994, o[:, 4] - 0.13349916
    assert dx.min() >= -1e-6 and dx.max() <= 0.02 + 1e-6 and dx.max() - dx.min() > 0.95 * 0.02
    assert dy.min() >= ylo - 1e-6 and dy.max() <= yhi + 1e-6 and dy.max() - dy.min() > 0.95 * (yhi - ylo)
    assert abs(np.corrcoef(dx, dy)[0, 1]) < 0.1                      # independent draws
    assert np.abs(o[:, 5] - 0.055111).max() < 1e-6                   # z untouched


def test_tier_choice_is_deterministic_and_shard_invariant(assets):
    """ADVICE r1: which size class steps an environment is decided per environment on the device, so float32 trajectories are
    bit-identical between two runs, between one batch of 2 n and two batches of n (world size 1 vs 2, RNG keyed by the global
    id) and between the device path and the chunked host path -- while a part of the batch is in grasp (full tier)."""
    n = 96
    cfg = dict(ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2, reset_key=1,
               term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500, reset_noise=lib.NOISE_LOW, auto_reset=1, lite_max_contacts=4)
    whole, again = make(assets, "main.xml", 2 * n, torch.float32, **cfg), make(assets, "main.xml", 2 * n, torch.float32, **cfg)
    lo, hi = make(assets, "main.xml", n, torch.float32, **cfg), make(assets, "main.xml", n, torch.float32, env_id_base=n, **cfg)
    o = whole.reset(seed=9).clone(); again.reset(seed=9); lo.reset(seed=9); hi.reset(seed=9)
    mug0 = o[:, 3:6].clone()
    full_seen = 0
    for k in range(260):
        a = torch.empty(2 * n, 4, device="cuda")
        a[:, 0:2] = whole.obs[:, 3:5]
        a[:, 2] = mug0[:, 2] + 0.02 + max(0.0, 0.1 - 0.002 * k)
        a[:, 3] = 1.0 if k > 90 else 0.0
        a[::3, 3] = 0.0                                               # a third of the batch never closes: mixed tiers
        a = a.contiguous()
        ow = whole.step(a)[0]; oa = again.step(a)[0]
        ol = lo.step(a[:n].contiguous())[0]; oh = hi.step(a[n:].contiguous())[0]
        assert torch.equal(ow, oa), k
        assert torch.equal(ow[:n], ol) and torch.equal(ow[n:], oh), k
        if k % 20 == 0:
            torch.cuda.synchronize()
            full_seen = max(full_seen, whole.kernel_info()["lite"]["last_overflow_envs"])
    assert 0 < full_seen < 2 * n        # some, not all, environments were stepped by the full tier


def test_host_entry_point(assets):
    n = 32
    b = make(assets, "main.xml", n, torch.float32, ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2,
             reset_key=1, term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500)
    o0 = b.reset().cpu().numpy()
    a = np.ascontiguousarray(np.hstack([o0[:, :3], np.zeros((n, 1))]).astype(np.float32))
    obs = np.zeros((n, 24), np.float32); rew = np.zeros(n, np.float32); te = np.zeros(n, np.uint8); tr = np.zeros(n, np.uint8)
    b.step_host(a, obs, rew, te, tr)
    assert np.isfinite(obs).all() and np.abs(obs[:, :3] - o0[:, :3]).max() < 1e-2


def test_host_entry_point_chunked_pipeline_matches_device_path(assets):
    """Batches >= 16384 environments go through the host entry point in four ranges on two streams (copies overlap the
    stepping); every environment's result is bit-identical to the single-launch device path, incl. a ragged last range."""
    n = 16384 + 77
    cfg = dict(ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2, reset_key=1,
               term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500, reset_noise=lib.NOISE_HIGH, auto_reset=1)
    bh = make(assets, "main.xml", n, torch.float32, **cfg); bd = make(assets, "main.xml", n, torch.float32, **cfg)
    o0 = bh.reset(seed=5); assert torch.equal(o0, bd.reset(seed=5))
    rng = np.random.default_rng(0)
    obs = np.zeros((n, 24), np.float32); rew = np.zeros(n, np.float32); te = np.zeros(n, np.uint8); tr = np.zeros(n, np.uint8)
    for k in range(3):
        a = np.ascontiguousarray(np.hstack([o0[:, :3].cpu().numpy() + rng.uniform(-0.05, 0.05, (n, 3)), rng.uniform(0, 1, (n, 1))]).astype(np.float32))
        bh.step_host(a, obs, rew, te, tr)
        od, rd, ted, trd = bd.step(torch.tensor(a, device="cuda"))
        assert np.array_equal(obs, od.cpu().numpy()) and np.array_equal(rew, rd.cpu().numpy())
        assert np.array_equal(te, ted.cpu().numpy()) and np.array_equal(tr, trd.cpu().numpy())


def test_bad_state_autoreset_and_masked_reset(assets):
    """mj_checkPos/Vel autoreset (SURVEY B.10, MUJOCO_LOG.TXT): an environment with NaN / huge state is reset to qpos0 inside the
    step and counted; the others are untouched.  Masked reset only touches the selected environments."""
    n = 16
    b = make(assets, "main.xml", n, torch.float32, ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2,
             reset_key=1, term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500)
    o0 = b.reset(seed=5).clone()
    qpos, qvel, _ = b.get_state()
    q2 = qpos.clone(); v2 = qvel.clone()
    v2[3, 2] = float("nan"); v2[7, 0] = 1e12
    b.set_state(q2, v2)
    a = torch.cat([o0[:, 0:3], torch.zeros(n, 1, device="cuda")], 1).contiguous()
    obs, rew, term, trunc = b.step(a)
    assert torch.isfinite(obs).all() and torch.isfinite(rew).all()
    st = b.stats_dict()
    assert st["unstable_resets"] == 2
    qp, qv, _ = b.get_state()
    assert torch.isfinite(qp).all() and torch.isfinite(qv).all()
    good = [i for i in range(n) if i not in (3, 7)]
    assert (qp[good] - qpos[good]).abs().max() < 1e-2                 # healthy environments moved by one small step only
    assert (qp[3, :6]).abs().max() < 0.05 and (qp[7, :6]).abs().max() < 0.05   # mj_resetData: back at qpos0 (arm joints 0), then one step
    # masked reset
    for _ in range(20):
        b.step(a)
    before, _, _ = b.get_state()
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda"); mask[2] = 1; mask[9] = 1
    b.reset(seed=5, mask=mask)
    after, _, _ = b.get_state()
    keep = [i for i in range(n) if i not in (2, 9)]
    assert torch.equal(after[keep], before[keep])
    assert (after[2, :14] - qpos[2, :14]).abs().max() < 1e-6 and (after[9, :14] - qpos[9, :14]).abs().max() < 1e-6


def test_state_roundtrip_and_determinism(assets):
    """get_state -> set_state reproduces the trajectory bit for bit (the stale-kinematics cache is rebuilt by the forward pass of
    set_state exactly as MujocoEnv.set_state does), and two batches with the same seed agree bitwise."""
    n = 32
    mk = lambda: make(assets, "main.xml", n, torch.float32, ctrl_mode=lib.CTRL_PID_TASK_ENV, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=4, gains=OE.GAINS_MUG, frame_skip=2,
                      reset_key=1, term_kind=lib.TERM_V2, reward_kind=lib.REW_V2, max_steps=2500, auto_reset=1, reset_noise=lib.NOISE_HIGH)
    b1, b2 = mk(), mk()
    o1 = b1.reset(seed=11).clone(); o2 = b2.reset(seed=11).clone()
    assert torch.equal(o1, o2)
    g = torch.Generator(device="cuda"); g.manual_seed(0)
    for k in range(30):
        a = (o1[:, 0:4] + 0.02 * torch.randn(n, 4, device="cuda", generator=g)).contiguous(); a[:, 3] = 0.5
        x1 = b1.step(a)[0].clone(); x2 = b2.step(a)[0].clone()
        assert torch.equal(x1, x2)
    o3 = b2.reset(seed=12)
    assert not torch.equal(o3[:, 3:5], o2[:, 3:5])                    # a different seed draws different mug positions


def test_model_smaller_than_its_size_class_f64(assets, tmp_path):
    """A 5-dof arm (ur3e_raw.xml without its last joint and motor) runs in the 6-dof size class: the register-resident
    solve pads the missing row with an identity row, the unrolled mat-vec / row dots take their generic fall-backs."""
    src = open(assets + "/ur3e_raw.xml").read().split("\n")
    src = [ln for ln in src if "wrist_3_joint" not in ln]          # drops the joint and its motor; the link stays, welded to wrist_2
    path = str(tmp_path / "ur3e_5dof.xml")
    open(path, "w").write("\n".join(src))
    m = Model(path)
    assert (m.nv, m.nu) == (5, 5)
    om = O.Model(path); d = O.Data(om)
    b = SimBatch(m, env_config(ctrl_mode=lib.CTRL_RAW, obs_kind=lib.OBS_STATE, obs_dim=10, act_dim=5), 2, 0, torch.float64)
    b.reset()
    d.reset()
    rng = np.random.default_rng(3)
    worst = 0.0
    for k in range(600):
        u = rng.uniform(-3, 3, 5) if k % 50 == 0 else u
        d.ctrl[:] = u; d.step(1)
        obs, *_ = b.step(torch.tensor(np.tile(u, (2, 1)), dtype=torch.float64, device="cuda"))
        o = obs[0].cpu().numpy()
        worst = max(worst, rel(o[:5], d.qpos), rel(o[5:], d.qvel))
    assert worst < 1e-9, worst


def test_logging_sensors_f64(assets):
    """actuatorfrc, the two pad touch sensors and the tcp pose of every step against the oracle (main.xml; the arm sags under zero
    torque while the gripper closes, so a pad lands on the table and later the fingers meet): SURVEY 8a row a17."""
    from scipy.spatial.transform import Rotation
    from ur3e_b200 import utils as U
    m = O.Model(assets + "/main.xml"); d = O.Data(m)
    b = make(assets, "main.xml", 2, torch.float64, ctrl_mode=lib.CTRL_RAW, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=7, frame_skip=1, reset_key=1)
    b.reset(); sens = b.enable_sensors()
    qp, qv = m.key("down"); d.reset(); d.set_state(qp, qv)
    u = np.zeros(7); u[6] = 255.0
    ut = torch.tensor(np.tile(u, (2, 1)), dtype=torch.float64, device="cuda")
    worst_f = worst_t = worst_p = worst_q = 0.0; touched = 0
    for k in range(700):
        if k % 20 == 0:                     # re-seed both sides from the oracle state (contact-rich: 1e-4 per step)
            q0, v0 = d.qpos.copy(), d.qvel.copy()
            d.set_state(q0, v0); d.arr("qacc_warmstart")[:] = 0
            b.set_state(torch.tensor(np.tile(q0, (2, 1)), device="cuda"), torch.tensor(np.tile(v0, (2, 1)), device="cuda"))
        d.ctrl[:] = u; d.forward(); ref_tq = d.torque_sensors().ravel()      # velocity-dependent: evaluated on the pre-integration state, like mj_step's sensors
        d.step(1)
        b.step(ut)
        ref = d.sensors(); got = sens[0].cpu().numpy()
        worst_f = max(worst_f, rel(got[:7], ref[:7], 1e-2))
        worst_t = max(worst_t, rel(got[7:9], ref[7:9], 1.0))
        tcp = m.id("site", "tcp")
        worst_p = max(worst_p, rel(got[9:12], d.site_xpos.reshape(-1, 3)[tcp]), rel(got[12:21], d.site_xmat.reshape(-1, 9)[tcp], 1.0))
        worst_q = max(worst_q, rel(got[28:46], ref_tq, 1e-2))        # the six <torque> site sensors (main.xml:384-391)
        assert np.array_equal(got[21:28], u)                                              # d.ctrl as the controller set it
        touched += int(ref[7] > 0.1 or ref[8] > 0.1)
        if k == 650:
            ts = U.get_task_space_state(b)[0].cpu().numpy()
            rv = Rotation.from_matrix(d.site_xmat.reshape(-1, 3, 3)[tcp]).as_rotvec()
            assert np.abs(ts[3:6] - rv).max() < 1e-6 and ts[6] == float(ref[8] > 0.1)
            assert bool(U.get_boolean_grasp_contact(b)[0].item()) == bool((ref[8], ref[7]) > (0.1, 0.1))
            assert np.abs(U.get_joint_space_state(b)[0, :6].cpu().numpy() - d.qpos[:6]).max() < 1e-6
            assert np.abs(U.get_jnt_torques(b)[0].cpu().numpy() - ref[:7]).max() < 1e-4
    assert touched > 100, touched           # the scenario does exercise the touch sensors
    assert worst_f < 1e-4 and worst_t < 1e-4 and worst_p < 1e-6 and worst_q < 1e-4, (worst_f, worst_t, worst_p, worst_q)
    assert torch.equal(sens[0], sens[1])
    b.enable_sensors(False); b.step(ut)     # detached again: stepping no longer writes


def test_long_random_rollout_is_stable_f32(assets):
    """Soak: 6 000 env-steps (12 000 mj_steps) of U(action_space) actions on 4 096 production (float32) environments with auto-reset,
    i.e. every environment runs through truncation twice: observations stay finite, the bad-state guard (mj_checkPos / Vel / Acc,
    the reference's MUJOCO_LOG.TXT lists 20 such events) never fires, nothing overflows the largest size class, and the episode
    counters are consistent."""
    from ur3e_b200 import presets
    n = 4096
    m = Model(assets + "/main.xml")
    _, kw, lo, hi = presets.ENV_SPECS["gymnasium_env/ur3e-v2"]
    b = SimBatch(m, presets.make_config(m, kw, auto_reset=1), n, 0, torch.float32)
    b.reset(seed=3)
    lo_t, hi_t = torch.tensor(lo, device="cuda", dtype=torch.float32), torch.tensor(hi, device="cuda", dtype=torch.float32)
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    acts = [(lo_t + (hi_t - lo_t) * torch.rand(n, 4, device="cuda", generator=g)).contiguous() for _ in range(64)]
    bad = torch.zeros((), device="cuda")
    for k in range(6000):
        obs, rew, term, trunc = b.step(acts[k % 64], want_final_obs=False)
        if k % 50 == 0:
            bad += (~torch.isfinite(obs)).sum() + (~torch.isfinite(rew)).sum()
    st = b.stats_dict()
    assert bad.item() == 0
    assert st["unstable_resets"] == 0 and st["overflow_steps"] == 0
    assert st["steps"] == n * 6000 and st["substeps"] == 2 * n * 6000
    assert st["truncations"] >= 2 * n * 0.5 and st["episodes"] >= st["truncations"]
    assert st["episodes"] == st["truncations"] + st["successes"] + st["term_reach"] + st["term_toppled"] + st["term_collision"]
