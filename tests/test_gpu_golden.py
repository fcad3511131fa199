"""GPU parity against the committed golden fixtures (tests/golden, made by the reference's own Python over the oracle)
and of the user-facing Python layers (vector env API, SB3 adapter, controller entry points)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import ur3e_b200._lib as lib
from ur3e_b200 import controller, presets
from ur3e_b200.batch import SimBatch
from ur3e_b200.envs import SB3VecEnv, UR3eVecEnv
from ur3e_b200.model import Model, asset

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
IDS = {"v2": "gymnasium_env/ur3e-v2", "v0": "gymnasium_env/ur3e-v0", "indirect": "gymnasium_env/imitation_indirect-v0",
       "direct": "gymnasium_env/imitation_direct-v0"}


def rel(a, b, floor=1e-3):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor)))


@pytest.mark.parametrize("kind", ["v2", "v0", "indirect", "direct"])
def test_env_episode_vs_reference_fixture_f64(kind):
    """A whole scripted approach-grasp-lift episode (260 env-steps, pad-mug contacts) from the fixture's initial state, no
    re-seeding: float64 build within 1e-4 relative of what the reference's env classes produced.  `direct`
    (imitation_env_direct.py:74-130: raw 7-vector actuator commands, obs 13 with the grasp count and the tcp linear velocity)
    starts with both pads on the mug and releases half way."""
    g = np.load(GOLD + "/env_%s.npz" % kind)
    env = UR3eVecEnv(IDS[kind], 2, dtype=torch.float64, auto_reset=False, reset_noise=lib.NOISE_NONE)
    env.reset()
    env.set_state(torch.tensor(np.tile(g["qpos0"], (2, 1)), device="cuda"), torch.tensor(np.tile(g["qvel0"], (2, 1)), device="cuda"))
    worst = 0.0
    for k in range(len(g["reward"])):
        obs, rew, term, trunc, _ = env.step(torch.tensor(np.tile(g["actions"][k], (2, 1)), device="cuda"))
        worst = max(worst, rel(obs[0].cpu().numpy(), g["obs"][k]), abs(rew[0].item() - g["reward"][k]) / max(1.0, abs(g["reward"][k])))
        assert bool(term[0]) == bool(g["terminated"][k]) and bool(trunc[0]) == bool(g["truncated"][k])
    assert worst < 1e-4, worst
    assert torch.equal(obs[0], obs[1])                       # identical inputs -> bitwise identical environments
    qpos, qvel, _ = env.get_state()
    assert rel(qpos[0].cpu().numpy(), g["qpos"][-1]) < 1e-4


def test_pick_place_expert_episode_vs_reference_fixture_f64():
    """BASELINE config 4 parity: the reference's scripted expert (move_l_mug.py targets, build_traj_l_pick_place) run through the
    reference's own UR3eEnv2 class for a whole episode -- approach, grasp (up to 16 contacts), lift 6 cm, carry towards the ghost,
    truncation at step 2500 -- tests/golden/env_v2_pick.npz.  float64 CUDA build from the fixture's initial state, NO re-seeding:
    every observation and reward of the 2500 steps within 1e-4 relative, same robust-grasp flags, same truncation step."""
    g = np.load(GOLD + "/env_v2_pick.npz")
    T = len(g["reward"])
    assert T == 2500 and g["truncated"][-1] and not g["terminated"].any() and g["ncon"].max() >= 12 and g["obs"][:, 5].max() > 0.1
    env = UR3eVecEnv(IDS["v2"], 2, dtype=torch.float64, auto_reset=False, reset_noise=lib.NOISE_NONE)
    env.reset()
    env.set_state(torch.tensor(np.tile(g["qpos0"], (2, 1)), device="cuda"), torch.tensor(np.tile(g["qvel0"], (2, 1)), device="cuda"))
    acts = torch.tensor(g["actions"], device="cuda")
    rec_o = torch.empty(T, 24, dtype=torch.float64, device="cuda"); rec_r = torch.empty(T, dtype=torch.float64, device="cuda")
    flags = torch.empty(T, 2, dtype=torch.uint8, device="cuda")
    for k in range(T):
        obs, rew, term, trunc, _ = env.step(acts[k].expand(2, 4).contiguous())
        rec_o[k] = obs[0]; rec_r[k] = rew[0]; flags[k, 0] = term[0]; flags[k, 1] = trunc[0]
    o, r, f = rec_o.cpu().numpy(), rec_r.cpu().numpy(), flags.cpu().numpy()
    err_o = np.abs(o - g["obs"]) / (np.abs(g["obs"]) + 1e-3)
    err_r = np.abs(r - g["reward"]) / np.maximum(1.0, np.abs(g["reward"]))
    assert np.array_equal(o[:, 23], g["obs"][:, 23])                       # robust-grasp flag on exactly the same 1511 steps
    assert err_o.max() < 1e-4 and err_r.max() < 1e-4, (err_o.max(), int(err_o.max(axis=1).argmax()), err_r.max())
    assert np.array_equal(f[:, 0].astype(bool), g["terminated"]) and np.array_equal(f[:, 1].astype(bool), g["truncated"])


def test_pick_place_expert_succeeds_on_production_f32():
    """The same script on the float32 production kernels (two tiers: the grasp runs on the full size class): the mug is grasped,
    lifted and carried like in the reference episode (chaotic contact switching forbids a per-step bound over 2500 steps; the
    stated bound is on the outcome: lift height within 5 mm, robust-grasp step count within 10 %, end position within 1 cm)."""
    g = np.load(GOLD + "/env_v2_pick.npz")
    T = len(g["reward"]); n = 8
    env = UR3eVecEnv(IDS["v2"], n, dtype=torch.float32, auto_reset=False, reset_noise=lib.NOISE_NONE)
    env.reset()
    env.set_state(torch.tensor(np.tile(g["qpos0"], (n, 1)), device="cuda", dtype=torch.float32), torch.tensor(np.tile(g["qvel0"], (n, 1)), device="cuda", dtype=torch.float32))
    acts = torch.tensor(g["actions"], device="cuda", dtype=torch.float32)
    zmax = torch.zeros(n, device="cuda"); robust = torch.zeros(n, device="cuda")
    for k in range(T):
        obs, rew, term, trunc, _ = env.step(acts[k].expand(n, 4).contiguous())
        zmax = torch.maximum(zmax, obs[:, 5]); robust += obs[:, 23]
    assert torch.equal(obs[0], obs[n - 1])
    assert abs(zmax[0].item() - g["obs"][:, 5].max()) < 5e-3
    assert abs(robust[0].item() - g["obs"][:, 23].sum()) < 0.1 * g["obs"][:, 23].sum()
    assert np.abs(obs[0, 3:6].cpu().numpy() - g["obs"][-1, 3:6]).max() < 1e-2
    info = env.batch.kernel_info()["lite"]
    assert info["lite_tier_steps"] == T and env.episode_stats()["overflow_steps"] == 0


@pytest.mark.parametrize("kind", ["v2", "v0"])
def test_collision_predicates_vs_reference_fixture(kind):
    """tests/golden/collision.npz: one step of the reference's own UR3eEnv2 / UR3eEnv (their get_self_collision / get_table_collision,
    utils/gym_utils.py:146-201, run verbatim) from five injected arm poses: keyframe, two folded elbows (self-collision: both classes
    terminate; v0's reward carries -40), pads pressed on the table and gripper base on the table (v0's -25, no termination).  float64
    CUDA build: same flags, observation and reward within 1e-4; the episode statistics count the collision terminations."""
    g = np.load(GOLD + "/collision.npz")
    n = len(g[kind + "_qpos"])
    assert list(g[kind + "_self_collision"]) == [0, 1, 1, 0, 0] and list(g[kind + "_table_collision"]) == [0, 0, 0, 1, 1]
    env = UR3eVecEnv(IDS[kind], n, dtype=torch.float64, auto_reset=False, reset_noise=lib.NOISE_NONE)
    env.reset()
    env.set_state(torch.tensor(g[kind + "_qpos"], device="cuda"), torch.tensor(np.tile(g["qvel"], (n, 1)), device="cuda"))
    obs, rew, term, trunc, _ = env.step(torch.tensor(g[kind + "_action"], device="cuda"))
    assert [bool(x) for x in term.cpu()] == [bool(x) for x in g[kind + "_terminated"]]
    for e in range(n):
        assert rel(obs[e].cpu().numpy(), g[kind + "_obs"][e]) < 1e-4, e
        assert abs(rew[e].item() - g[kind + "_reward"][e]) < 1e-4 * max(1.0, abs(g[kind + "_reward"][e])), (e, rew[e].item(), g[kind + "_reward"][e])
    st = env.episode_stats()
    assert st["term_collision"] == 2 and st["episodes"] == 2


@pytest.mark.parametrize("kind", ["v2", "v0"])
def test_folded_arm_self_collision_vs_oracle(kind):
    """SURVEY 8f-3: box hulls stand in for the arm's collision meshes; get_self_collision (gym_utils.py:146-172) fires when the elbow
    folds the wrist onto the shoulder / upper arm: ur3e-v2 and ur3e-v0 terminate (ur3e_env2.py:244-246, ur3e_env.py:441-443), v0's
    reward carries the -40 penalty (ur3e_env.py:340).  float64 CUDA build against the oracle env from the same injected state."""
    from oracle import envs as OE
    ref = OE.OracleEnv(asset("main.xml"), kind)
    qp, qv = ref.m.key("down")
    env = UR3eVecEnv(IDS[kind], 3, dtype=torch.float64, auto_reset=False, reset_noise=lib.NOISE_NONE)
    env.reset()
    Q = np.tile(qp, (3, 1)); Q[1, 2] = 2.8; Q[2, 2] = 2.9           # env 0 stays at 'down', 1 and 2 fold the elbow
    env.set_state(torch.tensor(Q, device="cuda"), torch.tensor(np.tile(qv, (3, 1)), device="cuda"))
    o0 = ref.reset()
    a = np.hstack([o0[:3], 0.0])
    obs, rew, term, trunc, _ = env.step(torch.tensor(np.tile(a, (3, 1)), device="cuda"))
    for e in range(3):
        ref.set_state(Q[e], qv)
        assert ref.self_collision() == (1 if e else 0)
        o, r, te, tr = ref.step(a)
        assert bool(term[e]) == te == bool(e), (e, te)
        assert rel(obs[e].cpu().numpy(), o) < 1e-4 and abs(rew[e].item() - r) < 1e-4 * max(1.0, abs(r))
    st = env.episode_stats()
    assert st["term_collision"] == 2 and st["episodes"] == 2


@pytest.mark.parametrize("kind", ["v2", "v0", "indirect"])
def test_truncation_step_vs_reference_fixture(kind):
    """SURVEY 8a row a15: ur3e-v2 increments t before the truncation test (first truncated step 2500), the other three test first
    (501 / 2501 / 1201).  tests/golden/truncation.npz holds what the reference's own classes reported under a hold-still action;
    the production float32 kernel, with the shipped max_steps, must truncate on exactly that step (and auto-reset right there)."""
    _check_truncation_vs_fixture(kind)


def test_direct_truncation_step_vs_reference_fixture():
    """The same for imitation_direct-v0, whose hold-still action is the gravity compensation at the keyframe (from mass_matrix)."""
    _check_truncation_vs_fixture("direct")


def _check_truncation_vs_fixture(kind):
    first_ref, term_ref = np.load(GOLD + "/truncation.npz")[kind]
    assert term_ref == 0
    env = UR3eVecEnv(IDS[kind], 3, dtype=torch.float32, auto_reset=True, reset_noise=lib.NOISE_NONE)
    obs, _ = env.reset()
    if kind == "direct":
        hold = torch.zeros(3, 7, device="cuda")
        hold[:, :6] = env.batch.mass_matrix(M=False, qfrc_bias=True)[1][0, :6]    # gravity compensation at the keyframe
    else:
        hold = torch.cat([obs[:, :3], torch.zeros(3, 1, device="cuda")], 1).contiguous()
    first = -1
    tr_all = []
    for k in range(1, int(first_ref) + 3):
        _, _, te, tr, _ = env.step(hold)
        tr_all.append(tr.clone())
        assert not te.any()
    tr_all = torch.stack(tr_all).cpu().numpy()
    for e in range(3):
        idx = np.nonzero(tr_all[:, e])[0]
        assert idx[0] + 1 == first_ref, (kind, idx[:3], first_ref)
        assert len(idx) == 1                       # auto-reset: t starts again at 0, so no second truncation two steps later
    assert env.episode_stats()["truncations"] == 3


def test_controllers_vs_reference_fixture():
    """pid_task_ctrl / move_j.ctrl of the reference on random ur3e_2f85.xml states: the kernel's ctrl is checked through the
    actuator it drives -- one mj_step from the fixture state with the fixture's target must match the oracle stepping with the
    reference's own u."""
    from oracle import oracle as O
    g = np.load(GOLD + "/controllers.npz")
    n = len(g["qpos"])
    m = Model(asset("ur3e_2f85.xml")); om = O.Model(asset("ur3e_2f85.xml")); od = O.Data(om)
    for mode, gains, tgt, u_ref in ((lib.CTRL_PID_TASK, g["gains_task"], g["traj"], g["u_task"]), (lib.CTRL_PD_JOINT, g["gains_j"], g["target_j"], g["u_joint"]),
                                    (lib.CTRL_PINV, g["gains_pinv"], g["traj"], g["u_pinv"])):
        cfg = presets.make_config(m, dict(ctrl_mode=mode, obs_kind=lib.OBS_STATE, obs_dim=28, act_dim=7, frame_skip=1, gains=gains, reset_key="down"))
        b = SimBatch(m, cfg, n, 0, torch.float64)
        b.reset()
        b.set_state(torch.tensor(g["qpos"], device="cuda"), torch.tensor(g["qvel"], device="cuda"))
        obs, *_ = b.step(torch.tensor(tgt, device="cuda"))
        for i in range(n):
            od.reset(); od.set_state(g["qpos"][i], g["qvel"][i]); od.forward(); od.ctrl[:] = u_ref[i]; od.step(1)
            assert rel(obs[i, :14].cpu().numpy(), od.qpos) < 1e-9 and rel(obs[i, 14:].cpu().numpy(), od.qvel, 1e-2) < 1e-8


def test_vec_env_api_and_sb3_adapter():
    env = UR3eVecEnv("gymnasium_env/ur3e-v2", 16)
    assert env.single_observation_space.shape == (24,) and env.single_action_space.shape == (4,) and env.metadata["render_fps"] == 500
    obs, info = env.reset(seed=3)
    assert obs.shape == (16, 24) and obs.is_cuda
    with pytest.raises(ValueError, match="Action dimension mismatch"):
        env.step(torch.zeros(16, 7, device="cuda"))
    sb = SB3VecEnv("gymnasium_env/ur3e-v2", 8, max_steps=4)
    o = sb.reset()
    assert o.shape == (8, 24) and o.dtype == np.float64
    rng = np.random.default_rng(0)
    seen = False
    for k in range(6):
        a = np.stack([sb.action_space.sample() if hasattr(sb.action_space, "sample") else np.zeros(4) for _ in range(8)])
        a[:, :3] = o[:, :3]
        o, r, done, infos = sb.step(a)
        if done.any():
            i = int(np.nonzero(done)[0][0]); seen = True
            assert "terminal_observation" in infos[i] and "episode" in infos[i] and infos[i]["episode"]["l"] <= 4
    assert seen
    direct = UR3eVecEnv("gymnasium_env/imitation_direct-v0", 4)
    o, _ = direct.reset()
    o, r, te, tr, _ = direct.step(torch.zeros(4, 7, device="cuda"))
    assert o.shape == (4, 13) and (r == -1).all() and not te.any()


def test_controller_entry_points_track_targets_via_query():
    """move_j on ur3e_raw.xml and move_l (pid_task_ctrl) on ur3e_2f85.xml converge to their targets (move_l's tcp read through a
    kinematics query)."""
    tgt = np.tile(np.array([0.3, -0.4, 0.5, -0.2, 0.1, 0.2, 0.0]), (3000, 1))
    q, v, _ = controller.move_j.run(tgt, n_envs=4, xml="ur3e_raw.xml", dtype=torch.float64, record_every=3000)
    err = (q[-1, 0] - torch.tensor(tgt[0, :6], device="cuda")).abs()            # 0.3 s of PD without gravity compensation
    assert torch.isfinite(q).all() and err.max() < 0.25 and err.norm() < 0.5 * float(np.linalg.norm(tgt[0, :6]))
    tcp = np.array([0.29799994, 0.13349916, 0.1682003])
    tl = np.tile(np.hstack([tcp + [0.03, 0.02, 0.03], presets.TOOL_ROTVEC, 0.0]), (1500, 1))
    q, v, b = controller.move_l.run(tl, n_envs=4, record_every=1500)
    tcp_pos = b.query([("site", "tcp")])()[0][0, 0].cpu().numpy()
    assert np.abs(tcp_pos - tl[0, :3]).max() < 0.02
    assert controller.task_space.pid_task_ctrl is controller.move_l.run


def test_device_built_per_env_trajectories_drive_move_l_via_query():
    """build_traj on the device -> [T, N, 7] per-environment waypoint streams -> the batched move_l loop, no host round trip."""
    tcp = torch.tensor([0.29799994, 0.13349916, 0.1682003], device="cuda", dtype=torch.float64)
    rot = torch.tensor(presets.TOOL_ROTVEC, device="cuda", dtype=torch.float64)
    off = torch.tensor([[0.03, 0.02, 0.03], [-0.02, 0.03, 0.02], [0.0, -0.03, 0.04], [0.02, 0.0, -0.01]], device="cuda", dtype=torch.float64)
    start = torch.cat([tcp.expand(4, 3), rot.expand(4, 3), torch.zeros(4, 1, device="cuda", dtype=torch.float64)], dim=1)
    stop = start.clone(); stop[:, :3] += off
    traj = controller.build_traj.build_traj_l_point_custom(start, stop, hold=100)                      # [1500, 4, 7] on the GPU
    assert traj.is_cuda and traj.shape == (1500, 4, 7)
    traj = torch.cat([traj, traj[-1:].expand(1000, 4, 7)])                                              # settle on the last waypoint
    q, v, b = controller.move_l.run(traj, n_envs=4, record_every=2500)
    tcp_pos = b.query([("site", "tcp")])()[0][:, 0].cpu().numpy()
    for e in range(4):
        assert np.abs(tcp_pos[e] - stop[e, :3].cpu().numpy()).max() < 0.02


def test_two_tier_stepping_f32():
    """float32 main.xml batches step with the lite size class and hand environments that exceed its caps (built-in: 8 contacts
    / 40 rows; lowered to 4 contacts here so that the fixture's grasp, 5-6 contacts, overflows) to the full class inside the
    same step call.  The result must equal full-only
    stepping, and the grasp episode of the v0 fixture must stay within the float32 drift bound of the reference trajectory."""
    g = np.load(GOLD + "/env_v0.npz")
    n = 64
    mk = lambda **kw: UR3eVecEnv(IDS["v0"], n, dtype=torch.float32, auto_reset=False, reset_noise=lib.NOISE_NONE, **kw)
    two, one = mk(lite_max_contacts=4), mk(single_tier=1)   # lite cap lowered to 4 contacts: any pad contact overflows
    qp = torch.tensor(np.tile(g["qpos0"], (n, 1)), device="cuda", dtype=torch.float32); qv = torch.tensor(np.tile(g["qvel0"], (n, 1)), device="cuda", dtype=torch.float32)
    for e in (two, one):
        e.reset(); e.set_state(qp, qv)
    handed_over, worst, worst_pair = 0, 0.0, 0.0
    T = 220
    for k in range(T):
        a = torch.tensor(np.tile(g["actions"][k], (n, 1)), device="cuda", dtype=torch.float32)
        # only an eighth of the batch grasps (below the quarter at which the full class takes over the whole batch): mixed
        # populations exercise the device-side overflow list
        a[n // 8:, 3] = 0.0
        o2, r2, *_ = two.step(a); o1, r1, *_ = one.step(a)
        torch.cuda.synchronize()
        handed_over = max(handed_over, two.batch.kernel_info()["lite"]["last_overflow_envs"])
        worst_pair = max(worst_pair, float((o2 - o1).abs().max()))
        worst = max(worst, float(np.abs(o2[0, :9].double().cpu().numpy() - g["obs"][k][:9]).max()))
    info = two.batch.kernel_info()["lite"]
    assert info["lite_tier_steps"] == T and info["full_only_steps"] == 0
    assert 0 < handed_over <= n // 8            # only the grasping environments ever overflow the lite caps
    assert one.batch.kernel_info()["lite"]["full_only_steps"] == T
    assert worst_pair < 1e-5, worst_pair         # two-tier == single-tier
    assert worst < 5e-3, worst                   # float32 drift vs the float64 reference episode (tcp / mug / ghost positions)
    assert int(o2[0, 9].item()) == int(g["obs"][T - 1][9])    # same grasp count as the reference at the end


def test_f32_production_build_per_step_drift_through_contacts():
    """float32 production kernels (exact-fit lite tier + full tier) against the float64 build on the fixture's scripted
    approach-grasp-lift episode, re-seeded from the float64 state before every step: stated per-step bound on the observation
    (positions 2e-4 m, velocities 2e-2 m/s or rad/s: one step of contact switching at float32 solver tolerances)."""
    g = np.load(GOLD + "/env_v2.npz")
    kw = dict(auto_reset=False, reset_noise=lib.NOISE_NONE)
    e64 = UR3eVecEnv(IDS["v2"], 2, dtype=torch.float64, **kw); e32 = UR3eVecEnv(IDS["v2"], 2, dtype=torch.float32, **kw)
    e64.reset(); e32.reset()
    e64.set_state(torch.tensor(np.tile(g["qpos0"], (2, 1)), device="cuda"), torch.tensor(np.tile(g["qvel0"], (2, 1)), device="cuda"))
    worst_p = worst_v = 0.0; max_ncon = 0.0
    for k in range(len(g["reward"])):
        qp, qv, ws = e64.get_state()
        e32.batch.set_state(qp.float(), qv.float(), ws.float())
        # set_state refreshes the stale-kinematics cache from the new state on both sides, so both controllers read the same pose
        e64.batch.set_state(qp, qv, ws)
        a = torch.tensor(np.tile(g["actions"][k], (2, 1)), device="cuda")
        o64, r64, t64, _, _ = e64.step(a); o32, r32, t32, _, _ = e32.step(a.float())
        d = (o32.double() - o64).abs()[0].cpu().numpy()
        worst_p = max(worst_p, d[:15].max(), d[21:27].max() if d.shape[0] > 27 else d[21:24].max())
        worst_v = max(worst_v, d[15:21].max())
        assert bool(t32[0]) == bool(t64[0])
        st = e32.episode_stats(reset=True)
        max_ncon = max(max_ncon, st["ncon_sum"] / st["substeps"])
    assert max_ncon >= 6, max_ncon                # beyond the four mug-table contacts: the pads do press on the mug in this episode
    assert worst_p < 2e-4 and worst_v < 2e-2, (worst_p, worst_v)


def test_batched_demo_collection_matches_oracle_loop(tmp_path):
    """collect_demos.py:86-189 batched: every demonstration's obs / acts equal what the reference's per-step loop
    (pid_task_ctrl -> d.ctrl -> mj_step -> get_obs) gives on the oracle for the same trajectory (float64 build, 1e-4), in both
    action modes; the pickle keeps the reference's list-of-Trajectory layout."""
    from oracle import envs as OE
    from ur3e_b200 import collect_demos as CD
    for mode in ("indirect", "direct"):
        d = CD.collect_expert_demonstrations(3, action_mode=mode, reset_mode="stochastic", noise_mag="low", down_sample=4, seed=5, dtype=torch.float64)
        T = d["traj"].shape[0]
        K = (T + 3) // 4
        assert d["obs"].shape == (3, K + 1, 24) and d["acts"].shape == (3, K, 4 if mode == "indirect" else 7)
        obs0 = d["obs"][:, 0].cpu().numpy()
        assert obs0[:, 4].std() > 0                                              # stochastic reset: different mug positions
        e = 1
        env = OE.OracleEnv(asset("main.xml"), "indirect")
        env.reset((obs0[e, 3] - 0.29799994, obs0[e, 4] - 0.13349916))
        traj = d["traj"][:, e].cpu().numpy()
        worst = 0.0
        for t in range(600):                                                     # approach and descent of demonstration 1
            u = env.d.pid_task_ctrl(env.tcp, traj[t], OE.GAINS_MUG)
            env.d.ctrl[:] = u; env.d.step(1)
            if t % 4 == 0:
                k = t // 4
                worst = max(worst, rel(d["obs"][e, k + 1].cpu().numpy(), env.obs()))
                want = np.hstack([traj[t, :3], u[-1]]) if mode == "indirect" else u
                worst = max(worst, rel(d["acts"][e, k].cpu().numpy(), want, 1e-2))
        assert worst < 1e-4, (mode, worst)
    trs = CD.to_trajectories(d)
    assert len(trs) == 3 and trs[0].obs.shape == (K + 1, 24) and len(trs[0]) == K and trs[0].terminal is True
    path = str(tmp_path / "demos" / "expert.pkl")
    assert CD.save_demos(trs, path) == 3 and CD.save_demos(trs, path, resume_collecting=True) == 6
    assert len(CD.load_demos(path)) == 6
