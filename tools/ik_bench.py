"""Inverse-kinematics timing (ur3e_batch_ik) on the float32 main.xml batch, beside one env-step for scale.

    python tools/ik_bench.py [--envs 65536] [--settle 1500] [--launches 20] [--out FILE]

The batch is query_bench.py's: the ur3e-v2 rollout of bench.py (U(action_space) actions, auto-reset, high reset noise), stepped
`--settle` untimed env-steps.  Targets are the tcp poses of random in-limit arm configurations (U(-2.5, 2.5) rad per arm joint), from
the batch's own kinematics query after set_state; the settled state is then restored, so every solve starts from it.  With CUDA events
around `--launches` back-to-back calls after a warm-up:
  a  every environment, tcp position + orientation targets, started from the stored state (default options, tol 1e-5)
  b  the same targets, position only
  c  a 4 096-environment trajectory conversion: a straight tcp line of T = 100 waypoints (build_traj_l_point_custom) from each
     environment's stored tcp pose to the tcp pose of its stored arm configuration moved by U(-0.3, 0.3) rad per joint, T calls each
     seeded from the previous solution, with the rotvec -> quaternion conversion in torch: time per waypoint
For each case: success fraction (status 0), mean / max steps.  The float32 noise floor of err_norm: case a's targets solved from their
own configurations moved by U(-0.3, 0.3) rad per arm joint, once at the default tol (success fraction) and once with tol = 0 and
max_steps = 100 (quantiles of the err_norm reached, over the problems that converged at the default tol).  Prints one JSON line with
the GPU's name, power limit and SM clock.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.query_bench import gpu_info  # noqa: E402


def mat2quat(R):
    """[m, 4] unit quaternions (w, x, y, z) of [m, 3, 3] rotations."""
    import torch
    d = torch.stack([R[:, 0, 0], R[:, 1, 1], R[:, 2, 2]], dim=1)
    w = 0.5 * (1 + d.sum(1)).clamp_min(0).sqrt()
    x = 0.5 * (1 + d[:, 0] - d[:, 1] - d[:, 2]).clamp_min(0).sqrt() * torch.sign(R[:, 2, 1] - R[:, 1, 2])
    y = 0.5 * (1 - d[:, 0] + d[:, 1] - d[:, 2]).clamp_min(0).sqrt() * torch.sign(R[:, 0, 2] - R[:, 2, 0])
    z = 0.5 * (1 - d[:, 0] - d[:, 1] + d[:, 2]).clamp_min(0).sqrt() * torch.sign(R[:, 1, 0] - R[:, 0, 1])
    q = torch.stack([w, x, y, z], dim=1)
    return q / q.norm(dim=1, keepdim=True)


def rotvec2quat(rv):
    import torch
    ang = rv.norm(dim=1, keepdim=True)
    axis = torch.where(ang > 0, rv / ang.clamp_min(1e-30), torch.zeros_like(rv))
    return torch.cat([torch.cos(ang / 2), axis * torch.sin(ang / 2)], dim=1).contiguous()


def quat2rotvec(q):
    import torch
    q = torch.where(q[:, :1] < 0, -q, q)
    s = q[:, 1:].norm(dim=1, keepdim=True)
    ang = 2 * torch.atan2(s, q[:, :1])
    return torch.where(s > 0, q[:, 1:] * ang / s.clamp_min(1e-30), torch.zeros_like(q[:, 1:]))


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--envs", type=int, default=65536)
    p.add_argument("--traj-envs", type=int, default=4096)
    p.add_argument("--T", type=int, default=100)
    p.add_argument("--settle", type=int, default=1500)
    p.add_argument("--launches", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = p.parse_args()
    import torch
    import ur3e_b200._lib as lib
    from ur3e_b200 import presets
    from ur3e_b200.batch import SimBatch
    from ur3e_b200.controller import build_traj as BT
    from ur3e_b200.model import Model, asset
    if not torch.cuda.is_available():
        raise SystemExit("ik_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    model = Model(asset("main.xml"))
    _, kw, _, _ = presets.ENV_SPECS["gymnasium_env/ur3e-v2"]
    b = SimBatch(model, presets.make_config(model, kw, auto_reset=1, reset_noise=lib.NOISE_HIGH), args.envs, 0, torch.float32)
    lo, hi = presets.action_bounds(model, "gymnasium_env/ur3e-v2")
    lo, hi = torch.tensor(lo, device=dev, dtype=torch.float32), torch.tensor(hi, device=dev, dtype=torch.float32)
    g = torch.Generator(device=dev); g.manual_seed(1234)
    acts = [(lo + (hi - lo) * torch.rand(args.envs, 4, device=dev, generator=g)).contiguous() for _ in range(16)]
    b.reset(seed=0)
    for k in range(args.settle):
        b.step(acts[k % 16])
    torch.cuda.synchronize()

    n = args.envs
    saved = [x.clone() for x in b.get_state()]
    tcp = b.query([("site", "tcp")])
    qr = saved[0].clone(); qr[:, :6] = (torch.rand(n, 6, device=dev, generator=g) * 5 - 2.5)
    b.set_state(qr, torch.zeros_like(saved[1]))
    pos, mat, _ = tcp(pos=True, mat=True)
    tpos, tquat = pos[:, 0].clone(), mat2quat(mat[:, 0].double()).float().contiguous()
    b.set_state(*saved)
    pos0, mat0, _ = tcp(pos=True, mat=True)
    start_pose = torch.cat([pos0[:, 0], quat2rotvec(mat2quat(mat0[:, 0].double())).float()], dim=1)
    torch.cuda.synchronize()

    def timed(fn, count):
        for _ in range(args.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(count):
            fn()
        e1.record(); e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / count   # us per call

    ik = b.ik(("site", "tcp"))
    res = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi(name, power.limit, clocks.sm, clocks.max.sm)": gpu_info(0),
           "envs": n, "settle_steps": args.settle, "launches": args.launches, "dtype": "float32"}

    def stats(r):
        info = r.info.cpu()
        return {"success_fraction": float((info[:, 1] == 0).double().mean()), "mean_steps": float(info[:, 0].double().mean()),
                "max_steps": int(info[:, 0].max()), "status_counts": {int(s): int((info[:, 1] == s).sum()) for s in info[:, 1].unique()}}

    for name, desc, kw in (("a", "all envs, tcp pos + quat targets from the stored state", dict(target_pos=tpos, target_quat=tquat)),
                           ("b", "all envs, tcp pos targets from the stored state", dict(target_pos=tpos))):
        us = timed(lambda: ik(**kw), args.launches)
        res[name] = dict(case=desc, us_per_call=us, **stats(ik(**kw)))
    near = qr.clone(); near[:, :6] += torch.rand(n, 6, device=dev, generator=g) * 0.6 - 0.3
    r = ik(tpos, tquat, qpos=near)
    conv = r.info[:, 1] == 0
    res["near_starts"] = dict(case="all envs, tcp pos + quat targets from their own configurations moved by up to 0.3 rad", **stats(r))
    floor = ik(tpos, tquat, qpos=near, tol=0.0).err_norm.double()[conv]
    res["f32_err_norm_floor(tol=0, max_steps=100)"] = {k: float(torch.quantile(floor, v)) for k, v in (("p50", 0.5), ("p90", 0.9), ("p99", 0.99), ("max", 1.0))}

    m, T = args.traj_envs, args.T
    qn = saved[0].clone(); qn[:, :6] += torch.rand(n, 6, device=dev, generator=g) * 0.6 - 0.3
    b.set_state(qn, torch.zeros_like(saved[1]))
    pos, mat, _ = tcp(pos=True, mat=True)
    stop = torch.cat([pos[:m, 0], quat2rotvec(mat2quat(mat[:m, 0].double())).float()], dim=1)
    b.set_state(*saved)
    traj = torch.cat([BT.build_traj_l_point_custom(start_pose[:m].double().cpu(), stop.double().cpu(), hold=1, num_points=T).to(dev, torch.float32),
                      torch.zeros(T, m, 1, device=dev)], dim=2)   # [T, m, 7]: pos, rotvec, grip
    ids = torch.arange(m, dtype=torch.int32, device=dev)
    out = {}

    def convert():
        r = ik(traj[0, :, :3].contiguous(), rotvec2quat(traj[0, :, 3:6]), env_ids=ids)
        q = r.qpos.clone()
        for t in range(1, T):
            r = ik(traj[t, :, :3].contiguous(), rotvec2quat(traj[t, :, 3:6]), qpos=q)
            q.copy_(r.qpos)
        out["r"] = r

    us = timed(convert, max(args.launches // 10, 2))
    res["c"] = dict(case="%d envs, T=%d trajectory conversion, seeded from the previous waypoint" % (m, T), us_per_waypoint=us / T,
                    us_per_trajectory=us, last_waypoint=stats(out["r"]))
    it = iter(range(10 ** 9))
    res["env_step_us"] = timed(lambda: b.step(acts[next(it) % 16]), 20)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
