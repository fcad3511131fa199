"""Rollout timing (ur3e_batch_rollout) on the float32 main.xml batch, beside the live env-step it reuses.

    python tools/rollout_bench.py [--envs 65536] [--settle 1500] [--reps 10] [--out FILE]

The batch is query_bench.py's: the ur3e-v2 rollout of bench.py (U(action_space) actions, auto-reset, high reset noise), stepped
`--settle` untimed env-steps so that episode phases and contact states are mixed.  Then, with CUDA events after a warm-up:
  a  branch every environment once: m = n, T = 32 with obs, reward, terminated and truncated, against the next 32 live steps with
     the same actions (the same kernels on the same records: the ratio is the rollout's own overhead, the gather and the scratch)
  b  one predictive-sampling planner step on a second batch of 1024 environments (settled the same way): 64 branches each
     (m = 65 536), T = 32, reward + terminated; then the argmax over branches of the reward summed up to the first termination, and
     one live step with the winning first action
  c  the launch-bound regime: m = 256 of the first batch, T = 64
Every rollout of a case starts from the same records (rollouts do not write them); case a's live steps advance the batch between
repetitions.  The 35 MB of records stay in the 126 MB L2 in both arms.  Prints one JSON line with the GPU's name, power limit and
SM clock.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--envs", type=int, default=65536)
    p.add_argument("--settle", type=int, default=1500)
    p.add_argument("--reps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = p.parse_args()
    import torch
    import ur3e_b200._lib as lib
    from query_bench import gpu_info
    from ur3e_b200 import presets
    from ur3e_b200.batch import SimBatch
    from ur3e_b200.model import Model, asset
    if not torch.cuda.is_available():
        raise SystemExit("rollout_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    model = Model(asset("main.xml"))
    _, kw, _, _ = presets.ENV_SPECS["gymnasium_env/ur3e-v2"]
    cfg = presets.make_config(model, kw, auto_reset=1, reset_noise=lib.NOISE_HIGH)
    lo, hi = presets.action_bounds(model, "gymnasium_env/ur3e-v2")
    lo, hi = torch.tensor(lo, device=dev, dtype=torch.float32), torch.tensor(hi, device=dev, dtype=torch.float32)
    g = torch.Generator(device=dev); g.manual_seed(1234)

    def uniform(*shape):
        return (lo + (hi - lo) * torch.rand(*shape, 4, device=dev, generator=g)).contiguous()

    def settled(n):
        b = SimBatch(model, cfg, n, 0, torch.float32)
        acts = [uniform(n) for _ in range(16)]
        b.reset(seed=0)
        for k in range(args.settle):
            b.step(acts[k % 16])
        return b

    def ms(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        return e0.elapsed_time(e1)

    def median(v):
        v = sorted(v)
        return v[len(v) // 2]

    b = settled(args.envs)
    n, T = args.envs, 32
    # (a) branch every environment once against the next T live steps
    acts = uniform(T, n)

    def live():
        for t in range(T):
            b.step(acts[t], want_final_obs=False)
    roll_ms, live_ms = [], []
    for r in range(args.warmup + args.reps):
        x = ms(lambda: b.rollout(acts))
        y = ms(live)
        if r >= args.warmup:
            roll_ms.append(x); live_ms.append(y)
    l0 = b.launch_count; b.rollout(acts); torch.cuda.synchronize()
    res = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi(name, power.limit, clocks.sm, clocks.max.sm)": gpu_info(0),
           "envs": n, "settle_steps": args.settle, "reps": args.reps, "dtype": "float32",
           "a_branch_all": {"m": n, "T": T, "outputs": "obs+reward+terminated+truncated", "rollout_ms": median(roll_ms),
                            "live_32_steps_ms": median(live_ms), "ratio": median(roll_ms) / median(live_ms),
                            "launches_per_call": b.launch_count - l0}}

    # (b) predictive sampling: 1024 environments x 64 branches
    E, K = 1024, 64
    p_b = settled(E)
    ids = torch.arange(E, dtype=torch.int32, device=dev).repeat_interleave(K)
    cand = uniform(T, E * K)
    rows = torch.arange(E, device=dev)

    def rollout_b():
        return p_b.rollout(cand, env_ids=ids, obs=False, reward=True, terminated=True, truncated=False)

    def planner():
        r = rollout_b()
        alive = (torch.cumsum(r.terminated, 0) - r.terminated) == 0   # steps up to and including the first termination
        score = (r.reward * alive).sum(0).view(E, K)
        best = score.argmax(1)
        p_b.step(cand[0].view(E, K, 4)[rows, best].contiguous(), want_final_obs=False)
    call_ms, plan_ms = [], []
    for r in range(args.warmup + args.reps):
        x = ms(rollout_b)
        y = ms(planner)
        if r >= args.warmup:
            call_ms.append(x); plan_ms.append(y)
    c = median(call_ms)
    res["b_planner"] = {"envs": E, "branches": K, "m": E * K, "T": T, "outputs": "reward+terminated", "rollout_us": c * 1e3,
                        "us_per_rollout_step": c * 1e3 / T, "ns_per_env_step": c * 1e6 / (E * K * T), "planner_step_us": median(plan_ms) * 1e3}

    # (c) launch-bound: 256 rollouts of 64 steps
    m, T2 = 256, 64
    ids_c = torch.arange(m, dtype=torch.int32, device=dev)
    acts_c = uniform(T2, m)
    small = []
    for r in range(args.warmup + args.reps):
        x = ms(lambda: b.rollout(acts_c, env_ids=ids_c))
        if r >= args.warmup:
            small.append(x)
    l0 = b.launch_count; b.rollout(acts_c, env_ids=ids_c); torch.cuda.synchronize()
    res["c_small"] = {"m": m, "T": T2, "rollout_us": median(small) * 1e3, "us_per_rollout_step": median(small) * 1e3 / T2,
                      "launches_per_call": b.launch_count - l0}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
