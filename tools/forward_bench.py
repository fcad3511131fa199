"""Forward-dynamics query timing (ur3e_batch_forward) on the float32 main.xml batch, beside one env-step for scale.

    python tools/forward_bench.py [--envs 65536] [--settle 1500] [--launches 500] [--out FILE]

The batch is the ur3e-v2 rollout of bench.py (U(action_space) actions, auto-reset, high reset noise), stepped `--settle` untimed
env-steps so that episode phases and contact states are mixed.  Then, with CUDA events around `--launches` back-to-back launches
after a warm-up:
  (a) contacts only: info, contact_geom and flags   (the contacts-only pass: kinematics and collision; what get_ncon and the
      collision predicates of ur3e_b200/utils.py run)
  (b) everything, with ctrl: qacc, qfrc_constraint, info, the five contact outputs, flags and sensordata   (the full mj_forward)
and one env-step over `--launches / 10` steps.  The byte floor counts what a call must move: the 544-byte record of every environment
read (the kernel loads it whole), ctrl read for (b), the outputs written.  Prints one JSON line with the GPU's name, power limit and
SM clock.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.query_bench import gpu_info   # noqa: E402


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--envs", type=int, default=65536)
    p.add_argument("--settle", type=int, default=1500)
    p.add_argument("--launches", type=int, default=500)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = p.parse_args()
    if args.launches < 500:
        p.error("--launches must be at least 500")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("forward_bench needs a CUDA device")
    import ur3e_b200._lib as lib
    from ur3e_b200 import presets
    from ur3e_b200.batch import SimBatch
    from ur3e_b200.model import Model, asset
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

    u = torch.zeros(args.envs, model.nu, device=dev)

    def timed(fn, count):
        for _ in range(args.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(count):
            fn()
        e1.record(); e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / count   # us per launch

    n, nv, nu, C = args.envs, model.nv, model.nu, b.max_contacts
    rec = int(b._L.ur3e_batch_state_bytes(b.ptr))
    res = {
        "gpu": torch.cuda.get_device_name(dev), "nvidia_smi(name, power.limit, clocks.sm, clocks.max.sm)": gpu_info(0),
        "envs": n, "settle_steps": args.settle, "launches": args.launches, "dtype": "float32", "max_contacts": C,
        "query_a": {"outputs": "info+contact_geom+flags",
                    "us_per_call": timed(lambda: b.forward(qacc=False, info=True, contact_geom=True, flags=True), args.launches),
                    "bytes_floor": n * (rec + 4 * (4 + 2 * C + 1))},
        "query_b": {"outputs": "all, with ctrl",
                    "us_per_call": timed(lambda: b.forward(ctrl=u, qacc=True, qfrc_constraint=True, info=True, contact_geom=True, contact_dist=True,
                                                           contact_pos=True, contact_frame=True, contact_force=True, flags=True, sensordata=True), args.launches),
                    "bytes_floor": n * (rec + 4 * nu + 4 * (2 * nv + 4 + C * (2 + 1 + 3 + 9 + 6) + 1 + lib.NSENSOR))},
    }
    info = b.forward(qacc=False, info=True).info.double()
    res["mean_ncon"] = info[:, 0].mean().item()
    res["mean_nefc"] = b.forward(qacc=True, info=True).info[:, 1].double().mean().item()
    it = iter(range(10 ** 9))
    res["env_step_us"] = timed(lambda: b.step(acts[next(it) % 16]), max(args.launches // 10, 10))
    for q in ("query_a", "query_b"):
        r = res[q]
        r["GB_per_s"] = r["bytes_floor"] / (r["us_per_call"] * 1e-6) / 1e9
        r["fraction_of_env_step"] = r["us_per_call"] / res["env_step_us"]
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
