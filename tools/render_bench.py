"""Offscreen-render timing (ur3e_batch_render) on the float32 main.xml batch, beside one env-step for scale.

    python tools/render_bench.py [--envs 65536] [--settle 1500] [--launches 100] [--out FILE]

The batch is query_bench.py's: the ur3e-v2 rollout of bench.py (U(action_space) actions, auto-reset, high reset noise), stepped
`--settle` untimed env-steps so that arm poses and mug positions are mixed.  Rendering never writes the record, so every case sees
that same state.  Then, with CUDA events around `--launches` back-to-back calls after a warm-up (each call is the pose pass and the
pixel pass), for the default geom list (every geom of main.xml):
  a  every environment, 64 x 64, world camera (UR3eEnv's default), rgb + depth + seg   (pixel-based RL)
  b  every environment, 64 x 64, wrist camera on site tcp, depth only
  c  one environment, 480 x 480, world camera, rgb   (UR3eEnv.render, video recording)
and one env-step over `--launches / 10` steps.  The byte floor is what a call must write: 3 B of rgb, 4 B of float32 depth and 4 B of
int32 seg per pixel asked for (the pose pass's reads are negligible beside it); at 65 536 x 64 x 64 with all three outputs that is
65 536 * 4 096 * 11 B = 2.95 GB.  Prints one JSON line with the GPU's name, power limit and SM clock.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.query_bench import gpu_info  # noqa: E402


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--envs", type=int, default=65536)
    p.add_argument("--settle", type=int, default=1500)
    p.add_argument("--launches", type=int, default=100)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = p.parse_args()
    import torch
    import ur3e_b200._lib as lib
    from ur3e_b200 import presets
    from ur3e_b200.batch import SimBatch
    from ur3e_b200.envs import DEFAULT_CAMERA_CONFIG
    from ur3e_b200.model import Model, asset
    if not torch.cuda.is_available():
        raise SystemExit("render_bench needs a CUDA device")
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

    def timed(fn, count):
        for _ in range(args.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(count):
            fn()
        e1.record(); e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / count   # us per call

    wrist = dict(pos=(0, 0, -0.1), xyaxes=(0, 1, 0, 1, 0, 0), site="tcp", fovy=70.0)
    one = torch.zeros(1, dtype=torch.int32, device=dev)
    cases = {
        "a": dict(desc="all envs, 64x64, world camera, rgb+depth+seg", r=b.renderer(64, 64, DEFAULT_CAMERA_CONFIG), ids=None, m=args.envs,
                  outs=dict(rgb=True, depth=True, seg=True), bpp=3 + 4 + 4),
        "b": dict(desc="all envs, 64x64, wrist camera on tcp, depth", r=b.renderer(64, 64, wrist), ids=None, m=args.envs,
                  outs=dict(rgb=False, depth=True, seg=False), bpp=4),
        "c": dict(desc="one env, 480x480, world camera, rgb", r=b.renderer(480, 480, DEFAULT_CAMERA_CONFIG), ids=one, m=1,
                  outs=dict(rgb=True, depth=False, seg=False), bpp=3),
    }
    res = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi(name, power.limit, clocks.sm, clocks.max.sm)": gpu_info(0),
           "envs": args.envs, "settle_steps": args.settle, "launches": args.launches, "dtype": "float32", "geoms": cases["a"]["r"].k}
    for name, c in cases.items():
        r, px = c["r"], c["r"].width * c["r"].height
        us = timed(lambda: r(c["ids"], **c["outs"]), args.launches)
        floor = c["m"] * px * c["bpp"]
        res[name] = {"case": c["desc"], "us_per_call": us, "Mpixel_per_s": c["m"] * px / us, "bytes_floor": floor, "GB_per_s": floor / (us * 1e-6) / 1e9}
    it = iter(range(10 ** 9))
    res["env_step_us"] = timed(lambda: b.step(acts[next(it) % 16]), max(args.launches // 10, 10))
    for name in cases:
        res[name]["fraction_of_env_step"] = res[name]["us_per_call"] / res["env_step_us"]
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
