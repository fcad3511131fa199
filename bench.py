#!/usr/bin/env python3
"""Headline benchmark: env-steps/s of the fused UR3e+2F85(+mug) step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload rollout|reach|mug] [--envs-per-gpu E] [--dtype f32|f64]
    python bench.py --impl reference ...      # the CPU arm: oracle port of the reference step on all host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's obs / reward / terminated / truncated as DIR/*.npy

One "step" = one Env.step for every environment on every rank.  Prints ONE JSON line.
Workloads (BASELINE.json configs):
  rollout = config 3 (gymnasium_env/ur3e-v2 semantics on main.xml, U(action_space) actions, auto-reset, 65536 envs per GPU), the
            configuration the 1e8 env-steps/s target is quoted on.  Measured in STEADY STATE: `--settle` (default 3000) untimed
            env-steps come first, so that every environment has been through truncation (2500 steps) + in-kernel auto-reset and
            the batch holds episodes at every phase; then W warm-up steps, then the K timed steps.
  mug     = config 4 (main.xml pick-and-lift through the ur3e-v2 wrapper, 16384 envs): the reference's scripted expert
            (controller/move_l_mug.py:36-41 + build_traj.py:28-59 build_traj_l_pick_place: approach, close, lift 0.15 m, carry
            to the ghost, release), per-environment targets; the approach is untimed, the timed steps are the grasp / lift /
            carry phase (contact_rich_frac = timed env-steps that ended with a pad-mug contact).
  reach   = config 2 (ur3e_2f85.xml, pid_task_ctrl every mj_step, 4096 envs, target re-drawn every 500 steps).
The default (rollout) line also carries a `workloads` block with short device-timed runs of mug and reach.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (UR3e+2F85, physics+controller)"
UNIT = "env-steps/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="rollout", choices=["rollout", "reach", "mug"])
    p.add_argument("--envs-per-gpu", type=int, default=0)
    p.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    p.add_argument("--settle", type=int, default=-1, help="untimed env-steps before the warm-up (-1 = the workload's default: rollout 3000, mug 1500, reach 1000)")
    p.add_argument("--cpu-steps", type=int, default=0, help="env-steps per CPU worker for the cpu_baseline sample (0 = auto)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-extra", action="store_true", help="skip the `workloads` block (mug / reach) of the default line")
    p.add_argument("--solver-iters", type=int, default=0, help="Newton iteration cap (0 = library default for the dtype)")
    p.add_argument("--no-l2-flush", action="store_true", help="profiling aid: skip the L2 flush between timed steps")
    p.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (rank 0's environments) as DIR/<name>.npy, "
                                                         "in the run's float dtype; inputs are seeded, so two builds can be compared output for output")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.warmup < 0:
        p.error("--warmup must not be negative")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    return a


WORKLOADS = {
    "rollout": dict(envs=65536, settle=3000, desc="config 3: gymnasium_env/ur3e-v2 rollout collection on main.xml, U(action_space) actions, auto-reset, frame_skip 2, dt 1 ms, steady state (episode phases staggered over the 2500-step horizon)"),
    "reach": dict(envs=4096, settle=1000, desc="config 2: ur3e_2f85.xml task-space reach, pid_task_ctrl every mj_step, target re-drawn every 500 steps, contact-free, frame_skip 1, dt 1 ms"),
    "mug": dict(envs=16384, settle=1500, desc="config 4: main.xml scripted pick-and-lift (move_l_mug.py / build_traj_l_pick_place targets; per-environment start delay, pick jitter, lift height) through the ur3e-v2 wrapper, frame_skip 2; approach untimed, timed region = grasp / lift / carry with gripper-mug contacts"),
}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, threading.Event(), []

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


def cpu_leg(workload, steps_per_proc, procs=None, warmup=20):
    """Oracle port of the reference step on the host cores: `warmup` untimed, then `steps_per_proc` timed env-steps per core."""
    from oracle import cpu_bench
    xml = os.path.join(ROOT, "ur3e_b200", "assets", "main.xml")
    # all three workloads' CPU legs run the v2 env step on main.xml, the reference's training env (train_rl.py:38-44), from reset
    # through truncation / auto-reset like the GPU arm's steady state; the reach workload (no mug) is cheaper per step, so this
    # is a conservative (slower) CPU number only for `reach`.
    return cpu_bench.run(xml, "v2", steps_per_proc, procs, warmup)


def flops_per_env_step(model_name, frame_skip, nefc, ncon, it):
    """SURVEY 8(d) algorithmic FLOP formula (FMA = 2) with measured mean nefc / ncon / Newton iterations."""
    C = dict(A=dict(nb=7, nv=6, nM=21, S2=91, grip=0), B=dict(nb=20, nv=14, nM=81, S2=543, grip=1), C=dict(nb=21, nv=20, nM=102, S2=634, grip=1))[model_name]
    nb, nv, nM, S2 = C["nb"], C["nv"], C["nM"], C["S2"]
    nbb, nbp = (4, 5) if model_name == "C" else (0, 0)
    f = 190 * nb + 100 * nb + 20 * nv + 10 * nb + 40 * nv + 11 * nM + 2 * S2 + 190 * nb + 40 * nv + 10 * nv + 4 * nM
    f += 1500 * nbb + 100 * nbp + 1820 * C["grip"] + 800 * ncon + nefc * (4 * nM + 2 * nv) + it * nefc * 4 * nv + 2 * S2 + 4 * nM + 4 * nv
    return frame_skip * f + 600 + 300


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  The reference runs on the mujoco wheel and meshes that
    this project does not ship (SURVEY F3/F4; probe log profiles/r2_mujoco_probe.log), so this is the oracle port (kind 'port'),
    one environment per host core.  Every core takes --warmup untimed env-steps, then --steps timed ones; one step = one env-step
    of every core's environment, timed by the slowest core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    value, procs, total, slowest, wall = cpu_leg(args.workload, args.steps, cores, warmup=args.warmup)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": slowest * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "impl": "reference", "config": {"workload": WORKLOADS[args.workload]["desc"], "timed_env_steps": total,
                                            "note": "one step here = one env-step of each of the %d CPU envs (one per host core); value aggregates them" % procs},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port",
                             "sample": "%d processes x %d timed ur3e-v2 env-steps after %d untimed (float64 oracle restatement of the reference step)" % (procs, args.steps, args.warmup)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


class Workload:
    """One benchmark configuration: the batch, its synthetic action stream (resident in HBM before the timed region) and the
    number of untimed steps that bring the batch to the state distribution being measured."""
    NBUF = 16

    def __init__(self, name, args, rank, local, n=None):
        import torch
        import ur3e_b200._lib as lib
        from ur3e_b200 import presets
        from ur3e_b200.batch import SimBatch
        from ur3e_b200.model import Model, asset
        self.name, self.torch = name, torch
        self.dev = dev = torch.device("cuda", local)
        self.dtype = dtype = torch.float32 if args.dtype == "f32" else torch.float64
        self.n = n = n or WORKLOADS[name]["envs"]
        self.settle = WORKLOADS[name]["settle"]
        if name == "reach":
            self.model = Model(asset("ur3e_2f85.xml")); self.mname = "B"
            self.cfg = presets.make_config(self.model, dict(ctrl_mode=lib.CTRL_PID_TASK, obs_kind=lib.OBS_STATE, obs_dim=28, act_dim=7, frame_skip=1, gains=presets.GAINS_L_TASK,
                                                            reset_key="down"), env_id_base=rank * n)
        else:
            self.model = Model(asset("main.xml")); self.mname = "C"
            _, kw, _, _ = presets.ENV_SPECS["gymnasium_env/ur3e-v2"]
            # mug: the reference script resets deterministically (move_l_mug.py:34 reset_with_mug(..., "deterministic", "down")); its open-loop
            # expert does not survive the env's reset noise.  Diversity between environments comes from per-environment script
            # delays, pick jitter and lift heights instead (see _mug_script_setup).
            self.cfg = presets.make_config(self.model, kw, auto_reset=1, env_id_base=rank * n, reset_noise=lib.NOISE_HIGH if name == "rollout" else lib.NOISE_NONE,
                                           solver_iterations=args.solver_iters)
        self.batch = SimBatch(self.model, self.cfg, n, local, dtype)
        self.obs0 = self.batch.reset(seed=0).clone()
        g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
        self.gen = g
        self.acts = None
        if name == "rollout":
            lo, hi = presets.action_bounds(self.model, "gymnasium_env/ur3e-v2")
            lo_t, hi_t = torch.tensor(lo, device=dev, dtype=dtype), torch.tensor(hi, device=dev, dtype=dtype)
            self.acts = [(lo_t + (hi_t - lo_t) * torch.rand(n, 4, device=dev, dtype=dtype, generator=g)).contiguous() for _ in range(self.NBUF)]
            self.period = 1            # i.i.d. per step (= action_space.sample() as in init_gym.py:35)
            self.stagger = int(self.cfg.max_steps)
            self.env_phase = torch.randint(0, self.stagger, (n,), generator=g, device=dev)
        elif name == "reach":
            tcp = torch.tensor([0.29799994, 0.13349916, 0.1682003], device=dev, dtype=dtype)   # tcp at keyframe 'down' (assets/main.xml:415)
            self.acts = []
            for _ in range(self.NBUF):
                a = torch.zeros(n, 7, device=dev, dtype=dtype)
                a[:, :3] = tcp + (torch.rand(n, 3, device=dev, dtype=dtype, generator=g) - 0.5) * 0.2
                a[:, 3:6] = torch.tensor(presets.TOOL_ROTVEC, device=dev, dtype=dtype)
                self.acts.append(a.contiguous())
            self.period = 500          # SURVEY 8d config 2: target re-drawn every 500 steps
        else:
            self._mug_script_setup()

    # ---- mug: the reference's scripted expert, per environment (move_l_mug.py:36-41, build_traj.py:28-59, 187-229)
    HOLD, NPTS = 60, 15                # hold 120 mj_steps per waypoint = 60 env-steps at frame_skip 2; 15 waypoints per segment
    MAX_DELAY = 300
    def _mug_script_setup(self):
        t = self.torch
        o = self.batch.obs
        n, kw = self.n, dict(device=self.dev, dtype=self.dtype)
        jit = (t.rand(n, 2, generator=self.gen, **kw) - 0.5) * 0.003                                      # pick jitter +-1.5 mm in x, y
        lift = 0.10 + 0.08 * t.rand(n, generator=self.gen, **kw)                                           # lift height 0.10 .. 0.18 m (the reference: 0.15)
        start = t.cat([o[:, 0:3], t.zeros(n, 1, **kw)], 1)                                                 # tcp at reset, gripper open
        pick = t.cat([o[:, 3:6], t.full((n, 1), 0.5, **kw)], 1); pick[:, 0:2] += jit                       # the mug's centre, gripper half closed
        up = pick.clone(); up[:, 2] += lift; up[:, 3] = 1.0                                                # lift, gripper closed
        place = t.cat([o[:, 6:9], t.ones(n, 1, **kw)], 1); place[:, 2] += 0.025
        drop = place.clone(); drop[:, 3] = 0.0
        self.way = t.stack([start, pick, up, place, drop])                                                 # [5, n, 4]
        self.delay = t.randint(0, self.MAX_DELAY, (n,), generator=self.gen, device=self.dev)               # every environment starts its script a little later
        self.script_len = 4 * self.HOLD * self.NPTS
        self.env_idx = t.arange(n, device=self.dev)

    def action(self, k):
        if self.acts is not None:
            return self.acts[(k // self.period) % self.NBUF]
        t = self.torch
        ke = (k % (self.script_len + self.MAX_DELAY) - self.delay).clamp(0, self.script_len - 1)
        seg = ke // (self.HOLD * self.NPTS)
        frac = (((ke % (self.HOLD * self.NPTS)) // self.HOLD + 1).to(self.dtype) / self.NPTS).unsqueeze(1)
        a, b = self.way[seg, self.env_idx], self.way[seg + 1, self.env_idx]
        return (a + (b - a) * frac).contiguous()

    def wrap(self, k):
        """mug: the script (plus the largest delay) is over -- start the next pick-and-place from a reset"""
        if self.acts is None and k > 0 and k % (self.script_len + self.MAX_DELAY) == 0:
            self.batch.reset(seed=k); self._mug_script_setup()

    def step(self, k):
        self.wrap(k)
        if self.name == "rollout" and k < self.stagger:
            # steady state of a long collection run: episode phases are spread over the 2500-step horizon (here by resetting 1/2500 of
            # the batch at each of the first 2500 settle steps), so that every step sees its share of truncations + auto-resets
            self.batch.reset(seed=1000 + k, mask=(self.env_phase == k))
        self.batch.step(self.action(k), want_final_obs=False)


def measure(w, steps, warmup, settle, flush, world, dist, sampler=None):
    """settle + warmup untimed steps, then `steps` timed ones: CUDA events on the launching stream around each step (the L2 flush
    sits outside the pairs), barrier + synchronize on both sides, max over ranks."""
    torch = w.torch
    b = w.batch
    k = 0
    for _ in range(settle + warmup):
        w.step(k); k += 1
    b.stats(reset=True)
    state0 = b.get_state() if w.name == "mug" else None
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.start()
    launches0 = b.launch_count
    b.kernel_timing(True)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    rec = []
    for i in range(steps):
        if flush is not None:
            flush.zero_()                   # L2 flush between timed iterations (outside the per-step event pair)
        w.wrap(k)
        a = w.action(k)
        if w.acts is None and len(rec) < 64:
            rec.append(a)
        ev[i][0].record()
        b.step(a, want_final_obs=False)
        ev[i][1].record()
        k += 1
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.stop_flag.set(); sampler.join(2)
    step_ms = [s.elapsed_time(e) for s, e in ev]
    kt = b.kernel_times(); b.kernel_timing(False)
    total_ms = float(sum(step_ms))
    t = torch.tensor([total_ms], device=w.dev, dtype=torch.float64)
    st = b.stats_dict(reset=True)
    if world > 1:
        import ur3e_b200._lib as lib
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sv = torch.tensor([st[kk] for kk in lib.STAT_NAMES], device=w.dev, dtype=torch.float64)
        dist.all_reduce(sv, op=dist.ReduceOp.SUM)      # the optional NCCL episode-stat all-reduce (SURVEY 8e), off the step path
        st = {kk: float(sv[i].item()) for i, kk in enumerate(lib.STAT_NAMES)}
    total_ms = float(t.item())
    sub = max(st["substeps"], 1.0)
    res = dict(total_ms=total_ms, value=w.n * world * steps / (total_ms * 1e-3), ms_per_step=total_ms / steps, launches=b.launch_count - launches0,
               stats=st, mean_nefc=st["nefc_sum"] / sub, mean_ncon=st["ncon_sum"] / sub, mean_it=st["solver_iter_sum"] / sub,
               contact_rich_frac=st["pad_contact_steps"] / max(st["steps"], 1.0), kernel_times=kt, k_end=k, state0=state0, rec=rec,
               kernel_ms=(kt["lite"][0] + kt["full"][0]) / steps, kernel_ms_lite=kt["lite"][0] / steps, kernel_ms_full=kt["full"][0] / steps,
               kernel_ms_side=kt["side"][0] / steps)
    return res


def rooflines(w, res, peaks):
    """FP32-pipe roofline (the bound SURVEY 8d names for this path) and the HBM one, both on the step kernels' own duration."""
    torch = w.torch
    esz = 4 if w.dtype == torch.float32 else 8
    ki = w.batch.kernel_info()
    fs = w.cfg.frame_skip
    bytes_per_env = 2 * ki["state_bytes"] + w.batch.act_dim * esz + w.batch.obs_dim * esz + esz + 2
    flops_env = flops_per_env_step(w.mname, fs, res["mean_nefc"], res["mean_ncon"], res["mean_it"])
    props = torch.cuda.get_device_properties(w.dev)
    sm_mhz = float(peaks.get("sm_max_mhz", 1965.0))
    fp32_peak = props.multi_processor_count * 128 * 2 * sm_mhz * 1e6 / 1e12
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    kms = max(res["kernel_ms"], 1e-9)
    r32 = {"bound": "fp32", "achieved": flops_env * w.n / (kms * 1e-3) / 1e12, "peak": fp32_peak, "unit": "TFLOP/s", "traffic": None,
           "kernel": "ur3e::step_kernel (the size-class launches on the step's critical path: lite tier + grasp / generic tier; the generic tier's side-stream launch overlaps them)", "kernel_ms": kms, "kernel_share_of_step": kms / res["ms_per_step"],
           "algorithmic_flops_per_env_step": flops_env, "units_per_launch": w.n, "mean_nefc": res["mean_nefc"], "mean_ncon": res["mean_ncon"], "mean_newton_iters": res["mean_it"],
           "peak_source": "SMs x 128 FP32 lanes x 2 x sm_max_mhz (%s)" % ("MEASURED_PEAKS.json" if "sm_max_mhz" in peaks else "fallback 1965 MHz")}
    r32["frac"] = r32["achieved"] / r32["peak"]
    traffic, cap = None, None
    try:   # dram__bytes_read + dram__bytes_write of the step kernels from the committed ncu capture of this same command (L2 flush on), per env-step
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        if w.name == tj.get("workload", "rollout") and w.dtype == torch.float32:
            traffic = (tj["dram_bytes_read"] + tj["dram_bytes_write"]) * w.n / tj["envs"]; cap = tj.get("capture")
    except Exception:
        pass
    rh = {"bound": "hbm", "achieved": bytes_per_env * w.n / (kms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s", "traffic": traffic, "traffic_capture": cap,
          "peak_source": peak_src, "algorithmic_bytes_per_env_step": bytes_per_env, "kernel_ms": kms}
    rh["frac"] = rh["achieved"] / rh["peak"]
    r32["traffic"] = traffic; r32["traffic_capture"] = cap
    return r32, rh, ki


DUMP_LIMIT = 64 * 10 ** 6       # bytes of all --dump-outputs files together, .npy headers included
NPY_HEADER = 256                # upper bound of np.save's header for these shapes


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """Write every [n, ...] array of `arrays` as out_dir/<name>.npy.  If they would exceed `limit` bytes together, the same fixed,
    seeded sample of rows (environments) is written from each, in ascending order, and env_index.npy holds the row numbers."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = len(next(iter(arrays.values())))
    row = sum(a.nbytes for a in arrays.values()) // n
    if n * row + NPY_HEADER * len(arrays) > limit:
        k = (limit - NPY_HEADER * (len(arrays) + 1)) // (row + 8)
        idx = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
        arrays = dict({name: a[idx] for name, a in arrays.items()}, env_index=idx.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: everything native libraries print while the job runs (NCCL's version banner comes out on
    # fd 1 at the first collective) is sent to stderr; the real stdout is restored just before the line is printed
    sys.stdout.flush()
    real_stdout = os.dup(1); os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    w = Workload(args.workload, args, rank, local, args.envs_per_gpu or None)
    n, dtype, batch = w.n, w.dtype, w.batch
    settle = args.settle if args.settle >= 0 else w.settle
    n_warm = max(args.warmup, 3)
    flush = None if args.no_l2_flush else torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    sampler = ClockSampler(local)
    res = measure(w, args.steps, n_warm, settle, flush, world, dist, sampler)
    value, total_ms = res["value"], res["total_ms"]
    if args.dump_outputs and rank == 0:
        # the batch-owned tensors SimBatch.step returns, as the last timed step left them; copied before the e2e leg steps the batch again
        last = (batch.obs, batch.reward, batch.terminated, batch.truncated)
        dump_outputs(args.dump_outputs, {name: t.to(dtype).cpu().numpy() for name, t in zip(("obs", "reward", "terminated", "truncated"), last)})

    # ---- e2e: the host-buffer C-ABI call, pinned host buffers, H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        ke = max(10, min(args.steps, 50))
        if w.acts is not None:
            hb = [torch.empty(n, batch.act_dim, dtype=dtype).pin_memory() for _ in range(4)]
            for i, h in enumerate(hb):
                h.copy_(w.acts[i % w.NBUF].cpu())
        else:
            # same phase as the device leg: back to the state the timed region started from, replaying its recorded actions
            ke = min(ke, len(res["rec"]))
            hb = [torch.empty(n, batch.act_dim, dtype=dtype).pin_memory() for _ in range(ke)]
            for h, a in zip(hb, res["rec"]):
                h.copy_(a.cpu())
            batch.set_state(*res["state0"])
        h_obs = torch.empty(n, batch.obs_dim, dtype=dtype).pin_memory(); h_rew = torch.empty(n, dtype=dtype).pin_memory()
        h_te = torch.empty(n, dtype=torch.uint8).pin_memory(); h_tr = torch.empty(n, dtype=torch.uint8).pin_memory()
        for k in range(3):
            batch.step_host(hb[k % len(hb)], h_obs, h_rew, h_te, h_tr)
        if w.acts is None:
            batch.set_state(*res["state0"])
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        batch.stats(reset=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(ke):
            batch.step_host(hb[k % len(hb)], h_obs, h_rew, h_te, h_tr)
        torch.cuda.synchronize()
        te = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        est = batch.stats_dict(reset=True)
        esz = 4 if dtype == torch.float32 else 8
        e2e = {"value": n * world * ke / float(te.item()), "unit": UNIT, "h2d_bytes_per_step": n * batch.act_dim * esz,
               "d2h_bytes_per_step": n * (batch.obs_dim * esz + esz + 2), "steps": ke,
               "mean_ncon": est["ncon_sum"] / max(est["substeps"], 1.0), "contact_rich_frac": est["pad_contact_steps"] / max(est["steps"], 1.0)}

    # ---- the other BASELINE configs, device-timed, short (default line only)
    extra = {}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    if args.workload == "rollout" and not args.no_extra and args.dtype == "f32" and not args.envs_per_gpu:
        for name in ("mug", "reach"):
            w2 = Workload(name, args, rank, local)
            k2 = max(20, min(args.steps, 200))
            r2 = measure(w2, k2, 3, w2.settle, flush, world, dist)
            if rank == 0:
                r32b, rhb, kib = rooflines(w2, r2, peaks)
                tiers = kib.get("lite", {})
                extra[name] = {"workload": WORKLOADS[name]["desc"], "value": r2["value"], "unit": UNIT, "ms_per_step": r2["ms_per_step"], "steps": k2, "settle": w2.settle,
                               "envs_per_gpu": w2.n, "frame_skip": w2.cfg.frame_skip, "mean_ncon": r2["mean_ncon"], "mean_nefc": r2["mean_nefc"],
                               "mean_newton_iters": r2["mean_it"], "contact_rich_frac": r2["contact_rich_frac"], "kernel_ms": r2["kernel_ms"],
                               "kernel_ms_lite_tier": r2["kernel_ms_lite"], "kernel_ms_full_tier": r2["kernel_ms_full"], "kernel_ms_side_stream": r2["kernel_ms_side"],
                               "full_tier_envs_last_step": tiers.get("last_overflow_envs"),
                               "fp32_frac": r32b["frac"], "fp32_tflops": r32b["achieved"], "hbm_frac": rhb["frac"], "episodes": r2["stats"]["episodes"],
                               "successes": r2["stats"]["successes"], "unstable_resets": r2["stats"]["unstable_resets"], "overflow_steps": r2["stats"]["overflow_steps"]}
            del w2
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    r32, rh, ki = rooflines(w, res, peaks)
    st = res["stats"]
    fs = w.cfg.frame_skip
    cpu = None
    if not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        per = args.cpu_steps or 80000
        rate, procs, total, _, wall = cpu_leg(args.workload, per, cores)
        cpu = {"value": rate, "unit": UNIT, "cores": procs, "kind": "port",
               "sample": "%d processes (one per host core) x %d ur3e-v2 env-steps of the float64 oracle restatement, resets included (%.1f s wall); MuJoCo 3.3.3 is not installable here" % (procs, per, wall)}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": n_warm,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload]["desc"], "envs_per_gpu": n, "total_envs": n * world, "frame_skip": fs, "substeps_per_s": value * fs,
                       "settle_steps": settle, "l2": "192 MiB buffer written between timed iterations (L2 flush), outside the per-step event pairs" if flush is not None else "no flush (profiling run)",
                       "parallelism": "independent env shards, one process per GPU, no step-path collective",
                       "kernel": ki, "episodes": st["episodes"], "truncations": st["truncations"], "successes": st["successes"], "term_toppled": st["term_toppled"],
                       "unstable_resets": st["unstable_resets"], "overflow_steps": st["overflow_steps"],
                       "mean_ncon": res["mean_ncon"], "mean_nefc": res["mean_nefc"], "contact_rich_frac": res["contact_rich_frac"],
                       "kernel_ms_lite_tier": res["kernel_ms_lite"], "kernel_ms_full_tier": res["kernel_ms_full"], "kernel_ms_side_stream": res["kernel_ms_side"]},
            "roofline": r32, "roofline_hbm": rh, "cpu_baseline": cpu, "e2e": e2e, "workloads": extra or None,
            "gpu_launches": res["launches"], "clocks": sampler.summary()}
    sys.stdout.flush(); os.dup2(real_stdout, 1)
    print(json.dumps(line)); sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
