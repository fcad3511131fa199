"""ORACLE-side CPU timing leg (test/bench infrastructure): the float64 restatement of the reference's
`gymnasium_env/ur3e-v2` step (controller -> mj_step x2 -> obs/reward/done) run one environment per
process over the host cores, the way the reference runs SubprocVecEnv workers (train_rl.py:38-44).
No torch import here: workers are spawned cheaply."""
import multiprocessing as mp
import os
import time

import numpy as np


def _worker(args):
    xml, kind, steps, warmup, seed = args
    from oracle.envs import OracleEnv
    env = OracleEnv(xml, kind)
    rng = np.random.default_rng(seed)
    lo = np.array([0.29799994 - 0.25, 0.13349916 - 0.25, 0.0, 0.0]); hi = np.array([0.29799994 + 0.25, 0.13349916 + 0.25, 0.5, 1.0])
    env.reset((rng.uniform(0, 0.02), rng.uniform(-0.25, 0.2)))
    for _ in range(warmup):
        env.step(lo + (hi - lo) * rng.random(4))
    t0 = time.perf_counter(); n = 0
    for _ in range(steps):
        _, _, te, tr = env.step(lo + (hi - lo) * rng.random(4)); n += 1
        if te or tr or env.d.warn_bad:
            env.reset((rng.uniform(0, 0.02), rng.uniform(-0.25, 0.2)))
    return n, time.perf_counter() - t0


def run(xml, kind="v2", steps_per_proc=3000, procs=None, warmup=20):
    """Every process steps one environment `warmup` untimed env-steps, then `steps_per_proc` timed ones.  Returns
    (timed env-steps per second aggregated over processes, procs, total timed env-steps, slowest timed window in s, wall seconds)."""
    procs = procs or (os.cpu_count() or 1)
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(procs) as pool:
        res = pool.map(_worker, [(xml, kind, steps_per_proc, warmup, 1000 + i) for i in range(procs)])
    wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    return total / slowest, procs, total, slowest, wall


if __name__ == "__main__":
    import sys
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, here)
    print(run(os.path.join(here, "ur3e_b200", "assets", "main.xml"), steps_per_proc=int(sys.argv[1]) if len(sys.argv) > 1 else 1000))
