"""Query timing (ur3e_batch_query, ur3e_batch_query_jac, ur3e_batch_forward, ur3e_batch_inverse, ur3e_batch_distance) on the float32 main.xml batch, beside one env-step for scale.

    python tools/query_bench.py [--envs 65536] [--settle 1500] [--launches 500] [--out FILE]

The batch is the ur3e-v2 rollout of bench.py (U(action_space) actions, auto-reset, high reset noise), stepped `--settle` untimed
env-steps so that episode phases and contact states are mixed.  The queries never write the record, so every case sees that same
state.  Then, with CUDA events around `--launches` back-to-back launches after a warm-up:
  kin_a  {site tcp, site handle_site, xbody ghost}, pos + vel      (what the v2 observation reads)
  kin_b  every body (both frames), geom and site: 77 objects, pos + mat + vel
  jac_a  tcp jacp + jacr, M and qfrc_bias   (Query.jac: the inputs of an operational-space controller)
  jac_b  M and qfrc_bias alone              (SimBatch.mass_matrix)
  fwd_a  contacts only: info, contact_geom and flags   (the contacts-only pass: kinematics and collision; what get_ncon and the
         collision predicates of ur3e_b200/utils.py run)
  fwd_b  everything, with ctrl: qacc, qfrc_constraint, info, the five contact outputs, flags and sensordata   (the full mj_forward)
  inv_a  qfrc_inverse at the stored state, qacc from a previous fwd_b   (SimBatch.inverse: mj_inverse, no solver iterations)
  inv_b  given states: a 16 x 4 096 rollout trajectory flattened to 65 536 states, discrete convention, qfrc_inverse + contact_force
         (inverse-dynamics labels along rollouts)
  dist_a the candidate pairs (SimBatch.distance(None): main.xml's 60) at the stored state, dist only, distmax = inf
         (the minimum clearance over everything the step can collide)
  dist_b the self and table pairs (robot geoms against each other and against the table) on the same 16 x 4 096 trajectory, given
         states, dist + fromto, distmax = inf   (a collision-avoidance cost along rollouts)
and one env-step over `--launches / 10` steps.  The byte floor counts what a call must move: the record fields it reads (qpos and
qvel for kin, jac and inv_a; the whole 544-byte record for fwd, which the kernel loads whole, and ctrl for fwd_b; the given qpos and
qvel for inv_b; qacc for inv; qpos for dist) and the outputs written.
The L2 is not flushed between launches: kin_a's working set (qpos + qvel of the records, 18 MB of outputs) stays in the 126 MB L2;
kin_b's 363 MB of outputs, jac_a's 142 MB and jac_b's 110 MB per call at 65 536 environments do not.  Prints one JSON line with the
GPU's name, power limit and SM clock.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True, timeout=10).stdout.strip()
    except Exception as e:   # the numbers still stand with the torch device name
        out = "nvidia-smi unavailable: %s" % e
    return out


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
    import ur3e_b200._lib as lib
    from ur3e_b200 import presets
    from ur3e_b200.batch import SimBatch
    from ur3e_b200.model import Model, asset
    if not torch.cuda.is_available():
        raise SystemExit("query_bench needs a CUDA device")
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

    small = b.query([("site", "tcp"), ("site", "handle_site"), ("xbody", "ghost")])
    objs = [(kind, i) for kind, n in (("body", model.nbody), ("xbody", model.nbody), ("geom", model.ngeom), ("site", model.nsite)) for i in range(n)]
    whole = b.query(objs)
    tcp = b.query([("site", "tcp")])
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

    n, nv, nq, nu, C = args.envs, model.nv, model.nq, model.nu, b.max_contacts
    state_bytes = 4 * (nq + nv)
    rec = int(b._L.ur3e_batch_state_bytes(b.ptr))
    res = {
        "gpu": torch.cuda.get_device_name(dev), "nvidia_smi(name, power.limit, clocks.sm, clocks.max.sm)": gpu_info(0),
        "envs": n, "settle_steps": args.settle, "launches": args.launches, "dtype": "float32", "max_contacts": C,
        "kin_a": {"objects": small.k, "outputs": "pos+vel", "us_per_call": timed(lambda: small(pos=True, vel=True), args.launches),
                  "bytes_floor": n * (state_bytes + 4 * small.k * 9)},
        "kin_b": {"objects": whole.k, "outputs": "pos+mat+vel", "us_per_call": timed(lambda: whole(pos=True, mat=True, vel=True), args.launches),
                  "bytes_floor": n * (state_bytes + 4 * whole.k * 18)},
        "jac_a": {"objects": "site tcp", "outputs": "jacp+jacr+M+qfrc_bias",
                  "us_per_call": timed(lambda: tcp.jac(jacp=True, jacr=True, M=True, qfrc_bias=True), args.launches),
                  "bytes_floor": n * (state_bytes + 4 * (2 * 3 * nv + nv * nv + nv))},
        "jac_b": {"objects": "none", "outputs": "M+qfrc_bias",
                  "us_per_call": timed(lambda: b.mass_matrix(M=True, qfrc_bias=True), args.launches),
                  "bytes_floor": n * (state_bytes + 4 * (nv * nv + nv))},
        "fwd_a": {"outputs": "info+contact_geom+flags",
                  "us_per_call": timed(lambda: b.forward(qacc=False, info=True, contact_geom=True, flags=True), args.launches),
                  "bytes_floor": n * (rec + 4 * (4 + 2 * C + 1))},
        "fwd_b": {"outputs": "all, with ctrl",
                  "us_per_call": timed(lambda: b.forward(ctrl=u, qacc=True, qfrc_constraint=True, info=True, contact_geom=True, contact_dist=True,
                                                         contact_pos=True, contact_frame=True, contact_force=True, flags=True, sensordata=True), args.launches),
                  "bytes_floor": n * (rec + 4 * nu + 4 * (2 * nv + 4 + C * (2 + 1 + 3 + 9 + 6) + 1 + lib.NSENSOR))},
    }
    # inverse dynamics: qacc of a previous forward (inv_a); a 16-step rollout of 4 096 branched environments, flattened (inv_b)
    fq = b.forward(ctrl=u, qacc=True).qacc.clone()
    res["inv_a"] = {"outputs": "qfrc_inverse, stored state", "us_per_call": timed(lambda: b.inverse(fq), args.launches),
                    "bytes_floor": n * (state_bytes + 4 * nv + 4 * nv)}
    T, mr = 16, n // 16
    ra = torch.stack([acts[k % 16][:mr] for k in range(T)]).contiguous()
    ids = torch.arange(mr, dtype=torch.int32, device=dev)
    r = b.rollout(ra, env_ids=ids, qpos=True, qvel=True, obs=False, reward=False, terminated=False, truncated=False)
    q0, v0, _ = b.get_state()
    tq = torch.cat([q0[:mr][None], r.qpos[:-1]]).reshape(-1, nq).contiguous()
    tv = torch.cat([v0[:mr][None], r.qvel[:-1]]).reshape(-1, nv).contiguous()
    ta = (torch.cat([v0[:mr][None], r.qvel]).diff(dim=0) / model.timestep).reshape(-1, nv).contiguous()
    res["inv_b"] = {"outputs": "qfrc_inverse+contact_force, given states (16 x %d trajectory), discrete" % mr,
                    "us_per_call": timed(lambda: b.inverse(ta, state=(tq, tv), discrete=True, qfrc_inverse=True, contact_force=True), args.launches),
                    "bytes_floor": T * mr * (4 * (nq + nv) + 4 * nv + 4 * (nv + 6 * C))}
    ib = b.inverse(ta, state=(tq, tv), discrete=True, qfrc_inverse=False, info=True).info
    res["inv_b"]["mean_ncon"] = ib[:, 0].double().mean().item(); res["inv_b"]["mean_nefc"] = ib[:, 1].double().mean().item()
    # geom distances: the candidate list at the stored state (dist_a); the self and table pairs along the trajectory (dist_b)
    da = b.distance()
    res["dist_a"] = {"pairs": da.k, "outputs": "dist, stored state", "us_per_call": timed(lambda: da(), args.launches),
                     "bytes_floor": n * (4 * nq + 4 * da.k)}
    name = lambda g: model.id2name(lib.OBJ_GEOM, g)
    pairs = [(a, c) for a, c in zip(da.geom1, da.geom2) if name(c) != "fish" and (name(a) == "table" or name(a) not in ("floor", "table"))]
    db = b.distance(pairs)
    res["dist_b"] = {"pairs": db.k, "outputs": "dist+fromto, given states (16 x %d trajectory)" % mr,
                     "us_per_call": timed(lambda: db(qpos=tq, fromto=True), args.launches), "bytes_floor": T * mr * (4 * nq + 4 * 7 * db.k)}
    res["dist_a"]["min_dist_mean"] = da()[0].min(dim=1).values.double().mean().item()
    res["mean_ncon"] = b.forward(qacc=False, info=True).info[:, 0].double().mean().item()
    res["mean_nefc"] = b.forward(qacc=True, info=True).info[:, 1].double().mean().item()
    it = iter(range(10 ** 9))
    res["env_step_us"] = timed(lambda: b.step(acts[next(it) % 16]), max(args.launches // 10, 10))
    for q in ("kin_a", "kin_b", "jac_a", "jac_b", "fwd_a", "fwd_b", "inv_a", "inv_b", "dist_a", "dist_b"):
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
