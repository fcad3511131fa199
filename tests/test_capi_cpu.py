"""CPU suite part 3: the C-ABI library loads without a GPU, exports every symbol of include/ur3e_b200.h, serves the model
arrays, refuses (loudly) to create a batch without a CUDA device; host-side sharding logic under gloo, world size 2."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import ur3e_b200._lib as lib
from oracle import oracle as O
from ur3e_b200 import dist as D
from ur3e_b200 import presets
from ur3e_b200.model import Model, asset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_header_symbol():
    L = lib.load()
    hdr = open(os.path.join(ROOT, "include", "ur3e_b200.h")).read()
    names = sorted(set(re.findall(r"\b(ur3e_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), n
    assert sorted(lib.EXPORTS) == names


def test_model_arrays_match_oracle_loader():
    for xml in ("ur3e_raw.xml", "ur3e_2f85.xml", "main.xml"):
        m = Model(asset(xml)); o = O.Model(asset(xml))
        assert (m.nq, m.nv, m.nu, m.nbody) == (o.nq, o.nv, o.nu, o.nbody)
        for f in ("body_mass", "jnt_range", "actuator_ctrlrange", "dof_invweight0", "body_invweight0", "eq_data", "geom_size"):
            assert np.allclose(np.asarray(m.array(f)).ravel(), np.asarray(o.arr(f)).ravel(), rtol=1e-12, atol=1e-14), (xml, f)
        assert m.opt.timestep == o.timestep
    m = Model(asset("main.xml"))
    assert m.body_id("fish") == 23 and m.site_id("tcp") >= 0 and m.id2name(lib.OBJ_BODY, 24) == "ghost"       # SURVEY App. A body order
    assert m.body_id("nope") == -1
    k = m.keyframe("down")
    assert np.allclose(k.qpos[14:17], [0.29799994, 0.13349916, 0.055111])
    with pytest.raises(KeyError):
        m.keyframe("missing")


def test_loader_errors_are_reported(tmp_path):
    with pytest.raises(ValueError, match="cannot open"):
        Model("/nonexistent/model.xml")
    bad = str(tmp_path / "_bad.xml")
    open(bad, "w").write("<mujoco><compiler angle='radian'/><worldbody><body><joint type='ball'/></body></worldbody></mujoco>")
    with pytest.raises(ValueError, match="not supported"):
        Model(bad)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    from ur3e_b200.batch import SimBatch
    m = Model(asset("main.xml"))
    cfg = presets.make_config(m, presets.ENV_SPECS["gymnasium_env/ur3e-v2"][1])
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        SimBatch(m, cfg, 4)
    L = lib.load()
    assert not L.ur3e_batch_create(m.ptr, C.byref(cfg), 4, 0, 0)
    assert b"no CUDA device" in L.ur3e_last_error()


def test_presets_match_reference_constants():
    m = Model(asset("main.xml"))
    lo, hi = presets.action_bounds(m, "gymnasium_env/ur3e-v2")
    x0, y0 = m.keyframe("down").qpos[14:16]                                   # ur3e_env2.py:57-59
    assert np.allclose(lo, [x0 - 0.25, y0 - 0.25, 0, 0]) and np.allclose(hi, [x0 + 0.25, y0 + 0.25, 0.5, 1])
    lo, hi = presets.action_bounds(m, "gymnasium_env/imitation_direct-v0")
    assert np.allclose(hi, [330, 330, 150, 54, 54, 54, 255]) and np.allclose(lo[:6], -hi[:6]) and lo[6] == 0
    for env_id, (xml, kw, _, _) in presets.ENV_SPECS.items():
        c = presets.make_config(m, kw)
        assert c.reset_key == 1 and c.frame_skip in (1, 2)
        assert round(1.0 / (m.opt.timestep * c.frame_skip)) in (500, 1000)    # metadata render_fps of the reference envs


def _gloo_worker(rank, world, port, total, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    a, b = D.shard(total, rank, world)
    stats = torch.zeros(16, dtype=torch.float64)
    stats[0] = b - a; stats[1] = float(sum(range(a, b)))
    D.all_reduce_stats(stats)
    if rank == 0:
        out.put((stats[0].item(), stats[1].item()))
    dist.destroy_process_group()


def test_sharding_and_stats_allreduce_gloo_world2():
    import torch.multiprocessing as mp
    total = 1001
    assert D.shard(total, 0, 2) == (0, 501) and D.shard(total, 1, 2) == (501, 1001)
    assert [D.shard(10, r, 4) for r in range(4)] == [(0, 3), (3, 6), (6, 8), (8, 10)]
    ctx = mp.get_context("spawn"); q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, 29731, total, q)) for r in range(2)]
    [p.start() for p in procs]
    n, s = q.get(timeout=120)
    [p.join(60) for p in procs]
    assert n == total and s == sum(range(total))
    d = D.summarize(torch.tensor([4.0, 10.0, 40.0, 1.0] + [0.0] * 12), lib.STAT_NAMES)
    assert len(lib.STAT_NAMES) == 16
    assert d["mean_return"] == 2.5 and d["mean_length"] == 10 and d["success_rate"] == 0.25
