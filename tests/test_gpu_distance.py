"""GPU suite for geom distances (ur3e_batch_distance, SimBatch.distance): the compiled sm_100a kernel against the host build and the
reference, the state sources, repeated and bad ids, untouched records and stats, identity with the forward query's contacts after
settling, float32 against float64, a side stream, and every rejected call."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as O
import ur3e_b200._lib as lib
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.model import Model
from tests import distance_reference as R
from tests.hostcheck import distance as HD

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "env_v2_pick.npz")


def _batch(assets, n, dtype):
    m = Model(assets + "/main.xml")
    return SimBatch(m, env_config(ctrl_mode=lib.CTRL_RAW, act_dim=m.nu, frame_skip=1, obs_kind=lib.OBS_V2, obs_dim=24), n, 0, dtype)


def _seeded(b, n):
    """[n, nq] float64 configurations: the golden's seeded states, cycled."""
    q = np.load(GOLD)["seed_qpos"]
    return q[np.arange(n) % len(q)]


def _set(b, qpos):
    b.set_state(torch.tensor(qpos, dtype=b.dtype, device=b.device), torch.zeros(b.n, b.model.nv, dtype=b.dtype, device=b.device))


def test_device_matches_host_and_reference(assets):
    """float64 device = the host build within 1e-12 at given states, for the candidate pairs (fromto where the closest points are
    unique); float32 within 1e-5 m of float64; the
    host build is itself pinned to the reference in test_distance_cpu.py, rechecked here on a few states."""
    n = 64
    q = _seeded(None, n)
    b = _batch(assets, n, torch.float64)
    d = b.distance()
    assert d.k == len(b.model.array("pair_geom1"))
    r = d(qpos=torch.tensor(q, dtype=torch.float64, device=b.device), fromto=True)
    dist, ft = r.dist.cpu().numpy(), r.fromto.cpu().numpy()
    xml = assets + "/main.xml"
    for e in range(0, n, 7):
        hd, hf = HD.distance(xml, d.geom1, d.geom2, q[e])
        assert np.abs(dist[e] - hd).max() <= 1e-12
        # fromto is the host build's, except where the closest points are not unique (parallel faces, a box face on the table):
        # there rounding may pick another closest pair, which must still be one
        same = np.abs(ft[e] - hf).max(axis=1) <= 1e-12
        gap = np.abs(np.linalg.norm(ft[e, :, 3:] - ft[e, :, :3], axis=1) - np.abs(dist[e]))
        assert (same | (gap <= 1e-12)).all()
        assert same.mean() >= 0.9
    om = O.Model(xml)
    for j in range(0, d.k, 5):
        ref, _, _ = R.pair(om, q[0], d.geom1[j], d.geom2[j])
        if ref is not None:
            assert abs(dist[0, j] - ref) <= 1e-9
    b32 = _batch(assets, n, torch.float32)
    d32 = b32.distance()
    r32 = d32(qpos=torch.tensor(q, dtype=torch.float32, device=b32.device), fromto=True)
    assert np.abs(r32.dist.double().cpu().numpy() - dist).max() <= 1e-5
    f32 = r32.fromto.double().cpu().numpy()
    same = np.abs(f32 - ft).max(axis=2) <= 1e-4
    gap = np.abs(np.linalg.norm(f32[..., 3:] - f32[..., :3], axis=2) - np.abs(r32.dist.double().cpu().numpy()))
    assert (same | (gap <= 1e-5)).all() and same.mean() >= 0.9   # another closest pair only where they are not unique


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_sources_ids_records_stream(assets, dtype):
    """The stored state, qpos = get_state()[0] and env_ids = arange(n) agree bit for bit; repeated ids repeat rows; a bad id gives NaN;
    the records and stats are unchanged; a side stream gives the same values."""
    n = 96
    b = _batch(assets, n, dtype)
    _set(b, _seeded(b, n))
    b.step(torch.zeros(n, b.act_dim, dtype=dtype, device=b.device))
    torch.cuda.synchronize()
    before = [x.clone() for x in b.get_state()]
    st0 = b.stats(reset=False).clone()
    d = b.distance()
    a = d(fromto=True)
    a = [x.clone() for x in a]
    qb = d(qpos=before[0].contiguous(), fromto=True)
    ids = torch.arange(n, dtype=torch.int32, device=b.device)
    ib = d(env_ids=ids, fromto=True)
    for x, y, z in zip(a, qb, ib):
        assert torch.equal(x, y) and torch.equal(x, z)
    rep = torch.tensor([5, 5, 0, n - 1, 5], dtype=torch.int32, device=b.device)
    rr = d(env_ids=rep, fromto=True)
    assert torch.equal(rr.dist, a[0][rep.long()]) and torch.equal(rr.fromto, a[1][rep.long()])
    bad = torch.tensor([3, -1, n, 7], dtype=torch.int32, device=b.device)
    rb = d(env_ids=bad, fromto=True)
    assert torch.isnan(rb.dist[1:3]).all() and torch.isnan(rb.fromto[1:3]).all()
    assert torch.equal(rb.dist[[0, 3]], a[0][[3, 7]])
    after = b.get_state()
    for x, y in zip(before, after):
        assert torch.equal(x, y)
    assert torch.equal(st0, b.stats(reset=False))
    s = torch.cuda.Stream(device=b.device)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        rs = d(dist=torch.empty(n, d.k, dtype=dtype, device=b.device))
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    assert torch.equal(rs.dist, a[0])


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_identity_with_forward_contacts(assets, dtype):
    """After settle steps, every candidate pair with a penetrating contact in forward() has dist < 0 equal to that pair's smallest
    contact_dist (1e-12 in float64, 2e-6 m in float32); a plane pair whose contacts fill plane_box's four points may be deeper."""
    n = 256
    b = _batch(assets, n, dtype)
    _set(b, _seeded(b, n))
    g = torch.Generator(device=b.device); g.manual_seed(7)
    for _ in range(60):
        b.step((torch.rand(n, b.act_dim, device=b.device, generator=g, dtype=dtype) - 0.5) * 20)
    d = b.distance()
    dist = d().dist.double().cpu().numpy()
    f = b.forward(qacc=False, info=True, contact_geom=True, contact_dist=True)
    ncon, cg, cd = f.info[:, 0].cpu().numpy(), f.contact_geom.cpu().numpy(), f.contact_dist.double().cpu().numpy()
    index = {(a, c): j for j, (a, c) in enumerate(zip(d.geom1, d.geom2))}
    gt = np.asarray(b.model.array("geom_type")).reshape(-1)
    tol = 1e-12 if dtype == torch.float64 else 2e-6
    checked = 0
    for e in range(n):
        per = {}
        for c in range(int(ncon[e])):
            per.setdefault(tuple(cg[e, c]), []).append(cd[e, c])
        for pair, ds in per.items():
            if min(ds) >= 0:
                continue
            j = index[pair]
            assert dist[e, j] < 0
            if gt[pair[0]] == 0 and len(ds) == 4:
                assert dist[e, j] <= min(ds) + tol
            else:
                assert abs(dist[e, j] - min(ds)) <= tol, (e, pair, dist[e, j], min(ds))
            checked += 1
    assert checked >= 50


def test_rejected_calls(assets):
    b = _batch(assets, 8, torch.float32)
    L, s = b._L, b._stream()
    m = b.model
    box, floor, table = m.geom_id("base"), m.geom_id("floor"), m.geom_id("table")
    arr = lambda *v: (C.c_int32 * max(len(v), 1))(*v)
    assert L.ur3e_batch_distance_create(b.ptr, arr(box), arr(m.ngeom), 1) < 0 and "out of range" in lib.last_error()
    assert L.ur3e_batch_distance_create(b.ptr, arr(floor), arr(table), 1) < 0 and "two planes" in lib.last_error()
    assert L.ur3e_batch_distance_create(b.ptr, arr(box), arr(box), 1) < 0 and "itself" in lib.last_error()
    assert L.ur3e_batch_distance_create(b.ptr, arr(box), arr(table), 0) < 0 and "outside [1, 256]" in lib.last_error()
    assert L.ur3e_batch_distance_create(b.ptr, arr(*[box] * 257), arr(*[table] * 257), 257) < 0 and "outside [1, 256]" in lib.last_error()
    with pytest.raises(ValueError, match="itself"):
        b.distance([("base", "base")])
    with pytest.raises(KeyError):
        b.distance([("base", "no_such_geom")])
    d = b.distance([("base", "table")])
    out = torch.empty(8, 1, device=b.device)
    p = lambda t: C.c_void_p(t.data_ptr())
    ids = torch.zeros(3, dtype=torch.int32, device=b.device)
    q = torch.zeros(3, m.nq, device=b.device)
    assert L.ur3e_batch_distance(b.ptr, d.id + 1, None, None, 8, 0.0, p(out), None, s) != 0 and "unknown distance id" in lib.last_error()
    assert L.ur3e_batch_distance(b.ptr, d.id, None, None, 8, 0.0, None, None, s) != 0 and "all outputs are null" in lib.last_error()
    assert L.ur3e_batch_distance(b.ptr, d.id, p(ids), p(q), 3, 0.0, p(out), None, s) != 0 and "not both" in lib.last_error()
    assert L.ur3e_batch_distance(b.ptr, d.id, None, None, 3, 0.0, p(out), None, s) != 0 and "m must equal n" in lib.last_error()
    assert L.ur3e_batch_distance(b.ptr, d.id, None, None, 8, float("nan"), p(out), None, s) != 0 and "NaN" in lib.last_error()
    with pytest.raises(ValueError, match="not both"):
        d(env_ids=ids, qpos=q)
    with pytest.raises(ValueError, match="at least one"):
        d(dist=False)
