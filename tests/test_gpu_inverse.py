"""GPU suite for the inverse-dynamics query (ur3e_batch_inverse, SimBatch.inverse): the compiled sm_100a kernel against the mj_inverse
restatement of tests/inverse_reference.py at the batch's stored state and at given states, the forward-inverse and step-inverse identities,
the two state sources, float32 against float64, non-interference with the step path and every rejected call."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as O
import ur3e_b200._lib as lib
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.model import Model
from tests import inverse_reference as R
from tests.test_gpu_forward_query import _batch_for, _np, _random_main_states
from tests.test_gpu_query import _run

SCENES = ["main.xml", "ur3e_2f85.xml", "ur3e_raw.xml"]


def rel(a, b, floor):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor))) if a.size else 0.0


def _t(x, b):
    return torch.tensor(np.ascontiguousarray(x), dtype=b.dtype, device=b.device)


def _raw(assets, xml, n, dtype):
    """CTRL_RAW, frame_skip 1: mujoco.rollout's semantics (one env-step = one mj_step with ctrl = the action)."""
    m = Model(assets + "/" + xml)
    obs = dict(obs_kind=lib.OBS_V2, obs_dim=24) if xml == "main.xml" else dict(obs_kind=lib.OBS_STATE, obs_dim=m.nq + m.nv)   # OBS_STATE holds at most 32 values
    return SimBatch(m, env_config(ctrl_mode=lib.CTRL_RAW, act_dim=m.nu, frame_skip=1, **obs), n, 0, dtype)


def _all(b):
    con = b.max_contacts > 0
    return dict(qfrc_inverse=True, qfrc_constraint=True, info=True, contact_geom=con, contact_force=con)


def _check(b, om, qp, qv, qacc, r, discrete, rows):
    """rows of the batch's result r at states (qp, qv, qacc) against the reference, to rounding."""
    seen = 0
    for e in rows:
        ref = R.inverse(om, qp[e], qv[e], qacc[e], discrete)
        n = ref["ncon"]
        assert list(r["info"][e]) == [n, ref["nefc"], 0]
        scale = np.abs(ref["qfrc_inverse"]).max() + 1.0
        assert np.abs(r["qfrc_inverse"][e] - ref["qfrc_inverse"]).max() <= 1e-9 * scale
        assert np.abs(r["qfrc_constraint"][e] - ref["qfrc_constraint"]).max() <= 1e-9 * scale
        if "contact_geom" in r:
            assert np.array_equal(r["contact_geom"][e][:n], ref["contact_geom"]) and (r["contact_geom"][e][n:] == -1).all()
            fs = np.abs(ref["contact_force"]).max(initial=0) + 1.0
            assert np.abs(r["contact_force"][e][:n] - ref["contact_force"]).max(initial=0) <= 1e-9 * fs
            assert not r["contact_force"][e][n:].any()
        seen += n > 0
    return seen


@pytest.mark.parametrize("discrete", [False, True], ids=["continuous", "discrete"])
@pytest.mark.parametrize("scene", SCENES)
def test_stored_state_matches_reference_f64(assets, scene, discrete):
    """float64, 300 seeded steps of each model family, random accelerations at the stored state."""
    b, lo, hi = _batch_for(assets, scene, 32, torch.float64)
    _run(b, lo, hi, 300, 3)
    om = O.Model(b.model.path)
    qp, qv, _ = (x.cpu().numpy() for x in b.get_state())
    qacc = np.random.default_rng(5).uniform(-5, 5, (b.n, b.model.nv))
    r = _np(b.inverse(_t(qacc, b), discrete=discrete, **_all(b)))
    _check(b, om, qp, qv, qacc, r, discrete, range(0, b.n, 3))


@pytest.mark.parametrize("discrete", [False, True], ids=["continuous", "discrete"])
def test_given_main_states_in_contact_f64(assets, discrete):
    """Random main.xml states with the mug pressed into the table, as given states (m != n)."""
    b, _, _ = _batch_for(assets, "main.xml", 4, torch.float64)
    om = O.Model(b.model.path)
    rng = np.random.default_rng(11)
    qp, qv = _random_main_states(om, rng, 24)
    qacc = rng.uniform(-5, 5, (24, om.nv))
    r = _np(b.inverse(_t(qacc, b), state=(_t(qp, b), _t(qv, b)), discrete=discrete, **_all(b)))
    assert _check(b, om, qp, qv, qacc, r, discrete, range(24)) >= 20


def test_forward_inverse_identity(assets):
    """forward(ctrl = u).qacc fed back: float64 gives forward's constraint and contact forces to rounding and the oracle's
    qfrc_actuator(u) within the solver's tolerance; float32's residual at the production solver settings is recorded."""
    res = {}
    for dtype in (torch.float64, torch.float32):
        b, lo, hi = _batch_for(assets, "main.xml", 256, dtype)
        _run(b, lo, hi, 300, 13)
        om = O.Model(b.model.path)
        u = np.random.default_rng(17).uniform(-5, 5, (b.n, om.nu)); u[:, 6] = np.random.default_rng(19).uniform(0, 255, b.n)
        f = b.forward(ctrl=_t(u, b), qacc=True, qfrc_constraint=True, info=True, contact_force=True)
        fq = f.qacc.clone()
        inv = _np(b.inverse(fq, qfrc_constraint=True, info=True, contact_force=True))
        fw = _np(f)
        qp, qv, _ = (x.double().cpu().numpy() for x in b.get_state())
        fa = np.zeros((b.n, om.nv))
        for e in range(b.n):
            d = O.Data(om); d.reset(); d.set_state(qp[e], qv[e]); d.ctrl[:] = u[e]; d.forward()
            fa[e] = d.qfrc_actuator
        if dtype == torch.float64:
            assert (inv["info"][:, :2] == fw["info"][:, :2]).all()
            assert rel(inv["qfrc_constraint"], fw["qfrc_constraint"], 1.0) < 1e-8
            assert rel(inv["contact_force"], fw["contact_force"], 1.0) < 1e-8
            assert rel(inv["qfrc_inverse"], fa, 1e-1) < 1e-6
        else:
            err = np.abs(inv["qfrc_inverse"] - fa).max(axis=1) / (np.abs(fa).max(axis=1) + 1.0)
            res["f32_residual_rel"] = dict(median=float(np.median(err)), p99=float(np.quantile(err, 0.99)), max=float(err.max()),
                                           mean_nefc=float(fw["info"][:, 1].mean()), mean_iters=float(fw["info"][:, 2].mean()))
            assert err.max() < 1e-3
    print("inverse: float32 forward-inverse residual", json.dumps(res))


@pytest.mark.parametrize("scene", ["main.xml", "ur3e_raw.xml"])
def test_step_identity_over_rollout(assets, scene):
    """A float64 CTRL_RAW, frame_skip 1 rollout of T = 20 steps from explicit states; one inverse call over all T x m states with the
    discrete convention and qacc = (qvel[t + 1] - qvel[t]) / h returns the oracle's qfrc_actuator(u_t) at each sampled state."""
    T, mm = 20, 16
    b = _raw(assets, scene, 4, torch.float64)
    om = O.Model(b.model.path)
    nq, nv, nu, h = om.nq, om.nv, om.nu, om.timestep
    rng = np.random.default_rng(23)
    if scene == "main.xml":
        q0, v0 = _random_main_states(om, rng, mm)
        u = rng.uniform(-5, 5, (T, mm, nu)); u[..., 6] = rng.uniform(0, 255, (T, mm))
    else:
        q0 = np.tile(np.array(om.arr("qpos0")), (mm, 1)) + rng.uniform(-1, 1, (mm, nq)); v0 = rng.uniform(-1, 1, (mm, nv))
        u = rng.uniform(-5, 5, (T, mm, nu))
    r = b.rollout(_t(u, b), state=(_t(q0, b), _t(v0, b)), qpos=True, qvel=True, obs=False, reward=False, terminated=False, truncated=False, info=True)
    assert not r.info.any()
    q = torch.cat([_t(q0, b)[None], r.qpos[:-1]]).reshape(-1, nq).contiguous()
    v = torch.cat([_t(v0, b)[None], r.qvel[:-1]]).reshape(-1, nv).contiguous()
    a = ((torch.cat([_t(v0, b)[None], r.qvel]).diff(dim=0)) / h).reshape(-1, nv).contiguous()
    tau = b.inverse(a, state=(q, v), discrete=True).qfrc_inverse.cpu().numpy().reshape(T, mm, nv)
    qn, vn = q.cpu().numpy().reshape(T, mm, nq), v.cpu().numpy().reshape(T, mm, nv)
    for t in range(0, T, 3):
        for j in range(0, mm, 3):
            d = O.Data(om); d.reset(); d.set_state(qn[t, j], vn[t, j]); d.ctrl[:] = u[t, j]; d.forward()
            assert rel(tau[t, j], d.qfrc_actuator, 1e-1) < 1e-6, (t, j)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_state_sources_agree(assets, dtype):
    """The stored state gives results bit-identical to state = get_state()[:2]; given states work with m > n, m < n and m = 1."""
    b, lo, hi = _batch_for(assets, "main.xml", 32, dtype)
    _run(b, lo, hi, 200, 29)
    qp, qv, _ = b.get_state()
    qacc = _t(np.random.default_rng(31).uniform(-5, 5, (b.n, b.model.nv)), b)
    want = {k: v.clone() for k, v in b.inverse(qacc, **_all(b))._asdict().items()}
    got = b.inverse(qacc, state=(qp, qv), **_all(b))._asdict()
    for k in want:
        assert torch.equal(want[k], got[k]), k
    for idx in (torch.arange(45) % b.n, torch.tensor([7]), torch.arange(5, 20)):
        idx = idx.to(b.device)
        r = b.inverse(qacc[idx].contiguous(), state=(qp[idx].contiguous(), qv[idx].contiguous()), **_all(b))._asdict()
        for k in want:
            assert torch.equal(r[k], want[k][idx]), (k, len(idx))


def test_undamped_model_conventions_identical(assets):
    """ur3e_raw.xml has no damping: the discrete and the continuous convention give bit-identical results."""
    for dtype in (torch.float32, torch.float64):
        b, lo, hi = _batch_for(assets, "ur3e_raw.xml", 16, dtype)
        _run(b, lo, hi, 100, 37)
        qacc = _t(np.random.default_rng(41).uniform(-5, 5, (b.n, b.model.nv)), b)
        x = b.inverse(qacc, discrete=False, qfrc_constraint=True, info=True)
        x = [t.clone() for t in x if t is not None]
        y = [t for t in b.inverse(qacc, discrete=True, qfrc_constraint=True, info=True) if t is not None]
        assert all(torch.equal(p, q) for p, q in zip(x, y))


@pytest.mark.parametrize("discrete", [False, True], ids=["continuous", "discrete"])
def test_float32_against_float64(assets, discrete):
    """The same states and accelerations through the float32 and the float64 batch."""
    rng = np.random.default_rng(43)
    om = O.Model(assets + "/main.xml")
    qp, qv = _random_main_states(om, rng, 64)
    qacc = rng.uniform(-5, 5, (64, om.nv))
    r = {}
    for dtype in (torch.float32, torch.float64):
        b, _, _ = _batch_for(assets, "main.xml", 8, dtype)
        r[dtype] = _np(b.inverse(_t(qacc, b), state=(_t(qp, b), _t(qv, b)), discrete=discrete, **_all(b)))
    a, c = r[torch.float32], r[torch.float64]
    same = (a["info"][:, :2] == c["info"][:, :2]).all(axis=1)
    assert same.mean() > 0.9
    err = np.abs(a["qfrc_inverse"] - c["qfrc_inverse"]).max(axis=1) / (np.abs(c["qfrc_inverse"]).max(axis=1) + 1.0)
    assert np.quantile(err[same], 0.9) < 1e-3


def test_non_interference(assets):
    """Records are untouched by a call; stepping with an inverse call between steps is bit-identical to stepping without; a non-default
    stream ordered after the default one gives the same results."""
    bs = []
    for _ in range(2):
        b, lo, hi = _batch_for(assets, "main.xml", 64, torch.float32)
        b.reset(seed=5)
        bs.append(b)
    rng = np.random.default_rng(47)
    qacc = _t(rng.uniform(-5, 5, (64, bs[0].model.nv)), bs[0])
    for k in range(30):
        a = _t(lo + (hi - lo) * rng.random((64, len(lo))), bs[0])
        before = [x.clone() for x in bs[0].get_state()]
        r = bs[0].inverse(qacc, discrete=bool(k & 1), **_all(bs[0]))
        after = bs[0].get_state()
        assert all(torch.equal(p, q) for p, q in zip(before, after))
        o0 = bs[0].step(a)[0].clone(); o1 = bs[1].step(a)[0].clone()
        assert torch.equal(o0, o1)
    assert all(torch.equal(p, q) for p, q in zip(bs[0].get_state(), bs[1].get_state()))
    want = {k: v.clone() for k, v in bs[0].inverse(qacc, **_all(bs[0]))._asdict().items()}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = {k: v.clone() for k, v in bs[0].inverse(qacc, **_all(bs[0]))._asdict().items()}
    torch.cuda.current_stream().wait_stream(side)
    for k in want:
        assert torch.equal(want[k], got[k]), k


def test_rejected_calls(assets):
    """Every rejected combination, through SimBatch and through the C entry point."""
    b, _, _ = _batch_for(assets, "main.xml", 8, torch.float64)
    nq, nv = b.model.nq, b.model.nv
    z = lambda *s: torch.zeros(*s, dtype=torch.float64, device=b.device)
    with pytest.raises(ValueError):
        b.inverse(z(9, nv))                                   # stored state, m != n
    with pytest.raises(ValueError):
        b.inverse(z(8, nv), state=(z(8, nq),))                # state without qvel
    with pytest.raises(ValueError):
        b.inverse(z(8, nv), state=(z(8, nq), z(7, nv)))       # mismatched shapes
    with pytest.raises(ValueError):
        b.inverse(z(8, nv).float())                           # wrong dtype
    with pytest.raises(ValueError):
        b.inverse(z(8, nv), qfrc_inverse=False)               # nothing asked for
    L, s = b._L, b._stream()
    qa, qp, qv = z(8, nv), z(8, nq), z(8, nv)
    o = torch.empty(8, nv, dtype=torch.float64, device=b.device)
    good = lib.InverseOut(o.data_ptr(), None, None, None, None)
    p = lambda t: C.c_void_p(t.data_ptr())
    assert L.ur3e_batch_inverse(b.ptr, None, None, 8, p(qa), 0, C.byref(good), s) == 0
    cases = [((p(qp), None, 8, p(qa), 0, C.byref(good)), "without qvel"), ((None, p(qv), 8, p(qa), 0, C.byref(good)), "without qpos"),
             ((None, None, 7, p(qa), 0, C.byref(good)), "stored state"), ((p(qp), p(qv), 0, p(qa), 0, C.byref(good)), "states"),
             ((p(qp), p(qv), 2 ** 31, p(qa), 0, C.byref(good)), "states"), ((None, None, 8, None, 0, C.byref(good)), "qacc is null"),
             ((None, None, 8, p(qa), 0, None), "out is null"), ((None, None, 8, p(qa), 0, C.byref(lib.InverseOut())), "all outputs")]
    for args, why in cases:
        assert L.ur3e_batch_inverse(b.ptr, *args, s) != 0
        assert why in lib.last_error(), (why, lib.last_error())
    torch.cuda.synchronize()
    raw, _, _ = _batch_for(assets, "ur3e_raw.xml", 4, torch.float64)
    assert raw.max_contacts == 0
    qa = torch.zeros(4, raw.model.nv, dtype=torch.float64, device=raw.device)
    for kw in (dict(contact_geom=True), dict(contact_force=True)):
        with pytest.raises(ValueError, match="no contact pairs"):
            raw.inverse(qa, **kw)
    g = torch.empty(4, 1, 2, dtype=torch.int32, device=raw.device)
    out = lib.InverseOut(None, None, None, g.data_ptr(), None)
    assert raw._L.ur3e_batch_inverse(raw.ptr, None, None, 4, p(qa), 0, C.byref(out), raw._stream()) != 0
    assert "contact outputs" in lib.last_error()
