"""GPU suite: the compiled sm_100a solves against the independent dual reference (tests/solver_reference.py) on the sample of
tests/test_solver_dual_cpu.py.

  forward float64    SimBatch.forward's qacc, qfrc_constraint and contact forces within 1e-8; at tolerance 1e-10 its iteration count
                     equals the host build's at the same state and warm start (the register-resident LDL^T and its arm / mug block
                     skip against the host build's chol_solve_aug); the same answer from a zero warm start and from the optimum
  forward float32    the generic arena, on states whose float32 row set is float64's, at the host float32 build's bounds
  step kernels       float32, CTRL_RAW, frame_skip 1: after set_state(q, v, ws) and step(u) the record's new warm start is the solve's
                     qacc (test_gpu_forward_query.py::test_forward_is_the_steps_forward_pass); per tier (lite: <= 8 contacts, grasp: the
                     pads on the mug, generic: single_tier), at the same bounds
  inverse float64    at the reference's qacc, contact_force and qfrc_constraint are f* and J^T f* within 1e-8
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import ur3e_b200._lib as lib
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.model import Model
from tests import test_solver_dual_cpu as T
from tests.hostcheck import build as HC


def _batch(xml, n, dtype, **kw):
    m = Model(xml)
    if os.path.basename(xml) == "main.xml":
        cfg = env_config(ctrl_mode=lib.CTRL_RAW, obs_kind=lib.OBS_V2, obs_dim=24, act_dim=m.nu, frame_skip=1, **kw)
    else:
        cfg = env_config(ctrl_mode=lib.CTRL_RAW, obs_kind=lib.OBS_STATE, obs_dim=m.nq + m.nv, act_dim=m.nu, frame_skip=1, **kw)
    b = SimBatch(m, cfg, n, 0, dtype)
    b.reset()
    return b


def _t(x, dtype):
    return torch.tensor(np.asarray(x), dtype=dtype, device="cuda")


def _np(r):
    return {k: (v.double().cpu().numpy() if v.is_floating_point() else v.cpu().numpy()) for k, v in r._asdict().items() if v is not None}


def _by_model(sample):
    out = {}
    for label, st in T._all(sample):
        out.setdefault(st[0], []).append((label, st))
    return out


@pytest.fixture(scope="module")
def sample(tmp_path_factory):
    tmp = str(tmp_path_factory.mktemp("solver_dual_gpu"))
    s = dict(pick=T.pick_states(), random_main=T.random_main_states(), gripper=T.gripper_states(), hinge=T.hinge_states(), box_pair=T.box_pair_states())
    s.update(T.box_variants(tmp))
    return s


def _forward(b, states, ws, dtype):
    qp, qv, u = (np.array([st[k] for _, st in states]) for k in (1, 2, 4))
    b.set_state(_t(qp, dtype), _t(qv, dtype), _t(ws, dtype))
    want = dict(qacc=True, qfrc_constraint=True, info=True)
    if b.max_contacts:
        want.update(contact_force=True, contact_geom=True)
    return _np(b.forward(ctrl=_t(u, dtype), **want))


def test_forward_f64_against_reference(sample):
    worst, mism, n_all, floor_mism = 0.0, [], 0, 0
    for xml, states in _by_model(sample).items():
        n = len(states)
        b = _batch(xml, n, torch.float64)
        ws = np.array([st[3] for _, st in states])
        r = _forward(b, states, ws, torch.float64)
        opt = np.zeros_like(ws)
        for e, (label, st) in enumerate(states):
            d, p = T.ref_at(st)
            ncon, nefc, it, ovf = r["info"][e]
            assert (ncon, nefc, ovf) == (d.ncon, d.nefc, 0), (label, e)
            err = T.errors(p, r["qacc"][e], r["qfrc_constraint"][e], r["contact_force"][e] if ncon else None)
            for k, v in err.items():
                assert v <= T.BOUND64, (label, e, k, v)
            worst = max(worst, *err.values())
            h = HC.forward(xml, st[1], st[2], st[3], st[4], info=True)
            floor_mism += it != h["info"][2]
            n_all += 1
            opt[e] = p.qacc(p.f)
        # the same Newton path as the host build's chol_solve_aug: equal iteration counts at a tolerance above the rounding floor
        # (at the build's 1e-15 the count depends on the last bits of the gradient, which FMA contraction changes: printed only)
        bt = _batch(xml, n, torch.float64, solver_tolerance=1e-10)
        it10 = _forward(bt, states, ws, torch.float64)["info"][:, 2]
        for e, (label, st) in enumerate(states):
            h = HC.run(xml, st[1], st[2], st[4], st[3], 0, tol=1e-10)["iters"]
            if it10[e] != h:
                mism.append((label, e, int(it10[e]), int(h)))
        for w in (np.zeros_like(ws), opt):                                 # warm-start independence
            r2 = _forward(b, states, w, torch.float64)
            for e, (label, _) in enumerate(states):
                assert T.rel(r2["qacc"][e], r["qacc"][e]) <= 1e-9, (label, e)
                assert T.rel(r2["qfrc_constraint"][e], r["qfrc_constraint"][e], 1e-3) <= 1e-9, (label, e)
    print("device float64 forward vs dual reference: worst %.1e over %d states; iteration counts unlike the host build's at tolerance "
          "1e-15: %d, at 1e-10: %s" % (worst, n_all, floor_mism, mism))
    assert not mism


def _f32_errors(states, qacc, fc, info, geom):
    """(errors, excluded, capped) of float32 results on float32-rounded states, keeping the states whose float32 contact list is the
    float64 one's (fc None: qacc alone)."""
    errs, excluded, capped = (dict(qacc=[], qfrc_constraint=[]) if fc is not None else dict(qacc=[])), 0, 0
    for e, st in enumerate(states):
        d, p = T.ref_at(st)
        og = np.array([[c.geom1, c.geom2] for c in d.contacts()], dtype=np.int64).reshape(-1, 2)
        if (info[e][0], info[e][1]) != (d.ncon, d.nefc) or not np.array_equal(geom[e][:d.ncon], og):
            excluded += 1
            continue
        capped += info[e][2] >= 8
        x = T.errors(p, qacc[e], fc[e] if fc is not None else p.J.T @ p.f, None)
        for k in errs:
            errs[k].append(x[k])
    return errs, excluded, capped


def _report(name, errs, excluded, capped, n):
    for k, v in errs.items():
        v = np.array(v)
        print("%s %-15s over %d states: median %.1e  p95 %.1e  max %.1e" % (name, k, len(v), np.median(v), np.percentile(v, 95), v.max()))
    print("  excluded for a different row set: %d of %d; solves at the 8-iteration cap: %d" % (excluded, n, capped))


def _main_f32_states():
    return [T.f32_state(st) for st in T.pick_states() + T.random_main_states(8, seed=11)]


def test_forward_f32_against_reference():
    states = _main_f32_states()
    n = len(states)
    b = _batch(states[0][0], n, torch.float32)
    r = _forward(b, [("", st) for st in states], np.array([st[3] for st in states]), torch.float32)
    errs, excluded, capped = _f32_errors(states, r["qacc"], r["qfrc_constraint"], r["info"], r["contact_geom"])
    _report("device float32 forward vs dual reference", errs, excluded, capped, n)
    assert excluded <= n // 10
    assert max(errs["qacc"]) <= T.F32_QACC and max(errs["qfrc_constraint"]) <= T.F32_FC


@pytest.mark.parametrize("tier", ["lite", "grasp", "generic"])
def test_step_kernels_against_reference(tier):
    """The step's solve by tier.  lite: states with at most 8 contacts (the mug on the table, no pad on it: no contact couples the arm
    and mug columns); grasp: states with more than 8 (the pads on the mug: the arm x mug block of H is not zero); generic: all of them
    on the generic size class alone (single_tier).  The row set is judged by the float32 forward query at the same state; the
    capped-solve count is the forward query's (the same solve on the generic arena, same state and warm start)."""
    states = _main_f32_states()
    q = _batch(states[0][0], len(states), torch.float32)
    r = _forward(q, [("", st) for st in states], np.array([st[3] for st in states]), torch.float32)
    if tier == "lite":
        keep = [e for e in range(len(states)) if r["info"][e][0] <= 8 and r["info"][e][1] <= 44]
    elif tier == "grasp":
        keep = [e for e in range(len(states)) if 8 < r["info"][e][0] <= 16 and r["info"][e][1] <= 68]
    else:
        keep = list(range(len(states)))
    assert len(keep) >= 20
    S = [states[e] for e in keep]
    n = len(S)
    b = _batch(S[0][0], n, torch.float32, single_tier=int(tier == "generic"))
    qp, qv, ws, u = (np.array([st[k] for st in S]) for k in (1, 2, 3, 4))
    b.set_state(_t(qp, torch.float32), _t(qv, torch.float32), _t(ws, torch.float32))
    b.step(_t(u, torch.float32))
    qacc = b.get_state()[2].double().cpu().numpy()
    torch.cuda.synchronize()
    b.step(_t(u, torch.float32))          # the tier counters of the first step are read back during the second
    torch.cuda.synchronize()
    info = b.kernel_info()["lite"]
    print(tier, info)
    if tier == "lite":
        assert info["lite_tier_steps"] == 2 and info["last_overflow_envs"] == 0, info
    elif tier == "grasp":
        assert info["lite_tier_steps"] == 2 and info["last_overflow_envs"] == n and "grasp_tier" in b.kernel_info(), info
    else:
        assert info["full_only_steps"] == 2 and info["lite_tier_steps"] == 0, info
    coupled = sum(r["info"][e][0] > 8 for e in keep)
    errs, excluded, capped = _f32_errors(S, qacc, None, r["info"][keep], r["contact_geom"][keep])
    _report("%s step kernel vs dual reference (%d states with a contact coupling arm and mug)" % (tier, coupled), errs, excluded, capped, n)
    assert excluded <= max(1, n // 10)
    assert max(errs["qacc"]) <= T.F32_QACC


def test_inverse_at_reference_qacc_f64(sample):
    """mj_inverse at the reference's qacc, from the given states: the constraint law at jar = J qacc* - aref returns f*."""
    worst = 0.0
    for xml, states in _by_model(sample).items():
        n = len(states)
        b = _batch(xml, n, torch.float64)
        qp, qv = (np.array([st[k] for _, st in states]) for k in (1, 2))
        a = np.array([T.ref_at(st)[1].qacc(T.ref_at(st)[1].f) for _, st in states])
        want = dict(qfrc_constraint=True, info=True)
        if b.max_contacts:
            want.update(contact_force=True)
        r = _np(b.inverse(_t(a, torch.float64), state=(_t(qp, torch.float64), _t(qv, torch.float64)), **want))
        for e, (label, st) in enumerate(states):
            d, p = T.ref_at(st)
            assert (r["info"][e][0], r["info"][e][1]) == (d.ncon, d.nefc), (label, e)
            fc = p.J.T @ p.f
            err = [T.rel(r["qfrc_constraint"][e], fc, 1e-3)]
            if d.ncon:
                err.append(T.rel(r["contact_force"][e][:d.ncon, :3], p.contact_forces(), 1e-3))
            assert max(err) <= T.BOUND64, (label, e, err)
            worst = max(worst, *err)
    print("device float64 inverse at the reference's qacc: worst %.1e" % worst)
