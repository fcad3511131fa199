"""GPU suite: the device-compiled narrow phase (box_box, plane_box) inside the batch's forward pass on tests/models/box_pair.xml, which
runs on the generic kernel of the main.xml size class.  Each environment holds one configuration of box_pair_states (set_state);
float64 must report exactly what the kernel's source compiled for the CPU gives at the batch's own geom poses, float32 must put every
contact on both boxes' surfaces and give float64's point set away from decision boundaries.  The octagon fills the 8-point stage in
both precisions."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import ur3e_b200._lib as lib
from ur3e_b200.batch import SimBatch, env_config
from ur3e_b200.model import Model
from tests.test_narrow_phase_cpu import (BOX_PAIR, GEOM_A, GEOM_B, GEOM_FLOOR, MARGIN, SIZE_A, SIZE_B, _pair_contacts, box_pair_states,
                                         narrow_phase_at, off_surface, same_set)

SIZES = {GEOM_A: SIZE_A, GEOM_B: SIZE_B}


def _run(dtype, states):
    m = Model(BOX_PAIR)
    assert (m.nq, m.nv, m.nu) == (15, 13, 1)
    b = SimBatch(m, env_config(ctrl_mode=lib.CTRL_RAW, obs_kind=lib.OBS_STATE, obs_dim=28, act_dim=1), len(states), 0, dtype)
    assert b.max_contacts == 24   # the main.xml size class
    qp = torch.tensor(np.stack([q for _, q, _ in states]), dtype=dtype, device="cuda")
    b.set_state(qp, torch.zeros(len(states), m.nv, dtype=dtype, device="cuda"))
    r = b.forward(qacc=False, info=True, contact_geom=True, contact_dist=True, contact_pos=True, contact_frame=True)
    pos, mat, _ = b.query([("geom", "floor"), ("geom", "a"), ("geom", "b")])(pos=True, mat=True)
    torch.cuda.synchronize()
    r = {k: getattr(r, k).double().cpu().numpy() if getattr(r, k).is_floating_point() else getattr(r, k).cpu().numpy()
         for k in ("info", "contact_geom", "contact_dist", "contact_pos", "contact_frame")}
    return r, pos.double().cpu().numpy(), mat.double().cpu().numpy().reshape(len(states), 3, 9)


def test_narrow_phase_f64_is_the_host_build():
    states = box_pair_states(5)
    r, pos, mat = _run(torch.float64, states)
    for e, (name, _, _) in enumerate(states):
        assert r["info"][e][3] == 0, name   # no overflow
        total = 0
        for g1, g2 in sorted(MARGIN):
            gp, gd, gn = _pair_contacts(r, e, g1, g2)
            hp, hd, hn = narrow_phase_at(pos[e], mat[e], g1, g2)
            assert len(gd) == len(hd), (name, g1, g2, len(gd), len(hd))
            for a, b_ in ((gp, hp), (gd, hd), (gn, hn)):
                assert np.abs(a - b_).max(initial=0) <= 1e-12, (name, g1, g2)
            total += len(gd)
        assert total == r["info"][e][0], name
    octagon = [e for e, (name, _, _) in enumerate(states) if name == "octagon"][0]
    assert len(_pair_contacts(r, octagon, GEOM_A, GEOM_B)[1]) == 8


def test_narrow_phase_f32_on_surface_and_sets():
    states = box_pair_states(5)
    r32, pos32, mat32 = _run(torch.float32, states)
    r64, _, _ = _run(torch.float64, states)
    for e, (name, _, clear) in enumerate(states):
        assert r32["info"][e][3] == 0, name
        for g1, g2 in sorted(MARGIN):
            p, d, nrm = _pair_contacts(r32, e, g1, g2)
            assert np.isfinite(p).all() and np.isfinite(d).all() and np.isfinite(nrm).all(), name
            R = [mat32[e][g].reshape(3, 3) for g in range(3)]
            for k in range(len(d)):
                assert abs(np.linalg.norm(nrm[k]) - 1) < 1e-5, name
                if g1 != GEOM_FLOOR:   # box 1 side of a box-box contact
                    assert off_surface(p[k] - d[k] / 2 * nrm[k], pos32[e][g1], R[g1], SIZES[g1]) <= 1e-5, (name, k)
                else:                  # the plane side
                    assert abs((p[k] - d[k] / 2 * nrm[k] - pos32[e][g1]) @ R[g1][:, 2]) <= 1e-5, (name, k)
                assert off_surface(p[k] + d[k] / 2 * nrm[k], pos32[e][g2], R[g2], SIZES[g2]) <= 1e-5, (name, k)
            if clear:
                p64, d64, _ = _pair_contacts(r64, e, g1, g2)
                assert same_set(p, p64, 1e-5) and np.allclose(np.sort(d), np.sort(d64), atol=1e-5), (name, g1, g2)
    octagon = [e for e, (name, _, _) in enumerate(states) if name == "octagon"][0]
    assert len(_pair_contacts(r32, octagon, GEOM_A, GEOM_B)[1]) == 8
