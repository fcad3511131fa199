"""The argument check of ur3e_batch_rollout (rollout.h rollout_check), compiled for the host: every accepted and rejected
combination of sizes, sources and outputs."""
import itertools

import pytest

from tests.hostcheck import rollout as HRO


def test_accepted_calls():
    assert HRO.rollout_check(1, 1) == ""
    assert HRO.rollout_check(65536 * 64, 32) == ""
    assert HRO.rollout_check(2 ** 31 - 1, 2 ** 31 - 1) == ""
    assert HRO.rollout_check(7, 3, src_ids=False, qpos0=True, qvel0=True) == ""
    assert HRO.rollout_check(7, 3, src_ids=False, qpos0=True, qvel0=True, ws0=True) == ""


@pytest.mark.parametrize("args, msg", [
    (dict(m=0, T=1), "m=0 rollouts"),
    (dict(m=-5, T=1), "m=-5 rollouts"),
    (dict(m=2 ** 31, T=1), "rollouts (1 .. 2^31 - 1"),
    (dict(m=4, T=0), "T=0 env-steps"),
    (dict(m=4, T=-1), "T=-1 env-steps"),
    (dict(m=4, T=2, actions=False), "actions is null"),
    (dict(m=4, T=2, qpos0=True, qvel0=True), "both sources"),
    (dict(m=4, T=2, qpos0=True, qvel0=True, ws0=True), "both sources"),
    (dict(m=4, T=2, src_ids=False), "no source"),
    (dict(m=4, T=2, src_ids=False, qpos0=True), "qpos0 is given without qvel0"),
    (dict(m=4, T=2, src_ids=False, qvel0=True), "qvel0 is given without qpos0"),
    (dict(m=4, T=2, src_ids=True, qvel0=True), "qvel0 is given without qpos0"),
    (dict(m=4, T=2, src_ids=False, ws0=True), "qacc_warmstart0 is given without qpos0"),
    (dict(m=4, T=2, src_ids=True, ws0=True), "qacc_warmstart0 is given without qpos0"),
    (dict(m=4, T=2, out=False, any_=False), "out is null"),
    (dict(m=4, T=2, any_=False), "all outputs are null"),
])
def test_rejected_calls(args, msg):
    assert msg in HRO.rollout_check(**args)


def test_full_matrix():
    """Every combination of the boolean inputs: accepted exactly when actions, exactly one source (ids, or qpos0 with qvel0 and an
    optional warm start) and at least one output are given."""
    for actions, src, qp, qv, ws, out, any_ in itertools.product((False, True), repeat=7):
        if any_ and not out:
            continue   # no output can be given without the struct
        want = actions and (src != qp) and qp == qv and (not ws or qp) and out and any_
        got = HRO.rollout_check(3, 2, actions, src, qp, qv, ws, out, any_)
        assert (got == "") == want, (actions, src, qp, qv, ws, out, any_, got)
