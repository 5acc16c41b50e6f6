"""Plan fingerprints of receiver state records (sdrb_plan_fingerprint): host only, no GPU. A record may only be loaded into a
bank whose plan computes the same samples, so the fingerprint covers everything that can change an output sample and
nothing that cannot (topics, addresses)."""
import glob
import os

import pytest

from conftest import plan_path
from sdrreceiver_b200 import binding as B


def all_plans(root):
    return sorted(glob.glob(os.path.join(root, "plans", "*.ini")))


def test_fingerprint_is_stable_and_distinct_per_plan(root):
    paths = all_plans(root)
    assert len(paths) >= 9
    fps = {}
    for p in paths:
        a, b = B.Plan(p).fingerprint, B.Plan(p).fingerprint
        assert a == b, p
        fps[os.path.basename(p)] = a
    assert len(set(fps.values())) == len(fps), fps


def rebuild(plan, mains=None, subs=None, correct_dc=None):
    return B.Plan.from_desc(plan.fs, plan.block, plan.bufsplit, plan.correct_dc if correct_dc is None else correct_dc,
                            plan.mains if mains is None else mains, plan.subs if subs is None else subs)


@pytest.mark.parametrize("name", ["25E", "54W_all", "FWD_test"])
def test_descriptor_changes(name):
    plan = B.Plan(plan_path(name))
    base = rebuild(plan).fingerprint
    assert rebuild(plan).fingerprint == base
    # the plan built from an ini and the same plan built from its numbers are one plan
    assert plan.fingerprint == base
    # names only: a renamed topic must not block a move
    subs = [dict(s, topic="Z%03d" % k) for k, s in enumerate(plan.subs)]
    mains = [dict(m, topic=("F%d" % k) if m["topic"] else "") for k, m in enumerate(plan.mains)]
    assert rebuild(plan, mains=mains, subs=subs).fingerprint == base
    # anything that changes a sample changes it
    changed = {
        "gain": rebuild(plan, subs=[dict(plan.subs[0], gain=plan.subs[0]["gain"] * 2)] + plan.subs[1:]),
        "sub mixer + 1 Hz": rebuild(plan, subs=[dict(plan.subs[0], mixer=plan.subs[0]["mixer"] + 1.0)] + plan.subs[1:]),
        "main mixer + 1 Hz": rebuild(plan, mains=[dict(plan.mains[0], mixer=plan.mains[0]["mixer"] + 1.0)] + plan.mains[1:]),
        "correct_dc": rebuild(plan, correct_dc=not plan.correct_dc),
    }
    s0 = plan.subs[0]
    if s0["decim"] > 0:
        changed["sub decimation"] = rebuild(plan, subs=[dict(s0, decim=s0["decim"] - 1)] + plan.subs[1:])
    fwd = [k for k, m in enumerate(plan.mains) if m["forward"]]
    if fwd:
        k = fwd[0]
        m = dict(plan.mains[k], scalecomp=plan.mains[k]["scalecomp"] + 1)
        changed["compress scale"] = rebuild(plan, mains=plan.mains[:k] + [m] + plan.mains[k + 1:])
    for what, p in changed.items():
        assert p.fingerprint != base, what
    assert len({p.fingerprint for p in changed.values()}) == len(changed)


def test_main_decimation_changes_it():
    main = lambda d: {"mixer": 0.0, "decim": d}
    a = B.Plan.from_desc(1536000, 384000, 4, False, [main(3)], [])
    b = B.Plan.from_desc(1536000, 384000, 4, False, [main(4)], [])
    assert a.fingerprint != b.fingerprint


def test_fingerprint_null_arguments():
    L = B.lib()
    assert L.sdrb_plan_fingerprint(None, None) == -1
    assert L.sdrb_bank_state_bytes(None) == 0
