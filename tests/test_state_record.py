"""Plan fingerprints of receiver state records (sdrb_plan_fingerprint): host only, no GPU. A record may only be loaded into a
bank whose plan computes the same samples, so the fingerprint covers everything that can change an output sample and
nothing that cannot (topics, addresses)."""
import glob
import os
import re

import numpy as np
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


def header_bounds(root):
    """The record bounds as include/sdrb200.h states them: (samples behind SDRB_STATE_MAX_BLOCKS_DONE, SDRB_STATE_MAX_DC)."""
    with open(os.path.join(root, "include", "sdrb200.h")) as f:
        h = f.read()
    shift = re.search(r"#define SDRB_STATE_MAX_BLOCKS_DONE\(block\) \(\(int64_t\)\(\(\(int64_t\)1 << (\d+)\) / \(int64_t\)\(block\)\)\)", h)
    dc = re.search(r"#define SDRB_STATE_MAX_DC ([0-9.]+)f", h)
    assert shift and dc
    return 1 << int(shift.group(1)), float(dc.group(1))


def test_counter_bound_leaves_headroom(root):
    samples, _ = header_bounds(root)
    assert samples == 2**62 and samples / 1536000 / (365.25 * 86400) > 95000      # years of signal at 1.536 MS/s
    for p in all_plans(root):
        block = B.Plan(p).block
        top = samples // block
        assert top * block <= 2**62 < (top + 1) * block
        # a receiver loaded at the bound still has 2^62 samples before (blocks_done + b) * block overflows
        assert (top + 2**62 // block) * block < 2**63


def test_dc_recursion_stays_inside_the_record_bound(root):
    """avept = avept * (1 - 1e-6) + 1e-6 * (x - 127) in float32 (sdrj.cpp:277-283), started at 0, on full-scale input: it
    rises monotonically to the fixed point of its rounding, +-124.2353, inside SDRB_STATE_MAX_DC = 128. The recursion is
    monotone in its input, so no byte sequence takes it further out than all 255 or all 0."""
    from oracle import oracle as O
    _, bound = header_bounds(root)
    n = 4_000_000                                            # 4 time constants; the state stops moving after about 3.5
    for v, sign in ((255, 1.0), (0, -1.0)):
        t = O.dc_trace(np.full(2 * n, v, np.uint8), every=1)
        for arm in (t.real, t.imag):
            assert np.all(np.isfinite(arm)) and np.all(sign * arm >= 0)
            peak = float(np.abs(arm).max())
            assert arm[-1] == arm[-n // 8] and abs(peak - 124.2353) < 1e-4, (v, peak)   # settled at its rounding fixed point
            assert peak <= bound
