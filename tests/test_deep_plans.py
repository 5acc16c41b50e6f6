"""Plans with deep decimation: main VFOs with 4..8 half-band stages, sub VFOs with 6..8 (vfo::decimate is decimate[9],
vfo.h:39), and sub VFOs whose callback is not a multiple of 32 samples. The plan compiler must agree with oracle/plan.py
on the three DEEP_* plans and refuse, naming the VFO, what the reference cannot run or the library cannot store."""
import numpy as np
import pytest

from conftest import plan_path
from oracle import plan as OP
from sdrreceiver_b200 import binding as B

DEEP = ["DEEP_1536", "DEEP_1920", "DEEP_288K"]


@pytest.mark.parametrize("name", DEEP)
def test_deep_plan_matches_oracle_plan(name):
    p = B.Plan(plan_path(name)); q = OP.build_plan(plan_path(name))
    assert (p.fs, p.block, p.bufsplit, p.correct_dc, p.center) == (q["Fs"], q["block"], q["bufsplit"], q["dc"], q["center"])
    assert len(p.mains) == len(q["mains"]) and len(p.subs) == len(q["subs"])
    for a, b in zip(p.mains, q["mains"]):
        assert (a["mixer"], a["decim"], a["out_rate"]) == (b["mixer"], b["decim"], b["out_rate"])
        assert a["block_out"] == q["block"] >> b["decim"]
    off = 0
    for a, b in zip(p.subs, q["subs"]):
        for k in ("topic", "main", "decim", "late", "filterbw", "mixer", "Fs", "out_rate", "samples_out", "freq"):
            assert a[k] == b[k], (k, a, b)
        assert np.float32(a["gain"]) == np.float32(b["gain"])
        assert a["pcm_offset"] == off
        off += a["samples_out"]
    assert p.pcm_per_block == off
    assert abs(p.alg_bytes - (2 + 2 * sum(s["out_rate"] for s in q["subs"]) / q["Fs"])) < 1e-12


def test_deep_plans_cover_the_new_ground():
    """What the three plans were chosen for: main tails of 1..4 stages, sub tails of 1..3, 5-stage sub VFOs under a
    full-rate parent, parents that are not whole 128-sample tiles or 32-sample chunks, mix-only subs on deep mains."""
    plans = {n: B.Plan(plan_path(n)) for n in DEEP}
    main_tails = {m["decim"] - 3 for p in plans.values() for m in p.mains if m["decim"] > 3}
    sub_tails = {s["decim"] - 5 for p in plans.values() for s in p.subs if s["decim"] > 5}
    assert main_tails == {1, 2, 3, 4} and sub_tails == {1, 2, 3}
    p = plans["DEEP_1536"]
    assert [m["decim"] for m in p.mains] == [5, 4, 0]
    assert [s["decim"] for s in p.subs] == [2, 0, 2, 7, 2, 5, 8, 5]
    assert p.pcm_per_block == 55500
    parents = {p.mains[s["main"]]["block_out"] for p in plans.values() for s in p.subs}
    assert {12000, 24000, 30000, 3600} <= parents                       # 12 000 / 24 000: not whole 128-sample tiles
    assert any(b % 32 for b in parents)
    q = plans["DEEP_288K"]
    assert (q.subs[0]["decim"], q.subs[0]["out_rate"], q.subs[0]["samples_out"]) == (0, 18000, 3600)
    assert [m["block_out"] for m in q.mains] == [3600, 450, 28800] and q.pcm_per_block == 10800
    assert [m["forward"] for m in q.mains] == [False, True, False]
    assert [m["forward"] for m in plans["DEEP_1920"].mains] == [False, True, False]
    assert plans["DEEP_1920"].pcm_per_block == 45000


def _ini(tmp_path, fs, mains, subs=()):
    lines = ["sample_rate=%d" % fs, "center_frequency=1545600000", "mix_offset=0", "[main_vfos]", "size=%d" % len(mains)]
    for k, (freq, rate) in enumerate(mains):
        lines += ["%d\\frequency=%d" % (k + 1, freq), "%d\\out_rate=%d" % (k + 1, rate)]
    lines += ["[vfos]", "size=%d" % len(subs)]
    for k, (freq, rate, topic) in enumerate(subs):
        lines += ["%d\\frequency=%d" % (k + 1, freq), "%d\\out_rate=%d" % (k + 1, rate), "%d\\gain=4" % (k + 1),
                  "%d\\topic=%s" % (k + 1, topic)]
    path = tmp_path / "p.ini"
    path.write_text("\n".join(lines) + "\n")
    return str(path)


def test_rejects_a_main_vfo_with_nine_stages(tmp_path):
    with pytest.raises(B.SdrbError, match=r"main VFO 1 needs 0\.\.8 half-band stages.*not 9"):
        B.Plan(_ini(tmp_path, 1536000, [(1545600000, 3000)]))


def test_rejects_an_odd_final_length(tmp_path):
    # 1.92 MS/s / 7 500 = 256: 8 stages, 480 000 >> 8 = 1 875 samples per callback
    with pytest.raises(B.SdrbError, match="main VFO 1 would store 1875 samples per callback"):
        B.Plan(_ini(tmp_path, 1920000, [(1545600000, 7500)]))


def test_rejects_a_half_band_stage_on_an_odd_input(tmp_path):
    # main at 15 kHz: 7 stages, 3 750 per callback (even); the sub VFO at 3 750 Hz needs 2 more, the second gets 1 875
    with pytest.raises(B.SdrbError, match="sub VFO 'VSUB1': half-band stage 2 would get 1875 samples per callback"):
        B.Plan(_ini(tmp_path, 1920000, [(1545600000, 15000)], [(1545601000, 3750, "VSUB1")]))


def test_the_same_rules_hold_for_plan_descriptions():
    main = lambda decim: {"mixer": 1000.0, "decim": decim}
    assert B.Plan.from_desc(1536000, 384000, 4, False, [main(8)], []).mains[0]["block_out"] == 1500
    assert B.Plan.from_desc(1536000, 384000, 4, False, [main(0)],
                            [{"main": 0, "mixer": 10.0, "decim": 8, "topic": "SUB8"}]).subs[0]["samples_out"] == 1500
    with pytest.raises(B.SdrbError, match="main VFO 1 needs 0..8 half-band stages"):
        B.Plan.from_desc(1536000, 384000, 4, False, [main(9)], [])
    with pytest.raises(B.SdrbError, match="sub VFO 'SUB9' needs 0..8 half-band stages"):
        B.Plan.from_desc(1536000, 384000, 4, False, [main(0)], [{"main": 0, "mixer": 10.0, "decim": 9, "topic": "SUB9"}])
    with pytest.raises(B.SdrbError, match="sub VFO 'NEG' needs 0..8"):
        B.Plan.from_desc(1536000, 384000, 4, False, [main(0)], [{"main": 0, "mixer": 10.0, "decim": -1, "topic": "NEG"}])
    # more than 3 main stages on k1_v2's third-stage output need a callback whose staged part outlasts the tail's reach
    with pytest.raises(B.SdrbError, match="main VFO 1 with more than 3 half-band stages needs at least 4096 samples"):
        B.Plan.from_desc(1536000, 2048, 4, False, [main(4)], [])
