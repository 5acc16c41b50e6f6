"""The exact DC recursion on inputs that drive every branch of k0_dc_walk (GPU).

The synthetic input of the other tests keeps the DC state within 8 LSB of zero: its bytes span 96..160, the state never
changes sign or binade, and most of the walk's integer model is never exercised. Here ten deterministic uint8 scenarios,
one per stream of one bank, push the state through the binades up to 128, across zero and across powers of two, onto
lock-in fixed points, and through the largest excursion one block can make. Each runs for at least 3 * 10^6 samples
(three time constants of the recursion) on the three sample rates of the sample plans, with DC removal on:

  * the block-start DC states and the DC-corrected input of every callback equal the plain-C restatement bit for bit;
  * whole-plan outputs of three of the scenarios agree with the restatement (+-1 LSB, 1e-4 rel-L2);
  * how the callbacks are grouped into calls and the input-ready overlap of process_device_ex give identical bits;
  * the walk's per-block mode bytes show that every path was taken (translations below and above T, integer solves,
    also in the ragged last batch of a callback, float steps), and that every block whose states leave the anchor's
    window was stepped in float -- a necessary condition of the algorithm, checked from the restatement's own trace."""
import os

import numpy as np
import pytest

from conftest import plan_path
from oracle import oracle as O, plan as OP
from sdrreceiver_b200 import binding as B
from test_dc_model import anchor

pytestmark = pytest.mark.gpu
DC_BLK = 128
BATCH = 32                      # blocks per batch of k0_dc_walk (DCW_BATCH)
TAU = 1_000_000                 # samples: time constant of the recursion, 1 / (1 - a)
MIN_SAMPLES = 3 * TAU

# plan -> (ini, callbacks per stream, irregular call split)
PLANS = {
    "25E": ("25E", 8, [3, 1, 2, 2]),
    "54W_all": ("54W_all", 7, [2, 3, 1, 1]),
    "54W_288K": ("54W_288K", 53, [7, 1, 13, 2, 9, 21]),
}
WHOLE_PLAN = ("full_scale", "staircase", "neg_offset")


# ---- scenarios: deterministic uint8 I and Q of n samples ----------------------------------------------------------------
def _noise(rng, n, mean, sigma):
    return np.clip(np.rint(mean + sigma * rng.standard_normal(n)), 0, 255).astype(np.uint8)


def _dither(rng, n, mean):
    """Bytes floor(mean) or floor(mean) + 1 with the right odds: a DC of `mean` without noise."""
    lo = np.floor(mean)
    return (lo + (rng.random(n) < mean - lo)).astype(np.uint8)


def _slew(n, byte, length, then):
    """`length` samples of `byte` (the fastest way to a high binade), then the array `then`."""
    out = then.copy()
    out[:length] = byte
    return out


def _segments(n, seg, fn):
    """Concatenation of fn(k, length) over segments of `seg` samples."""
    parts, k, at = [], 0, 0
    while at < n:
        m = min(seg, n - at)
        parts.append(fn(k, m))
        k, at = k + 1, at + m
    return np.concatenate(parts)


def sc_full_scale(rng, n):
    """sigma = 45 around 127.5: both rails clip, the increments span the whole table."""
    return _noise(rng, n, 127.5, 45.0), _noise(rng, n, 127.5, 45.0)


def sc_pos_offset(rng, n):
    """Lock-in near +73 (binade 64..128) and near +58 (32..64) after a slew of 255s."""
    return (_slew(n, 255, 840_000, _noise(rng, n, 200.0, 3.0)), _slew(n, 255, 600_000, _noise(rng, n, 185.0, 2.0)))


def sc_neg_offset(rng, n):
    """Lock-in near -107 and near -67 after a slew of 0s."""
    return (_slew(n, 0, 1_850_000, _noise(rng, n, 20.0, 3.0)), _slew(n, 0, 1_000_000, _noise(rng, n, 60.0, 3.0)))


def sc_dither_pow2(rng, n):
    """DC a little above 1.0, then a little above 2.0 (I; the mirror image below zero on Q), dithered by +-0.03: the
    state sits on the power of two and changes binade about a hundred times, inside calls and between them."""
    t = np.arange(n)
    wobble = 0.03 * np.sin(t / 9000.0)
    i = np.where(t < 1_500_000, _dither(rng, n, 128.015 + wobble), _dither(rng, n, 129.02 + wobble))
    q = np.where(t < 1_200_000, _dither(rng, n, 125.985 - wobble), _dither(rng, n, 124.98 - wobble))
    i[:7_961] = 255; i[1_500_000:1_508_000] = 255                 # slews: 0 -> 1.0 and 1.0 -> 2.0
    q[:7_961] = 0; q[1_200_000:1_208_000] = 0
    return i, q


def sc_staircase(rng, n):
    """DC jumps every ~0.4 callbacks of 25E, off block and callback boundaries: +60, +3, -3 (sign change), -60, +0.5."""
    lv = [60.0, 3.0, -3.0, -60.0, 0.5]
    i = _segments(n, 153_637, lambda k, m: _noise(rng, m, 127.0 + lv[k % 5], 2.0))
    q = _segments(n, 149_999, lambda k, m: _noise(rng, m, 127.0 + lv[(k + 2) % 5], 1.0))
    return i, q


def sc_decay(rng, n):
    """Slew to ~+100 (and ~-88), then bytes of exactly 127: every threshold crossing is deterministic and straddles a
    block, so it is an integer solve."""
    return (_slew(n, 255, 1_520_000, np.full(n, 127, np.uint8)), _slew(n, 0, 1_200_000, np.full(n, 127, np.uint8)))


def sc_constant(rng, n):
    """sigma = 0: the state runs onto a lock-in fixed point (from below on I, which then sits exactly on T; from above
    on Q) and stays there: long runs of translations by D = 0."""
    return (_slew(n, 255, 500_000, np.full(n, 190, np.uint8)), _slew(n, 0, 1_100_000, np.full(n, 64, np.uint8)))


def excursion_blocks(n):
    """The DC blocks of sc_excursion that are one whole dip: every 29th after the slew."""
    b = np.arange(n // DC_BLK)
    return b[(b % 29 == 28) & (b * DC_BLK >= 400_000)]


def sc_excursion(rng, n):
    """A drifting state with, every 29th 128-sample block, a whole block of I = 0 / Q = 255: the largest dip towards
    zero one block can make, met at every depth of the window, its low margin included (checked in
    test_walk_paths_are_all_taken)."""
    i = _slew(n, 255, 400_000, _noise(rng, n, 147.0, 2.0))
    q = _slew(n, 0, 400_000, _noise(rng, n, 107.0, 2.0))
    hit = np.isin(np.arange(n) // DC_BLK, excursion_blocks(n))
    i[hit], q[hit] = 0, 255
    return i, q


def sc_near_zero(rng, n):
    """DC 127.02 / 126.98, sigma = 1: |state| stays below 2^-3, where the anchor is never ok."""
    return _noise(rng, n, 127.02, 1.0), _noise(rng, n, 126.98, 1.0)


def sc_square(rng, n):
    """Rail square wave 0/255 with a period of 37 samples, which does not divide 128."""
    t = np.arange(n)
    return (np.where(t % 37 < 18, 0, 255).astype(np.uint8), np.where((t + 11) % 37 < 19, 0, 255).astype(np.uint8))


SCENARIOS = {f.__name__[3:]: f for f in (sc_full_scale, sc_pos_offset, sc_neg_offset, sc_dither_pow2, sc_staircase,
                                         sc_decay, sc_constant, sc_excursion, sc_near_zero, sc_square)}


def make_streams(n):
    out = np.empty((len(SCENARIOS), 2 * n), np.uint8)
    for k, (name, fn) in enumerate(SCENARIOS.items()):
        i, q = fn(np.random.default_rng(1000 + k), n)
        out[k, 0::2], out[k, 1::2] = i, q
    return out


# ---- plans and runs -----------------------------------------------------------------------------------------------------
def dc_plan(tmp_dir, name):
    """A copy of a sample plan with correct_dc_bias=1."""
    with open(plan_path(name)) as f:
        lines = [x for x in f.read().splitlines() if not x.startswith("correct_dc_bias")]
    at = next(k for k, x in enumerate(lines) if x.startswith("sample_rate"))
    lines.insert(at + 1, "correct_dc_bias=1")
    path = os.path.join(tmp_dir, name + "_dc.ini")
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
    return path


def run_bank(plan, iq, splits, inputs=False, want_tap=False):
    """Process iq [streams, bytes] in calls of `splits` callbacks. Returns pcm, tap, the DC trace and mode bytes of every
    callback, and (inputs=True) the DC-corrected input of every callback."""
    import torch
    ns, row = iq.shape[0], plan.block * 2
    per = plan.block // DC_BLK
    bank = B.Bank(plan, ns, max(splits))
    pcm, tap, trace, modes, ins, b0 = [], [], [], [], [], 0
    for nb in splits:
        p, t = bank.process_numpy(iq[:, b0 * row:(b0 + nb) * row], nb, want_tap=want_tap)
        tr = torch.empty((ns, nb * per, 2), dtype=torch.float32, device="cuda")
        md = torch.empty((ns, nb * per), dtype=torch.uint8, device="cuda")
        bank.copy_dc_trace(nb, tr.data_ptr(), md.data_ptr())
        torch.cuda.synchronize()
        pcm.append(p); tap.append(t); trace.append(tr.cpu().numpy()); modes.append(md.cpu().numpy())
        if inputs:
            ins.append(np.stack([bank.read_input(cb, plan.block) for cb in range(nb)], axis=1))
        b0 += nb
    bank.close()
    cat = lambda xs: np.concatenate(xs, axis=1) if xs and xs[0] is not None else None
    return dict(pcm=cat(pcm), tap=cat(tap), trace=cat(trace), modes=cat(modes), inputs=cat(ins))


def run_bank_overlapped(plan, iq, splits):
    """The same through process_device_ex, every call queued back to back on one stream with an input-ready event, so
    that the DC pre-pass of call k + 1 (anchor, block statistics, walk) may run while call k is still filtering: the
    anchor and table are double-buffered by call parity. The DC trace of call k is gathered on the stream right after
    it; call k + 2, which reuses that buffer, is handed an input-ready event recorded after the gather, so the gather
    never races with it while call k + 1 still overlaps call k. Host reads happen after the last call."""
    import torch
    ns, row = iq.shape[0], plan.block * 2
    per = plan.block // DC_BLK
    bounds = np.cumsum([0] + list(splits))
    d_iq = [torch.from_numpy(np.ascontiguousarray(iq[:, a * row:b * row])).cuda() for a, b in zip(bounds, bounds[1:])]
    d_pcm = [torch.zeros((ns, nb, plan.pcm_per_block), dtype=torch.int16, device="cuda") for nb in splits]
    d_tr = [torch.empty((ns, nb * per, 2), dtype=torch.float32, device="cuda") for nb in splits]
    d_md = [torch.empty((ns, nb * per), dtype=torch.uint8, device="cuda") for nb in splits]
    torch.cuda.synchronize()
    bank = B.Bank(plan, ns, max(splits))
    st = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in splits]
    for e in ready[:2]:
        e.record(st)
    for k, nb in enumerate(splits):
        bank.process_device(d_iq[k].data_ptr(), nb * row, nb, d_pcm[k].data_ptr(), None, st.cuda_stream,
                            ready[k].cuda_event)
        bank.copy_dc_trace(nb, d_tr[k].data_ptr(), d_md[k].data_ptr(), st.cuda_stream)
        if k + 2 < len(splits):
            ready[k + 2].record(st)
    st.synchronize()
    torch.cuda.synchronize()
    out = dict(pcm=np.concatenate([x.cpu().numpy() for x in d_pcm], axis=1), tap=None,
               trace=np.concatenate([x.cpu().numpy() for x in d_tr], axis=1),
               modes=np.concatenate([x.cpu().numpy() for x in d_md], axis=1))
    bank.close()
    return out


class Case:
    def __init__(self, tmp_dir, key):
        ini, self.n_cb, self.split = PLANS[key]
        self.ini = dc_plan(tmp_dir, ini)
        self.op, self.plan = OP.build_plan(self.ini), B.Plan(self.ini)
        assert self.op["dc"] and self.plan.correct_dc and sum(self.split) == self.n_cb
        self.n = self.n_cb * self.plan.block
        assert self.n >= MIN_SAMPLES and self.plan.block % DC_BLK == 0
        self.iq = make_streams(self.n)
        self.main = run_bank(self.plan, self.iq, self.split, inputs=True, want_tap=True)


@pytest.fixture(scope="module", params=list(PLANS))
def case(request, tmp_path_factory):
    return Case(str(tmp_path_factory.mktemp("dcplans")), request.param)


def bits(x):
    return np.ascontiguousarray(x).view(np.uint32)


# ---- bit identity with the restatement ------------------------------------------------------------------------------------
def test_dc_trace_bit_identical(case):
    got = case.main["trace"]
    for k, name in enumerate(SCENARIOS):
        want = O.dc_trace(case.iq[k], DC_BLK).view(np.float32).reshape(-1, 2)
        bad = np.flatnonzero((bits(got[k]) != bits(want)).any(axis=1))
        assert bad.size == 0, (name, "first bad block", int(bad[0]), got[k][bad[0]], want[bad[0]],
                               "mode", int(case.main["modes"][k][bad[0]]))


def test_dc_corrected_input_bit_identical(case):
    got = case.main["inputs"]                                   # [stream, callback, sample]
    for k, name in enumerate(SCENARIOS):
        want = O.input_samples(case.iq[k], True).reshape(case.n_cb, -1)
        eq = bits(got[k].view(np.float32)) == bits(want.view(np.float32))
        assert eq.all(), (name, "callback, sample:", np.argwhere(~eq.reshape(case.n_cb, -1, 2).any(axis=2))[0])


@pytest.mark.parametrize("scenario", WHOLE_PLAN)
def test_whole_plan_outputs(case, scenario):
    """int16 within +-1 LSB (modulo 2^16: full-scale input can wrap int16 in both implementations -- the reference's
    (short) of a double, here __float2int_rz and truncation) and float tap within 1e-4 rel-L2 of the restatement."""
    k = list(SCENARIOS).index(scenario)
    orc = O.Oracle(case.op)
    orc.process(case.iq[k])
    gp, gt = B.split_pcm(case.plan, case.main["pcm"][k]), B.split_pcm(case.plan, case.main["tap"][k])
    for j, s in enumerate(case.op["subs"]):
        rp, rt = orc.pcm(j), orc.tap(j)
        assert rp.size == gp[s["topic"]].size
        d = (gp[s["topic"]].astype(np.int64) - rp.astype(np.int64)) % 65536
        assert np.minimum(d, 65536 - d).max() <= 1, (scenario, s["topic"])
        rel = np.linalg.norm(gt[s["topic"]] - rt) / np.linalg.norm(rt)
        assert rel <= 1e-4, (scenario, s["topic"], rel)
    orc.close()


# ---- invariance -----------------------------------------------------------------------------------------------------------
def same_bits(a, b, what):
    assert np.array_equal(bits(a["trace"]), bits(b["trace"])), what + ": DC trace"
    assert np.array_equal(a["pcm"], b["pcm"]), what + ": int16"
    if a["tap"] is not None and b["tap"] is not None:
        assert np.array_equal(bits(a["tap"]), bits(b["tap"])), what + ": tap"


def test_call_shape_does_not_matter(case):
    """One call, one callback per call, the irregular split, and the irregular split queued back to back through
    process_device_ex with input-ready events (each call's DC pre-pass free to overlap the previous call's filters):
    identical bits, DC trace included."""
    same_bits(case.main, run_bank(case.plan, case.iq, [case.n_cb], want_tap=True), "one call")
    same_bits(case.main, run_bank(case.plan, case.iq, [1] * case.n_cb, want_tap=True), "single-callback calls")
    same_bits(case.main, run_bank_overlapped(case.plan, case.iq, case.split), "process_device_ex, overlapped")


# ---- the scenarios do what they say --------------------------------------------------------------------------------------
# per arm: least max |state|, most max |state|, least number of sign changes, least number of binade changes
FACTS = {"pos_offset": [(64.0, 128.0, 0, 0), (32.0, 64.0, 0, 0)], "neg_offset": [(100.0, 128.0, 0, 0), (64.0, 128.0, 0, 0)],
         "dither_pow2": [(1.9, 2.1, 0, 50), (1.9, 2.1, 0, 50)], "staircase": [(2.0, 64.0, 2, 0), (2.0, 64.0, 2, 0)],
         "decay": [(64.0, 128.0, 0, 0), (64.0, 128.0, 0, 0)], "constant": [(32.0, 128.0, 0, 0), (32.0, 128.0, 0, 0)],
         "near_zero": [(0.0, 0.125, 0, 0), (0.0, 0.125, 0, 0)]}


@pytest.mark.parametrize("name", list(FACTS))
def test_scenario_reaches_its_regime(name):
    """From the restatement's per-sample trace: the state reaches the binades, sign changes and binade changes its
    scenario is written for, so that a change to a generator cannot quietly turn it into plain noise."""
    n = PLANS["25E"][1] * 384_000
    k = list(SCENARIOS).index(name)
    i, q = SCENARIOS[name](np.random.default_rng(1000 + k), n)
    iq = np.empty(2 * n, np.uint8)
    iq[0::2], iq[1::2] = i, q
    tr = O.dc_trace(iq, 1).view(np.float32).reshape(-1, 2)
    for arm, (lo, hi, signs, binades) in enumerate(FACTS[name]):
        s = tr[:, arm]
        peak = float(np.abs(s).max())
        n_sign = int((np.diff(np.signbit(s[1:]).astype(np.int8)) != 0).sum())
        n_bin = int((np.diff((np.abs(s[1:]).view(np.uint32) >> 23).astype(np.int32)) != 0).sum())
        assert lo <= peak < hi and n_sign >= signs and n_bin >= binades, (name, arm, peak, n_sign, n_bin)


# ---- which path each block took -------------------------------------------------------------------------------------------
def block_classes(iq_stream, split, block):
    """From the restatement's per-sample trace and the restated k0_dc_anchor of every call, per DC block and arm:
    `must_step` -- the anchor is not ok, the block starts outside the window (lo, hi), or one of its states reaches hi,
    leaves the anchor's binade or has the other sign: no translation or solve applies, the walk must step it in float;
    `solvable` -- all its states and the next block's start inside the window, some below T and some at or above it:
    the one-block integer solve (if not a run of 2 or 4) must take it, so it may not be stepped in float;
    `near_lo` -- the block starts inside the window within DC_BLK * qmax of lo, the margin the anchor keeps for one
    block's dip. (States below lo but in the binade are allowed in a translation below T: the margin covers them.)"""
    n = iq_stream.size // 2
    tr = O.dc_trace(iq_stream, 1).view(np.float32).reshape(-1, 2)
    nblk = n // DC_BLK
    per = block // DC_BLK
    must_step = np.zeros((nblk, 2), bool)
    solvable = np.zeros((nblk, 2), bool)
    near_lo = np.zeros((nblk, 2), bool)
    b0 = 0
    for nb in split:
        j0, j1 = b0 * per, (b0 + nb) * per
        for arm in range(2):
            A = anchor(tr[j0 * DC_BLK, arm])
            if not A["ok"]:
                must_step[j0:j1, arm] = True
                continue
            s = tr[j0 * DC_BLK:j1 * DC_BLK + 1, arm]                          # + the state after the call's last block
            m = np.abs(s).view(np.uint32).astype(np.int64)
            right = ((s < 0) == (A["sgn"] < 0)) & (s != 0)
            in_binade = right & ((m >> 23) == A["ef"])
            in_win = right & (m > A["lo"]) & (m < A["hi"])
            k = nb * per
            blk = lambda v: v[:k * DC_BLK].reshape(k, DC_BLK)
            nxt = np.append(in_win[DC_BLK::DC_BLK], in_win[-1])                # start of the next block
            must_step[j0:j1, arm] = ~in_win[:k * DC_BLK:DC_BLK] | ~blk(in_binade).all(1) | (blk(m) >= A["hi"]).any(1)
            above = blk(m) >= A["T"]
            solvable[j0:j1, arm] = blk(in_win).all(1) & nxt[:k] & above.any(1) & ~above.all(1)
            start = m[:k * DC_BLK:DC_BLK]
            near_lo[j0:j1, arm] = in_win[:k * DC_BLK:DC_BLK] & (start <= A["lo"] + DC_BLK * A["qmax"])
        b0 += nb
    if n % DC_BLK == 0 and nblk:
        solvable[-1] = False                                                  # its end state is not in the trace
    return must_step, solvable, near_lo


def test_walk_paths_are_all_taken(case):
    per = case.plan.block // DC_BLK
    last = per % BATCH                             # blocks in the ragged last batch of a callback (0: none)
    ragged = (np.arange(case.n // DC_BLK) % per >= per - last) if last else np.zeros(case.n // DC_BLK, bool)
    tot = dict(m1=0, m2=0, solves=0, ragged_solves=0)
    for k, name in enumerate(SCENARIOS):
        must_step, solvable, near_lo = block_classes(case.iq[k], case.split, case.plan.block)
        md = case.main["modes"][k]
        mode = np.stack([md & 15, md >> 4], axis=1)
        assert set(np.unique(mode)) <= {0, 1, 2}, name
        c = dict(m0=(mode == 0).mean(), m1=(mode == 1).mean(), m2=(mode == 2).mean(), solves=int(solvable.sum()),
                 ragged_solves=int((solvable & ragged[:, None]).sum()))
        print("DCMODES %7d Hz %-11s blocks %6d  mode0 %.4f  mode1 %.4f  mode2 %.4f  integer solves %6d (%d in a ragged "
              "last batch)" % (case.plan.fs, name, mode.size, c["m0"], c["m1"], c["m2"], c["solves"], c["ragged_solves"]))
        bad = np.argwhere(must_step & (mode != 2))
        assert bad.size == 0, (name, "block, arm", bad[0], "must be stepped, mode", int(mode[tuple(bad[0])]))
        bad = np.argwhere(solvable & (mode != 0))
        assert bad.size == 0, (name, "block, arm", bad[0], "must be solved, mode", int(mode[tuple(bad[0])]))
        if name in ("near_zero", "dither_pow2"):
            assert c["m2"] > 0.999, name                # no usable anchor / never inside a window
        else:
            assert c["m1"] > 0 and c["solves"] > 0, name
        if name == "excursion":                         # whole-block dips that start in the window's low margin
            dips = excursion_blocks(case.n)
            for arm in range(2):
                assert near_lo[dips, arm].any(), (name, arm)
        tot["m1"] += int((mode == 1).sum()); tot["m2"] += int((mode == 2).sum())
        tot["solves"] += c["solves"]; tot["ragged_solves"] += c["ragged_solves"]
    assert tot["m1"] > 0 and tot["m2"] > 0 and tot["solves"] > 0, tot
    if last:
        assert tot["ragged_solves"] > 0, tot
