"""Receivers that have run for hours, days or millennia, built in microseconds from shifted state records.

Every phase-dependent index of the hot path comes from one 64-bit counter per stream, blocks_done: the NCO table index of a
VFO is (blocks_done * samples per callback + i) mod L, L = (int) the VFO's input rate. The rest of the suite never takes that
counter past a few dozen callbacks; here it crosses the sample counts where index arithmetic typically breaks: 2^24 (a float
index loses integers), 2^31 (a 32-bit signed product overflows), 2^32 (unsigned 32-bit arithmetic wraps), 2^53 (a double
loses integers) and the largest counter a record may carry (include/sdrb200.h, SDRB_STATE_MAX_BLOCKS_DONE).

Shifting a counter by a multiple of the plan's period P changes no table index and no choice of k2a_v3's mixing path, so a
shifted receiver must produce the unshifted one's outputs bit for bit."""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import plan_path
from sdrreceiver_b200 import binding as B
from test_state_gpu import ALL_PLANS, cut, device_call, make_inputs, refused

pytestmark = pytest.mark.gpu

INT64_MIN, INT64_MAX = -2**63, 2**63 - 1
DONE_OFF, DC_OFF = 24, 32                       # header offsets of blocks_done (i64) and dc_state (2 x f32)
WARM, SPLITS = 3, (2, 1, 3)                     # callbacks before the records are read, then the calls both banks run


@pytest.fixture
def stream():
    import torch
    return torch.cuda.Stream()


def max_blocks_done(plan):
    return 2**62 // plan.block                  # SDRB_STATE_MAX_BLOCKS_DONE(block)


def period(plan):
    """Callbacks after which every NCO table index of the plan repeats: lcm over all VFOs of L / gcd(L, samples per
    callback), L = (int) the VFO's input rate = its Oscillator table length."""
    table_len = lambda kind, k: B.lib().sdrb_plan_copy_table(plan.h, kind, k, None, 0)
    vfos = [(int(plan.fs), plan.block, table_len(0, k)) for k in range(len(plan.mains))]
    vfos += [(int(s["Fs"]), plan.mains[s["main"]]["block_out"], table_len(1, k)) for k, s in enumerate(plan.subs)]
    p = 1
    for L, spc, n_table in vfos:
        assert n_table == L
        p = math.lcm(p, L // math.gcd(L, spc))
    assert plan.bufsplit % p == 0               # block * bufsplit = sample_rate: one second of signal is a whole period
    return p


def thresholds(plan):
    """(name, samples per callback at that rate, sample count to cross) for the six shifted streams."""
    deepest = min(plan.subs, key=lambda s: s["Fs"])                 # the sub VFO whose parent runs at the lowest rate
    sub_spc = plan.mains[deepest["main"]]["block_out"]
    out = [("2^24 in", plan.block, 2**24), ("2^31 in", plan.block, 2**31), ("2^32 in", plan.block, 2**32)]
    if sub_spc != plan.block:
        out.append(("2^31 at %d Hz" % deepest["Fs"], sub_spc, 2**31))
    else:                                       # the parent is not decimated: that count is the input's, take 2^40 instead
        out.append(("2^40 in", plan.block, 2**40))
    out.append(("2^53 in", plan.block, 2**53))
    return out


def shifted_counts(plan, P):
    """Per shifted stream its counter when the records are loaded, WARM + M * P, with the crossing inside the six callbacks
    both banks then run; the last stream starts at the largest counter a record may carry."""
    counts, names = [], []
    for name, spc, T in thresholds(plan):
        M = (2 * T - (2 * WARM + 1) * spc) // (2 * P * spc)         # T / spc - start in [1/2, P + 1/2)
        start = WARM + M * P
        assert M > 0 and start * spc < T < (start + sum(SPLITS)) * spc, (name, start)
        counts.append(start); names.append(name)
    top = WARM + (max_blocks_done(plan) - WARM) // P * P
    counts.append(top); names.append("max")
    assert len(set(counts)) == len(counts)
    return counts, names


def inspect_subs(bank, nb):
    """The z of every sub VFO with more than five half-band stages (vfo::decimate[decimateCount], sdrb_bank_read_sub)."""
    return {"z%d" % k: bank.read_sub(k, nb) for k, s in enumerate(bank.plan.subs) if s["decim"] > 5}


def call(bank, x, st, mode):
    """One call of nb callbacks through the device path or one of the host paths; everything it can be inspected by."""
    plan, ns = bank.plan, bank.n_streams
    nb = x.shape[1] // (plan.block * 2)
    if mode == "device":
        out = device_call(bank, x, st)
    elif mode == "host":
        pcm, tap = bank.process_numpy(x, nb, want_tap=True)
        out = {"pcm": pcm, "tap": tap}
    else:
        inp = B.PinnedBuffer(x.size)
        pcm = B.PinnedBuffer(ns * nb * plan.pcm_per_block * 2)
        tap = B.PinnedBuffer(ns * nb * plan.pcm_per_block * 4)
        inp.array[:] = x.reshape(-1)
        bank.process_host_async(inp.ptr, x.shape[1], nb, pcm.ptr, tap.ptr)
        bank.host_wait(0)
        out = {"pcm": pcm.view(np.int16).reshape(ns, nb, -1).copy(), "tap": tap.view(np.float32).reshape(ns, nb, -1).copy()}
        for p in (inp, pcm, tap):
            p.close()
    out.update(inspect_subs(bank, nb))
    out["blocks_done"] = np.array([bank.blocks_done(s) for s in range(ns)])
    return out


def shift_scenario(name, st, mode="device"):
    """Bank A (3 streams) runs WARM callbacks from reset, so the sample-0 path lies behind it. Its records, each loaded twice
    with its counter shifted by a different multiple of the period, become the six streams of bank S. A and S then run the
    same SPLITS calls; everything S produces must be A's, bit for bit, and S's counters the shifted ones plus the callbacks."""
    plan = B.Plan(plan_path(name))
    P = period(plan)
    counts, names = shifted_counts(plan, P)
    iq = make_inputs(plan, WARM + sum(SPLITS), [0, 1, 2])
    A = B.Bank(plan, 3, max(SPLITS))
    call(A, cut(iq, plan, 0, 1), st, mode)
    call(A, cut(iq, plan, 1, WARM - 1), st, mode)
    rows = [0, 1, 2, 0, 1, 2]                   # S's stream k continues A's stream rows[k]
    rec = A.read_state([0, 1, 2])[rows]
    rec[:, DONE_OFF:DONE_OFF + 8] = np.array(counts, "<i8").view(np.uint8).reshape(-1, 8)
    S = B.Bank(plan, len(rows), max(SPLITS))
    S.write_state(list(range(len(rows))), rec)
    b0 = WARM
    for nb in SPLITS:
        x = cut(iq, plan, b0, nb)
        want, got = call(A, x, st, mode), call(S, x[rows], st, mode)
        b0 += nb
        assert np.array_equal(want["blocks_done"], [b0] * 3)
        assert np.array_equal(got.pop("blocks_done"), np.array(counts) + (b0 - WARM)), (name, mode, b0)
        for key in want:
            if key != "blocks_done":
                a, b = got[key], want[key][rows]
                assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), (name, mode, b0, key)
    # the whole carried state agrees too, apart from the counter
    ra, rs = A.read_state([0, 1, 2])[rows], S.read_state(list(range(len(rows))))
    assert np.array_equal(np.delete(ra, np.s_[DONE_OFF:DONE_OFF + 8], axis=1), np.delete(rs, np.s_[DONE_OFF:DONE_OFF + 8], axis=1))
    A.close(); S.close()
    return P, counts, names


@pytest.mark.parametrize("name", ALL_PLANS)
def test_shifted_counters_continue_bit_for_bit(name, stream):
    P, counts, names = shift_scenario(name, stream)
    plan = B.Plan(plan_path(name))
    first, last = [c * plan.block for c in counts], [(c + sum(SPLITS)) * plan.block - 1 for c in counts]
    print("%s: P = %d; input samples crossed: %s" % (name, P, "; ".join(
        "%s [%d .. %d]" % (n, a, b) for n, a, b in zip(names, first, last))))


@pytest.mark.parametrize("mode", ["host", "host_async"])
def test_shifted_counters_host_paths(mode, stream):
    shift_scenario("25E", stream, mode)


def test_shifted_counters_per_callback_launches(stream, monkeypatch):
    monkeypatch.setenv("SDRB_PER_CB", "1")
    shift_scenario("25E", stream)


def with_header(records, k, done=None, dc=None):
    bad = records.copy()
    if done is not None:
        bad[k, DONE_OFF:DONE_OFF + 8] = np.array([done], "<i8").view(np.uint8)
    if dc is not None:
        bad[k, DC_OFF:DC_OFF + 8] = np.array(dc, "<f4").view(np.uint8)
    return bad


def bad_records(plan):
    top = max_blocks_done(plan)
    past = float(np.nextafter(np.float32(128.0), np.float32(np.inf)))
    for done in (-1, INT64_MIN, top + 1, INT64_MAX):
        yield dict(done=done), r"blocks_done is %d, this bank needs 0\.\.%d" % (done, top)
    for arm, a in (("I", 0), ("Q", 1)):
        for v in (np.nan, np.inf, -np.inf, past, -past):
            dc = [0.5, -0.5]
            dc[a] = v
            yield dict(dc=dc), r"dc_state %s is" % arm


def test_refuses_counters_and_dc_states_no_kernel_can_run(stream):
    """A record with a negative or too large counter, or a DC state the recursion cannot reach, is refused by write_state and
    load_state: the error names the record, the stream and the field, nothing of the batch is loaded, and the bank's next call
    is its untouched twin's."""
    import torch
    plan = B.Plan(plan_path("25E"))
    bank, twin, donor = (B.Bank(plan, 3, 2) for _ in range(3))
    iq, other = make_inputs(plan, 4, [0, 1, 2]), make_inputs(plan, 1, [5, 6, 7])
    for b in (bank, twin):
        call(b, cut(iq, plan, 0, 2), stream, "device")
    call(donor, other, stream, "device")
    good = donor.read_state([0, 1, 2])          # another state: had any record of the batch been loaded, the bank would show it
    n = 0
    for change, field in bad_records(plan):
        bad = with_header(good, 1, **change)
        match = r"record 1 \(for stream 0\): " + field + ".*nothing was loaded"
        refused(bank, lambda: bank.write_state([2, 0, 1], bad), "sdrb_bank_write_state: " + match)
        d = torch.from_numpy(bad).cuda()
        refused(bank, lambda: bank.load_state([2, 0, 1], d.data_ptr(), stream.cuda_stream), "sdrb_bank_load_state: " + match)
        n += 1
    assert n == 14
    x = cut(iq, plan, 2, 2)
    got, want = call(bank, x, stream, "device"), call(twin, x, stream, "device")
    for key in want:
        assert np.array_equal(got[key].view(np.uint8), want[key].view(np.uint8)), key
    for b in (bank, twin, donor):
        b.close()


def test_accepts_the_bounds_themselves():
    plan = B.Plan(plan_path("54W_288K"))
    bank = B.Bank(plan, 2, 1)
    edge = with_header(bank.read_state([0, 1]), 0, done=max_blocks_done(plan), dc=[-128.0, 128.0])
    edge = with_header(edge, 1, done=0, dc=[128.0, -128.0])
    bank.write_state([0, 1], edge)
    assert np.array_equal(bank.read_state([0, 1]), edge)
    assert bank.blocks_done(0) == max_blocks_done(plan)
    bank.close()


def test_nco_mix_at_large_sample_counts():
    """sdrb_nco_mix (Oscillator::tick indexing) with windows of 300 samples across 2^24, 2^31, 2^32, a table wrap beyond
    2^40 and just below 2^62, against table[(n0 + i) mod L] * x in float64 from the float32 operands. Per component the
    error may be that of one complex product with one fused multiply-add: 2^-22 |t| |x|."""
    import torch
    fs, f, n, n_ch = 1536000, -123457.0, 300, 2
    L = B.lib()
    tab = np.zeros(2 * fs, np.float32)
    assert L.sdrb_nco_table(float(fs), f, tab.ctypes.data_as(C.c_void_p), fs) == fs
    t = tab.view(np.complex64)
    k = 2**40 // fs + 1
    starts = [2**24 - 5, 2**31 - 100, 2**32 - 100, k * fs + (fs - 50), 2**62 - 1000]
    rng = np.random.default_rng(11)
    x = (rng.standard_normal((n_ch, n)) + 1j * rng.standard_normal((n_ch, n))).astype(np.complex64) * 50
    d_tab, d_x = torch.from_numpy(tab).cuda(), torch.from_numpy(x.view(np.float32).copy()).cuda()
    d_y = torch.empty_like(d_x)
    for n0 in starts:
        assert L.sdrb_nco_mix(d_tab.data_ptr(), fs, n0, d_x.data_ptr(), d_y.data_ptr(), n_ch, n, None) == 0
        got = d_y.cpu().numpy().view(np.complex64).astype(np.complex128)
        tt = t[(n0 + np.arange(n, dtype=np.int64)) % fs].astype(np.complex128)
        want = tt[None, :] * x.astype(np.complex128)
        bound = 2.0**-22 * np.abs(tt)[None, :] * np.abs(x)
        assert np.all(np.abs(got.real - want.real) <= bound) and np.all(np.abs(got.imag - want.imag) <= bound), n0
