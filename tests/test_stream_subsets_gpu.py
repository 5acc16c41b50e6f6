"""Stream-list calls (sdrb_bank_process_streams_device / _host): n_blocks callbacks for the listed receivers only, every other
receiver of the bank left exactly as it was. Live dongles do not deliver callbacks in lockstep; these calls let a server
process whoever has a callback ready."""
import ctypes as C

import numpy as np
import pytest

from conftest import plan_path
from sdrreceiver_b200 import binding as B
from test_state_gpu import ALL_PLANS, assert_rows_close, assert_rows_equal, cut, make_inputs

pytestmark = pytest.mark.gpu
SENT_PCM, SENT_TAP = -12345, -7.25


@pytest.fixture
def stream():
    import torch
    return torch.cuda.Stream()


def list_call(bank, streams, iq, st, input_ready=None, sync=True, bufs=None):
    """One stream-list call on device buffers of all n_streams rows (rows of unlisted streams hold a sentinel), and everything
    it can be inspected by, as numpy (rows = bank streams). streams=None: one sdrb_bank_process_device_ex call."""
    import torch
    plan, ns = bank.plan, bank.n_streams
    nb = iq.shape[1] // (plan.block * 2)
    d_iq = torch.from_numpy(iq).cuda()
    d_pcm = torch.full((ns, nb, plan.pcm_per_block), SENT_PCM, dtype=torch.int16, device="cuda")
    d_tap = torch.full((ns, nb, plan.pcm_per_block), SENT_TAP, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    if streams is None:
        bank.process_device(d_iq.data_ptr(), iq.shape[1], nb, d_pcm.data_ptr(), d_tap.data_ptr(), st.cuda_stream, input_ready)
    else:
        bank.process_streams_device(streams, d_iq.data_ptr(), iq.shape[1], nb, d_pcm.data_ptr(), d_tap.data_ptr(), st.cuda_stream,
                                    input_ready)
    out = {"pcm": d_pcm, "tap": d_tap}
    for k, m in enumerate(plan.mains):
        out["main%d" % k] = torch.empty((ns, nb * m["block_out"] * 2), dtype=torch.float32, device="cuda")
        bank.copy_main(k, nb, out["main%d" % k].data_ptr(), st.cuda_stream)
        if m["forward"]:
            out["fwd%d" % k] = torch.empty((ns, nb * m["fwd_bytes"]), dtype=torch.uint8, device="cuda")
            bank.copy_forward(k, nb, out["fwd%d" % k].data_ptr(), st.cuda_stream)
    if plan.correct_dc:
        n = nb * plan.block // 128
        out["dc"] = torch.empty((ns, n * 2), dtype=torch.float32, device="cuda")
        out["modes"] = torch.empty((ns, n), dtype=torch.uint8, device="cuda")
        bank.copy_dc_trace(nb, out["dc"].data_ptr(), out["modes"].data_ptr(), st.cuda_stream)
    st.synchronize()
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res["blocks_done"] = np.array([bank.blocks_done(s) for s in range(ns)])
    return res


def split_rounds(name, st, rounds=(2, 1, 2), lists=([3, 0], [1, 4, 2])):
    """Bank S runs every round as stream-list calls that together list each stream once; bank F runs one process_device call
    per round. Every output and the final records must be bit-identical."""
    plan = B.Plan(plan_path(name))
    iq = make_inputs(plan, sum(rounds), [0, 1, 2, 3, 4])
    S, F = B.Bank(plan, 5, max(rounds)), B.Bank(plan, 5, max(rounds))
    b0 = 0
    for nb in rounds:
        x = cut(iq, plan, b0, nb)
        want = list_call(F, None, x, st)
        for lst in lists:
            got = list_call(S, lst, x, st)
            assert_rows_equal(got, lst, want, lst, (name, b0, lst))
            unl = [s for s in range(5) if s not in lst]
            assert (got["pcm"][unl] == SENT_PCM).all() and (got["tap"][unl] == SENT_TAP).all(), (name, "unlisted rows written")
        b0 += nb
    assert np.array_equal(S.read_state(range(5)), F.read_state(range(5))), name
    S.close(); F.close()


@pytest.mark.parametrize("name", ALL_PLANS)
def test_split_rounds_equal_full_calls(name, stream):
    split_rounds(name, stream)


@pytest.mark.parametrize("env", ["SDRB_PER_CB", "SDRB_K2A_V3"])
def test_split_rounds_other_launch_paths(env, stream, monkeypatch):
    monkeypatch.setenv(env, "1" if env == "SDRB_PER_CB" else "0")
    split_rounds("25E", stream)


def schedule(n_streams, n_calls, seed):
    """Per call: (streams ready, n_blocks). Every stream skips 1, 2 and 3 consecutive calls at least once."""
    rng = np.random.default_rng(seed)
    skip = {s: set() for s in range(n_streams)}
    for s in range(n_streams):
        at = 1 + s % 2
        for gap in (1, 2, 3):
            skip[s].update(range(at, at + gap))
            at += gap + 1 + int(rng.integers(0, 2))
    calls = []
    for c in range(n_calls):
        ready = [s for s in rng.permutation(n_streams).tolist() if c not in skip[s]]
        if ready:                                   # a tick at which nobody is ready makes no call
            calls.append((ready, 1 + int(rng.integers(0, 2))))
    return calls


@pytest.mark.parametrize("name", ["25E", "CBAND_143E", "54W_all", "DEEP_1536"])
def test_staggered_schedule_matches_receivers_run_alone(name, stream):
    """Each stream gets its own callbacks at its own pace; it must match a one-stream bank fed the same callbacks: bit for bit
    except audio, audio within +-1 LSB (the sub-VFO cascade's path choice is per group of streams). The same schedule with two
    calls in flight (input_ready_event) gives identical results."""
    import torch
    plan = B.Plan(plan_path(name))
    ns, n_calls = 4, 14
    calls = schedule(ns, n_calls, 2)
    for s in range(ns):                             # gaps of 1, 2 and 3 calls in every stream's history
        hist = "".join("x" if s in r else "." for r, _ in calls)
        assert all(("x" + "." * g + "x") in hist for g in (1, 2, 3)), (s, hist)
    total = {s: sum(nb for r, nb in calls if s in r) for s in range(ns)}
    iq = make_inputs(plan, max(total.values()), list(range(ns)))
    S = B.Bank(plan, ns, 2)
    solo = [B.Bank(plan, 1, 2) for _ in range(ns)]
    pos = [0] * ns
    results = []
    for ready, nb in calls:
        x = np.zeros((ns, nb * plan.block * 2), np.uint8)
        for s in ready:
            x[s] = cut(iq[s:s + 1], plan, pos[s], nb)[0]
        got = list_call(S, ready, x, stream)
        results.append(got)
        for s in ready:
            want = list_call(solo[s], None, x[s:s + 1], stream)
            assert_rows_close(got, [s], want, [0], (name, s, pos[s]))
            pos[s] += nb
    for s in range(ns):
        assert S.blocks_done(s) == total[s]
        assert np.array_equal(S.read_state([s]), solo[s].read_state([0])), (name, s)
    # again, with every call's input landing on a copy stream and the DC pre-pass allowed to overlap the previous call
    T = B.Bank(plan, ns, 2)
    copy = torch.cuda.Stream()
    pos = [0] * ns
    held = []
    for c, (ready, nb) in enumerate(calls):
        x = np.zeros((ns, nb * plan.block * 2), np.uint8)
        for s in ready:
            x[s] = cut(iq[s:s + 1], plan, pos[s], nb)[0]
            pos[s] += nb
        h = torch.from_numpy(x).pin_memory()
        with torch.cuda.stream(copy):
            d_iq = torch.empty_like(h, device="cuda")
            d_iq.copy_(h, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy)
        d_pcm = torch.full((ns, nb, plan.pcm_per_block), SENT_PCM, dtype=torch.int16, device="cuda")
        d_tap = torch.full((ns, nb, plan.pcm_per_block), SENT_TAP, dtype=torch.float32, device="cuda")
        stream.wait_stream(torch.cuda.current_stream())
        T.process_streams_device(ready, d_iq.data_ptr(), x.shape[1], nb, d_pcm.data_ptr(), d_tap.data_ptr(), stream.cuda_stream,
                                 ev.cuda_event)
        held.append((h, d_iq, d_pcm, d_tap, ev))
    stream.synchronize()
    for c, (h, d_iq, d_pcm, d_tap, ev) in enumerate(held):
        assert np.array_equal(d_pcm.cpu().numpy(), results[c]["pcm"]), (name, "in flight", c)
        assert np.array_equal(d_tap.cpu().numpy().view(np.uint32), results[c]["tap"].view(np.uint32)), (name, "in flight", c)
    assert np.array_equal(T.read_state(range(ns)), S.read_state(range(ns))), name
    for b in [S, T] + solo:
        b.close()


@pytest.mark.parametrize("name", ["25E", "CBAND_143E", "DEEP_1536"])
def test_unlisted_receivers_are_untouched(name, stream):
    """Records of a skipped stream are byte-identical before and after 1, 2 and 3 skipped calls (odd gaps move the DC halo
    between the two table buffers), and its spectrum display does not change."""
    import torch
    plan = B.Plan(plan_path(name))
    ns = 3
    iq = make_inputs(plan, 16, [0, 1, 2])
    S = B.Bank(plan, ns, 2)
    list_call(S, None, cut(iq, plan, 0, 2), stream)
    sp = B.Spectrum(ns)
    pos, skip = 2, 2
    for gap in (1, 2, 3):
        before = S.read_state([skip])
        pwr0 = sp.read()
        for _ in range(gap):
            x = cut(iq, plan, pos, 1)
            got = list_call(S, [1, 0], x, stream)
            assert (got["pcm"][skip] == SENT_PCM).all() and (got["tap"][skip] == SENT_TAP).all()
            for src in (-1, 0):
                S.spectrum_feed(sp, src, 0, None, stream.cuda_stream)
            stream.synchronize()
            pos += 1
        after = sp.read()
        assert np.array_equal(S.read_state([skip]), before), (name, gap)
        for a, b in zip(pwr0, after):
            if a is not None and np.ndim(a) >= 2:
                assert np.array_equal(np.asarray(a)[skip], np.asarray(b)[skip]), (name, gap, "spectrum")
                assert not np.array_equal(np.asarray(a)[0], np.asarray(b)[0]), (name, gap, "listed display unchanged")
        x = cut(iq, plan, pos, 1)
        list_call(S, [skip], x, stream)              # the skipped stream resumes
        pos += 1
    sp.close(); S.close()


def test_host_call_matches_device_call(stream):
    """process_streams_host with pinned and pageable rows gives exactly the listed rows of the device call; it is ordered after
    a process_host_async still in flight and after a load_state."""
    import torch
    plan = B.Plan(plan_path("25E"))
    ns, lst = 5, [4, 1, 3]
    iq = make_inputs(plan, 6, list(range(ns)))
    D, H = B.Bank(plan, ns, 2), B.Bank(plan, ns, 2)
    # a full host call still in flight on H, the same call on D
    x0 = cut(iq, plan, 0, 2)
    inp = B.PinnedBuffer(x0.size); pcm = B.PinnedBuffer(ns * 2 * plan.pcm_per_block * 2)
    inp.array[:] = x0.reshape(-1)
    H.process_host_async(inp.ptr, x0.shape[1], 2, pcm.ptr, None)
    list_call(D, None, x0, stream)
    x = cut(iq, plan, 2, 2)
    pinned = [B.PinnedBuffer(x.shape[1]) for _ in lst]
    for p, s in zip(pinned, lst):
        p.array[:] = x[s]
    got_p, tap_p = H.process_streams_host(lst, [p.ptr for p in pinned], 2, want_tap=True)
    want = list_call(D, lst, x, stream)
    assert np.array_equal(got_p, want["pcm"][lst]) and np.array_equal(tap_p.view(np.uint32), want["tap"][lst].view(np.uint32))
    x = cut(iq, plan, 4, 1)
    got, tap = H.process_streams_host(lst, [x[s].copy() for s in lst], 1, want_tap=True)     # pageable rows
    want = list_call(D, lst, x, stream)
    assert np.array_equal(got, want["pcm"][lst]) and np.array_equal(tap.view(np.uint32), want["tap"][lst].view(np.uint32))
    # after a load_state: H's stream 0 takes D's stream 4, then one more call lists it
    rec = torch.empty((1, D.state_bytes), dtype=torch.uint8, device="cuda")
    D.save_state([4], rec.data_ptr(), stream.cuda_stream)
    H.load_state([0], rec.data_ptr(), stream.cuda_stream)
    x = cut(iq, plan, 5, 1)
    got, _ = H.process_streams_host([0], [x[4].copy()], 1)
    want = list_call(D, [4], x, stream)
    assert np.array_equal(got[0], want["pcm"][4])
    for p in pinned + [inp, pcm]:
        p.close()
    D.close(); H.close()


def test_refusals_leave_the_bank_unchanged(stream):
    import torch
    plan = B.Plan(plan_path("25E"))
    ns = 4
    bank = B.Bank(plan, ns, 2)
    iq = make_inputs(plan, 2, list(range(ns)))
    list_call(bank, None, cut(iq, plan, 0, 1), stream)
    rec0 = bank.read_state(range(ns))
    x = cut(iq, plan, 1, 1)
    d_iq = torch.from_numpy(x).cuda()
    d_pcm = torch.zeros((ns, 1, plan.pcm_per_block), dtype=torch.int16, device="cuda")
    L = B.lib()
    cases = [([], "n must be 1..n_streams"), ([0, 1, 2, 3, 0], "n must be 1..n_streams"), ([1, 2, 1], "streams[2] = 1 is listed twice"),
             ([0, -1], "streams[1] = -1 is outside"), ([3, 4], "streams[1] = 4 is outside")]
    for lst, what in cases:
        s = np.array(lst, dtype=np.int32)
        sp = s.ctypes.data_as(C.c_void_p)
        rc = L.sdrb_bank_process_streams_device(bank.h, sp, s.size, d_iq.data_ptr(), x.shape[1], 1, d_pcm.data_ptr(), None,
                                                stream.cuda_stream, None)
        assert rc == -1 and what in L.sdrb_last_error().decode(), (lst, L.sdrb_last_error())
        rows = (C.c_void_p * max(s.size, 1))(*([x[0].ctypes.data] * max(s.size, 1)))
        pcm = np.zeros((max(s.size, 1), 1, plan.pcm_per_block), np.int16)
        rc = L.sdrb_bank_process_streams_host(bank.h, sp, s.size, C.cast(rows, C.c_void_p), 1, pcm.ctypes.data_as(C.c_void_p), None)
        assert rc == -1 and what in L.sdrb_last_error().decode(), (lst, L.sdrb_last_error())
    s = np.array([0, 1], dtype=np.int32)
    sp = s.ctypes.data_as(C.c_void_p)
    assert L.sdrb_bank_process_streams_device(bank.h, None, 2, d_iq.data_ptr(), x.shape[1], 1, d_pcm.data_ptr(), None, None, None) == -1
    assert L.sdrb_bank_process_streams_device(bank.h, sp, 2, None, x.shape[1], 1, d_pcm.data_ptr(), None, None, None) == -1
    assert L.sdrb_bank_process_streams_device(bank.h, sp, 2, d_iq.data_ptr(), x.shape[1], 1, None, None, None, None) == -1
    assert L.sdrb_bank_process_streams_device(None, sp, 2, d_iq.data_ptr(), x.shape[1], 1, d_pcm.data_ptr(), None, None, None) == -1
    rows = (C.c_void_p * 2)(x[0].ctypes.data, None)
    pcm = np.zeros((2, 1, plan.pcm_per_block), np.int16)
    assert L.sdrb_bank_process_streams_host(bank.h, sp, 2, C.cast(rows, C.c_void_p), 1, pcm.ctypes.data_as(C.c_void_p), None) == -1
    assert "h_iq[1] is NULL" in L.sdrb_last_error().decode()
    assert L.sdrb_bank_process_streams_host(bank.h, sp, 2, None, 1, pcm.ctypes.data_as(C.c_void_p), None) == -1
    assert L.sdrb_bank_process_streams_host(bank.h, sp, 2, C.cast(rows, C.c_void_p), 1, None, None) == -1
    torch.cuda.synchronize()
    assert [bank.blocks_done(s) for s in range(ns)] == [1] * ns
    assert np.array_equal(bank.read_state(range(ns)), rec0)
    bank.close()
