"""Receiver state records on the GPU (sdrb_bank_save_state / load_state / read_state / write_state): a receiver moved into
another bank of the same plan continues bit for bit as if it had never moved -- same kernels, same inputs, same state."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

from conftest import plan_path
from sdrreceiver_b200 import binding as B

pytestmark = pytest.mark.gpu
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
ALL_PLANS = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(ROOT, "plans", "*.ini")))


def make_inputs(plan, n_cb, lanes):
    """uint8 IQ [len(lanes), n_cb*block*2]: per lane a seeded noise floor, a carrier near every sub VFO and a DC offset."""
    n = plan.block * n_cb
    t = np.arange(n, dtype=np.float64) / plan.fs
    tone = np.zeros(n, np.complex128)
    for s in plan.subs[:8]:
        tone += 6.0 * np.exp(2j * np.pi * (s["freq"] + 1500.0 - plan.center if plan.center else -s["mixer"] + 1500.0) * t)
    out = np.empty((len(lanes), 2 * n), np.uint8)
    for k, lane in enumerate(lanes):
        rng = np.random.default_rng(1000 + int(lane))
        x = tone + rng.normal(0, 6, n) + 1j * rng.normal(0, 6, n) + complex(1.7 + 0.3 * lane, -2.1 + 0.2 * lane)
        out[k, 0::2] = np.clip(np.rint(127.5 + x.real), 0, 255)
        out[k, 1::2] = np.clip(np.rint(127.5 + x.imag), 0, 255)
    return out


def cut(iq, plan, b0, nb):
    row = plan.block * 2
    return np.ascontiguousarray(iq[:, b0 * row:(b0 + nb) * row])


def device_call(bank, iq, st, input_ready=None):
    """One sdrb_bank_process_device_ex call and everything it can be inspected by, as numpy."""
    import torch
    plan, ns = bank.plan, bank.n_streams
    nb = iq.shape[1] // (plan.block * 2)
    d_iq = torch.from_numpy(iq).cuda()
    d_pcm = torch.zeros((ns, nb, plan.pcm_per_block), dtype=torch.int16, device="cuda")
    d_tap = torch.zeros((ns, nb, plan.pcm_per_block), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    bank.process_device(d_iq.data_ptr(), iq.shape[1], nb, d_pcm.data_ptr(), d_tap.data_ptr(), st.cuda_stream, input_ready)
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


def assert_rows_equal(got, got_rows, want, want_rows, what):
    for key in want:
        a, b = got[key][got_rows], want[key][want_rows]
        assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), (what, key)


@pytest.fixture
def stream():
    import torch
    return torch.cuda.Stream()


def move_scenario(name, st, splits_a=(2, 1), splits_b=(2, 1), dirty=None, check=None):
    """Bank A (3 streams, max_blocks 3) runs splits_a; its streams [0, 1, 2] move into slots [4, 0, 2] of bank B (5 streams,
    max_blocks 5), which has already run one call of `dirty` callbacks of other data (default: as many as A ran, in fewer
    calls, so B's DC buffer parity differs from A's); B runs splits_b. R runs all calls uninterrupted, Bo is B without the
    load. check(got, got_rows, want, want_rows, what) compares (default: bit for bit)."""
    import torch
    check = check or assert_rows_equal
    plan = B.Plan(plan_path(name))
    n_a, n_b = sum(splits_a), sum(splits_b)
    dirty = n_a if dirty is None else dirty
    iq_a = make_inputs(plan, n_a + n_b, [0, 1, 2])
    iq_o = make_inputs(plan, dirty + n_b, [10, 11, 12, 13, 14])
    slots = [4, 0, 2]
    A, R = B.Bank(plan, 3, 3), B.Bank(plan, 3, 3)
    Bk, Bo = B.Bank(plan, 5, 5), B.Bank(plan, 5, 5)
    b0 = 0
    for nb in splits_a:
        device_call(A, cut(iq_a, plan, b0, nb), st)
        device_call(R, cut(iq_a, plan, b0, nb), st)
        b0 += nb
    for bank in (Bk, Bo):
        device_call(bank, cut(iq_o, plan, 0, dirty), st)
    rec = torch.empty((3, A.state_bytes), dtype=torch.uint8, device="cuda")
    A.save_state([0, 1, 2], rec.data_ptr(), st.cuda_stream)
    Bk.load_state(slots, rec.data_ptr(), st.cuda_stream)
    o0 = dirty
    for nb in splits_b:
        xb = cut(iq_o, plan, o0, nb)
        xb[slots] = cut(iq_a, plan, b0, nb)
        got, ref, own = device_call(Bk, xb, st), device_call(R, cut(iq_a, plan, b0, nb), st), device_call(Bo, xb, st)
        check(got, slots, ref, [0, 1, 2], (name, "moved", b0))
        check(got, [1, 3], own, [1, 3], (name, "untouched", b0))
        b0 += nb; o0 += nb
    for bank in (A, R, Bk, Bo):
        bank.close()


@pytest.mark.parametrize("name", ALL_PLANS)
def test_seamless_move(name, stream):
    """PCM, tap, every main VFO's output, forwarder bytes, DC trace and modes, blocks_done: all bit-identical to an
    uninterrupted run for the moved streams, and to B's own run for the streams the load did not list."""
    move_scenario(name, stream)


def test_seamless_move_per_callback_launches(stream, monkeypatch):
    monkeypatch.setenv("SDRB_PER_CB", "1")
    move_scenario("25E", stream)


def assert_rows_close(got, got_rows, want, want_rows, what):
    """Everything but the sub-VFO cascade's products bit for bit; audio within the parity criteria (+-1 LSB, rel-L2 1e-5)."""
    for key in want:
        a, b = got[key][got_rows], want[key][want_rows]
        if key == "pcm":
            assert np.abs(a.astype(np.int32) - b.astype(np.int32)).max() <= 1, (what, key)
        elif key == "tap":
            assert np.linalg.norm(a - b) <= 1e-5 * np.linalg.norm(b), (what, key)
        else:
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), (what, key)


@pytest.mark.parametrize("name", ["25E", "DEEP_1536"])
def test_move_into_bank_at_another_callback_count(name, stream):
    """k2a_v3 picks its table-anchored or its exact mixing path per warp, for all the streams the warp holds, and the two
    round differently: next to streams at another callback count a stream's audio may differ in the last bits, moved or
    not (as next to a stream reset with sdrb_bank_reset). The state itself moves exactly: main outputs, forwarder bytes,
    DC trace and counters stay bit-identical."""
    move_scenario(name, stream, dirty=1, check=assert_rows_close)


@pytest.mark.parametrize("split", [1, 13])
def test_dc_trace_across_split(split):
    """25E: moved while the DC recursion still steps (callback 1) and near its lock-in (callback 13), host records."""
    plan = B.Plan(plan_path("25E"))
    iq = make_inputs(plan, 16, [3])
    import torch
    st = torch.cuda.Stream()
    A, R, Bk = B.Bank(plan, 1, 16), B.Bank(plan, 1, 16), B.Bank(plan, 2, 16)
    device_call(A, cut(iq, plan, 0, split), st)
    device_call(R, cut(iq, plan, 0, split), st)
    device_call(Bk, np.concatenate([cut(make_inputs(plan, split, [9]), plan, 0, split)] * 2), st)   # dirty
    Bk.write_state([1], A.read_state([0]))
    x = np.concatenate([cut(make_inputs(plan, 16, [9]), plan, 0, 16 - split), cut(iq, plan, split, 16 - split)])
    got, ref = device_call(Bk, x, st), device_call(R, cut(iq, plan, split, 16 - split), st)
    assert_rows_equal(got, [1], ref, [0], split)
    for bank in (A, R, Bk):
        bank.close()


def test_process_device_ex_save_between_overlapping_calls():
    """Call n, a save and call n+1 (input_ready: its DC pre-pass may start at once) enqueued back to back without a host
    synchronise: the record is the one of a fully synchronised run, and call n+1 is unchanged."""
    import torch
    plan = B.Plan(plan_path("25E"))
    iq = make_inputs(plan, 4, [0, 1])
    st, side = torch.cuda.Stream(), torch.cuda.Stream()
    X, Y = B.Bank(plan, 2, 2), B.Bank(plan, 2, 2)
    d0 = torch.from_numpy(cut(iq, plan, 0, 2)).cuda()
    d1 = torch.from_numpy(cut(iq, plan, 2, 2)).cuda()
    pcm = [torch.zeros((2, 2, plan.pcm_per_block), dtype=torch.int16, device="cuda") for _ in range(2)]
    rec = torch.zeros((2, X.state_bytes), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ready = torch.cuda.Event()
    ready.record(side)
    X.process_device(d0.data_ptr(), d0.shape[1], 2, pcm[0].data_ptr(), None, st.cuda_stream, ready.cuda_event)
    X.save_state([1, 0], rec.data_ptr(), st.cuda_stream)
    X.process_device(d1.data_ptr(), d1.shape[1], 2, pcm[1].data_ptr(), None, st.cuda_stream, ready.cuda_event)
    st.synchronize()
    device_call(Y, cut(iq, plan, 0, 2), st)
    want = Y.read_state([1, 0])
    assert np.array_equal(rec.cpu().numpy(), want)
    y1 = device_call(Y, cut(iq, plan, 2, 2), st)
    assert np.array_equal(pcm[1].cpu().numpy(), y1["pcm"])
    X.close(); Y.close()


def test_host_paths():
    """process_host, process_host_async with calls still in flight when read_state runs, and write_state before host calls."""
    plan = B.Plan(plan_path("54W_288K"))
    iq = make_inputs(plan, 6, [0, 1])
    row = plan.block * 2
    R, A, Bk = B.Bank(plan, 2, 2), B.Bank(plan, 2, 2), B.Bank(plan, 3, 4)
    r = [R.process_numpy(cut(iq, plan, 2 * k, 2), 2, want_tap=True) for k in range(3)]
    pins = [B.PinnedBuffer(2 * 2 * row) for _ in range(2)]
    outs = [B.PinnedBuffer(2 * 2 * plan.pcm_per_block * 2) for _ in range(2)]
    for k in range(2):
        pins[k].array[:] = cut(iq, plan, 2 * k, 2).reshape(-1)
        A.process_host_async(pins[k].ptr, row * 2, 2, outs[k].ptr)
    rec = A.read_state([0, 1])                                    # both calls may still be in flight
    for k in range(2):
        assert np.array_equal(outs[k].view(np.int16).reshape(2, 2, -1), r[k][0])
    Bk.process_numpy(make_inputs(plan, 4, [7, 8, 9]), 4)          # A's callback count, the other DC parity
    Bk.write_state([2, 0], rec)
    x = np.concatenate([cut(iq, plan, 4, 2)[1:2], make_inputs(plan, 2, [5]), cut(iq, plan, 4, 2)[0:1]])
    pcm, tap = Bk.process_numpy(x, 2, want_tap=True)
    assert np.array_equal(pcm[[2, 0]], r[2][0]) and np.array_equal(tap[[2, 0]].view(np.uint32), r[2][1].view(np.uint32))
    for p in pins + outs:
        p.close()
    for bank in (R, A, Bk):
        bank.close()


def cf32_call(bank, x, nb):
    plan = bank.plan
    pcm = np.zeros((bank.n_streams, nb, plan.pcm_per_block), np.int16)
    x = np.ascontiguousarray(x, np.complex64)
    B._check(B.lib().sdrb_bank_process_cf32_host(bank.h, x.ctypes.data_as(C.c_void_p), x.shape[1], nb,
                                                  pcm.ctypes.data_as(C.c_void_p), None), "cf32")
    return pcm


def test_cf32_path_carries_cf_tail():
    plan = B.Plan(plan_path("54W_all"))
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((1, 4 * plan.block)) + 1j * rng.standard_normal((1, 4 * plan.block))).astype(np.complex64) * 20
    R, A, Bk = B.Bank(plan, 1, 2), B.Bank(plan, 1, 2), B.Bank(plan, 2, 2)
    cf32_call(R, x[:, :2 * plan.block], 2)
    want = cf32_call(R, x[:, 2 * plan.block:], 2)
    cf32_call(A, x[:, :2 * plan.block], 2)
    cf32_call(Bk, np.concatenate([x[:, 2 * plan.block:]] * 2), 2)
    Bk.write_state([1], A.read_state([0]))
    got = cf32_call(Bk, np.concatenate([x[:, :2 * plan.block], x[:, 2 * plan.block:]]), 2)
    assert np.array_equal(got[1], want[0])
    for bank in (R, A, Bk):
        bank.close()


@pytest.mark.parametrize("name", ALL_PLANS)
def test_layout_and_determinism(name):
    plan = B.Plan(plan_path(name))
    small, big = B.Bank(plan, 1, 1), B.Bank(plan, 4, 5)
    assert small.state_bytes == big.state_bytes and small.state_bytes % 16 == 0
    print("record %s: %d bytes" % (name, small.state_bytes))
    fresh = small.read_state([0])
    iq = make_inputs(plan, 2, [0, 1, 2, 3])
    big.process_numpy(iq, 2)
    a, b = big.read_state([0, 1, 2, 3]), big.read_state([0, 1, 2, 3])
    assert np.array_equal(a, b)                                   # two saves of one state
    hdr = a[0, :64].copy()
    assert hdr[:4].tobytes() == b"SBST" and int.from_bytes(hdr[8:16].tobytes(), "little") == big.state_bytes
    assert int.from_bytes(hdr[16:24].tobytes(), "little") == plan.fingerprint
    assert int.from_bytes(hdr[24:32].tobytes(), "little") == 2 and not hdr[44:].any()
    big.reset(1)
    assert np.array_equal(big.read_state([1]), fresh)           # reset == fresh
    big.write_state([2], fresh)                                  # loading a fresh record == reset
    assert np.array_equal(big.read_state([2]), fresh)
    pcm, tap = big.process_numpy(np.stack([iq[3], iq[3], iq[3], iq[3]]), 2, want_tap=True)
    assert np.array_equal(pcm[1], pcm[2]) and np.array_equal(tap[1].view(np.uint32), tap[2].view(np.uint32))
    small.close(); big.close()


def test_across_devices():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    plan = B.Plan(plan_path("25E"))
    iq = make_inputs(plan, 4, [0])
    R, A, Bk = B.Bank(plan, 1, 2, device=0), B.Bank(plan, 1, 2, device=0), B.Bank(plan, 1, 2, device=1)
    R.process_numpy(cut(iq, plan, 0, 2), 2)
    want = R.process_numpy(cut(iq, plan, 2, 2), 2, want_tap=True)
    A.process_numpy(cut(iq, plan, 0, 2), 2)
    Bk.write_state([0], A.read_state([0]))
    got = Bk.process_numpy(cut(iq, plan, 2, 2), 2, want_tap=True)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))
    for bank in (R, A, Bk):
        bank.close()


def refused(bank, fn, match):
    before = bank.read_state(list(range(bank.n_streams)))
    with pytest.raises(B.SdrbError, match=match):
        fn()
    assert np.array_equal(bank.read_state(list(range(bank.n_streams))), before)


def test_refusals():
    import torch
    plan = B.Plan(plan_path("25E"))
    other = B.Plan.from_desc(plan.fs, plan.block, plan.bufsplit, plan.correct_dc, plan.mains,
                             [dict(plan.subs[0], gain=plan.subs[0]["gain"] * 2)] + plan.subs[1:])
    bank, ob = B.Bank(plan, 3, 2), B.Bank(other, 1, 1)
    assert ob.state_bytes == bank.state_bytes
    bank.process_numpy(make_inputs(plan, 2, [0, 1, 2]), 2)
    good = bank.read_state([0, 1])
    refused(bank, lambda: bank.write_state([0], ob.read_state([0])), r"record 0 \(for stream 0\): plan fingerprint")
    for off, field in ((0, "magic"), (4, "version"), (8, "record_bytes")):
        bad = good.copy()
        bad[1, off] ^= 1
        refused(bank, lambda: bank.write_state([2, 0], bad), r"record 1 \(for stream 0\): %s" % field)   # one bad among good
        d = torch.from_numpy(bad).cuda()
        refused(bank, lambda: bank.load_state([2, 0], d.data_ptr()), r"record 1 \(for stream 0\): %s" % field)
    for streams, match in (([3], "outside"), ([-1], "outside"), ([1, 1], "listed twice"), ([], "n must be"),
                           ([0, 1, 2, 0], "n must be")):
        recs = np.zeros((max(len(streams), 1), bank.state_bytes), np.uint8)
        refused(bank, lambda: bank.write_state(streams, recs[:len(streams)]) if streams else
                B._check(B.lib().sdrb_bank_write_state(bank.h, recs.ctypes.data_as(C.c_void_p), 0,
                                                       recs.ctypes.data_as(C.c_void_p)), "write_state"), match)
    sentinel = torch.full((2, bank.state_bytes), 0xA5, dtype=torch.uint8, device="cuda")
    with pytest.raises(B.SdrbError, match="outside"):
        bank.save_state([0, 5], sentinel.data_ptr())
    torch.cuda.synchronize()
    assert bool((sentinel == 0xA5).all())
    s = (C.c_int32 * 1)(0)
    assert B.lib().sdrb_bank_read_state(bank.h, s, 1, None) == -1
    assert B.lib().sdrb_bank_load_state(bank.h, None, 1, sentinel.data_ptr(), None) == -1
    assert B.lib().sdrb_bank_save_state(None, s, 1, sentinel.data_ptr(), None) == -1
    bank.close(); ob.close()


def test_fused_late_setting_is_refused(monkeypatch):
    plan = B.Plan(plan_path("54W_all"))
    fused = B.Bank(plan, 1, 1)
    monkeypatch.setenv("SDRB_FUSE_LATE", "0")
    plain = B.Bank(plan, 1, 1)
    assert fused.state_bytes == plain.state_bytes
    refused(plain, lambda: plain.write_state([0], fused.read_state([0])), "record 0 .*flags")
    refused(fused, lambda: fused.write_state([0], plain.read_state([0])), "record 0 .*flags")
    fused.close(); plain.close()
