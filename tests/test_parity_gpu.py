"""Parity tests proper: the CUDA path, called through the C ABI (libsdrb200.so via ctypes),
against the oracle on the same seeded bytes. Criteria (BASELINE.json north_star):
  pre-quantisation float audio  rel-L2 <= 1e-4 per VFO
  int16 output                  within +-1 LSB
Integer-exactness is not claimed: the kernels use FMA and re-associated sums (~1e-7)."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import PLANS, level_for, plan_path
from oracle import oracle as O, plan as OP
from sdrreceiver_b200 import binding as B, synth

pytestmark = pytest.mark.gpu
TOL_REL_L2 = 1e-4
TOL_LSB = 1
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def make_input(op, n_blocks, stream=0):
    return synth.make_iq(op["Fs"], op["block"] * n_blocks, synth.carriers_for_plan(op["center"], op["subs"]),
                         stream=stream, level=level_for(op))


def run_gpu(plan, iq, splits, want_main=False):
    """iq [n_streams, bytes]; returns pcm, tap [n_streams, blocks, rec] (+ per-main cf32)."""
    import torch
    n_streams = iq.shape[0]
    bank = B.Bank(plan, n_streams, max(splits))
    row = plan.block * 2
    pcm, tap, mains, b0 = [], [], [[] for _ in plan.mains], 0
    for nb in splits:
        p, t = bank.process_numpy(iq[:, b0 * row:(b0 + nb) * row], nb, want_tap=True)
        pcm.append(p); tap.append(t)
        if want_main:
            for k, m in enumerate(plan.mains):
                out = torch.empty((n_streams, nb * m["block_out"], 2), dtype=torch.float32, device="cuda")
                bank.copy_main(k, nb, out.data_ptr())
                torch.cuda.synchronize()
                mains[k].append(out.cpu().numpy().view(np.complex64)[..., 0])
        b0 += nb
    bank.close()
    mains = [np.concatenate(m, axis=1) for m in mains] if want_main else None
    return np.concatenate(pcm, axis=1), np.concatenate(tap, axis=1), mains


def check_against_oracle(plan, op, iq_stream, pcm_s, tap_s, mains_s=None):
    orc = O.Oracle(op, main_tap=mains_s is not None)
    orc.process(iq_stream)
    gp, gt = B.split_pcm(plan, pcm_s), B.split_pcm(plan, tap_s)
    worst = 0.0
    for k, s in enumerate(op["subs"]):
        rp, rt = orc.pcm(k), orc.tap(k)
        assert rp.size == gp[s["topic"]].size
        rel = np.linalg.norm(gt[s["topic"]] - rt) / np.linalg.norm(rt)
        dl = np.abs(gp[s["topic"]].astype(np.int32) - rp.astype(np.int32)).max()
        assert rel <= TOL_REL_L2, (s["topic"], rel)
        assert dl <= TOL_LSB, (s["topic"], dl)
        worst = max(worst, rel)
    if mains_s is not None:
        for k in range(len(op["mains"])):
            r = orc.main_tap(k)
            assert np.linalg.norm(mains_s[k] - r) / np.linalg.norm(r) <= 1e-5
    orc.close()
    return worst


@pytest.mark.parametrize("name", PLANS)
def test_plan_parity_16_callbacks(name):
    """4 s of signal: crosses every NCO table wrap 4x and 15 callback edges per half-band stage;
    three process calls so the carried state (DC, tails, counters) is exercised too."""
    op = OP.build_plan(plan_path(name)); plan = B.Plan(plan_path(name))
    iq = make_input(op, 16)
    pcm, tap, mains = run_gpu(plan, iq[None, :], [6, 6, 4], want_main=True)
    check_against_oracle(plan, op, iq, pcm[0], tap[0], [m[0] for m in mains])


@pytest.mark.parametrize("name", ["25E", "CBAND_143E"])
def test_gpu_against_the_unmodified_reference_16_callbacks(name):
    """No restatement in between: the CUDA path against the reference's own translation units over 4 s of signal -- table
    wraps, DC approach and lock-in, 15 callback edges per half-band stage. The reference's int16 and float tap are stored
    in tests/golden/ref_<plan>_16blocks.npz as every `stride`-th sample of every sub VFO (tools/make_golden.py runs);
    the GPU's outputs are compared on those samples."""
    ini = plan_path(name)
    op = OP.build_plan(ini); plan = B.Plan(ini)
    iq = make_input(op, 16)
    g = np.load(os.path.join(GOLD, "ref_%s_16blocks.npz" % name))
    assert np.array_equal(np.frombuffer(hashlib.sha256(iq.tobytes()).digest(), np.uint8), g["input_sha256"])
    stride = int(g["stride"])
    pcm, tap, _ = run_gpu(plan, iq[None, :], [5, 4, 7])
    gp, gt = B.split_pcm(plan, pcm[0]), B.split_pcm(plan, tap[0])
    for s in op["subs"]:
        rp, rt = g["pcm_" + s["topic"]], g["tap_" + s["topic"]]
        assert int(g["n_" + s["topic"]]) == gp[s["topic"]].size
        got_p, got_t = gp[s["topic"]][::stride], gt[s["topic"]][::stride]
        assert got_p.size == rp.size and got_t.size == rt.size
        rel = np.linalg.norm(got_t - rt) / np.linalg.norm(rt)
        dl = np.abs(got_p.astype(np.int32) - rp.astype(np.int32)).max()
        assert rel <= TOL_REL_L2 and dl <= TOL_LSB, (s["topic"], rel, dl)


def test_split_invariance_bitwise():
    """How the callbacks are batched into calls must not change a single bit."""
    op = OP.build_plan(plan_path("25E")); plan = B.Plan(plan_path("25E"))
    iq = make_input(op, 6)[None, :]
    a = run_gpu(plan, iq, [6])
    b = run_gpu(plan, iq, [1] * 6)
    c = run_gpu(plan, iq, [2, 4])
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[0], c[0])
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[1], c[1])


def test_streams_are_independent_and_ragged_bank():
    op = OP.build_plan(plan_path("CBAND_143E")); plan = B.Plan(plan_path("CBAND_143E"))
    iq = np.stack([make_input(op, 3, stream=s) for s in range(3)])      # 3 streams: not a multiple of the host groups
    pcm, tap, _ = run_gpu(plan, iq, [2, 1])
    solo_pcm, solo_tap, _ = run_gpu(plan, iq[1:2], [3])
    assert np.array_equal(pcm[1], solo_pcm[0]) and np.array_equal(tap[1], solo_tap[0])
    for s in (0, 2):
        check_against_oracle(plan, op, iq[s], pcm[s], tap[s])


def test_reset_and_per_stream_reset():
    op = OP.build_plan(plan_path("54W_all")); plan = B.Plan(plan_path("54W_all"))
    iq = np.stack([make_input(op, 2, stream=s) for s in range(2)])
    bank = B.Bank(plan, 2, 2)
    first, _ = bank.process_numpy(iq, 2)
    assert bank.blocks_done(0) == 2
    cont, _ = bank.process_numpy(iq, 2)              # state carried: differs from a fresh start
    assert not np.array_equal(first, cont)
    bank.reset(1)                                    # only stream 1 starts over
    assert (bank.blocks_done(0), bank.blocks_done(1)) == (4, 0)
    mixed, _ = bank.process_numpy(iq, 2)
    assert np.array_equal(mixed[1], first[1]) and not np.array_equal(mixed[0], first[0])
    bank.reset()
    again, _ = bank.process_numpy(iq, 2)
    assert np.array_equal(again, first)
    bank.close()


def test_device_entry_point_equals_host_entry_point():
    import torch
    op = OP.build_plan(plan_path("54W_288K")); plan = B.Plan(plan_path("54W_288K"))
    iq = np.stack([make_input(op, 2, stream=s) for s in range(4)])
    pcm_h, tap_h, _ = run_gpu(plan, iq, [2])
    bank = B.Bank(plan, 4, 2)
    d_iq = torch.from_numpy(iq).cuda()
    d_pcm = torch.zeros((4, 2, plan.pcm_per_block), dtype=torch.int16, device="cuda")
    d_tap = torch.zeros((4, 2, plan.pcm_per_block), dtype=torch.float32, device="cuda")
    st = torch.cuda.Stream()
    bank.process_device(d_iq.data_ptr(), iq.shape[1], 2, d_pcm.data_ptr(), d_tap.data_ptr(), st.cuda_stream)
    st.synchronize()
    assert bank.last_launches >= 4
    assert np.array_equal(d_pcm.cpu().numpy(), pcm_h) and np.array_equal(d_tap.cpu().numpy(), tap_h)
    bank.close()


def test_overlapped_device_calls_with_input_ready_event():
    """sdrb_bank_process_device_ex: six back-to-back calls on a DC-removing plan, each handed an
    'input ready' event so that its DC pre-pass runs while the previous call is still filtering
    (double-buffered anchor/table). Must be bit-identical to the serialised calls, DC trace included."""
    import torch
    op = OP.build_plan(plan_path("25E")); plan = B.Plan(plan_path("25E"))
    n_streams, calls, nb = 3, 6, 2
    iq = np.stack([make_input(op, calls * nb, stream=s) for s in range(n_streams)])
    row = plan.block * 2 * nb
    d_iq = [torch.from_numpy(np.ascontiguousarray(iq[:, k * row:(k + 1) * row])).cuda() for k in range(calls)]
    n_dc = nb * plan.block // 128

    def run(overlap):
        bank = B.Bank(plan, n_streams, nb)
        st = torch.cuda.Stream()
        ready = torch.cuda.Event()
        ready.record(st)
        ready.synchronize()
        pcm = [torch.zeros((n_streams, nb, plan.pcm_per_block), dtype=torch.int16, device="cuda") for _ in range(calls)]
        trace = torch.zeros((n_streams, n_dc, 2), dtype=torch.float32, device="cuda")
        for k in range(calls):
            bank.process_device(d_iq[k].data_ptr(), row, nb, pcm[k].data_ptr(), None, st.cuda_stream,
                                ready.cuda_event if overlap else None)
        bank.copy_dc_trace(nb, trace.data_ptr(), None, st.cuda_stream)     # DC states of the last call
        st.synchronize()
        torch.cuda.synchronize()
        out = np.concatenate([p.cpu().numpy() for p in pcm], axis=1), trace.cpu().numpy()
        bank.close()
        return out

    pcm_a, tr_a = run(False)
    pcm_b, tr_b = run(True)
    assert np.array_equal(pcm_a, pcm_b)
    assert np.array_equal(tr_a.view(np.uint32), tr_b.view(np.uint32))
    pcm_h, _, _ = run_gpu(plan, iq, [nb] * calls)
    assert np.array_equal(pcm_a, pcm_h)


def test_async_host_calls_pipeline_bit_identical():
    """sdrb_bank_process_host_async: eight calls, up to three in flight (shared staging buffers ordered chunk by
    chunk), rotating host buffers -- bit-identical to the synchronous calls, tap included."""
    op = OP.build_plan(plan_path("25E")); plan = B.Plan(plan_path("25E"))
    n_streams, calls, nb = 5, 8, 2
    iq = np.stack([make_input(op, calls * nb, stream=s) for s in range(n_streams)])
    row = plan.block * 2 * nb
    pcm_s, tap_s, _ = run_gpu(plan, iq, [nb] * calls)
    bank = B.Bank(plan, n_streams, nb)
    depth = 3
    ins = [B.PinnedBuffer(n_streams * row) for _ in range(depth)]
    outs = [B.PinnedBuffer(n_streams * nb * plan.pcm_per_block * 2) for _ in range(depth)]
    taps = [B.PinnedBuffer(n_streams * nb * plan.pcm_per_block * 4) for _ in range(depth)]
    got_p, got_t = [], []

    def collect(k):
        got_p.append(outs[k % depth].view(np.int16).reshape(n_streams, nb, -1).copy())
        got_t.append(taps[k % depth].view(np.float32).reshape(n_streams, nb, -1).copy())

    for k in range(calls):
        if k >= depth:
            bank.host_wait(depth - 1)                        # call k-depth is complete: its buffers may be reused
            collect(k - depth)
        ins[k % depth].array.reshape(n_streams, row)[:] = iq[:, k * row:(k + 1) * row]
        bank.process_host_async(ins[k % depth].ptr, row, nb, outs[k % depth].ptr, taps[k % depth].ptr)
    bank.host_wait()
    for k in range(max(calls - depth, 0), calls):
        collect(k)
    assert np.array_equal(np.concatenate(got_p, axis=1), pcm_s)
    assert np.array_equal(np.concatenate(got_t, axis=1), tap_s)
    # a synchronous call right after asynchronous ones drains them first
    bank.process_host_async(ins[0].ptr, row, nb, outs[0].ptr, None)
    pcm2, _ = bank.process_numpy(iq[:, :row], nb)
    assert bank.blocks_done(0) == (calls + 2) * nb
    bank.close()
    for b in ins + outs + taps:
        b.close()


def test_argument_errors():
    plan = B.Plan(plan_path("54W_288K"))
    bank = B.Bank(plan, 1, 2)
    buf = np.zeros(plan.block * 2 * 3 + 16, np.uint8)
    out = np.zeros(3 * plan.pcm_per_block, np.int16)
    with pytest.raises(B.SdrbError, match="max_blocks"):
        bank.process_host(buf.ctypes.data_as(C.c_void_p), plan.block * 6, 3, out.ctypes.data_as(C.c_void_p))
    with pytest.raises(B.SdrbError, match="aligned"):
        bank.process_host(buf.ctypes.data + 1, plan.block * 4, 2, out.ctypes.data_as(C.c_void_p))
    with pytest.raises(B.SdrbError, match="bad argument"):
        bank.reset(5)
    bank.close()


def test_silence_in_silence_out():
    """Bytes of 127 are exactly zero after the (x-127) conversion: with DC correction off every
    output sample must be exactly 0 (and, with the start-up transient of the NCO tables,
    nothing may become NaN)."""
    plan = B.Plan(plan_path("54W_288K"))
    bank = B.Bank(plan, 2, 2)
    iq = np.full((2, plan.block * 2 * 2), 127, np.uint8)
    pcm, tap = bank.process_numpy(iq, 2, want_tap=True)
    assert not pcm.any() and not tap.any()
    bank.close()


def test_golden_vectors_from_the_reference():
    """Committed outputs of the unmodified reference (tools/make_golden.py)."""
    g = np.load(os.path.join(GOLD, "plan_54W_288K_3blocks.npz"))
    op = OP.build_plan(plan_path("54W_288K")); plan = B.Plan(plan_path("54W_288K"))
    iq = make_input(op, 3)
    pcm, tap, mains = run_gpu(plan, iq[None, :], [2, 1], want_main=True)
    gp, gt = B.split_pcm(plan, pcm[0]), B.split_pcm(plan, tap[0])
    for s in op["subs"]:
        assert np.abs(gp[s["topic"]].astype(np.int32) - g["pcm_" + s["topic"]].astype(np.int32)).max() <= TOL_LSB
        ref = g["tap_" + s["topic"]]
        assert np.linalg.norm(gt[s["topic"]][::16] - ref) / np.linalg.norm(ref) <= TOL_REL_L2
    assert np.linalg.norm(mains[0][0][::64] - g["main0"]) / np.linalg.norm(g["main0"]) <= 1e-5
    dig = json.load(open(os.path.join(GOLD, "plan_digests.json")))
    for name in ("25E", "CBAND_143E"):
        op = OP.build_plan(plan_path(name)); plan = B.Plan(plan_path(name))
        iq = make_input(op, 2)
        assert hashlib.sha256(iq.tobytes()).hexdigest() == dig[name]["input_sha256"]
        pcm, tap, _ = run_gpu(plan, iq[None, :], [2])
        gp, gt = B.split_pcm(plan, pcm[0]), B.split_pcm(plan, tap[0])
        for s in op["subs"]:
            head = np.array(dig[name]["pcm_head"][s["topic"]])
            assert np.abs(gp[s["topic"]][:8].astype(np.int32) - head).max() <= TOL_LSB
            l2 = float(np.linalg.norm(gt[s["topic"]].astype(np.float64)))
            assert abs(l2 - dig[name]["tap_l2"][s["topic"]]) <= 1e-4 * dig[name]["tap_l2"][s["topic"]]


def test_full_size_bank_properties():
    """BASELINE configuration per GPU: 128 streams x 25E x 4 callbacks. Too large for the oracle
    to walk completely in a unit test, so: (1) streams that carry identical bytes must produce
    identical outputs wherever they sit in the bank, (2) two spot-checked streams match the
    oracle, (3) a second run from reset reproduces the same digest."""
    op = OP.build_plan(plan_path("25E")); plan = B.Plan(plan_path("25E"))
    n_streams, nb = 128, 4
    base = [make_input(op, nb, stream=s) for s in range(2)]
    iq = np.empty((n_streams, base[0].size), np.uint8)
    for s in range(n_streams):
        iq[s] = np.roll(base[s % 2], 2 * 977 * (s // 2))
    iq[77] = base[0]; iq[126] = base[1]; iq[5] = base[1]
    bank = B.Bank(plan, n_streams, nb)
    pcm, tap = bank.process_numpy(iq, nb, want_tap=True)
    assert np.array_equal(pcm[0], pcm[77]) and np.array_equal(pcm[1], pcm[126]) and np.array_equal(pcm[1], pcm[5])
    check_against_oracle(plan, op, iq[77], pcm[77], tap[77])
    check_against_oracle(plan, op, iq[100], pcm[100], tap[100])
    d1 = hashlib.sha256(pcm.tobytes()).hexdigest()
    bank.reset()
    pcm2, _ = bank.process_numpy(iq, nb)
    assert hashlib.sha256(pcm2.tobytes()).hexdigest() == d1
    bank.close()


@pytest.mark.parametrize("dc,sigma,n_blocks,splits", [(127.5, 2.5, 12, [4, 4, 4]), (129.3, 2.5, 8, [3, 3, 2]),
                                                      (125.3, 4.0, 8, [4, 4]), (127.02, 1.0, 6, [2, 4]),
                                                      (134.9, 3.0, 6, [6])])
def test_dc_state_is_bit_identical(dc, sigma, n_blocks, splits):
    """The reference's float DC recursion locks onto a mantissa step of its rounded decay and
    ends up to 6 % away from the ideal low-pass value; the kernels must follow it bit for bit,
    whatever the DC level and however the callbacks are grouped into calls."""
    import torch
    op = OP.build_plan(plan_path("CBAND_143E")); plan = B.Plan(plan_path("CBAND_143E"))
    car = synth.carriers_for_plan(op["center"], op["subs"])
    iq = np.stack([synth.make_iq(op["Fs"], op["block"] * n_blocks, car, stream=s, sigma=sigma, dc=dc + 0.37 * s)
                   for s in range(2)])
    bank = B.Bank(plan, 2, max(splits))
    row, per = plan.block * 2, plan.block // 128
    got, b0 = [], 0
    for nb in splits:
        bank.process_numpy(iq[:, b0 * row:(b0 + nb) * row], nb)
        out = torch.empty((2, nb * per, 2), dtype=torch.float32, device="cuda")
        bank.copy_dc_trace(nb, out.data_ptr())
        torch.cuda.synchronize()
        got.append(out.cpu().numpy())
        b0 += nb
    got = np.concatenate(got, axis=1)
    for s in range(2):
        want = O.dc_trace(iq[s], 128).view(np.float32).reshape(-1, 2)
        assert np.array_equal(got[s].view(np.uint32), want.view(np.uint32)), (s, np.abs(got[s] - want).max())
    bank.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k1_threads,k2a_threads,extra", [(128, 64, {}), (96, 96, {"SDRB_K2A_V3": "0"}), (64, 128, {"SDRB_K1_BULK": "0"}),
                                                          (64, 64, {"SDRB_K2A_V3": "0", "SDRB_FUSE_LATE": "0", "SDRB_PER_CB": "1"}),
                                                          (64, 64, {}),
                                                          (64, 64, {"SDRB_LATE_GENERIC": "1"})])
def test_every_cta_size_of_the_cascade_kernels(k1_threads, k2a_threads, extra):
    """k1_v2 / k2a_v2 exist for 64-, 96- and 128-thread CTAs and the host picks one per launch
    (api.cu: v2_pick_threads). SDRB_K1_THREADS / SDRB_K2A_THREADS force a size: every instantiation
    must pass the same oracle comparison as the default (smoke(): 54W_288K and 25E, 1e-4 rel-L2, +-1 LSB).
    The other switches select the kernels the defaults replaced (k2a_v2 instead of k2a_v3, per-thread cp.async instead of
    the bulk-copy prefetch, unfused /late mixer, run-time tap count in the /late FIR, per-callback launches): they
    stay selectable for A/B measurements and must stay correct."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, SDRB_K1_THREADS=str(k1_threads), SDRB_K2A_THREADS=str(k2a_threads), **extra)
    r = subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], cwd=root, env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "smoke 25E: 27 sub VFOs" in r.stdout


@pytest.mark.gpu
def test_bench_line_on_the_gpu():
    """bench.py's B200 arm on a small bank: one JSON line with the keys the driver reads (value, e2e with the
    bytes it moved, gpu_launches > 0, clocks, roofline with achieved/peak/frac/traffic) and a digest."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "bench.py", "--steps", "3", "--warmup", "3", "--streams", "8", "--blocks", "2",
                        "--no-cpu-baseline"], cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    lines = [x for x in r.stdout.splitlines() if x.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["unit"] == "MS/s" and d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3 and d["dtype"] == "f32"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["gpu_launches"] > 0
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 8 * 2 * 384000 * 2 and d["e2e"]["d2h_bytes_per_step"] > 0
    rf = d["roofline"]
    # the binding axis of the dominant kernel class is reported as the headline, the other one beside it
    assert (rf["bound"], rf["unit"]) in (("fp32", "TFLOP/s"), ("hbm", "GB/s"))
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert rf["frac"] == max(rf["fp32"]["frac"], rf["hbm"]["frac"])
    assert rf["hbm"]["peak"] > 1000 and 25.0 < rf["fp32"]["peak_tflops"] < 90.0
    assert set(rf["per_class"]) >= {"dc_scan", "ingest_main", "sub_cascade", "usb_audio"}       # dc_scan is no longer hidden
    assert rf["longest_class_any_stream"] in rf["per_class"]
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    # parity verdict: canary against the reference's golden output, canary digest equal on every rank
    assert d["parity_ok"] is True and d["parity"]["canary_max_lsb_vs_reference"] <= 1 and d["parity"]["checked_against_golden"]
    assert d["digests"] and len(d["digests"][0]) == 7
    # the other BASELINE configurations ride along with short runs
    assert set(d["plans"]) == {"54W_288K", "54W_all", "CBAND_143E"} and all(v.get("value", 0) > 0 for v in d["plans"].values())
    assert d["plans"]["CBAND_143E"]["spectrum_feed_ms_per_step"] > 0
    assert d["e2e_zmq"]["value"] > 0 and d["e2e_zmq"]["messages_received"] > 0


@pytest.mark.gpu
def test_twenty_sub_vfos_on_one_main_vfo(tmp_path):
    """A plan the sample inis do not contain: 20 sub VFOs on ONE main VFO (the sub-VFO kernels take at most 16 per launch, so the
    parent's subs are split into a group of 16 and a group of 4, whose warps then own 8 streams each) with 5-, 4-, 3- and 2-stage
    cascades side by side, plus a second main VFO with a single sub. 3 ragged streams, 6 callbacks in two calls, DC removal on."""
    lines = ["sample_rate=1536000", "center_frequency=1545600000", "zmq_address=tcp://*:6003", "correct_dc_bias=1", "mix_offset=0", "",
             "[main_vfos]", "size=2", "1\\frequency=1545116000", "1\\out_rate=384000", "2\\frequency=1546096000", "2\\out_rate=192000", "",
             "[vfos]", "size=21"]
    rates = [600, 600, 1200, 600, 10500, 1200, 600, 600, 8400, 600, 1200, 600, 600, 10500, 600, 600, 1200, 600, 8400, 600]
    for k, dr in enumerate(rates):
        f = 1545116000 - 150000 + 15000 * k + 137 * k
        lines += ["%d\\frequency=%d" % (k + 1, f), "%d\\gain=5" % (k + 1), "%d\\data_rate=%d" % (k + 1, dr), "%d\\topic=V%02d" % (k + 1, k + 1)]
    lines += ["21\\frequency=1546096000", "21\\gain=3", "21\\data_rate=10500", "21\\topic=V21"]
    ini = tmp_path / "many.ini"
    ini.write_text("\n".join(lines) + "\n")
    op = OP.build_plan(str(ini)); plan = B.Plan(str(ini))
    assert sum(1 for s in op["subs"] if s["main"] == 0) == 20 and {s["decim"] for s in op["subs"]} == {2, 3, 4, 5}
    n_streams = 3
    iqs = np.stack([make_input(op, 6, stream=s) for s in range(n_streams)])
    pcm, tap, _ = run_gpu(plan, iqs, [4, 2])
    for s in range(n_streams):
        check_against_oracle(plan, op, iqs[s], pcm[s], tap[s], None)


@pytest.mark.gpu
def test_ten_seconds_in_uneven_calls():
    """40 callbacks (10 s of signal: every Oscillator table wraps ten times, the DC recursion spends seven seconds in its lock-in
    regime) handed over in calls of 1..4 callbacks in an irregular order -- the span geometry of the sub-VFO kernels, the DC
    double buffering and every carried tail change from call to call -- against the restatement over the whole run."""
    op = OP.build_plan(plan_path("25E")); plan = B.Plan(plan_path("25E"))
    splits = [1, 3, 4, 2, 4, 4, 1, 4, 2, 3, 4, 4, 1, 3]
    assert sum(splits) == 40
    iq = make_input(op, 40)
    pcm, tap, _ = run_gpu(plan, iq[None, :], splits)
    check_against_oracle(plan, op, iq, pcm[0], tap[0], None)
