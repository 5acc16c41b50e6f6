"""Deep decimation on the GPU: main VFOs with 4..8 half-band stages (k1_v2 / k1_ingest_main run 3, k_hb_tail the rest),
sub VFOs with 6..8 (k2a_v3 / k2a_v2 run 5, k_hb_tail the rest) and sub VFOs on parents whose callback is not a multiple of
32 samples (k2a_v2's masked instantiation). The C restatement is the oracle, with the criteria of test_parity_gpu.py:
tap rel-L2 <= 1e-4 per VFO, int16 within +-1 LSB, main-VFO outputs rel-L2 <= 1e-5."""
import ctypes as C

import numpy as np
import pytest

from conftest import level_for, plan_path
from oracle import oracle as O, plan as OP
from sdrreceiver_b200 import binding as B, synth

pytestmark = pytest.mark.gpu
DEEP = ["DEEP_1536", "DEEP_1920", "DEEP_288K"]
TOL_REL_L2, TOL_LSB, TOL_MAIN = 1e-4, 1, 1e-5


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def load(name):
    return OP.build_plan(plan_path(name)), B.Plan(plan_path(name))


def make_input(op, n_blocks, stream=0):
    return synth.make_iq(op["Fs"], op["block"] * n_blocks, synth.carriers_for_plan(op["center"], op["subs"]),
                         stream=stream, level=level_for(op))


def deep_subs(plan):
    return [k for k, s in enumerate(plan.subs) if s["decim"] > 5]


def fwd_mains(plan):
    return [k for k, m in enumerate(plan.mains) if m["topic"]]


def run_device(plan, iq, splits, inspect=False):
    """Device-resident calls (sdrb_bank_process_device_ex) on one CUDA stream. Returns pcm, tap [n_streams, blocks, rec]
    and, with inspect, per main VFO its output, per forwarding main VFO its payload bytes and per deep sub VFO its z."""
    import torch
    ns, row = iq.shape[0], plan.block * 2
    bank = B.Bank(plan, ns, max(splits))
    st = torch.cuda.Stream()
    pcm, tap, b0 = [], [], 0
    mains = {k: [] for k in range(len(plan.mains))}
    fwd = {k: [] for k in fwd_mains(plan)}
    z = {k: [] for k in deep_subs(plan)}
    for nb in splits:
        d_iq = torch.from_numpy(np.ascontiguousarray(iq[:, b0 * row:(b0 + nb) * row])).cuda()
        d_pcm = torch.zeros((ns, nb, plan.pcm_per_block), dtype=torch.int16, device="cuda")
        d_tap = torch.zeros((ns, nb, plan.pcm_per_block), dtype=torch.float32, device="cuda")
        bank.process_device(d_iq.data_ptr(), nb * row, nb, d_pcm.data_ptr(), d_tap.data_ptr(), st.cuda_stream)
        if inspect:
            outs = {}
            for k, m in enumerate(plan.mains):
                outs[k] = torch.empty((ns, nb * m["block_out"], 2), dtype=torch.float32, device="cuda")
                bank.copy_main(k, nb, outs[k].data_ptr(), st.cuda_stream)
            fo = {}
            for k in fwd:
                fo[k] = torch.empty((ns, nb * plan.mains[k]["fwd_bytes"]), dtype=torch.uint8, device="cuda")
                bank.copy_forward(k, nb, fo[k].data_ptr(), st.cuda_stream)
            st.synchronize()
            for k in outs:
                mains[k].append(outs[k].cpu().numpy().view(np.complex64)[..., 0])
            for k in fo:
                fwd[k].append(fo[k].cpu().numpy())
            for k in z:
                z[k].append(bank.read_sub(k, nb))
        st.synchronize()
        pcm.append(d_pcm.cpu().numpy()); tap.append(d_tap.cpu().numpy())
        b0 += nb
    bank.close()
    cat = lambda d: {k: np.concatenate(v, axis=1) for k, v in d.items() if v}
    return np.concatenate(pcm, axis=1), np.concatenate(tap, axis=1), cat(mains), cat(fwd), cat(z)


def check_audio(plan, op, orc, pcm_s, tap_s):
    gp, gt = B.split_pcm(plan, pcm_s), B.split_pcm(plan, tap_s)
    for k, s in enumerate(op["subs"]):
        rp, rt = orc.pcm(k), orc.tap(k)
        assert rp.size == gp[s["topic"]].size
        rel = np.linalg.norm(gt[s["topic"]] - rt) / np.linalg.norm(rt)
        dl = np.abs(gp[s["topic"]].astype(np.int32) - rp.astype(np.int32)).max()
        assert rel <= TOL_REL_L2 and dl <= TOL_LSB, (s["topic"], rel, dl)


def sub_z_restated(op, orc, k):
    """vfo::decimate[decimateCount] of sub VFO k (vfo.cpp:237-251) from the restatement's parts: its Oscillator on the
    parent's output, then decimateCount half-band stages with the carried, one-slot-early history of each."""
    L = O.lib()
    s = op["subs"][k]
    parent = orc.main_tap(s["main"])
    n, spb = parent.size, s["samples_per_buffer"]
    osc = np.zeros(2 * n, np.float32)
    L.orc_oscillator(float(s["Fs"]), float(s["mixer"]), _p(osc), n)
    x = np.ascontiguousarray(osc.view(np.complex64) * parent)
    for a in range(s["decim"]):
        blk = spb >> a
        y = np.zeros(x.size // 2, np.complex64)
        L.orc_halfband(_p(x.view(np.float32)), blk, x.size // blk, _p(y.view(np.float32)))
        x = y
    return x


@pytest.mark.parametrize("name", DEEP)
def test_deep_plan_parity_16_callbacks(name):
    """16 callbacks in three calls: audio of every sub VFO, every main VFO's output, the forwarders' bytes and the z of the
    6..8-stage sub VFOs against the restatement."""
    op, plan = load(name)
    iq = make_input(op, 16)
    pcm, tap, mains, fwd, z = run_device(plan, iq[None, :], [6, 6, 4], inspect=True)
    orc = O.Oracle(op, main_tap=True)
    orc.process(iq)
    check_audio(plan, op, orc, pcm[0], tap[0])
    for k in range(len(op["mains"])):
        r = orc.main_tap(k)
        assert mains[k][0].size == r.size
        assert np.linalg.norm(mains[k][0] - r) / np.linalg.norm(r) <= TOL_MAIN, k
    for k, got in fwd.items():
        m = op["mains"][k]
        assert np.array_equal(got[0], O.compress(mains[k][0], m["scalecomp"], 1))      # vfo::compress of the GPU's output
        want = O.compress(orc.main_tap(k), m["scalecomp"], 1)                          # and of the restatement's, to a step
        assert got[0].size == want.size
        dre = ((got[0] >> 4).astype(np.int32) - (want >> 4).astype(np.int32)) % 16
        dim = ((got[0] & 15).astype(np.int32) - (want & 15).astype(np.int32)) % 16
        assert np.isin(dre, (0, 1, 15)).all() and np.isin(dim, (0, 1, 15)).all()
        assert np.mean(got[0] != want) < 2e-3
    for k, got in z.items():
        want = sub_z_restated(op, orc, k)
        assert got[0].size == want.size
        assert np.linalg.norm(got[0] - want) / np.linalg.norm(want) <= TOL_REL_L2, plan.subs[k]["topic"]
    orc.close()


def test_seven_and_eight_stage_sub_vfos_are_covered():
    _, plan = load("DEEP_1536")
    assert {plan.subs[k]["decim"] for k in deep_subs(plan)} == {7, 8}


@pytest.mark.parametrize("name", DEEP)
def test_deep_outputs_do_not_depend_on_call_shape_or_launch_order(name, monkeypatch):
    op, plan = load(name)
    iq = np.stack([make_input(op, 16, stream=s) for s in range(2)])
    ref = run_device(plan, iq, [16], inspect=True)
    for splits in ([1] * 16, [5, 4, 7]):
        got = run_device(plan, iq, splits, inspect=True)
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), splits
        for a, b in zip(got[2:], ref[2:]):
            assert all(np.array_equal(a[k], b[k]) for k in b), splits
    monkeypatch.setenv("SDRB_PER_CB", "1")                  # read when the bank is created
    got = run_device(plan, iq, [5, 4, 7])
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])


@pytest.mark.parametrize("name", DEEP)
def test_host_paths_equal_the_device_path(name):
    """process_host and process_host_async with two calls in flight, 3 streams (not a multiple of the host groups)."""
    op, plan = load(name)
    ns, nb, calls = 3, 2, 4
    iq = np.stack([make_input(op, nb * calls, stream=s) for s in range(ns)])
    pcm_d, tap_d = run_device(plan, iq, [nb] * calls)[:2]
    bank = B.Bank(plan, ns, nb)
    row = plan.block * 2 * nb
    got = [bank.process_numpy(iq[:, k * row:(k + 1) * row], nb, want_tap=True) for k in range(calls)]
    assert np.array_equal(np.concatenate([g[0] for g in got], axis=1), pcm_d)
    assert np.array_equal(np.concatenate([g[1] for g in got], axis=1), tap_d)
    bank.reset()
    depth = 2
    ins = [B.PinnedBuffer(ns * row) for _ in range(depth)]
    outs = [B.PinnedBuffer(ns * nb * plan.pcm_per_block * 2) for _ in range(depth)]
    taps = [B.PinnedBuffer(ns * nb * plan.pcm_per_block * 4) for _ in range(depth)]
    got_p, got_t = [], []

    def collect(k):
        got_p.append(outs[k % depth].view(np.int16).reshape(ns, nb, -1).copy())
        got_t.append(taps[k % depth].view(np.float32).reshape(ns, nb, -1).copy())

    for k in range(calls):
        if k >= depth:
            bank.host_wait(depth - 1)
            collect(k - depth)
        ins[k % depth].array.reshape(ns, row)[:] = iq[:, k * row:(k + 1) * row]
        bank.process_host_async(ins[k % depth].ptr, row, nb, outs[k % depth].ptr, taps[k % depth].ptr)
    bank.host_wait()
    for k in range(calls - depth, calls):
        collect(k)
    assert np.array_equal(np.concatenate(got_p, axis=1), pcm_d)
    assert np.array_equal(np.concatenate(got_t, axis=1), tap_d)
    bank.close()
    for b in ins + outs + taps:
        b.close()


def test_per_stream_reset_on_a_deep_plan():
    op, plan = load("DEEP_1920")
    iq = np.stack([make_input(op, 2, stream=s) for s in range(2)])
    bank = B.Bank(plan, 2, 2)
    first, _ = bank.process_numpy(iq, 2)
    cont, _ = bank.process_numpy(iq, 2)
    assert not np.array_equal(first, cont)
    bank.reset(1)
    mixed, _ = bank.process_numpy(iq, 2)
    assert np.array_equal(mixed[1], first[1]) and not np.array_equal(mixed[0], first[0])
    bank.reset()
    again, _ = bank.process_numpy(iq, 2)
    assert np.array_equal(again, first)
    bank.close()


def test_cf32_entry_point_on_deep_mains():
    """sdrb_bank_process_cf32_host (k1_ingest_main: 3 stages, then the tails) fed the restatement's DC-corrected samples."""
    import torch
    op, plan = load("DEEP_1536")
    nb, calls = 4, 2
    iq = make_input(op, nb * calls)
    x = O.input_samples(iq, op["dc"])
    orc = O.Oracle(op, main_tap=True)
    orc.process(iq)
    bank = B.Bank(plan, 1, nb)
    L = B.lib()
    mains = {k: [] for k in range(len(plan.mains))}
    pcm, tap = [], []
    for c in range(calls):
        xin = np.ascontiguousarray(x[c * nb * plan.block:(c + 1) * nb * plan.block])
        p = np.zeros((1, nb, plan.pcm_per_block), np.int16); t = np.zeros(p.shape, np.float32)
        assert L.sdrb_bank_process_cf32_host(bank.h, _p(xin.view(np.float32)), xin.size, nb, _p(p), _p(t)) == 0
        pcm.append(p); tap.append(t)
        for k, m in enumerate(plan.mains):
            out = torch.empty((1, nb * m["block_out"], 2), dtype=torch.float32, device="cuda")
            bank.copy_main(k, nb, out.data_ptr())
            torch.cuda.synchronize()
            mains[k].append(out.cpu().numpy().view(np.complex64)[0, :, 0])
    bank.close()
    for k in mains:
        got, r = np.concatenate(mains[k]), orc.main_tap(k)
        assert got.size == r.size and np.linalg.norm(got - r) / np.linalg.norm(r) <= TOL_MAIN, k
    check_audio(plan, op, orc, np.concatenate(pcm, axis=1)[0], np.concatenate(tap, axis=1)[0])
    orc.close()


def test_k2a_v2_runs_the_five_stage_subs_under_a_full_rate_parent(monkeypatch):
    monkeypatch.setenv("SDRB_K2A_V3", "0")
    op, plan = load("DEEP_1536")
    iq = make_input(op, 16)
    pcm, tap, _, _, z = run_device(plan, iq[None, :], [6, 6, 4], inspect=True)
    orc = O.Oracle(op, main_tap=True)
    orc.process(iq)
    check_audio(plan, op, orc, pcm[0], tap[0])
    for k, got in z.items():
        want = sub_z_restated(op, orc, k)
        assert np.linalg.norm(got[0] - want) / np.linalg.norm(want) <= TOL_REL_L2
    orc.close()
