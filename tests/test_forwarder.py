"""IQ forwarder (vfo::compress, vfo.cpp:389-424): a main VFO without sub VFOs re-publishes its
decimated IQ as packed bytes. None of the reference's sample plans uses it; plans/FWD_test.ini does.

CPU: the oracle's restatement is pinned to the UNMODIFIED reference (oracle/_ref driven headless; its
outputs stored as digests), and the product's plan compiler reads the main-VFO keys. GPU: the kernel is bit-exact on identical
input (including values whose int8 conversion wraps) and the bank's payloads match the oracle."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import plan_path
from oracle import oracle as O, plan as OP
from sdrreceiver_b200 import binding as B, synth

NAME = "FWD_test"


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def make_input(op, n_blocks):
    return synth.make_iq(op["Fs"], op["block"] * n_blocks, synth.carriers_for_plan(op["center"], op["subs"]), level=1.0)


def test_oracle_compress_is_the_reference():
    """The reference's run of this plan is stored as SHA-256 digests of its outputs and its wire frames
    (tests/golden/ref_runs.json, tools/make_golden.py runs)."""
    op = OP.build_plan(plan_path(NAME))
    iq = make_input(op, 3)
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_runs.json")) as f:
        ref = json.load(f)[NAME + "/3"]
    assert _sha(iq) == ref["input_sha256"], "synthetic input differs from the golden file's"
    frames = [(bytes.fromhex(t), r, n, p) for t, r, n, p in ref["frames"]]
    orc = O.Oracle(op, main_tap=True)
    orc.process(iq)
    assert len(ref["main_sha256"]) == len(op["mains"])
    for k, m in enumerate(op["mains"]):
        assert _sha(orc.main_tap(k)) == ref["main_sha256"][str(k)]
        if not m["topic"]:
            continue
        payload = O.compress(orc.main_tap(k), m["scalecomp"], 1)
        assert _sha(payload) == ref["pcm_sha256"][m["topic"]]
        # the wire: [5-byte topic][u32 rate = main out_rate][block_out bytes], one per callback
        mine = [f for f in frames if f[0] == m["topic"].encode()]
        assert len(mine) == 3 and all(f[1] == m["out_rate"] and f[2] == op["block"] >> m["decim"] and f[3] == 3 for f in mine)
        if m["topic"] == "IQ003":
            # main 3 runs at scale 1: the conversion to signed char wraps, and the oracle wraps like the reference
            assert np.unique(payload).size > 200
    assert "IQ003" in ref["pcm_sha256"]
    orc.close()


def test_compress_known_answers():
    x = np.array([0.0 + 0.0j, 0.999 - 0.999j, 0.1249 + 0.126j, -0.126 - 0.1249j, 1.0 + 0.5j, -1.0 - 0.5j, 2.5 - 3.0j],
                 dtype=np.complex64)
    got = O.compress(x, 1, 1)
    # (int)(v*128) & 0xF0 per arm: 127 -> 0x70, -127 -> 0x81 & 0xF0 = 0x80, 15 -> 0x00, 16 -> 0x10, -16 -> 0xF0,
    # -15 -> 0xF1 & 0xF0 = 0xF0, 128 -> wraps to -128 -> 0x80, 64 -> 0x40, -128 -> 0x80, -64 -> 0xC0,
    # 320 -> 0x140 -> 0x40, -384 -> 0x...E80 -> 0x80
    assert list(got) == [0x00, 0x78, 0x01, 0xFF, 0x84, 0x8C, 0x48]
    got8 = O.compress(x[:2], 1, 0)
    assert list(got8.view(np.int8)) == [0, 0, 127, -127]
    assert list(O.compress(np.array([8.0 + 4.0j], np.complex64), 16, 1)) == [0x42]


def test_plan_compiler_reads_the_forwarder_keys():
    op = OP.build_plan(plan_path(NAME))
    plan = B.Plan(plan_path(NAME))
    assert [m["n_subs"] for m in plan.mains] == [2, 0, 0]
    assert [m["forward"] for m in plan.mains] == [False, True, True]
    for pm, om in zip(plan.mains, op["mains"]):
        assert pm["topic"] == om["topic"] and pm["zmq_address"] == om["zmq_address"] and pm["scalecomp"] == om["scalecomp"]
        assert pm["cstyle"] == 1 and pm["fwd_bytes"] == op["block"] >> om["decim"]
    # from a description: same plan; a style other than 1 (0 = default 1) sends int8 I,Q pairs, twice the payload
    d = B.Plan.from_desc(plan.fs, plan.block, plan.bufsplit, plan.correct_dc,
                         [dict(m, cstyle=2) for m in plan.mains], plan.subs)
    assert [m["fwd_bytes"] for m in d.mains] == [2 * m["fwd_bytes"] for m in plan.mains]
    assert [m["forward"] for m in d.mains] == [False, True, True]


@pytest.mark.gpu
@pytest.mark.parametrize("scale,style", [(1, 1), (16, 1), (3, 1), (1, 0), (7, 2)])
@pytest.mark.parametrize("n", [1, 5, 4096, 100003])
def test_compress_kernel_bit_exact(scale, style, n):
    import torch
    rng = np.random.default_rng(n + scale)
    x = (rng.standard_normal((2, n, 2)) * rng.choice([0.05, 0.9, 4.0, 300.0], size=(2, n, 1))).astype(np.float32)
    x[0, 0] = [127.0 / 128, -1.0]
    d_x = torch.from_numpy(x).cuda()
    per = 1 if style == 1 else 2
    d_y = torch.zeros((2, n * per), dtype=torch.uint8, device="cuda")
    assert B.lib().sdrb_compress_iq(d_x.data_ptr(), d_y.data_ptr(), 2, n, scale, style, None) == 0
    got = d_y.cpu().numpy()
    for ch in range(2):
        want = O.compress(x[ch].view(np.complex64)[:, 0], scale, style)
        assert np.array_equal(got[ch], want)


@pytest.mark.gpu
def test_bank_forwarder_payloads_match_the_oracle():
    op = OP.build_plan(plan_path(NAME)); plan = B.Plan(plan_path(NAME))
    n_blocks = 3
    iq = np.stack([make_input(op, n_blocks), np.roll(make_input(op, n_blocks), 2 * 4321)])
    bank = B.Bank(plan, 2, n_blocks)
    pcm, tap = bank.process_numpy(iq, n_blocks, want_tap=True)
    fwd = {k: bank.read_forward(k, n_blocks) for k in (1, 2)}
    import torch
    main_gpu = {}
    for k in (1, 2):
        out = torch.empty((2, n_blocks * plan.mains[k]["block_out"], 2), dtype=torch.float32, device="cuda")
        bank.copy_main(k, n_blocks, out.data_ptr())
        torch.cuda.synchronize()
        main_gpu[k] = out.cpu().numpy().view(np.complex64)[..., 0]
    bank.close()
    for s in range(2):
        orc = O.Oracle(op, main_tap=True)
        orc.process(iq[s])
        gp = B.split_pcm(plan, pcm[s])
        for k, sub in enumerate(op["subs"]):                      # the USB side of the same plan still holds
            assert np.abs(gp[sub["topic"]].astype(np.int32) - orc.pcm(k).astype(np.int32)).max() <= 1
        for k in (1, 2):
            m = op["mains"][k]
            got = fwd[k][s].reshape(-1)
            # (a) exactly vfo::compress of the GPU's own main-VFO output
            assert np.array_equal(got, O.compress(main_gpu[k][s], m["scalecomp"], 1))
            # (b) against the oracle's bytes: the main outputs agree to ~1e-6, so a nibble can only differ
            # where a sample sits on a quantisation step -- by one step (mod 16), in a tiny fraction of bytes
            want = O.compress(orc.main_tap(k), m["scalecomp"], 1)
            assert got.size == want.size
            dre = ((got >> 4).astype(np.int32) - (want >> 4).astype(np.int32)) % 16
            dim = ((got & 15).astype(np.int32) - (want & 15).astype(np.int32)) % 16
            assert np.isin(dre, (0, 1, 15)).all() and np.isin(dim, (0, 1, 15)).all()
            assert np.mean(got != want) < 2e-3, np.mean(got != want)
        orc.close()
