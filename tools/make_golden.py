#!/usr/bin/env python
"""Generate tests/golden/* from the UNMODIFIED reference (oracle/_ref, needs /root/reference to
have been built). The fixtures let a box without oracle/_ref still pin the C restatement and
the CUDA path to reference outputs. Inputs are regenerated from sdrreceiver_b200.synth (seeded,
library-RNG free), so only outputs/digests are stored. `make_golden.py runs` writes only what
write_reference_runs() writes, from sdr_ref_i16 and sdr_ref_f32."""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from oracle import oracle as O, plan as OP  # noqa: E402
from sdrreceiver_b200 import synth  # noqa: E402

PLANS = ["25E", "98W", "54W_all", "54W_288K", "CBAND_143E"]
GOLD = os.path.join(ROOT, "tests", "golden")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def plan_input(name, n_blocks):
    op = OP.build_plan(os.path.join(ROOT, "plans", name + ".ini"))
    level = 0.5 if any(s["late"] for s in op["subs"]) else 1.0
    return op, synth.make_iq(op["Fs"], op["block"] * n_blocks, synth.carriers_for_plan(op["center"], op["subs"]), level=level)


def write_canaries(names=("25E", "54W_288K", "54W_all", "CBAND_143E")):
    for name in names:
        op, iq = plan_input(name, 1)
        outs, _, _ = O.run_ref(os.path.join(ROOT, "plans", name + ".ini"), iq)
        np.savez_compressed(os.path.join(GOLD, "canary_%s_1block.npz" % name),
                            input_sha256=np.frombuffer(hashlib.sha256(iq.tobytes()).digest(), np.uint8),
                            **{"pcm_" + k: v for k, v in outs.items()})


RUN_STRIDE = 257      # prime, so the sample does not lock onto a callback or half-band period


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def write_reference_runs():
    """Whole runs of the reference binaries alone (sdr_ref_i16 / sdr_ref_f32, no libref_prims.so needed):
    ref_runs.json  -- SHA-256 of every sub VFO's int16 and float tap (IQ forwarders: their payload bytes) and of every
                      main-VFO tap, and the wire frames, for the runs tests/test_oracle_vs_ref.py and
                      tests/test_forwarder.py hold the restatement to bit for bit;
    ref_<plan>_16blocks.npz -- every RUN_STRIDE-th int16 and float-tap sample of every sub VFO over 16 callbacks, what
                      tests/test_parity_gpu.py holds the CUDA path to."""
    runs = {}
    for name, n_blocks in [(p, 2) for p in PLANS] + [("25E", 16), ("CBAND_143E", 13), ("54W_all", 9), ("54W_288K", 12),
                                                     ("FWD_test", 3)]:
        op, iq = plan_input(name, n_blocks)
        ini = os.path.join(ROOT, "plans", name + ".ini")
        outs, frames, mains = O.run_ref(ini, iq, main_tap=True)
        taps, _, _ = O.run_ref(ini, iq, float_tap=True)
        runs["%s/%d" % (name, n_blocks)] = {
            "input_sha256": digest(iq),
            "pcm_sha256": {k: digest(v) for k, v in outs.items()},
            "tap_sha256": {k: digest(v) for k, v in taps.items()},
            "main_sha256": {str(k): digest(v) for k, v in mains.items()},
            "frames": [[t.hex(), r, n, p] for t, r, n, p in frames],
        }
    with open(os.path.join(GOLD, "ref_runs.json"), "w") as f:
        json.dump(runs, f, sort_keys=True, separators=(",", ":"))
    for name in ("25E", "CBAND_143E"):
        op, iq = plan_input(name, 16)
        ini = os.path.join(ROOT, "plans", name + ".ini")
        outs, _, _ = O.run_ref(ini, iq)
        taps, _, _ = O.run_ref(ini, iq, float_tap=True)
        np.savez_compressed(os.path.join(GOLD, "ref_%s_16blocks.npz" % name),
                            input_sha256=np.frombuffer(hashlib.sha256(iq.tobytes()).digest(), np.uint8),
                            stride=np.int64(RUN_STRIDE),
                            **{"pcm_" + k: v[::RUN_STRIDE].copy() for k, v in outs.items()},
                            **{"tap_" + k: v[::RUN_STRIDE].copy() for k, v in taps.items()},
                            **{"n_" + k: np.int64(v.size) for k, v in outs.items()})


def main():
    if sys.argv[1:] == ["runs"]:
        assert all(os.path.exists(os.path.join(O.REF_DIR, f)) for f in ("sdr_ref_i16", "sdr_ref_f32")), \
            "build oracle/_ref/sdr_ref_i16 and sdr_ref_f32 first (make -C oracle)"
        write_reference_runs()
        return
    assert O.have_ref(), "build oracle/_ref first (make -C oracle)"
    os.makedirs(GOLD, exist_ok=True)
    R = O.ref_prims()
    # ---- class-level known answers ----
    ka = {}
    for fs, f in ((1536000, 484000), (384000, 110854), (192000, -73244)):
        v = np.zeros(2 * (fs + 16), np.float32)
        R.ref_oscillator(fs, f, _p(v), fs + 16)
        v = v.view(np.complex64)
        ka["osc_%d_%d_head" % (fs, f)] = v[:16].copy()
        ka["osc_%d_%d_wrap" % (fs, f)] = v[fs - 8:fs + 16].copy()
        ka["osc_%d_%d_stride" % (fs, f)] = v[::4099].copy()
    rng = np.random.default_rng(20261017)
    x = rng.standard_normal(2 * 64 * 4).astype(np.float32)
    y = np.zeros(64 * 4, np.float32)
    R.ref_halfband(11, 64, _p(x), 64, 4, _p(y))
    ka["hb_in"], ka["hb_out"] = x, y
    for fs in (3000, 12000):
        pts = np.zeros(125, np.float32)
        R.ref_hilbert_points(125, fs, _p(pts))
        ka["hilbert_%d" % fs] = pts
    for key, args in (("lp_48k_10k", (2, 48000, 10000, 2500)), ("lp_dec5", (2, 60000, 6000, 3000)),
                      ("lp_dec6", (2, 288000, 24000, 9600)), ("lp_48k_3k", (2, 48000, 3000, 750))):
        t = np.zeros(512, np.float32)
        n = R.ref_low_pass(*args, _p(t), 512)
        ka[key] = t[:n].copy()
    u_in = rng.standard_normal(2 * 400).astype(np.float32)
    u = np.zeros(400, np.float32)
    R.ref_usb(125, 12000, _p(u_in), 400, _p(u))
    ka["usb_in"], ka["usb_out"] = u_in, u
    np.savez_compressed(os.path.join(GOLD, "known_answers.npz"), **ka)

    # ---- whole-plan: full int16 + float tap for the small plan, digests for the others ----
    op, iq = plan_input("54W_288K", 3)
    ini = os.path.join(ROOT, "plans", "54W_288K.ini")
    outs, frames, mains = O.run_ref(ini, iq, main_tap=True)
    taps, _, _ = O.run_ref(ini, iq, float_tap=True)
    np.savez_compressed(os.path.join(GOLD, "plan_54W_288K_3blocks.npz"),
                        **{"pcm_" + k: v for k, v in outs.items()},
                        **{"tap_" + k: v[::16].copy() for k, v in taps.items()},
                        main0=mains[0][::64].copy())
    dig = {}
    for name in PLANS:
        op, iq = plan_input(name, 2)
        ini = os.path.join(ROOT, "plans", name + ".ini")
        outs, frames, _ = O.run_ref(ini, iq)
        taps, _, _ = O.run_ref(ini, iq, float_tap=True)
        dig[name] = {
            "input_sha256": hashlib.sha256(iq.tobytes()).hexdigest(),
            "frames": [[t.decode("latin1"), r, n, p] for t, r, n, p in frames[:len(op["subs"])]],
            "pcm_sha256": {k: hashlib.sha256(v.tobytes()).hexdigest() for k, v in outs.items()},
            "tap_l2": {k: float(np.linalg.norm(v.astype(np.float64))) for k, v in taps.items()},
            "pcm_head": {k: v[:8].tolist() for k, v in outs.items()},
        }
    # ---- the bench's canaries: first callback of stream 0 of a plan from a reset receiver, full int16 (bench.py canary_check) ----
    write_canaries()
    write_reference_runs()
    with open(os.path.join(GOLD, "plan_digests.json"), "w") as f:
        json.dump(dig, f, indent=1, sort_keys=True)
    print("golden written to", GOLD)


if __name__ == "__main__":
    main()
