"""What stream-list calls cost: device time per call (CUDA events, input resident in HBM) of a 128-receiver 25E bank for the
full-bank call, a shuffled list of all streams, lists of 64, 32 and 1, and a live-like schedule: every receiver's callbacks
arrive at its own random phase, and every 25 ms one call (n_blocks = 1) processes whoever is ready, through the synchronous host
call. For the schedule it prints the margin against real time (seconds of signal per second of wall clock).

    python tools/subset_time.py [--plan 25E] [--streams 128] [--blocks 4] [--reps 20] [--live-seconds 5]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from sdrreceiver_b200 import binding as B  # noqa: E402
from state_move_time import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--plan", default="25E")
    ap.add_argument("--streams", type=int, default=128)
    ap.add_argument("--blocks", type=int, default=4)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--live-seconds", type=float, default=5.0)
    ap.add_argument("--settle", type=int, default=8, help="full calls before timing: the DC recursion leaves its start-up path")
    a = ap.parse_args()
    import torch

    plan = B.Plan(os.path.join(ROOT, "plans", a.plan + ".ini"))
    ns, nb = a.streams, a.blocks
    bank = B.Bank(plan, ns, nb)
    rng = np.random.default_rng(1)
    row = nb * plan.block * 2
    # bench.py's input: a few synthesised streams (carriers at the plan's sub VFOs, noise, DC offset), the rest time-rotated copies
    from sdrreceiver_b200 import synth
    car = synth.carriers_for_plan(plan.center, plan.subs)
    base = [synth.make_iq(plan.fs, nb * plan.block, car, stream=s) for s in range(8)]
    iq = np.stack([np.roll(base[s % 8], 2 * 997 * (s // 8)) for s in range(ns)])
    d_iq = torch.from_numpy(iq).cuda()
    d_pcm = torch.empty((ns, nb, plan.pcm_per_block), dtype=torch.int16, device="cuda")
    st = torch.cuda.Stream()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def timed(streams):
        ms = []
        for r in range(a.reps + 3):                               # three warm-up calls
            ev[0].record(st)
            if streams is None:
                bank.process_device(d_iq.data_ptr(), row, nb, d_pcm.data_ptr(), None, st.cuda_stream)
            else:
                bank.process_streams_device(streams, d_iq.data_ptr(), row, nb, d_pcm.data_ptr(), None, st.cuda_stream)
            ev[1].record(st)
            st.synchronize()
            if r >= 3:
                ms.append(ev[0].elapsed_time(ev[1]))
        return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms))}

    for _ in range(a.settle):
        bank.process_device(d_iq.data_ptr(), row, nb, d_pcm.data_ptr(), None, st.cuda_stream)
    st.synchronize()
    res = {"gpu": gpu_info(), "plan": a.plan, "streams": ns, "n_blocks": nb, "reps": a.reps}
    perm = rng.permutation(ns).tolist()
    order = [("full_call", None), ("list_all_shuffled", perm)] + [("list_%d" % k, perm[:k]) for k in (64, 32, 1) if k <= ns]
    for _ in range(2):                                            # two alternating rounds: the spread between them is the noise
        for name, lst in order:
            res.setdefault(name, []).append(timed(lst))

    # live-like: callback period 1/bufsplit s, each receiver at its own phase; one host call every 25 ms for whoever is ready
    period, tick = 1.0 / plan.bufsplit, 0.025
    phase = rng.uniform(0, period, ns)
    rows = [iq[s, :plan.block * 2] for s in range(ns)]
    pinned = [B.PinnedBuffer(plan.block * 2) for _ in range(ns)]
    for p, r in zip(pinned, rows):
        p.array[:] = r
    n_ticks = int(a.live_seconds / tick)
    due = phase.copy()
    call_ms, listed = [], []
    t_wall = 0.0
    for k in range(n_ticks):
        now = (k + 1) * tick
        ready = [s for s in range(ns) if due[s] <= now]
        if not ready:
            continue
        due[ready] += period
        t0 = time.perf_counter()
        bank.process_streams_host(ready, [pinned[s].ptr for s in ready], 1)
        dt = time.perf_counter() - t0
        t_wall += dt
        call_ms.append(dt * 1e3); listed.append(len(ready))
    signal_s = n_ticks * tick
    res["live"] = {"tick_ms": tick * 1e3, "calls": len(call_ms), "mean_listed": float(np.mean(listed)),
                   "median_call_ms": float(np.median(call_ms)), "max_call_ms": float(np.max(call_ms)),
                   "busy_s": t_wall, "signal_s": signal_s, "x_real_time": signal_s / t_wall}
    for p in pinned:
        p.close()
    print(json.dumps(res, indent=1))
    bank.close()


if __name__ == "__main__":
    main()
