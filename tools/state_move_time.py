"""What moving receivers costs: time to save every receiver of a bank into state records and load them into another bank,
with CUDA events (device-resident records) and with a host clock (host records, read_state / write_state). Also prints
the record size of every plan in plans/.

    python tools/state_move_time.py [--plan 25E] [--streams 128] [--max-blocks 4] [--reps 20]
"""
import argparse
import glob
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from sdrreceiver_b200 import binding as B  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--plan", default="25E")
    ap.add_argument("--streams", type=int, default=128)
    ap.add_argument("--max-blocks", type=int, default=4)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    import torch

    sizes = {}
    for p in sorted(glob.glob(os.path.join(ROOT, "plans", "*.ini"))):
        bank = B.Bank(B.Plan(p), 1, 1)
        sizes[os.path.basename(p)[:-4]] = bank.state_bytes
        bank.close()

    plan = B.Plan(os.path.join(ROOT, "plans", a.plan + ".ini"))
    ns, nb = a.streams, a.max_blocks
    src, dst = B.Bank(plan, ns, nb), B.Bank(plan, ns, nb)
    rng = np.random.default_rng(1)
    iq = rng.integers(100, 156, size=(ns, nb * plan.block * 2), dtype=np.uint8)
    src.process_numpy(iq, nb)                                   # a receiver state that is not the reset one
    streams = list(range(ns))
    rec = torch.empty((ns, src.state_bytes), dtype=torch.uint8, device="cuda")
    st = torch.cuda.Stream()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    save_ms, load_ms, pair_ms = [], [], []
    for r in range(a.reps + 2):                                 # two warm-up rounds
        t0 = time.perf_counter()
        e[0].record(st)
        src.save_state(streams, rec.data_ptr(), st.cuda_stream)
        e[1].record(st)
        dst.load_state(streams, rec.data_ptr(), st.cuda_stream)   # synchronises st to check the headers
        e[2].record(st)
        st.synchronize()
        t1 = time.perf_counter()
        if r >= 2:
            save_ms.append(e[0].elapsed_time(e[1])); load_ms.append(e[1].elapsed_time(e[2])); pair_ms.append((t1 - t0) * 1e3)
    host_ms = []
    for r in range(max(3, a.reps // 4) + 1):
        t0 = time.perf_counter()
        dst.write_state(streams, src.read_state(streams))
        if r >= 1:
            host_ms.append((time.perf_counter() - t0) * 1e3)
    assert np.array_equal(dst.read_state(streams), src.read_state(streams))
    med = lambda v: float(np.median(v))
    print(json.dumps({
        "gpu": gpu_info(), "plan": a.plan, "streams": ns, "max_blocks": nb, "record_bytes": src.state_bytes,
        "device_save_ms": med(save_ms), "device_load_ms": med(load_ms), "device_save_load_wall_ms": med(pair_ms),
        "host_read_write_wall_ms": med(host_ms), "record_bytes_per_plan": sizes}, indent=1))
    src.close(); dst.close()


if __name__ == "__main__":
    main()
