"""k2a_v3's warp body executed on the CPU (tests/cpp/k3_sim.cu: the same __host__ __device__ template the
kernel instantiates, 32 host threads per warp) against a plain restatement of vfo::process's front end
(vfo.cpp:237-251, halfbanddecimator.cpp:43-72, dsp.cpp:163-173): table wrap, start-up transient, stream
sample 0, callback heads, ragged stream groups, several spans per callback, state carried over three calls, and streams that
start at large or mixed callback counts.

Per VFO the simulation asserts rel-L2 <= 2e-6 and a worst sample error |d| <= 9e-6 x the RMS of the reference output. On the
first eight geometries below the worst sample is 1.3e-6 .. 2.2e-6 x RMS (2.19e-6 for 4-2-7-16 and 4-2-3-15), so the bound is
4x the measured worst; a wrong table index or a wrong start-up sample is off by O(1) x RMS."""
import os
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, ".."))
EXE = os.path.join(HERE, "cpp", "k3_sim")


@pytest.fixture(scope="module")
def sim(built):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    src = os.path.join(HERE, "cpp", "k3_sim.cu")
    hdr = os.path.join(ROOT, "sdrreceiver_b200", "csrc", "kernels_v3.cuh")
    if not os.path.exists(EXE) or os.path.getmtime(EXE) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        if not os.path.exists(nvcc):
            pytest.skip("nvcc not available")
        r = subprocess.run([nvcc, "-std=c++20", "-O1", "-w", "-gencode", "arch=compute_100a,code=sm_100a", "-o", EXE, src,
                            os.path.join(ROOT, "sdrreceiver_b200", "csrc", "plan_host.o"), "-Xcompiler", "-pthread"],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
    return EXE


# fs, callback size, streams, streams per warp, spans per callback, sub VFOs[, callback count of each stream at the start]
@pytest.mark.parametrize("args", [
    (30720, 7680, 3, 2, 4, 6),       # two stream groups, the second one half empty
    (30720, 7680, 5, 3, 1, 6),       # odd streams per warp (a pair with one member), one span
    (30720, 7680, 4, 2, 7, 16),      # 16 sub VFOs, ragged last span
    (30720, 7680, 3, 8, 3, 4),       # eight streams per warp
    (30720, 7680, 2, 1, 5, 16),      # one stream per warp
    (30720, 7680, 4, 2, 3, 15),      # 15 sub VFOs, two lanes without a row (25E's two-stage group)
    (30720, 7680, 9, 8, 2, 1),       # one sub VFO, eight streams per warp, a second group with one stream
    (30000, 6144, 3, 2, 3, 6),       # the table wraps inside a tile (sample 30000 of 36864)
    # eight streams per warp at counts 0..7: in every callback one stream takes the exact start-up path, the others the
    # table-anchored one, each at its own table position
    (30720, 7680, 8, 8, 3, 4, "0,1,2,3,4,5,6,7"),
    # one warp at counts 0, floor(2^31/B) - 1 (crosses sample 2^31 in the first call), floor(2^32/B) + 3 (past 2^32) and
    # 2^40: a table index computed in 32 bits is wrong for the last two
    (30720, 7680, 4, 4, 3, 6, "0,%d,%d,%d" % (2**31 // 7680 - 1, 2**32 // 7680 + 3, 2**40)),
    # the table wraps inside a tile at large counts: samples 14256, 28368 and 30000 of 36864
    (30000, 6144, 3, 2, 3, 6, "%d,%d,%d" % (2**40, 2**32 // 6144 + 3, 10**12)),
], ids=lambda a: "-".join(str(x) for x in a).replace(",", "_"))
def test_k3_unit_matches_the_plain_cascade(sim, args):
    r = subprocess.run([sim] + [str(a) for a in args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout[-3000:]
