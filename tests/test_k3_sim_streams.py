"""k2a_v3's stream-list form (k3_unit<MAXS, true>: warp-local stream s of stream group g is bank stream map[g*nsw + s]) executed
on the CPU by tests/cpp/k3_sim_streams.cu against the same plain cascade and within the same bounds as tests/test_k3_sim.py:
rel-L2 <= 2e-6 and worst |d| <= 9e-6 x RMS per VFO. The lists are permuted and non-contiguous, leave a ragged last group, and
the streams start at mixed and large callback counts. Streams left out of the list must keep their output rows untouched."""
import os
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, ".."))
EXE = os.path.join(HERE, "cpp", "k3_sim_streams")
B30 = 7680


@pytest.fixture(scope="module")
def sim(built):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    srcs = [os.path.join(HERE, "cpp", f) for f in ("k3_sim_streams.cu", "k3_sim.cu")]
    hdr = os.path.join(ROOT, "sdrreceiver_b200", "csrc", "kernels_v3.cuh")
    if not os.path.exists(EXE) or os.path.getmtime(EXE) < max(os.path.getmtime(f) for f in srcs + [hdr]):
        if not os.path.exists(nvcc):
            pytest.skip("nvcc not available")
        r = subprocess.run([nvcc, "-std=c++20", "-O1", "-w", "-gencode", "arch=compute_100a,code=sm_100a", "-o", EXE, srcs[0],
                            os.path.join(ROOT, "sdrreceiver_b200", "csrc", "plan_host.o"), "-Xcompiler", "-pthread"],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
    return EXE


# fs, callback size, streams, streams per warp, spans per callback, sub VFOs, callback count of each stream, the list
@pytest.mark.parametrize("args", [
    # 12 streams, 7 listed out of order, two per warp: a one-stream last group
    (30720, B30, 12, 2, 3, 6, ",".join(["0"] * 12), "9,2,7,0,11,4,5"),
    # eight per warp over a permuted full list at counts 0..7 (every warp mixes the exact and the table-anchored path)
    (30720, B30, 8, 8, 3, 4, "0,1,2,3,4,5,6,7", "6,1,7,3,0,5,2,4"),
    # 25E's two-stage group shape (15 VFOs, two streams per warp), a ragged list of 3 at large counts
    (30720, B30, 6, 2, 3, 15, "%d,0,%d,5,%d,1" % (2**40, 2**32 // B30 + 3, 2**31 // B30 - 1), "4,0,2"),
    # one listed stream, past 2^32 samples, the table wrapping inside a tile
    (30000, 6144, 5, 2, 3, 6, "0,0,0,%d,0" % (10**12), "3"),
    # three per warp, descending list with gaps, large mixed counts
    (30720, B30, 10, 3, 2, 6, "1,%d,3,%d,5,6,%d,8,9,10" % (2**40, 2**33, 2**31 // B30 + 1), "8,6,3,1"),
], ids=lambda a: "-".join(str(x) for x in a[:6]) + "-list" + a[7].replace(",", "_"))
def test_k3_unit_over_a_stream_list_matches_the_plain_cascade(sim, args):
    r = subprocess.run([sim] + [str(a) for a in args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout[-3000:]
