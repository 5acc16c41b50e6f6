"""sdrb_publisher_pool_send_streams: the compact result of a stream-list call (record k = receiver streams[k]) goes out like a
whole call would: receiver s on socket s % n_sockets, its callbacks in order, every message the reference's three frames
(zmqpublisher.cpp:82-96). Host-only: no GPU needed."""
import ctypes as C
import pathlib
import shutil
import tempfile
import time

import numpy as np
import pytest

from conftest import plan_path
from sdrreceiver_b200 import binding as B

zmq = pytest.importorskip("zmq")


@pytest.fixture
def sock_dir():
    d = tempfile.mkdtemp(prefix="sdrb-", dir="/tmp")         # ipc:// paths must stay short
    yield pathlib.Path(d)
    shutil.rmtree(d, ignore_errors=True)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def test_listed_receivers_go_out_on_their_sockets_in_order(sock_dir):
    L = B.lib()
    base = "ipc://" + str(sock_dir / "pool.sock")
    pool = C.c_void_p()
    rc = L.sdrb_publisher_pool_open(base.encode(), 1, 3, C.byref(pool))
    if rc == -5:
        pytest.skip("libzmq not loadable here: " + L.sdrb_last_error().decode())
    assert rc == 0, L.sdrb_last_error()
    ctx = zmq.Context()
    subs = []
    for k in range(3):
        buf = C.create_string_buffer(256)
        assert L.sdrb_publisher_pool_address(pool, k, buf, 256) == 0
        sub = ctx.socket(zmq.SUB)
        sub.setsockopt(zmq.SUBSCRIBE, b"")
        sub.setsockopt(zmq.RCVTIMEO, 5000)
        sub.connect(buf.value.decode())
        subs.append(sub)
    time.sleep(0.4)
    plan = B.Plan(plan_path("54W_288K"))
    streams = np.array([5, 2, 7], dtype=np.int32)           # sockets 2, 2 and 1; socket 0 gets nothing
    n_blocks = 2
    pcm = (np.arange(streams.size * n_blocks * plan.pcm_per_block, dtype=np.int64) % 30011 - 15000).astype(np.int16)
    pcm = pcm.reshape(streams.size, n_blocks, plan.pcm_per_block)
    try:
        for rep in range(2):
            assert L.sdrb_publisher_pool_send_streams(pool, plan.h, _ptr(pcm), _ptr(streams), streams.size, n_blocks) == 0, \
                L.sdrb_last_error()
            for k, sub in enumerate(subs):
                for i, s in enumerate(streams):
                    if s % 3 != k:
                        continue
                    for cb in range(n_blocks):
                        for v in plan.subs:
                            topic, rate, payload = sub.recv_multipart()
                            assert topic == v["topic"].encode()[:5].ljust(5, b"\0")
                            assert int.from_bytes(rate, "little") == v["out_rate"]
                            want = pcm[i, cb, v["pcm_offset"]:v["pcm_offset"] + v["samples_out"]]
                            assert np.frombuffer(payload, dtype="<i2").tobytes() == want.tobytes()
            with pytest.raises(zmq.Again):                  # socket 0 has no listed receiver: nothing extra anywhere
                subs[0].setsockopt(zmq.RCVTIMEO, 200)
                subs[0].recv_multipart()
            subs[0].setsockopt(zmq.RCVTIMEO, 5000)

        # refusals: nothing is sent, the error names the problem
        def refused(pcm_p, streams_arr, n, nb, what):
            sp = _ptr(streams_arr) if streams_arr is not None else None
            assert L.sdrb_publisher_pool_send_streams(pool, plan.h, pcm_p, sp, n, nb) == -1
            assert what in L.sdrb_last_error().decode()
        refused(None, streams, 3, n_blocks, "NULL")
        refused(_ptr(pcm), None, 3, n_blocks, "NULL")
        assert L.sdrb_publisher_pool_send_streams(pool, None, _ptr(pcm), _ptr(streams), 3, n_blocks) == -1
        refused(_ptr(pcm), np.array([5, 2, 5], dtype=np.int32), 3, n_blocks, "streams[2] = 5 is listed twice")
        refused(_ptr(pcm), np.array([5, -1, 7], dtype=np.int32), 3, n_blocks, "streams[1] = -1 is negative")
        refused(_ptr(pcm), streams, 0, n_blocks, "positive")
        refused(_ptr(pcm), streams, 3, 0, "positive")
        for sub in subs:
            sub.setsockopt(zmq.RCVTIMEO, 200)
            with pytest.raises(zmq.Again):
                sub.recv_multipart()
    finally:
        L.sdrb_publisher_pool_close(pool)
        for sub in subs:
            sub.close(0)
        ctx.term()
