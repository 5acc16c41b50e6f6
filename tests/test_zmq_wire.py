"""ZMQ wire format: the product's publisher (sdrb_publisher_*, libzmq loaded at run time) must
put on the wire exactly what ZmqPublisher::publish does (zmqpublisher.cpp:82-96):
[topic, 5 bytes][uint32 LE rate][int16 LE PCM], nothing for an empty payload. A pyzmq SUB
socket plays JAERO. Host-only: no GPU needed."""
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
    """Directory for ipc:// endpoints. A Unix socket path holds at most 107 bytes, which a deep tmp_path can exceed, so the
    sockets live in a fresh directory directly under /tmp."""
    d = tempfile.mkdtemp(prefix="sdrb-", dir="/tmp")
    yield pathlib.Path(d)
    shutil.rmtree(d, ignore_errors=True)


def _open(addr, bind):
    h = C.c_void_p()
    rc = B.lib().sdrb_publisher_open(addr.encode(), int(bind), C.byref(h))
    if rc == -5:
        pytest.skip("libzmq not loadable here: " + B.lib().sdrb_last_error().decode())
    assert rc == 0, B.lib().sdrb_last_error()
    return h


def test_three_frame_messages_reach_a_subscriber(sock_dir):
    addr = "ipc://" + str(sock_dir / "sdrb.sock")
    pub = _open(addr, True)
    ctx = zmq.Context()
    sub = ctx.socket(zmq.SUB)
    sub.setsockopt(zmq.SUBSCRIBE, b"VFO")
    sub.setsockopt(zmq.RCVTIMEO, 5000)
    sub.connect(addr)
    time.sleep(0.3)                                   # PUB/SUB slow joiner
    L = B.lib()
    pcm = (np.arange(3000, dtype=np.int16) - 1500)
    assert L.sdrb_publisher_send(pub, b"VFO01", 12000, pcm.ctypes.data_as(C.c_void_p), pcm.nbytes) == 0
    assert L.sdrb_publisher_send(pub, b"VFO02", 48000, pcm.ctypes.data_as(C.c_void_p), 0) == 0       # len 0: nothing sent
    assert L.sdrb_publisher_send(pub, b"VFO123456", 24000, pcm.ctypes.data_as(C.c_void_p), 10) == 0   # topic cut to 5 bytes
    m1 = sub.recv_multipart()
    m2 = sub.recv_multipart()
    assert [len(p) for p in m1] == [5, 4, 6000]
    assert m1[0] == b"VFO01" and int.from_bytes(m1[1], "little") == 12000
    assert np.array_equal(np.frombuffer(m1[2], dtype="<i2"), pcm)
    assert m2[0] == b"VFO12" and int.from_bytes(m2[1], "little") == 24000 and len(m2[2]) == 10
    L.sdrb_publisher_close(pub)
    sub.close(0)
    ctx.term()


def test_send_block_emits_one_message_per_vfo_in_plan_order(sock_dir):
    addr = "ipc://" + str(sock_dir / "sdrb2.sock")
    pub = _open(addr, True)
    ctx = zmq.Context()
    sub = ctx.socket(zmq.SUB)
    sub.setsockopt(zmq.SUBSCRIBE, b"")
    sub.setsockopt(zmq.RCVTIMEO, 5000)
    sub.connect(addr)
    time.sleep(0.3)
    plan = B.Plan(plan_path("54W_all"))
    rec = np.arange(plan.pcm_per_block, dtype=np.int32).astype(np.int16)
    assert B.lib().sdrb_publisher_send_block(pub, plan.h, rec.ctypes.data_as(C.c_void_p)) == 0
    for s in plan.subs:
        topic, rate, payload = sub.recv_multipart()
        assert topic == s["topic"].encode()[:5].ljust(5, b"\0")
        assert int.from_bytes(rate, "little") == s["out_rate"]
        want = rec[s["pcm_offset"]:s["pcm_offset"] + s["samples_out"]]
        assert np.array_equal(np.frombuffer(payload, dtype="<i2"), want)
    B.lib().sdrb_publisher_close(pub)
    sub.close(0)
    ctx.term()


def test_bad_address_is_an_error_code_not_a_crash():
    h = C.c_void_p()
    rc = B.lib().sdrb_publisher_open(b"notaproto://x", 1, C.byref(h))
    assert rc == -5 and not h.value


def test_publisher_pool_keeps_format_and_per_receiver_order(sock_dir):
    """sdrb_publisher_pool_*: n sockets, one sender thread each; receiver s on socket s % n, its callbacks in order, every message
    the reference's three frames (zmqpublisher.cpp:82-96). One SUB socket per pool address plays the decoders."""
    L = B.lib()
    base = "ipc://" + str(sock_dir / "pool.sock")
    pool = C.c_void_p()
    rc = L.sdrb_publisher_pool_open(base.encode(), 1, 3, C.byref(pool))
    if rc == -5:
        pytest.skip("libzmq not loadable here: " + L.sdrb_last_error().decode())
    assert rc == 0, L.sdrb_last_error()
    assert L.sdrb_publisher_pool_sockets(pool) == 3
    ctx = zmq.Context()
    subs = []
    for k in range(3):
        buf = C.create_string_buffer(256)
        assert L.sdrb_publisher_pool_address(pool, k, buf, 256) == 0
        assert buf.value.decode() == base + ".%d" % k
        sub = ctx.socket(zmq.SUB)
        sub.setsockopt(zmq.SUBSCRIBE, b"")
        sub.setsockopt(zmq.RCVTIMEO, 5000)
        sub.connect(buf.value.decode())
        subs.append(sub)
    time.sleep(0.4)
    plan = B.Plan(plan_path("54W_288K"))
    n_streams, n_blocks = 5, 2
    pcm = (np.arange(n_streams * n_blocks * plan.pcm_per_block, dtype=np.int64) % 30011 - 15000).astype(np.int16)
    pcm = pcm.reshape(n_streams, n_blocks, plan.pcm_per_block)
    for rep in range(2):                                         # the workers are reused from call to call
        assert L.sdrb_publisher_pool_send_call(pool, plan.h, pcm.ctypes.data_as(C.c_void_p), n_streams, n_blocks) == 0
        for k, sub in enumerate(subs):
            for s in range(k, n_streams, 3):                     # a worker sends its receivers one after the other
                for cb in range(n_blocks):
                    for v in plan.subs:
                        topic, rate, payload = sub.recv_multipart()
                        assert topic == v["topic"].encode()[:5].ljust(5, b"\0")
                        assert int.from_bytes(rate, "little") == v["out_rate"]
                        want = pcm[s, cb, v["pcm_offset"]:v["pcm_offset"] + v["samples_out"]]
                        assert np.array_equal(np.frombuffer(payload, dtype="<i2"), want)
    assert L.sdrb_publisher_pool_send_call(pool, plan.h, None, 0, 0) == 0          # nothing to send
    assert L.sdrb_publisher_pool_send_call(pool, plan.h, None, 2, 2) == -1         # NULL records
    L.sdrb_publisher_pool_close(pool)
    for sub in subs:
        sub.close(0)
    ctx.term()


def test_publisher_pool_address_rules(sock_dir):
    L = B.lib()
    for base, want in (("ipc://" + str(sock_dir / "a%d.sock"), "ipc://" + str(sock_dir / "a1.sock")),
                       ("tcp://127.0.0.1:45731", "tcp://127.0.0.1:45732")):
        pool = C.c_void_p()
        rc = L.sdrb_publisher_pool_open(base.encode(), 1, 2, C.byref(pool))
        if rc == -5 and b"libzmq" in L.sdrb_last_error():
            pytest.skip("libzmq not loadable here")
        assert rc == 0, L.sdrb_last_error()
        buf = C.create_string_buffer(256)
        assert L.sdrb_publisher_pool_address(pool, 1, buf, 256) == 0 and buf.value.decode() == want
        assert L.sdrb_publisher_pool_address(pool, 2, buf, 256) == -1
        L.sdrb_publisher_pool_close(pool)
    pool = C.c_void_p()
    assert L.sdrb_publisher_pool_open(b"ipc:///tmp/x", 1, 0, C.byref(pool)) == -1 and not pool.value


def test_pool_delivers_a_whole_call_to_the_counting_sink(sock_dir):
    """A call's burst (here 8 receivers x 2 callbacks x 27 messages on 2 sockets, three times) reaches tools/zmq_sink.cpp -- the
    counting subscriber bench.py uses for its publish leg -- completely: message count and payload bytes."""
    import json
    import os
    import subprocess
    sink_bin = os.path.join(os.path.dirname(os.path.abspath(B.__file__)), "zmq_sink")
    if not os.access(sink_bin, os.X_OK):
        pytest.skip("zmq_sink not built (make -C sdrreceiver_b200/csrc)")
    L = B.lib()
    pool = C.c_void_p()
    rc = L.sdrb_publisher_pool_open(("ipc://" + str(sock_dir / "sink%d.sock")).encode(), 1, 2, C.byref(pool))
    if rc == -5:
        pytest.skip("libzmq not loadable here")
    assert rc == 0, L.sdrb_last_error()
    addrs = []
    for k in range(2):
        buf = C.create_string_buffer(256)
        assert L.sdrb_publisher_pool_address(pool, k, buf, 256) == 0
        addrs.append(buf.value.decode())
    sink = subprocess.Popen([sink_bin] + addrs, stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)
    assert sink.stdout.readline().strip() == "ready"
    time.sleep(0.4)
    plan = B.Plan(plan_path("25E"))
    pcm = np.ones((8, 2, plan.pcm_per_block), dtype=np.int16)
    for _ in range(3):
        assert L.sdrb_publisher_pool_send_call(pool, plan.h, pcm.ctypes.data_as(C.c_void_p), 8, 2) == 0
    time.sleep(0.5)
    out, _ = sink.communicate("", timeout=20)
    got = json.loads(out.strip().splitlines()[-1])
    L.sdrb_publisher_pool_close(pool)
    assert got["messages"] == 3 * 8 * 2 * len(plan.subs)
    assert got["payload_bytes"] == 3 * 8 * 2 * 2 * sum(v["samples_out"] for v in plan.subs)
