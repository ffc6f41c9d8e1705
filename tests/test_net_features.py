"""Transport features: raw KV apps, SimpleApp, reliable delivery under injected
message loss, heartbeats / dead-node detection, colocated shm IPC, UDS signalling."""
import os
import threading
import time

import numpy as np
import pytest

from _cluster import Cluster
from _mp import free_port


def _core():
    from byteps_b200 import _native

    return _native.core()


def _echo_cluster(c, nw=2, ns=1, extra=None):
    port = free_port()
    extra = extra or {}
    pos, apps = {}, {}
    errs = []

    def node(role, rank):
        try:
            po = c.Postoffice(role, nw, ns, "127.0.0.1", port, "127.0.0.1", rank, extra)
            pos[(role, rank)] = po
            if role == "server":
                apps[(role, rank)] = c.EchoKVServer(po)
            elif role == "worker":
                apps[(role, rank)] = c.KVWorker(po)
            po.start(0, True)
        except Exception as e:  # noqa: BLE001
            errs.append(e)
    ts = [threading.Thread(target=node, args=("scheduler", -1))]
    ts += [threading.Thread(target=node, args=("server", i)) for i in range(ns)]
    ts += [threading.Thread(target=node, args=("worker", i)) for i in range(nw)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(60)
    assert not errs, errs
    return pos, apps


def _finalize(pos, apps):
    for k, a in apps.items():
        if k[0] == "server":
            pass
    ts = [threading.Thread(target=lambda p=p: p.finalize(0, True)) for p in pos.values()]
    for t in ts:
        t.start()
    for t in ts:
        t.join(60)
    for k, a in apps.items():
        if k[0] == "server":
            a.stop()


def test_raw_push_pull_and_simple_app():
    c = _core()
    pos, apps = _echo_cluster(c, 2, 2)
    w0 = apps[("worker", 0)]
    x = np.arange(100_000, dtype=np.float32)
    for server in (0, 1):
        w0.push(server, 42 + server, x.ctypes.data, x.nbytes)
        y = np.zeros_like(x)
        assert w0.pull(server, 42 + server, y.ctypes.data, y.nbytes) == x.nbytes
        np.testing.assert_array_equal(x, y)
    w0.request(7, "hello", c.GROUP_SERVER)
    assert all("hello" in apps[("server", i)].simple_bodies() for i in range(2))
    assert pos[("worker", 0)].my_id() == 9 and pos[("worker", 1)].my_id() == 11
    assert pos[("server", 1)].my_id() == 10 and pos[("scheduler", -1)].my_id() == 1
    kr = pos[("worker", 0)].server_key_ranges()
    assert len(kr) == 2 and kr[0][1] == kr[1][0]
    assert pos[("worker", 0)].send_bytes() > x.nbytes
    _finalize(pos, apps)


@pytest.mark.parametrize("van", ["tcp", "shm"])
def test_resender_survives_message_drops(van):
    """PS_DROP_MSG-style fault injection with PS_RESEND-style retransmission."""
    c = _core()
    cl = Cluster(2, 1, extra={"resend": True, "resend_timeout_ms": 100, "drop_msg_pct": 10, "van_type": van}).start()
    out = {}

    def work(rank, w, po):
        key = c.make_key(0, 0)
        z = np.zeros(5000, dtype=np.float32)
        w.init_key(key, z.ctypes.data, z.nbytes, c.F32)
        for it in range(10):
            x = np.full(5000, float(rank + it), dtype=np.float32)
            assert w.wait(w.push_pull("g", x.ctypes.data, c.F32, [(key, 0, x.nbytes)], 0, 0, 1.0), 60_000)
            assert np.all(x == (0 + it) + (1 + it)), (it, x[:3])
        out[rank] = True
    cl.run_workers(work)
    assert len(out) == 2
    cl.stop()


@pytest.mark.parametrize("van", ["tcp", "shm"])
def test_heartbeat_and_dead_node_detection(van):
    c = _core()
    cl = Cluster(1, 1, extra={"heartbeat_interval_s": 1, "heartbeat_timeout_s": 2, "van_type": van}).start(
        make_worker=False)
    time.sleep(1.5)
    assert cl.sched.dead_nodes(2) == []          # everyone is beating
    assert cl.sched.dead_nodes(0) == []          # timeout 0 = detection off
    cl.stop()


def test_colocated_ipc_moves_payload_through_shm():
    c = _core()
    cl = Cluster(2, 1, extra={"enable_ipc": True}).start()
    sent = {}

    def work(rank, w, po):
        name = "bps_test_shm_%d_%d" % (po.my_port(), rank)
        n = 200_000
        ptr = c.shm_create(name, n * 4)
        import ctypes

        x = np.frombuffer((ctypes.c_float * n).from_address(ptr), dtype=np.float32)
        key = c.make_key(0, 0)
        x[:] = 0
        w.init_key(key, ptr, n * 4, c.F32)
        before = po.send_bytes()
        for it in range(3):
            x[:] = rank + 1 + it
            assert w.wait(w.push_pull("g", ptr, c.F32, [(key, 0, n * 4)], 0, 0, 1.0))
            assert np.all(x == (1 + it) + (2 + it))
        sent[rank] = po.send_bytes() - before
        del x
        c.shm_release(name)
    cl.run_workers(work)
    # 3 pushes of 800 KB each went through shared memory: only metas crossed the socket
    assert all(v < 100_000 for v in sent.values()), sent
    cl.stop()


def test_uds_local_signalling(sock_dir):
    c = _core()
    members = [0, 1, 2]
    comms = {}

    def make(r):
        comms[r] = c.LocalComm(r, members, sock_dir, "t")
    ts = [threading.Thread(target=make, args=(r,)) for r in members]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    root = comms[2]
    assert root.is_root() and comms[0].root == 2
    rt = c.ReadyTable(2, "reduce")
    root.set_tables(rt)
    assert comms[0].send_to_root(c.SIG_REDUCE_READY, 77) and comms[1].send_to_root(c.SIG_REDUCE_READY, 77)
    for _ in range(100):
        if rt.is_key_ready(77):
            break
        time.sleep(0.01)
    assert rt.is_key_ready(77) and root.received() == 2
    assert root.broadcast(c.SIG_DO_REDUCE, 77) and root.broadcast(c.SIG_DO_GROUP, 0)
    for r in (0, 1):
        assert comms[r].recv_from_root(2000) == (2, c.SIG_DO_REDUCE, 77)
        assert comms[r].recv_from_root(2000) == (2, c.SIG_DO_GROUP, 0)
    assert comms[0].recv_from_root(300) is None
    comms.clear()


def test_uds_path_too_long_is_an_error():
    c = _core()
    with pytest.raises(RuntimeError, match="socket path too long"):
        c.LocalComm(0, [0, 1], "/tmp/" + "d" * 120, "t")


def test_multi_lane_connections_stripe_keys():
    """DMLC_NUM_PORTS-style parallel connections: 4 lanes per peer, 16 keys, several rounds;
    sums stay exact and per-key order holds (same key -> same lane)."""
    import numpy as np

    from _cluster import Cluster

    c = _core()
    nw = 2
    cl = Cluster(nw, 2, extra={"num_lanes": 4}).start()
    n = 50_000
    parts = [(c.make_key(0, i), i * n * 4, n * 4) for i in range(16)]
    results = {}

    def work(rank, w, po):
        for key, off, ln in parts:
            z = np.zeros(ln // 4, dtype=np.float32)
            w.init_key(key, z.ctypes.data, ln, c.F32)
        for it in range(4):
            x = (np.arange(n * 16, dtype=np.float32) % 89) * (rank + 1) + it
            h = w.push_pull("g", x.ctypes.data, c.F32, parts, 0, 0, 1.0)
            assert w.wait(h)
            results[(rank, it)] = x
    cl.run_workers(work)
    for it in range(4):
        expect = sum((np.arange(n * 16, dtype=np.float32) % 89) * (r + 1) + it for r in range(nw))
        for r in range(nw):
            np.testing.assert_allclose(results[(r, it)], expect, rtol=1e-6)
    cl.stop()


def test_dmlc_local_unix_domain_transport():
    """DMLC_LOCAL=1 (ps-lite's ipc:// mode): scheduler bootstrap, barriers, multi-lane data and colocated shm IPC
    all work over Unix-domain stream sockets; nothing listens on TCP."""
    import socket

    import numpy as np

    from _cluster import Cluster

    c = _core()
    nw = 2
    cl = Cluster(nw, 2, extra={"local": True, "num_lanes": 2}).start()
    s = socket.socket()
    s.settimeout(1)
    assert s.connect_ex(("127.0.0.1", cl.port)) != 0, "the scheduler must not listen on TCP in local mode"
    s.close()
    with open("/proc/net/unix") as f:
        assert "@byteps_van_%d" % cl.port in f.read()
    n = 300_000
    parts = [(c.make_key(0, i), i * n * 4, n * 4) for i in range(4)]
    results = {}

    def work(rank, w, po):
        for key, off, ln in parts:
            z = np.zeros(ln // 4, dtype=np.float32)
            w.init_key(key, z.ctypes.data, ln, c.F32)
        for it in range(3):
            x = (np.arange(n * 4, dtype=np.float32) % 61) * (rank + 1) + it
            h = w.push_pull("g", x.ctypes.data, c.F32, parts, 0, 0, 1.0)
            assert w.wait(h)
            results[(rank, it)] = x
    cl.run_workers(work)
    for it in range(3):
        expect = sum((np.arange(n * 4, dtype=np.float32) % 61) * (r + 1) + it for r in range(nw))
        for r in range(nw):
            np.testing.assert_allclose(results[(r, it)], expect, rtol=1e-6)
    cl.stop()


@pytest.mark.parametrize("ipc_windows", [False, True])
def test_shm_van_socket_free_transport(ipc_windows, monkeypatch):
    """DMLC_PS_VAN_TYPE=shm: bootstrap, barriers, small (inline), medium (arena), oversized (one-off segment) and
    registered-window (by reference) payloads all travel through shared memory; nothing is left in /dev/shm."""
    import glob
    import socket

    import numpy as np

    from _cluster import Cluster

    monkeypatch.setenv("BYTEPS_SHMVAN_ARENA_MB", "4")       # 4 MB arena: the 3 MB key goes through a one-off segment
    c = _core()
    nw = 2
    before = set(glob.glob("/dev/shm/bps_shmvan_*"))
    cl = Cluster(nw, 2, extra={"van_type": "shm"}).start()
    s = socket.socket()
    s.settimeout(1)
    assert s.connect_ex(("127.0.0.1", cl.port)) != 0, "no TCP listener in shm mode"
    s.close()
    assert os.path.exists("/dev/shm/bps_shmvan_%d" % cl.port)
    sizes = [16, 1000, 300_000, 750_000]        # floats: 64 B, 4 KB (inline), 1.2 MB (arena), 3 MB (one-off)
    offs = np.cumsum([0] + sizes)
    parts = [(c.make_key(0, i), int(offs[i]) * 4, sizes[i] * 4) for i in range(len(sizes))]
    total = int(offs[-1])
    results = {}

    def work(rank, w, po):
        if ipc_windows:     # registered window: pushes go by reference, pulls are written into it by the server
            ptr = c.shm_create("BytePS_ShM_test_shmvan_%d_%d" % (os.getpid(), rank), total * 4)
            x = np.ctypeslib.as_array((__import__("ctypes").c_float * total).from_address(ptr))
        else:
            x = np.zeros(total, dtype=np.float32)
        for key, off, ln in parts:
            w.init_key(key, x.ctypes.data + off, ln, c.F32)
        for it in range(5):
            x[:] = (np.arange(total, dtype=np.float32) % 53) * (rank + 1) + it
            h = w.push_pull("g", x.ctypes.data, c.F32, parts, 0, 0, 1.0)
            assert w.wait(h)
            results[(rank, it)] = x.copy()
    cl.run_workers(work)
    for it in range(5):
        expect = sum((np.arange(total, dtype=np.float32) % 53) * (r + 1) + it for r in range(nw))
        for r in range(nw):
            np.testing.assert_allclose(results[(r, it)], expect, rtol=1e-6)
    cl.stop()
    if ipc_windows:
        for r in range(nw):
            c.shm_release("BytePS_ShM_test_shmvan_%d_%d" % (os.getpid(), r))
    assert set(glob.glob("/dev/shm/bps_shmvan_*")) <= before, "shm van left objects behind"


def test_shm_van_sweeps_objects_of_dead_processes(tmp_path):
    """Leftovers of a killed job (arena named after a dead pid, queue whose header names a dead owner) disappear the
    next time a process binds a shm van; objects of live processes stay."""
    import struct
    import subprocess
    import sys

    dead = subprocess.Popen([sys.executable, "-c", "pass"])
    dead.wait()
    stale_arena = "/dev/shm/bps_shmvan_11111_to_22222_%d_0" % dead.pid
    stale_queue = "/dev/shm/bps_shmvan_33333"
    live_arena = "/dev/shm/bps_shmvan_11111_to_22222_%d_7" % os.getpid()
    for path in (stale_arena, live_arena):
        open(path, "wb").write(b"\0" * 4096)
    open(stale_queue, "wb").write(struct.pack("<II", 0x62707351, dead.pid) + b"\0" * 4088)
    try:
        code = ("import sys; sys.path[:0] = [%r, %r]\n"
                "from _cluster import Cluster\n"
                "Cluster(1, 1, extra={'van_type': 'shm'}).start(make_worker=False).stop()\n"
                % (os.path.dirname(os.path.abspath(__file__)), os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
        subprocess.check_call([sys.executable, "-c", code], timeout=120)
        assert not os.path.exists(stale_arena) and not os.path.exists(stale_queue)
        assert os.path.exists(live_arena)
    finally:
        for path in (stale_arena, stale_queue, live_arena):
            if os.path.exists(path):
                os.unlink(path)
