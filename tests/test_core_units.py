"""Unit tests of the native runtime pieces the reference never tested
(scheduler, ready table, partitioning, registry, hashing, reducer, timeline)."""
import json
import os
import threading
import time

import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def c():
    from byteps_b200 import _native

    return _native.core()


def test_dtype_table_and_command_pairing(c):
    assert [c.dtype_size(d) for d in (c.F32, c.F64, c.F16, c.U8, c.I32, c.I8, c.I64, c.BF16)] == [4, 8, 2, 1, 4, 1, 8, 2]
    for req in range(3):
        for dt in range(8):
            assert c.command_decode(c.command_encode(req, dt)) == (req, dt)
    assert c.stage_name(c.REDUCE) == "REDUCE" and c.stage_name(c.BROADCAST) == "BROADCAST"


def test_partitioning_and_keys(c):
    parts = c.partition_bytes(10_000_000, 4_096_000)
    assert parts == [(0, 4096000), (4096000, 4096000), (8192000, 1808000)]
    assert c.partition_bytes(0, 100) == [(0, 0)]
    k = c.make_key(513, 7)
    assert c.key_declared(k) == 513 and c.key_part(k) == 7
    assert c.align_payload(10, c.F32) == 128 and c.round_up(5, 4) == 8


def test_registry_declaration_order_is_stable(c):
    r = c.Registry()
    assert [r.declare(n) for n in ("b", "a", "b", "c")] == [0, 1, 0, 2]
    assert r.declared_names() == ["b", "a", "c"]
    keys = r.init_tensor("a", 9_000_000, c.F32, 4_096_000, 4096)
    assert keys == [c.make_key(1, i) for i in range(3)]
    r.reset_contexts()          # suspend/resume keeps names and keys
    assert r.declare("a") == 1 and r.is_declared("c")
    with pytest.raises(RuntimeError):
        r.init_tensor("nope", 4, c.F32, 4, 4)


def test_hash_family_and_placement_balance(c):
    assert c.hash_naive((3 << 16) + 5) == (3 + 5) * 9973
    assert c.hash_djb2(0) == 5381 * 33 + ord("0")
    for fn in ("naive", "built_in", "djb2", "sdbm"):
        kp = c.KeyPlacer(fn, 4, 4)
        keys = [c.make_key(t, p) for t in range(50) for p in range(4)]
        servers = [kp.server_of(k, 1000) for k in keys]
        assert [kp.server_of(k, 1000) for k in keys] == servers          # memoised / deterministic
        assert sum(kp.load()) == 1000 * len(keys) and min(kp.load()) > 0
    kp = c.KeyPlacer("mixed", 6, 4, True, 101)        # 2 non-colocated + 4 colocated servers
    assert all(0 <= kp.server_of(k, 1) < 6 for k in range(1000))
    with pytest.raises(RuntimeError):
        c.KeyPlacer("bogus", 2, 2).server_of(1, 1)


def test_scheduler_priority_then_key_order(c):
    q = c.ScheduledQueue(c.REDUCE, True, 0)
    for key, prio in [(5, 0), (3, 1), (1, 0), (9, 1), (2, -1)]:
        q.add(c.Task(key, prio, 100))
    assert [q.get().key for _ in range(5)] == [3, 9, 1, 5, 2]
    assert q.get() is None and q.pending() == 0


def test_scheduler_fifo_when_not_scheduled(c):
    q = c.ScheduledQueue(c.PUSH, False, 0)
    for key, prio in [(5, 0), (3, 9), (1, 4)]:
        q.add(c.Task(key, prio, 1))
    assert [q.get().key for _ in range(3)] == [5, 3, 1]


def test_scheduler_byte_credits(c):
    q = c.ScheduledQueue(c.REDUCE, True, 250)
    for k in range(4):
        q.add(c.Task(k, 0, 100))
    a, b = q.get(), q.get()
    assert (a.key, b.key) == (0, 1) and q.credits() == 50
    assert q.get() is None                   # third does not fit in the window
    q.report_finish(100)
    assert q.get().key == 2
    big = c.ScheduledQueue(c.REDUCE, True, 50)
    big.add(c.Task(7, 0, 1000))             # larger than the whole window: allowed when idle
    assert big.get().key == 7


def test_scheduler_ready_predicate_and_ready_table(c):
    flag = {"ok": False}
    q = c.ScheduledQueue(c.REDUCE, True, 0)
    q.add(c.Task(1, 5, 10, lambda: flag["ok"]))
    q.add(c.Task(2, 0, 10))
    assert q.get().key == 2                  # higher priority task is not ready yet
    assert q.get() is None
    flag["ok"] = True
    assert q.get().key == 1
    rt = c.ReadyTable(2, "t")
    q2 = c.ScheduledQueue(c.PUSH, True, 0, rt)
    q2.add(c.Task(11, 0, 10))
    assert q2.get() is None
    rt.add_ready_count(11)
    assert q2.get() is None
    rt.add_ready_count(11)
    assert rt.is_key_ready(11) and q2.get().key == 11
    assert rt.count(11) == 0                 # consumed
    q2.add(c.Task(12, 0, 1))
    assert q2.get_by_key(12).key == 12 and q2.get_by_key(12) is None


def test_handle_manager_wait_blocks_until_done(c):
    hm = c.HandleManager()
    h = hm.allocate()
    assert not hm.poll(h) and hm.outstanding() == 1
    assert hm.wait_and_release(h, 10)[0] == 5          # ST_IN_PROGRESS on timeout
    threading.Timer(0.05, lambda: hm.mark_done(h, 0, "")).start()
    t0 = time.time()
    assert hm.wait_and_release(h, -1)[0] == 0 and time.time() - t0 < 2
    assert hm.poll(h)                                    # released handles read as complete


@pytest.mark.parametrize("dt,code", [(torch.float32, "F32"), (torch.float64, "F64"), (torch.float16, "F16"),
                                     (torch.bfloat16, "BF16"), (torch.int32, "I32"), (torch.int64, "I64"),
                                     (torch.uint8, "U8"), (torch.int8, "I8")])
def test_cpu_reducer_all_dtypes(c, dt, code):
    red = c.CpuReducer(3)
    n = 10_007
    torch.manual_seed(0)
    if dt.is_floating_point:
        a, b = torch.randn(n).to(dt), torch.randn(n).to(dt)
    else:
        a, b = torch.randint(0, 50, (n,)).to(dt), torch.randint(0, 50, (n,)).to(dt)
    nbytes = n * a.element_size()
    d = a.clone()
    red.sum(d.data_ptr(), b.data_ptr(), nbytes, getattr(c, code))
    ref = (a.double() + b.double()).to(dt) if dt.is_floating_point else a + b
    if dt in (torch.float16, torch.bfloat16):
        ref = (a.float() + b.float()).to(dt)
    assert torch.equal(d, ref)
    out = torch.zeros_like(a)
    red.sum3(out.data_ptr(), a.data_ptr(), b.data_ptr(), nbytes, getattr(c, code))
    assert torch.equal(out, ref)
    if dt.is_floating_point:
        d = a.clone()
        red.sum_scaled(d.data_ptr(), b.data_ptr(), nbytes, getattr(c, code), 0.5)
        assert torch.allclose(d.float(), (a.float() + 0.5 * b.float()).to(dt).float(), rtol=1e-6, atol=1e-6)
        d = a.clone()
        red.scale(d.data_ptr(), nbytes, getattr(c, code), 0.25)
        assert torch.equal(d, (a.float() * 0.25).to(dt))
    else:
        d = (a.clone() * 3)
        red.scale(d.data_ptr(), nbytes, getattr(c, code), 1.0 / 4)
        assert torch.equal(d, torch.floor_divide(a * 3, 4))
    big = torch.arange(3_000_000, dtype=torch.float32)
    dst = torch.empty_like(big)
    red.copy(dst.data_ptr(), big.data_ptr(), big.numel() * 4)
    assert torch.equal(dst, big)


def test_half_conversions_match_torch(c):
    xs = torch.tensor([0.0, -0.0, 1.0, -2.5, 65504.0, 70000.0, 1e-8, 6.1e-5, 3.14159, float("inf")])
    for x in xs.tolist():
        assert c.f32_to_f16(x) == int(torch.tensor(x).to(torch.float16).view(torch.int16).item()) & 0xffff
        assert c.f32_to_bf16(x) == int(torch.tensor(x).to(torch.bfloat16).view(torch.int16).item()) & 0xffff
    for h in (0x3c00, 0x0001, 0x7bff, 0xc000, 0x0400):
        assert c.f16_to_f32(h) == torch.tensor(h - (1 << 16) if h >= (1 << 15) else h, dtype=torch.int16).view(torch.float16).float().item()


def test_timeline_chrome_trace_and_window(c, tmp_path):
    t = c.Timeline()
    t.configure(True, 2, 4, str(tmp_path), 3)
    assert not t.active(1) and t.active(2) and t.active(3) and not t.active(4)
    t.record("Gradient.w", "PUSH", c.make_key(1, 0), 1000, 50)
    t.record("Gradient.w", "", (1 << 64) - 1, 900, 400)
    js = json.loads(t.to_json())
    ev = js["traceEvents"]
    assert ev[0]["name"] == "Comm.Gradient.w.PUSH" and ev[0]["ph"] == "X" and ev[0]["tid"] == str(c.make_key(1, 0))
    assert ev[1]["tid"] == "total" and ev[1]["dur"] == 400 and ev[0]["cat"] == "Comm"
    path = t.dump()
    assert path.endswith(os.path.join("3", "comm.json")) and os.path.exists(path)


def test_telemetry_speed_samples(c):
    tel = c.Telemetry(True, 0.05)
    assert tel.get() == (0, -5.0)              # the reference's "no data" sentinel
    tel.record(1_000_000)
    time.sleep(0.08)
    tel.record(1_000_000)
    ts, mbps = tel.get()
    assert ts > 0 and mbps > 0 and tel.total_bytes() == 2_000_000


def test_xorshift_stream_matches_reference_definition(c):
    rng = c.XorShift128Plus()
    rng.set_seed(2020)
    a = b = 2020
    mask = (1 << 64) - 1
    for _ in range(5):
        t, s = a, b
        a = s
        t ^= (t << 23) & mask
        t ^= t >> 17
        t ^= s ^ (s >> 26)
        b = t
        assert rng.next() == (t + s) & mask


def test_compressor_numpy_models(c):
    """onebit / topk / randomk against independent numpy models (the reference's test idea)."""
    n = 4096
    rng = np.random.RandomState(1)
    g = rng.randn(n).astype(np.float32)
    buf = np.zeros(n * 16 + 64, dtype=np.uint8)
    out = np.zeros(n, dtype=np.float32)
    comp = c.Compressor({"compressor_type": "onebit", "compressor_onebit_scaling": "true"}, n * 4, c.F32)
    gc = g.copy()
    m = comp.compress(gc.ctypes.data, buf.ctypes.data)
    assert m == n // 32 * 4 + 4
    comp.decompress(buf.ctypes.data, m, out.ctypes.data)
    np.testing.assert_allclose(out, np.where(g < 0, -1, 1) * np.abs(g).mean(), rtol=1e-5)
    words = buf[:n // 8].view(np.uint32)
    assert ((words[0] >> 31) & 1) == int(g[0] < 0)        # MSB first
    comp = c.Compressor({"compressor_type": "topk", "compressor_k": "0.01"}, n * 4, c.F32)
    gc = g.copy()
    m = comp.compress(gc.ctypes.data, buf.ctypes.data)
    k = int(0.01 * n)
    assert m == k * 8
    comp.decompress(buf.ctypes.data, m, out.ctypes.data)
    idx = np.argsort(-np.abs(g))[:k]
    ref = np.zeros(n, dtype=np.float32)
    ref[idx] = g[idx]
    np.testing.assert_array_equal(out, ref)
    comp = c.Compressor({"compressor_type": "randomk", "compressor_k": "16", "seed": "99"}, n * 4, c.F32)
    gc = g.copy()
    m = comp.compress(gc.ctypes.data, buf.ctypes.data)
    comp.decompress(buf.ctypes.data, m, out.ctypes.data)
    r = c.XorShift128Plus()
    r.set_seed(99)
    ref = np.zeros(n, dtype=np.float32)
    for _ in range(16):
        i = r.randint(0, n)
        ref[i] = g[i]
    np.testing.assert_array_equal(out, ref)
    # error feedback: e = corrected - D(C(corrected)); second step adds e back
    comp = c.Compressor({"compressor_type": "topk", "compressor_k": "8", "ef_type": "vanilla"}, n * 4, c.F32)
    g1 = g.copy()
    m = comp.compress(g1.ctypes.data, buf.ctypes.data)
    comp.decompress(buf.ctypes.data, m, out.ctypes.data)
    err = g - out
    g2 = np.zeros(n, dtype=np.float32)
    m = comp.compress(g2.ctypes.data, buf.ctypes.data)
    comp.decompress(buf.ctypes.data, m, out.ctypes.data)
    idx = np.argsort(-np.abs(err))[:8]
    ref = np.zeros(n, dtype=np.float32)
    ref[idx] = err[idx]
    np.testing.assert_allclose(out, ref, rtol=1e-6)
    assert sorted(c.compressor_names()) == ["dithering_compressor_type", "nesterov_momentum_type",
                                            "onebit_compressor_type", "randomk_compressor_type",
                                            "topk_compressor_type", "vanilla_ef_type"]
    kw = {"compressor_type": "topk", "compressor_k": "3"}
    assert c.kwargs_deserialize(c.kwargs_serialize(kw)) == kw


@pytest.mark.parametrize("partition,normalize", [(0, 0), (1, 1)])
def test_dithering_roundtrip_is_unbiased(c, partition, normalize):
    n = 2048
    rng = np.random.RandomState(3)
    g = rng.randn(n).astype(np.float32)
    kw = {"compressor_type": "dithering", "compressor_k": "8", "seed": "7", "dithering_partition": str(partition),
          "dithering_normalize": str(normalize)}
    comp = c.Compressor(kw, n * 4, c.F32)
    buf = np.zeros(comp.max_compressed_bytes(), dtype=np.uint8)
    acc = np.zeros(n, dtype=np.float64)
    out = np.zeros(n, dtype=np.float32)
    trials = 300
    for _ in range(trials):
        gc = g.copy()
        m = comp.compress(gc.ctypes.data, buf.ctypes.data)
        assert m < n * 4                     # it does compress
        comp.decompress(buf.ctypes.data, m, out.ctypes.data)
        acc += out
    assert np.abs(acc / trials - g).mean() < 0.05


def test_resender_stress_many_rounds():
    """Regression for two shutdown bugs found by fault injection: (1) one Message object sent to
    several nodes kept its first signature, so later copies were neither tracked nor accepted;
    (2) a reader fd closed early stayed registered and StopTransport() shut down whichever socket
    had inherited the number.  Five clusters in a row with 15 % drops must all finalize."""
    import numpy as np

    from _cluster import Cluster
    from byteps_b200 import _native

    c = _native.core()
    for rnd in range(5):
        cl = Cluster(2, 1, extra={"resend": True, "resend_timeout_ms": 50, "drop_msg_pct": 15}).start()

        def work(rank, w, po):
            key = c.make_key(0, 0)
            z = np.zeros(2000, dtype=np.float32)
            w.init_key(key, z.ctypes.data, z.nbytes, c.F32)
            for it in range(5):
                x = np.full(2000, float(rank + it), dtype=np.float32)
                assert w.wait(w.push_pull("g", x.ctypes.data, c.F32, [(key, 0, x.nbytes)], 0, 0, 1.0), 60_000)
                assert np.all(x == 2 * it + 1)
        cl.run_workers(work)
        cl.stop()


ROOT = __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__)))


def test_env_knobs_interface_port_hash_coef(monkeypatch):
    """DMLC_INTERFACE / DMLC_PORT / BYTEPS_BUILT_IN_HASH_COEF / BYTEPS_NUMA_ROOT_QUOTA are honoured."""
    import subprocess
    import sys

    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "from byteps_b200 import _native\n"
        "c = _native.core()\n"
        "p = c.KeyPlacer('built_in', 7, 7)\n"
        "print([p.server_of(c.make_key(i, 0), 100) for i in range(12)])\n" % ROOT)
    outs = []
    for coef in ("1", "3"):
        env = dict(__import__("os").environ, BYTEPS_BUILT_IN_HASH_COEF=coef)
        outs.append(subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env).stdout)
    assert outs[0] and outs[1] and outs[0] != outs[1]
    from byteps_b200.launcher import launch

    monkeypatch.setenv("BYTEPS_NUMA_ROOT_QUOTA", "6")
    alloc = launch.allocate_cpu(2, nodes=[list(range(8)), list(range(8, 16))], multithreaded=False, blacklist=set())
    assert alloc[0] == list(range(8)) and alloc[1] == list(range(8, 14))


def test_advertised_node_host_resolution(monkeypatch):
    """What a node advertises to the scheduler (ps-lite van.cc:520-562): an explicit host wins, then
    DMLC_NODE_HOST, then DMLC_INTERFACE's address, then the first non-loopback IPv4 - except that a job whose
    scheduler is on the loopback interface stays on 127.0.0.1.  (Round 1 ignored DMLC_INTERFACE because the
    python callers always passed DMLC_NODE_HOST-or-127.0.0.1 explicitly.)"""
    import socket

    from byteps_b200 import _native

    c = _native.core()
    monkeypatch.delenv("DMLC_NODE_HOST", raising=False)
    monkeypatch.delenv("DMLC_INTERFACE", raising=False)
    assert c.resolve_node_host("127.0.0.1", "") == "127.0.0.1"
    assert c.resolve_node_host("localhost", "") == "127.0.0.1"
    assert c.resolve_node_host("10.1.2.3", "host-a") == "host-a"
    auto = c.resolve_node_host("10.1.2.3", "")
    socket.inet_aton(auto)                                 # a dotted quad
    externals = [a for a in _ipv4_addresses() if not a.startswith("127.")]
    assert auto == (externals[0] if externals else "127.0.0.1")
    monkeypatch.setenv("DMLC_INTERFACE", "lo")
    assert c.resolve_node_host("10.1.2.3", "") == "127.0.0.1"
    monkeypatch.setenv("DMLC_NODE_HOST", "1.2.3.4")
    assert c.resolve_node_host("10.1.2.3", "") == "1.2.3.4"
    assert c.resolve_node_host("10.1.2.3", "5.6.7.8") == "5.6.7.8"


def _ipv4_addresses():
    """IPv4 addresses of the interfaces that are up, in getifaddrs order (what the native code walks)."""
    import ctypes
    import ctypes.util
    import socket

    class sockaddr(ctypes.Structure):
        _fields_ = [("sa_family", ctypes.c_ushort), ("sa_data", ctypes.c_ubyte * 14)]

    class ifaddrs(ctypes.Structure):
        pass
    ifaddrs._fields_ = [("ifa_next", ctypes.POINTER(ifaddrs)), ("ifa_name", ctypes.c_char_p),
                        ("ifa_flags", ctypes.c_uint), ("ifa_addr", ctypes.POINTER(sockaddr)),
                        ("ifa_netmask", ctypes.POINTER(sockaddr)), ("ifa_ifu", ctypes.POINTER(sockaddr)),
                        ("ifa_data", ctypes.c_void_p)]
    libc = ctypes.CDLL(ctypes.util.find_library("c"), use_errno=True)
    head = ctypes.POINTER(ifaddrs)()
    if libc.getifaddrs(ctypes.byref(head)) != 0:
        return []
    out, p = [], head
    while p:
        ifa = p.contents
        if ifa.ifa_addr and ifa.ifa_addr.contents.sa_family == socket.AF_INET and (ifa.ifa_flags & 1):
            out.append(socket.inet_ntoa(bytes(ifa.ifa_addr.contents.sa_data[2:6])))
        p = ifa.ifa_next
    libc.freeifaddrs(head)
    return out


def test_shard_geometry_properties():
    """Host/device agreement on shard boundaries: for any (groups, world) the per-rank ranges returned by
    the CUDA module's shard_units() (the function the kernels use) tile [0, groups) exactly, in rank order,
    with sizes that differ by at most one chunk, and equal BucketedGradSync.shard_range()'s arithmetic."""
    from hypothesis import given, settings
    from hypothesis import strategies as st

    from byteps_b200 import _native

    cu = _native.cuda()          # imports on CPU: driver entry points are resolved lazily

    @settings(max_examples=300, deadline=None)
    @given(groups=st.integers(0, 1 << 26), world=st.integers(1, 16))
    def check(groups, world):
        prev_end = 0
        per = (groups + world - 1) // world
        for r in range(world):
            b, e = cu.shard_units(groups, world, r)
            assert b == prev_end and b <= e <= groups
            assert (b, e) == (min(per * r, groups), min(min(per * r, groups) + per, groups))
            prev_end = e
        assert prev_end == groups

    check()
    assert cu.SEG_DESC_BYTES == 32 and cu.OPT_HPARAMS_BYTES == 64


def test_compressor_edge_sizes_properties(c):
    """Random sizes (1 .. 5000, not multiples of the word size), k up to and beyond n, constant and zero inputs:
    payload never exceeds max_compressed_bytes(), decompression is finite and obeys each scheme's definition."""
    from hypothesis import given, settings
    from hypothesis import strategies as st

    @settings(max_examples=400, deadline=None)
    @given(n=st.integers(1, 5000), kind=st.sampled_from(["onebit", "onebit_scaled", "topk", "randomk", "dithering"]),
           kfrac=st.floats(0.001, 1.5), seed=st.integers(1, 2 ** 31), fill=st.sampled_from(["randn", "zeros", "const"]))
    def check(n, kind, kfrac, seed, fill):
        rng = np.random.RandomState(seed % (2 ** 31))
        g = {"randn": rng.randn(n), "zeros": np.zeros(n), "const": np.full(n, -2.5)}[fill].astype(np.float32)
        k = max(1, int(kfrac * n))
        kw = {"onebit": {"compressor_type": "onebit"},
              "onebit_scaled": {"compressor_type": "onebit", "compressor_onebit_scaling": "true"},
              "topk": {"compressor_type": "topk", "compressor_k": str(k)},
              "randomk": {"compressor_type": "randomk", "compressor_k": str(k), "seed": str(seed)},
              "dithering": {"compressor_type": "dithering", "compressor_k": "4", "seed": str(seed)}}[kind]
        comp = c.Compressor(kw, n * 4, c.F32)
        cap = comp.max_compressed_bytes()
        buf = np.full(cap + 64, 0xAB, dtype=np.uint8)
        out = np.full(n, np.nan, dtype=np.float32)
        gc = g.copy()
        m = comp.compress(gc.ctypes.data, buf.ctypes.data)
        assert 0 < m <= cap, (kind, n, m, cap)
        assert (buf[cap:] == 0xAB).all()                       # nothing written past the declared capacity
        comp.decompress(buf.ctypes.data, m, out.ctypes.data)
        assert np.isfinite(out).all(), (kind, n)
        if kind == "onebit":
            np.testing.assert_array_equal(out, np.where(g < 0, -1.0, 1.0).astype(np.float32))
        elif kind == "onebit_scaled":
            np.testing.assert_allclose(out, np.where(g < 0, -1.0, 1.0) * np.abs(g).mean(), rtol=1e-5, atol=1e-7)
        elif kind == "topk":
            kk = min(k, n)
            nz = np.flatnonzero(out)
            assert len(nz) <= kk
            assert np.array_equal(out[nz], g[nz])
            if fill == "randn" and kk < n:                    # everything kept is at least as large as anything dropped
                dropped = np.delete(np.abs(g), nz)
                assert np.abs(g[nz]).min() >= dropped.max() - 1e-12
        elif kind == "randomk":
            nz = np.flatnonzero(out)
            assert np.array_equal(out[nz], g[nz]) and len(nz) <= k
        else:
            assert np.abs(out).max() <= np.abs(g).max() * 1.0001 + 1e-6

    check()


def test_meta_decoder_fuzz(c):
    """The wire decoder never trusts lengths: random bytes, truncations and bit flips of valid encodings are
    either decoded or rejected (this test is also part of the AddressSanitizer run, tools/sanitize.sh)."""
    from hypothesis import given, settings
    from hypothesis import strategies as st

    good = c.meta_pack_sample(3, "payload-description")
    assert c.meta_unpack_bytes(good) == (True, 3, len("payload-description"))

    @settings(max_examples=500, deadline=None)
    @given(data=st.binary(min_size=0, max_size=300), cut=st.integers(0, len(good)), flip=st.integers(0, len(good) * 8 - 1))
    def check(data, cut, flip):
        c.meta_unpack_bytes(data)                                   # garbage
        ok, _, _ = c.meta_unpack_bytes(good[:cut])                  # truncation
        assert ok == (cut == len(good))
        b = bytearray(good)
        b[flip // 8] ^= 1 << (flip % 8)
        c.meta_unpack_bytes(bytes(b))                               # single bit flip: any verdict, no crash
        c.meta_unpack_bytes(good + data)                            # trailing bytes

    check()


def test_cpu_reducer_sizes_and_alignment_properties(c):
    """SIMD kernels with scalar tails: any element count (including 0 and non-multiples of the vector width)
    and pointers offset by a few elements from the allocation give the same result as torch."""
    from hypothesis import given, settings
    from hypothesis import strategies as st

    red = c.CpuReducer(2)
    table = {"F32": torch.float32, "F64": torch.float64, "F16": torch.float16, "BF16": torch.bfloat16,
             "I32": torch.int32, "I64": torch.int64, "U8": torch.uint8}

    @settings(max_examples=250, deadline=None)
    @given(n=st.integers(0, 3000), off=st.integers(0, 7), code=st.sampled_from(sorted(table)), seed=st.integers(0, 10 ** 6),
           alpha=st.sampled_from([0.5, -1.25, 2.0]))
    def check(n, off, code, seed, alpha):
        dt = table[code]
        g = torch.Generator().manual_seed(seed)
        def mk():
            base = torch.randn(n + 8, generator=g).to(dt) if dt.is_floating_point else \
                torch.randint(0, 40, (n + 8,), generator=g).to(dt)
            return base, base[off:off + n]
        (_, a), (_, b) = mk(), mk()
        nbytes = n * a.element_size()
        ref = (a.float() + b.float()).to(dt) if dt in (torch.float16, torch.bfloat16) else a + b
        d_base = torch.zeros(n + 8, dtype=dt)
        d = d_base[off:off + n]
        d.copy_(a)
        red.sum(d.data_ptr(), b.data_ptr(), nbytes, getattr(c, code))
        assert torch.equal(d, ref)
        out_base = torch.zeros(n + 8, dtype=dt)
        out = out_base[off:off + n]
        red.sum3(out.data_ptr(), a.data_ptr(), b.data_ptr(), nbytes, getattr(c, code))
        assert torch.equal(out, ref)
        assert (out_base[:off] == 0).all() and (out_base[off + n:] == 0).all()      # nothing outside the range
        if dt.is_floating_point:
            d.copy_(a)
            red.sum_scaled(d.data_ptr(), b.data_ptr(), nbytes, getattr(c, code), alpha)
            want = (a.double() + alpha * b.double()).to(dt)
            tol = 1e-6 if dt in (torch.float32, torch.float64) else 2e-2
            assert torch.allclose(d.double(), want.double(), rtol=tol, atol=tol)

    check()


@pytest.mark.parametrize("code,tdt", [("F16", torch.float16), ("BF16", torch.bfloat16), ("F64", torch.float64)])
def test_compressors_other_float_dtypes(c, code, tdt):
    """The compressors are templated over the element type: onebit / topk / randomk / dithering on half, bfloat16
    and double tensors obey the same definitions as on float (payload record sizes differ per dtype)."""
    n = 3001
    torch.manual_seed(4)
    g = torch.randn(n).to(tdt)
    nbytes = n * g.element_size()
    cases = [{"compressor_type": "onebit", "compressor_onebit_scaling": "true"},
             {"compressor_type": "topk", "compressor_k": "37"},
             {"compressor_type": "randomk", "compressor_k": "37", "seed": "5"},
             {"compressor_type": "dithering", "compressor_k": "8", "seed": "5"},
             {"compressor_type": "topk", "compressor_k": "37", "ef_type": "vanilla"}]
    for kw in cases:
        comp = c.Compressor(kw, nbytes, getattr(c, code))
        cap = comp.max_compressed_bytes()
        buf = torch.full((cap + 32,), 0x5A, dtype=torch.uint8)
        out = torch.full((n,), float("nan")).to(tdt)
        src = g.clone()
        m = comp.compress(src.data_ptr(), buf.data_ptr())
        assert 0 < m <= cap and (buf[cap:] == 0x5A).all(), (kw, m, cap)
        comp.decompress(buf.data_ptr(), m, out.data_ptr())
        assert torch.isfinite(out.float()).all(), kw
        kind = kw["compressor_type"]
        if kind == "onebit":
            scale = g.float().abs().mean()
            want = torch.where(g < 0, -scale, scale).to(tdt)
            assert torch.allclose(out.float(), want.float(), rtol=1e-2), kw
        elif kind == "topk":
            nz = out.float().nonzero().flatten()
            assert len(nz) <= 37 and torch.equal(out[nz], g[nz])
            dropped = g.float().abs().clone()
            dropped[nz] = 0
            assert g.float().abs()[nz].min() >= dropped.max()
        elif kind == "randomk":
            nz = out.float().nonzero().flatten()
            assert len(nz) <= 37 and torch.equal(out[nz], g[nz])
        else:
            assert out.float().abs().max() <= g.float().abs().max() * 1.01 + 1e-6


def test_config_from_env_precedence(monkeypatch):
    """torchrun variables and the BytePS/DMLC variables map onto the same Config; BYTEPS_LOCAL_RANK selects the
    BytePS reading; is_distributed follows the reference's rule; partition bound is rounded per local_size."""
    from byteps_b200.config import Config

    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE", "GROUP_RANK", "BYTEPS_LOCAL_RANK",
              "BYTEPS_LOCAL_SIZE", "DMLC_WORKER_ID", "DMLC_NUM_WORKER", "DMLC_NUM_SERVER", "BYTEPS_GLOBAL_RANK",
              "BYTEPS_FORCE_DISTRIBUTED", "BYTEPS_PARTITION_BYTES"):
        monkeypatch.delenv(k, raising=False)
    c = Config.from_env()
    assert (c.rank, c.size, c.local_rank, c.local_size) == (0, 1, 0, 1) and not c.is_distributed
    monkeypatch.setenv("RANK", "5")
    monkeypatch.setenv("WORLD_SIZE", "16")
    monkeypatch.setenv("LOCAL_RANK", "5")
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "8")
    c = Config.from_env()
    assert (c.rank, c.size, c.local_rank, c.local_size, c.worker_id, c.num_worker) == (5, 16, 5, 8, 0, 2)
    # the launcher's variables win as soon as BYTEPS_LOCAL_RANK is present
    monkeypatch.setenv("BYTEPS_LOCAL_RANK", "3")
    monkeypatch.setenv("BYTEPS_LOCAL_SIZE", "4")
    monkeypatch.setenv("DMLC_WORKER_ID", "2")
    monkeypatch.setenv("DMLC_NUM_WORKER", "3")
    c = Config.from_env()
    assert (c.rank, c.size, c.local_rank, c.local_size) == (3 + 2 * 4, 12, 3, 4)
    assert not c.is_distributed                             # no servers
    monkeypatch.setenv("DMLC_NUM_SERVER", "2")
    assert Config.from_env().is_distributed
    monkeypatch.setenv("DMLC_NUM_WORKER", "1")
    assert not Config.from_env().is_distributed             # one box: NVLink path ...
    monkeypatch.setenv("BYTEPS_FORCE_DISTRIBUTED", "1")
    assert Config.from_env().is_distributed                 # ... unless forced through the servers
    monkeypatch.setenv("BYTEPS_GLOBAL_RANK", "7")
    assert Config.from_env().rank == 7
    monkeypatch.setenv("BYTEPS_PARTITION_BYTES", "1000001")
    c = Config.from_env()
    assert c.partition_bound() % (4 * 4096) == 0 and c.partition_bound() >= 1000001


def test_topk_large_fp32_selection_is_exact(c):
    """Large fp32 tensors take the sampled-threshold path of top-k: the selected set must still be THE k largest
    magnitudes on gaussian, heavy-tailed, tied, mostly-zero and sorted inputs (and ties go to the lower index)."""
    rng = np.random.RandomState(3)
    n = 300_000
    cases = [
        ("0.01", rng.randn(n)),
        ("0.001", rng.standard_cauchy(n)),
        ("5000", rng.randn(n) * np.exp(rng.randn(n) * 3)),
        ("0.02", np.round(rng.randn(n) * 4) / 4),                          # many equal magnitudes
        ("0.01", np.where(rng.rand(n) < 0.003, rng.randn(n), 0.0)),         # fewer non-zeros than k
        ("0.01", np.sort(rng.randn(n))),
    ]
    for kk, g in cases:
        g = g.astype(np.float32)
        comp = c.Compressor({"compressor_type": "topk", "compressor_k": kk}, n * 4, c.F32)
        buf = np.zeros(comp.max_compressed_bytes() + 64, dtype=np.uint8)
        out = np.zeros(n, dtype=np.float32)
        gc = g.copy()
        m = comp.compress(gc.ctypes.data, buf.ctypes.data)
        comp.decompress(buf.ctypes.data, m, out.ctypes.data)
        k = m // 8
        idx = buf[:m].view(np.uint32).reshape(-1, 2)[:, 0]
        assert len(set(idx.tolist())) == k
        a = np.abs(g)
        kth = np.sort(a)[-k]
        sel = np.zeros(n, bool)
        sel[idx] = True
        assert a[sel].min() >= kth and a[~sel].max() <= kth
        assert np.array_equal(out[sel], g[sel]) and not out[~sel].any()
    # deterministic tie rule on the sampled path: equal magnitudes -> lower indices win
    g = np.ones(n, dtype=np.float32)
    g[::2] = -1.0
    g[1000:1200] = 5.0
    comp = c.Compressor({"compressor_type": "topk", "compressor_k": "0.01"}, n * 4, c.F32)
    buf = np.zeros(comp.max_compressed_bytes() + 64, dtype=np.uint8)
    m = comp.compress(g.copy().ctypes.data if False else g.ctypes.data, buf.ctypes.data)
    idx = np.sort(buf[:m].view(np.uint32).reshape(-1, 2)[:, 0])
    assert set(range(1000, 1200)) <= set(idx.tolist()) and len(idx) == 3000


def test_elias_delta_multibit_codec_roundtrip(c):
    """dithering payloads written with the multi-bit writer decode to what was encoded (all four variants, odd sizes)."""
    rng = np.random.RandomState(11)
    for n in (1, 31, 1000, 70001):
        g = (rng.randn(n) * np.exp(rng.randn(n))).astype(np.float32)
        for part in ("linear", "natural"):
            kw = {"compressor_type": "dithering", "compressor_k": "7", "seed": "5",
                  "dithering_partition": "0" if part == "linear" else "1"}
            comp = c.Compressor(kw, n * 4, c.F32)
            buf = np.zeros(comp.max_compressed_bytes() + 64, dtype=np.uint8)
            out = np.zeros(n, dtype=np.float32)
            m = comp.compress(g.ctypes.data, buf.ctypes.data)
            comp.decompress(buf.ctypes.data, m, out.ctypes.data)
            scale = np.abs(g).max()
            levels = 7 if part == "linear" else 64
            q = np.abs(out) / scale * levels
            assert np.allclose(q, np.round(q), atol=1e-3)                  # every value sits on a quantisation level
            assert np.all(np.sign(out[out != 0]) == np.sign(g[out != 0]))
            if part == "linear":                                           # stochastic rounding moves < one level
                assert np.all(np.abs(np.abs(out) - np.abs(g)) <= scale / levels + 1e-6)
            else:                                                          # natural: levels are powers of two
                nz = q[q > 0]
                assert np.allclose(np.log2(nz), np.round(np.log2(nz)), atol=1e-3)


@pytest.mark.parametrize("code,tdt", [("F32", "float32"), ("F64", "float64"), ("F16", "float16"), ("BF16", "bfloat16")])
def test_decompress_add_equals_decompress_then_sum(c, code, tdt):
    """The server's accumulate-in-place path (dst += D(payload)) is bit-identical to decompressing into a scratch
    buffer and adding it, for every compressor and dtype - including random-k payloads that repeat an index."""
    import torch

    dt = getattr(torch, tdt)
    rng = np.random.RandomState(21)
    for n in (7, 64, 1000, 70003):
        configs = [{"compressor_type": "onebit", "compressor_onebit_scaling": "true"},
                   {"compressor_type": "topk", "compressor_k": "0.05"},
                   {"compressor_type": "randomk", "compressor_k": str(max(2, n // 2)), "seed": "3"},   # many duplicates
                   {"compressor_type": "dithering", "compressor_k": "5", "seed": "3"},
                   {"compressor_type": "topk", "compressor_k": "0.05", "ef_type": "vanilla"}]
        for kw in configs:
            g = torch.from_numpy(rng.randn(n).astype(np.float32)).to(dt)
            base = torch.from_numpy(rng.randn(n).astype(np.float32)).to(dt)
            es = g.element_size()
            comp = c.Compressor(kw, n * es, getattr(c, code), True)
            buf = np.zeros(comp.max_compressed_bytes() + 64, dtype=np.uint8)
            m = comp.compress(g.clone().data_ptr() if False else g.data_ptr(), buf.ctypes.data)
            dense = torch.zeros(n, dtype=dt)
            comp.decompress(buf.ctypes.data, m, dense.data_ptr())
            want = base.clone()
            c.CpuReducer(1).sum(want.data_ptr(), dense.data_ptr(), n * es, getattr(c, code))
            got = base.clone()
            comp.decompress_add(buf.ctypes.data, m, got.data_ptr())
            assert torch.equal(got.view(torch.uint8), want.view(torch.uint8)), (kw, n, code)


def test_every_environment_variable_read_by_the_code_is_documented():
    """docs/env.md is the configuration reference: a knob the code reads but the page does not name is a bug."""
    import glob
    import re

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = set()
    for f in glob.glob(os.path.join(root, "byteps_b200", "**", "*"), recursive=True):
        if not f.endswith((".py", ".cc", ".h", ".cu", ".cuh")) or os.sep + "build" + os.sep in f:
            continue
        s = open(f, errors="ignore").read()
        names.update(re.findall(r'env_(?:int|str|bool|has)\(\s*"([A-Z0-9_]+)"', s))
        names.update(re.findall(r'(?:environ\.get|getenv|environ\.setdefault)\(\s*[\'"]((?:BYTEPS|DMLC|PS)_[A-Z0-9_]+)[\'"]', s))
    page = os.path.join(root, "docs", "env.md")
    if not os.path.exists(page):
        pytest.skip("docs/ is not part of this copy of the tree")
    doc = open(page).read()
    missing = sorted(n for n in names if n not in doc)
    assert len(names) > 60 and not missing, missing


def test_numa_helpers_degrade_gracefully(c, monkeypatch):
    """core/numa.h: sysfs parsing, the init-push hint codec, and the syscalls must never fail hard - the build
    container has one node and may forbid mbind / move_pages altogether."""
    import ctypes

    assert c.parse_cpu_list("0-3,8,10-11") == [0, 1, 2, 3, 8, 10, 11]
    assert c.parse_cpu_list("") == [] and c.parse_cpu_list("5") == [5]
    for pushers, node in ((0, -1), (2, 0), (8, 1), (65535, 7), (3, 254)):
        h = c.numa_pack_head(pushers, node)
        assert c.numa_head_pushers(h) == pushers and c.numa_head_node(h) == node
    assert c.numa_head_node(c.numa_pack_head(4, 300)) == -1          # out of range: no hint rather than a wrong one
    assert c.numa_num_nodes() >= 1
    monkeypatch.setenv("BYTEPS_NUMA_FAKE_NODES", "2")
    assert c.numa_num_nodes() == 2
    monkeypatch.delenv("BYTEPS_NUMA_FAKE_NODES")
    assert c.numa_node_of_pci("ffff:ff:1f.7") == -1                  # no such device
    assert not c.numa_aware()
    monkeypatch.setenv("BYTEPS_NUMA_AWARE", "1")
    assert c.numa_aware()
    buf = ctypes.create_string_buffer(1 << 20)
    addr = ctypes.addressof(buf)
    ok = c.numa_bind_memory(addr, 1 << 20, 0)                        # node 0 always exists; a sandbox may still refuse
    assert ok in (True, False)
    buf[0] = b"x"
    assert c.numa_node_of_addr(addr) in (-1, 0) or c.numa_num_nodes() > 1
    assert c.numa_bind_memory(addr, 1 << 20, 1000) is False          # no such node: refused, not fatal
    assert c.numa_bind_memory(0, 0, 0) is False
    cpus = c.numa_cpus_of_node(0)
    assert c.numa_cpus_of_node(999) == []
    if cpus:
        assert c.numa_pin_thread_to_node(0) in (True, False)
    assert c.numa_pin_thread_to_node(999) is False
    assert c.numa_prefer_node_for_process(999) == 0
    if cpus:
        assert c.numa_prefer_node_for_process(0) in (0, 1, 2, 3)       # 3 = CPUs and memory policy set


def test_shm_registry_lookup_and_stale_reaping(c, tmp_path):
    """ShmRegistry: address -> (name, offset) for any pointer inside a mapped object (ordered by base address),
    and objects named after a pid that no longer exists are reaped while live ones stay."""
    import os
    import subprocess
    import sys

    names = ["BytePS_ShM_%d_unit%d" % (os.getpid(), i) for i in range(5)]
    ptrs = [c.shm_create(n, 8192) for n in names]
    try:
        for n, p in zip(names, ptrs):
            assert c.shm_lookup(p, 8192) == (n, 0)
            assert c.shm_lookup(p + 4096, 4096) == (n, 4096)
            assert c.shm_lookup(p + 4096, 8192) is None          # runs past the end of the object
        assert c.shm_lookup(min(ptrs) - 4096, 16) is None or c.shm_lookup(min(ptrs) - 4096, 16)[0] not in names
    finally:
        for n in names:
            c.shm_release(n)
    assert c.shm_lookup(ptrs[0], 16) is None
    # a pid that certainly is dead: a child that has exited and been waited for
    child = subprocess.Popen([sys.executable, "-c", "pass"])
    child.wait()
    d = str(tmp_path)
    dead = ["BytePS_ShM_%d_x" % child.pid, "BytePS_SrvStore_%d_7_0" % child.pid]
    live = ["BytePS_ShM_%d_y" % os.getpid(), "BytePS_SrvStore_%d_7_1" % os.getpid(), "unrelated_%d" % child.pid,
            "BytePS_ShM_notapid"]
    for n in dead + live:
        open(os.path.join(d, n), "w").close()
    assert c.shm_reap_stale(d) == len(dead)
    left = sorted(os.listdir(d))
    assert left == sorted(live)


def test_ready_table_blocking_wait(c):
    import threading
    import time

    t = c.ReadyTable(2, "unit")
    assert not t.wait_ready(5, 20)                     # times out: nobody has arrived
    threading.Thread(target=lambda: (time.sleep(0.05), t.add_ready_count(5), t.add_ready_count(5))).start()
    assert t.wait_ready(5, 5000) and t.is_key_ready(5)
    t.clear_ready_count(5)
    assert not t.is_key_ready(5)


def _host_reduce_rank(rank, world, tag, tmp):
    import numpy as np

    from byteps_b200 import _native

    c = _native.core()
    hr = c.HostLocalReduce(rank, world, tag, 2, tmp)
    assert hr.is_root() == (rank == world - 1)
    for key, n, dt, code in ((11, 100_003, np.float32, c.F32), (12, 4097, np.float64, c.F64), (13, 33, np.int32, c.I32)):
        for rnd in range(3):
            x = ((np.arange(n) + rnd) % 13).astype(dt) * (rank + 1)
            out = np.zeros_like(x)
            assert hr.contribute(key, x.ctypes.data, x.nbytes, 20000)
            if hr.is_root():
                win = hr.reduce(key, x.nbytes, code, 20000)
                assert win and win == hr.window(key)
                assert hr.publish(key, out.ctypes.data, x.nbytes, 20000)
            else:
                assert hr.collect(key, out.ctypes.data, x.nbytes, 20000, code)
            ref = ((np.arange(n) + rnd) % 13).astype(dt) * sum(r + 1 for r in range(world))
            np.testing.assert_array_equal(out, ref)
    if hr.is_root():
        assert hr.signals_received() == 3 * 9 * (world - 1)       # READY, shard done and BCAST_READY per follower per round


def test_host_local_reduce_three_ranks(sock_dir):
    """csrc/core/host_reduce.h by itself: slots in shared memory, READY / DO_BROADCAST / BCAST_READY datagrams,
    CpuReducer sum on the root, window reuse across rounds."""
    import os

    from _mp import run_workers

    run_workers(_host_reduce_rank, world=3, args=("unit%d" % os.getpid(), sock_dir), timeout=120)


def _host_reduce_timeouts(rank, world, tag, tmp):
    import time

    import numpy as np

    from byteps_b200 import _native

    c = _native.core()
    hr = c.HostLocalReduce(rank, world, tag, 1, tmp)
    x = np.ones(1000, dtype=np.float32)
    out = np.zeros_like(x)
    if hr.is_root():
        # the follower never contributes to key 1: the root's wait ends with "no window", not with a hang
        assert hr.contribute(1, x.ctypes.data, x.nbytes, 5000)
        t0 = time.time()
        assert hr.reduce(1, x.nbytes, c.F32, 300) == 0
        assert 0.2 < time.time() - t0 < 5
        # key 2 is a normal round, so both sides leave in step
        assert hr.contribute(2, x.ctypes.data, x.nbytes, 5000) and hr.reduce(2, x.nbytes, c.F32, 20000)
        assert hr.publish(2, out.ctypes.data, x.nbytes, 20000)
    else:
        # nothing was ever announced for key 3: collect gives up after its timeout
        t0 = time.time()
        assert not hr.collect(3, out.ctypes.data, x.nbytes, 300)
        assert 0.2 < time.time() - t0 < 5
        assert hr.contribute(2, x.ctypes.data, x.nbytes, 20000) and hr.collect(2, out.ctypes.data, x.nbytes, 20000, c.F32)
    assert np.all(out == world)


def test_host_local_reduce_timeouts_do_not_hang(sock_dir):
    import os

    from _mp import run_workers

    run_workers(_host_reduce_timeouts, world=2, args=("tmo%d" % os.getpid(), sock_dir), timeout=120)
