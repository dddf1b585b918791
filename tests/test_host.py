"""Host side of the product through the C ABI vs the oracle: worker protocol, reader stack, layout, errors.

CPU only (no kernels are launched).  Scenarios follow the reference's own tests:
  curvine-server/tests/worker_test.rs:49-176   hand-built Open -> Running x N -> Complete, sum-crc both sides
  orpc/tests/file_test.rs:44-134               100 x 64 KiB frames
  curvine-tests/tests/block_test.rs:33-103,209-302   full stack, {short-circuit, remote} x {parallel 1, 4} x chunk sizes
"""
import ctypes
import os
import socket
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import pytest

from curvine_b200 import _lib, fs as F
from oracle import clib, layout, synth
from oracle import reader_model as RM
from oracle import wire as W


@pytest.fixture(scope="module")
def cluster(tmp_path_factory):
    d = tmp_path_factory.mktemp("worker")
    w = F.MiniWorker(["[MEM:10MB]" + str(d / "mem"), "[SSD]" + str(d / "ssd")], cluster_id="curvine")
    yield w, d
    w.stop()


def test_library_exports_every_declared_symbol():
    L = _lib.lib()
    for name in _lib.EXPORTS:
        assert hasattr(L, name), name
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    declared = set()
    for h in ("curvine_b200.h", "curvine_b200_kernels.h"):
        declared |= set(re.findall(r"\b(cv[kh]?_[a-z0-9_]+)\s*\(", open(os.path.join(root, "include", h)).read()))
    declared -= {"cv_stream_t", "cv_event_t"}
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)


def test_null_handles_and_out_pointers_are_errors_not_crashes():
    """include/curvine_b200.h: entry points never throw or abort.  Every cv_* function called with NULL for every pointer argument
    (and 0 for every integer) must come back -- with a negative ErrorKind where a handle or a required out-pointer is missing -- in a
    subprocess, so a crash is a test failure and not the end of the test run."""
    import subprocess
    import sys
    code = """
import ctypes, sys
sys.path.insert(0, %r)
from curvine_b200 import _lib
L = _lib.lib()
bad = []
for name in _lib.EXPORTS:
    if not name.startswith("cv_"):
        continue
    fn = getattr(L, name)
    args = []
    for t in (fn.argtypes or []):
        args.append(None if (t in (ctypes.c_void_p, ctypes.c_char_p) or hasattr(t, "contents") or hasattr(t, "_type_") and isinstance(t._type_, type)) else 0)
    rc = fn(*args)
    if name in ("cv_open", "cv_read", "cv_seek", "cv_verify", "cv_read_device", "cv_fs_load_namespace_string", "cv_worker_hbm_load", "cv_writer_open",
                "cv_write", "cv_device_stats", "cv_fs_pool_stats", "cv_worker_metrics", "cv_shard_plan", "cv_read_many_device") and not (isinstance(rc, int) and rc < 0):
        bad.append((name, rc))
print("survived", bad)
assert not bad, bad
""" % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert r.returncode == 0 and "survived []" in r.stdout, (r.returncode, r.stdout[-1500:])


def test_tuning_hook_validates_its_arguments_without_a_gpu():
    """cvk_tune only flips process-wide launch choices: legal values are accepted, everything else is cudaErrorInvalidValue (1)."""
    L = _lib.lib()
    for what, value in ((0, 2), (0, 4), (1, 4), (1, 2), (3, 1), (3, 0)):
        assert L.cvk_tune(what, value) == 0
    for what, value in ((0, 3), (1, 8), (2, 1), (3, 2), (9, 0)):
        assert L.cvk_tune(what, value) == 1
    assert L.cvk_tune(0, 4) == 0 and L.cvk_tune(1, 2) == 0 and L.cvk_tune(3, 0) == 0  # back to the defaults


def test_host_crc_and_generator_match_oracle():
    L = _lib.lib()
    rng = np.random.default_rng(0)
    for n in (0, 1, 7, 8, 9, 4095, 4096, 1 << 20):
        d = rng.bytes(n)
        for p in (0, 1):
            assert L.cv_host_crc(p, d, n) == clib.crc(p, d)
    buf = ctypes.create_string_buffer(100003)
    L.cv_synth_block(1001, 7, buf, 100003)
    assert buf.raw == synth.block_bytes(1001, 7, 100003)


def _recv(sock, n):
    out = bytearray()
    while len(out) < n:
        c = sock.recv(n - len(out))
        assert c, "connection closed"
        out += c
    return bytes(out)


def _rpc(sock, msg):
    sock.sendall(W.encode(msg))
    code, rq, rs, req_id, seq_id, hsz, dsz = W.decode_protocol(_recv(sock, 22))
    return W.Message(code, rq, rs, req_id, seq_id, _recv(sock, hsz), _recv(sock, dsz))


@pytest.mark.parametrize("chunk,count", [(1024, 100), (65536, 100)])
def test_worker_protocol_hand_built_messages(cluster, chunk, count):
    """worker_test.rs:49-176 / file_test.rs:44-134: the oracle codec drives the product worker over TCP."""
    w, d = cluster
    n = chunk * count + 37
    ino = 2000 + chunk
    man = w.create_file("/wt/%d" % chunk, ino, n, 1 << 30, storage_type=0)
    want = synth.block_bytes(ino, 0, n)
    bid = layout.create_block_id(ino, 0)
    # on-disk layout is the reference's (block_meta.rs:199-237); [MEM:10MB] dir chosen for storage_type Mem
    path = layout.block_path(str(d / "mem" / "curvine"), bid)
    assert os.path.getsize(path) == n and open(path, "rb").read() == want
    assert (" %d " % 0) in man.splitlines()[2]
    s = socket.create_connection(("127.0.0.1", w.port))
    rid = 0x1122334455667788
    o = _rpc(s, W.request(81, W.REQ_OPEN, rid, 0, W.BlockReadRequest(bid, 0, n, chunk, False, True, 1 << 20, 1 << 20).encode()))
    assert (o.code, o.req_status, o.resp_status, o.req_id, o.seq_id) == (81, W.REQ_OPEN, W.RESP_SUCCESS, rid, 0)
    r = W.BlockReadResponse.decode(o.header)
    assert (r.id, r.len, r.path, r.storage_type) == (bid, n, None, W.STORAGE_MEM)
    got, seq, rsum = bytearray(), 0, 0
    while len(got) < n:
        seq += 1
        m = _rpc(s, W.request(81, W.REQ_RUNNING, rid, seq))
        assert m.is_success() and m.seq_id == seq and m.req_id == rid and m.header == b""
        assert len(m.data) == min(chunk, n - len(got))  # local_file.rs:103-117
        rsum += zlib.crc32(m.data)
        got += m.data
    assert bytes(got) == want
    assert rsum == sum(zlib.crc32(want[i:i + chunk]) for i in range(0, n, chunk))  # write-side sum == read-side sum
    # reading past the end is an error *response* (0x13), not a dropped connection (block_handler.rs:57-60)
    e = _rpc(s, W.request(81, W.REQ_RUNNING, rid, seq + 1))
    assert e.resp_status == W.RESP_ERROR and e.status_byte() == 19 and "offset exceeds file length" in W.decode_error(e.data)[1]
    # seek piggy-backed on a Running request (DataHeaderProto.offset is absolute in the block file)
    m = _rpc(s, W.request(81, W.REQ_RUNNING, rid, seq + 2, W.DataHeaderProto(12345).encode()))
    assert m.data == want[12345:12345 + chunk]
    c = _rpc(s, W.request(81, W.REQ_COMPLETE, rid, seq + 3, W.BlockReadRequest(id=bid).encode()))
    assert c.is_success() and c.req_status == W.REQ_COMPLETE and c.data == b"" and c.header == b""
    # short-circuit open returns the block file path and no data is served (read_handler.rs:87-95,115-120)
    o = _rpc(s, W.request(81, W.REQ_OPEN, rid + 1, 0, W.BlockReadRequest(bid, 0, n, chunk, True).encode()))
    assert W.BlockReadResponse.decode(o.header).path == path
    e = _rpc(s, W.request(81, W.REQ_RUNNING, rid + 1, 1))
    assert e.resp_status == W.RESP_ERROR
    # errors: unknown block, bad chunk size, oversized read-ahead, unsupported code
    e = _rpc(s, W.request(81, W.REQ_OPEN, 5, 0, W.BlockReadRequest(424242, 0, 1, chunk).encode()))
    assert e.resp_status == W.RESP_ERROR and W.decode_error(e.data)[0] == 10000
    e = _rpc(s, W.request(81, W.REQ_OPEN, 5, 0, W.BlockReadRequest(bid, 0, n, 0).encode()))
    assert "chunk_size must be greater than 0" in W.decode_error(e.data)[1]
    e = _rpc(s, W.request(81, W.REQ_OPEN, 5, 0, W.BlockReadRequest(bid, 0, n, chunk, False, True, (16 << 20) + 1).encode()))
    assert e.resp_status == W.RESP_ERROR
    e = _rpc(s, W.request(81, W.REQ_OPEN, 5, 0, W.BlockReadRequest(bid, n + 1, n, chunk).encode()))
    assert "exceeds the maximum length" in W.decode_error(e.data)[1]
    e = _rpc(s, W.request(99, W.REQ_OPEN, 5, 0))
    assert e.resp_status == W.RESP_ERROR
    # heartbeats are skipped (rpc_frame.rs:255-259)
    s.sendall(W.encode(W.Message(0, W.REQ_HEARTBEAT, W.RESP_UNDEFINED, -1, -1)))
    assert _rpc(s, W.request(81, W.REQ_COMPLETE, 9, 9)).is_success()
    s.close()
    assert w.metrics()["read_count"] >= count


def _model_for(ino, n, bs, conf, hole_every=0):
    data = bytearray(synth.file_bytes(ino, n, bs))
    blocks = []
    for i in range((n + bs - 1) // bs):
        blen = min(bs, n - i * bs)
        hole = hole_every > 0 and i % hole_every == hole_every - 1
        if hole:
            data[i * bs:i * bs + blen] = bytes(blen)
        blocks.append(RM.BlockSpec(layout.create_block_id(ino, i), blen, hole))
    return RM.ReaderModel(RM.FileModel(blocks, bytes(data)), conf), bytes(data)


@pytest.mark.parametrize("short_circuit", [True, False])
@pytest.mark.parametrize("chunk_kb,chunk_num,parallel", [(128, 8, 1), (64, 1, 1), (64, 4, 4)])
def test_block_test_scenario_matrix(cluster, short_circuit, chunk_kb, chunk_num, parallel):
    """block_test.rs:33-103,209-302: 1 MiB blocks, 1 KiB reads, sum-crc + length, then seeks across block/chunk edges."""
    w, _ = cluster
    bs, n = 1 << 20, 10240 * 1024 + 13
    ino = 3000 + chunk_kb + parallel + (500 if short_circuit else 0)
    man = w.create_file("/bt/%d" % ino, ino, n, bs)
    conf = F.client_conf(short_circuit=short_circuit, read_chunk_size="%dKB" % chunk_kb, read_chunk_num=chunk_num, read_parallel=parallel)
    mconf = RM.ClientConf(read_chunk_size=chunk_kb * 1024, read_chunk_num=chunk_num, read_parallel=parallel, short_circuit=short_circuit)
    model, data = _model_for(ino, n, bs, mconf)
    with F.CurvineFileSystem(conf) as fs:
        fs.load_namespace(man)
        r = fs.open("/bt/%d" % ino)
        assert r.len() == n and r.chunk_size() == chunk_kb * 1024
        total, cks = 0, 0
        while True:
            b = r.read(1024)
            assert b == model.read(1024)  # same bytes AND the same short reads at chunk boundaries
            if not b:
                break
            total += len(b)
            cks += zlib.crc32(b)
        assert total == n and r.pos() == n == model.pos
        assert cks & (2 ** 64 - 1) == sum(zlib.crc32(data[i:i + 1024]) for i in range(0, n, 1024))
        for pos in (bs, bs, bs - 1, bs + 64 * 1024 - 1024, bs + 64 * 1024, 0, n - 5, n):
            r.seek(pos)
            model.seek(pos)
            got = r.read_full(1024)
            assert got == data[pos:pos + 1024] == model.read_full(1024)
            assert r.pos() == min(n, pos + 1024) == model.pos
        # fuse-shaped read: whole chunks after a seek (reader.rs:101-124)
        segs = r.fuse_read(3 * bs + 4096, 300000)
        assert segs == model.fuse_read(3 * bs + 4096, 300000) and b"".join(segs) == data[3 * bs + 4096:3 * bs + 4096 + 300000]
        # blocking_read hands out the whole current chunk
        r.seek(5 * bs - 100)
        model.seek(5 * bs - 100)
        assert r.read_chunk() == model.blocking_read() == data[5 * bs - 100:5 * bs]
        r.seek(n + 1)  # clamped by FsReaderParallel::seek in the reference: no error, reads return nothing
        assert r.read(10) == b"" and r.pos() == n + 1
        with pytest.raises(F.FsError):
            r.seek(-1)
        r.complete()
        assert fs.metrics()["read_bytes"] >= n


def test_hole_blocks_read_as_zeros(cluster):
    """block_reader_hole.rs:69-79."""
    w, _ = cluster
    bs, n, ino = 1 << 20, (5 << 20) + 100, 4100
    man = w.create_file("/holes", ino, n, bs, mode=2, hole_every=2)
    model, data = _model_for(ino, n, bs, RM.ClientConf(), hole_every=2)
    assert data[bs:2 * bs] == bytes(bs)
    with F.CurvineFileSystem(F.client_conf()) as fs:
        fs.load_namespace(man)
        with fs.open("/holes") as r:
            assert r.read_full(n) == data


def test_az_mode_and_bench_checksum(cluster):
    """curvine-bench shape: repeated a-z buffer, 128 KiB read_full loop, sum of crc32 (curvine_bench.rs:212-236)."""
    w, _ = cluster
    n = 3 * (1 << 20) + 128 * 1024
    man = w.create_file("/az", 4200, n, 1 << 20, mode=1)
    with F.CurvineFileSystem(F.client_conf(short_circuit=False)) as fs:
        fs.load_namespace(man)
        with fs.open("/az") as r:
            cks, total, whole = 0, 0, bytearray()
            while True:
                b = r.read_full(128 * 1024)
                if not b:
                    break
                cks += zlib.crc32(b)
                total += len(b)
                whole += b
    assert total == n and set(whole) <= set(range(ord("a"), ord("z") + 1))
    assert whole[:131072] == whole[131072:262144]
    assert cks == clib.bench_checksum(bytes(whole), 128 * 1024)


def test_errors_map_to_reference_error_kinds(cluster):
    w, d = cluster
    with F.CurvineFileSystem(F.client_conf()) as fs:
        with pytest.raises(F.FsError) as ei:
            fs.open("/nope")
        assert ei.value.kind == 8  # FileNotFound
        # chunk_size must be a multiple of 4 KiB; slice a multiple of chunk (fs_reader_parallel.rs:62-71)
    man = w.create_file("/e1", 4300, 1 << 20, 1 << 20)
    with F.CurvineFileSystem(F.client_conf(read_chunk_size="5000")) as fs:
        fs.load_namespace(man)
        with pytest.raises(F.FsError) as ei:
            fs.open("/e1")
        assert "integer multiple" in ei.value.msg
    # a block file that vanished: short-circuit open fails on the client, remote gets an error response; kind Common / IO
    bid = layout.create_block_id(4300, 0)
    os.remove(layout.block_path(str(d / "mem" / "curvine"), bid))
    for sc in (True, False):
        with F.CurvineFileSystem(F.client_conf(short_circuit=sc)) as fs:
            fs.load_namespace(man)
            r = fs.open("/e1")
            with pytest.raises(F.FsError) as ei:
                r.read(10)
            assert ei.value.kind in (1, 10000)
    # a worker that is not there
    man2 = man.replace(":%d:" % w.port, ":1:")
    with F.CurvineFileSystem(F.client_conf()) as fs:
        fs.load_namespace(man2)
        r = fs.open("/e1")
        with pytest.raises(F.FsError) as ei:
            r.read(10)
        assert ei.value.kind == 1  # IO


def test_conf_parsing_matches_reference_rules():
    """ByteUnit binary sizes (byte_unit.rs:29-34,76-125); read_slice/read_ahead defaults (client_conf.rs:228-281)."""
    with F.CurvineFileSystem('[client]\nread_chunk_size = "64kb"\nread_chunk_num = 4\n') as fs:
        pass
    with pytest.raises(F.FsError):
        F.CurvineFileSystem('[client]\nread_chunk_size = "64XB"\n')


def test_duration_strings_and_block_conn_pool_semantics(cluster):
    """block_client_pool.rs:102-168 + client_conf.rs:406-413 + duration_unit.rs:66-108: connections are reused LIFO per worker;
    the pool keeps at most block_conn_idle_size idle connections over all workers (extra ones are closed on release); a pooled
    connection that sat idle for block_conn_idle_time or longer is dropped at the next acquire."""
    import time
    w, _ = cluster
    man = "".join(w.create_file("/pool/f%d" % i, 4800 + i, 1 << 20, 1 << 18) for i in range(3))  # 3 files x 4 blocks

    def read_all(fs, name):
        r = fs.open(name)
        got = r.read_full(1 << 20)
        r.complete()
        return got

    for bad in ("10x", "abc", "-5s"):
        with pytest.raises(F.FsError):
            F.CurvineFileSystem('[client]\nblock_conn_idle_time = "%s"\n' % bad)
    for ok in ("60s", "5m", "2h", "1d", "250ms", "250", "1.5s"):
        F.CurvineFileSystem('[client]\nblock_conn_idle_time = "%s"\n' % ok).close()
    # reuse: sequential block readers of one file and of the next file share one pooled connection
    with F.CurvineFileSystem(F.client_conf(short_circuit=False)) as fs:
        fs.load_namespace(man)
        assert read_all(fs, "/pool/f0") == synth.file_bytes(4800, 1 << 20, 1 << 18)
        read_all(fs, "/pool/f1")
        st = fs.pool_stats()
        # (the reader opens block k+1 while block k's reader is still alive, so two connections alternate for any number of blocks)
        assert 1 <= st["opened"] <= 2 and st["idle"] == st["opened"] and st["expired"] == 0, st
    # global idle cap: 4 parallel sub-readers open 4 connections, only block_conn_idle_size = 2 stay pooled
    with F.CurvineFileSystem(F.client_conf(short_circuit=False, read_parallel=4, read_chunk_size="64KB", read_chunk_num=1,
                                           extra_client="block_conn_idle_size = 2")) as fs:
        fs.load_namespace(man)
        read_all(fs, "/pool/f2")
        st = fs.pool_stats()
        assert st["opened"] >= 2 and st["idle"] <= 2, st
    # idle-time expiry: the pooled connection is 80 ms old when the next reader asks, the limit is 50 ms -> dropped, a new one opened
    with F.CurvineFileSystem(F.client_conf(short_circuit=False, extra_client='block_conn_idle_time = "50ms"')) as fs:
        fs.load_namespace(man)
        read_all(fs, "/pool/f0")
        st0 = fs.pool_stats()
        assert st0["idle"] == st0["opened"] >= 1 and st0["expired"] == 0, st0
        time.sleep(0.08)
        r = fs.open("/pool/f1")
        r.read(10)
        st = fs.pool_stats()
        # every stale one met was dropped and a fresh connection opened (on a loaded machine the prefetcher's next block may already have needed
        # a second one: the connection released in between has aged past 50 ms too)
        assert st["expired"] >= st0["idle"] and st["opened"] >= st0["opened"] + 1, (st0, st)
        r.complete()
    # pool disabled: nothing is kept
    with F.CurvineFileSystem(F.client_conf(short_circuit=False, extra_client="enable_block_conn_pool = false")) as fs:
        fs.load_namespace(man)
        read_all(fs, "/pool/f0")
        st = fs.pool_stats()
        assert st["idle"] == 0 and st["opened"] == 4, st  # one connection per block reader


def test_pooled_connections_to_a_restarted_worker_are_not_reused(tmp_path):
    """A worker restart leaves the client's pooled sockets with a FIN queued.  The pool checks a connection (non-blocking
    peek) before handing it out, so the first read after the restart opens a fresh connection instead of failing on a dead
    one (the reference only has the 60 s idle expiry for this; every stale connection there costs one failed read)."""
    d = tmp_path / "w"
    n, ino = (3 << 20) + 7, 4900
    w = F.MiniWorker(["[MEM]" + str(d)])
    try:
        man = w.create_file("/restart", ino, n, 1 << 20)
        want = synth.file_bytes(ino, n, 1 << 20)
        for sc in (False, True):
            with F.CurvineFileSystem(F.client_conf(short_circuit=sc)) as fs:
                fs.load_namespace(man)
                r = fs.open("/restart")
                assert r.read_full(n) == want
                r.complete()
                st0 = fs.pool_stats()
                assert st0["idle"] >= 1
                port = w.port
                w.stop()
                w = F.MiniWorker(["[MEM]" + str(d)], port=port)
                r = fs.open("/restart")
                assert r.read_full(n) == want
                r.complete()
                st = fs.pool_stats()
                assert st["expired"] >= 1 and st["opened"] > st0["opened"], (st0, st)
    finally:
        w.stop()


def test_storage_tier_selection(cluster):
    """storage policy: blocks go to a dir of the file's storage type, falling back to Disk dirs (policy.rs:56-105)."""
    w, d = cluster
    w.create_file("/ssd1", 4400, 1 << 20, 1 << 20, storage_type=1)
    assert os.path.exists(layout.block_path(str(d / "ssd" / "curvine"), layout.create_block_id(4400, 0)))


@pytest.mark.parametrize("sc", [True, False])
@pytest.mark.parametrize("parallel", [1, 3])
def test_oracle_cpu_reader_against_product_worker(cluster, sc, parallel):
    """The C restatement of the reference client (oracle/cpu_reader.c) reads the product worker's blocks and
    reproduces the curvine-bench checksum (sum of crc32 over 128 KiB buffers) of the oracle generator's bytes."""
    w, _ = cluster
    bs, n, ino = 1 << 20, (7 << 20) + 4096 * 3, 4500 + parallel
    w.create_file("/cpu%d" % ino, ino, n, bs)
    ids = [layout.create_block_id(ino, i) for i in range((n + bs - 1) // bs)]
    data = synth.file_bytes(ino, n, bs)
    got, cks, threads = clib.cpu_read_file(w.port, sc, n, bs, ids, 131072, 8, parallel, 131072)
    assert got == n and threads == parallel + 1 and cks == clib.bench_checksum(data, 131072)
    got, cks, _ = clib.cpu_read_file(w.port, sc, n, bs, ids, 65536, 4, parallel, 131072, limit=3 << 20, checksum=0)
    assert got == 3 << 20 and cks == clib.bench_checksum(data[:3 << 20], 131072)
    assert clib.crc32_pclmul(data) == zlib.crc32(data)


def test_replica_failover_on_read_error(tmp_path):
    """block_reader.rs:217-254: a read error drops that worker and reopens at pos on the next replica.
    (Open-time errors are NOT failed over in the reference -- the `?` inside get_reader's block propagates,
    block_reader.rs:168-215 -- so the test kills the worker that serves the block being read, mid-block.)"""
    import shutil
    d1, d2 = tmp_path / "w1", tmp_path / "w2"
    n, ino = (4 << 20) + 99, 4600
    w1 = F.MiniWorker(["[MEM]" + str(d1)])
    man = w1.create_file("/ha", ino, n, 8 << 20)  # one block
    shutil.copytree(str(d1), str(d2))
    w2 = F.MiniWorker(["[MEM]" + str(d2)])  # rescans active/ on start (vfs_dir.rs:339-362)
    assert w2.metrics()["num_blocks"] == 1
    want = synth.file_bytes(ino, n, 8 << 20)
    man2 = "\n".join(l + ",localhost:%d:2" % w2.port if l.startswith("block ") else l for l in man.splitlines())
    try:
        with F.CurvineFileSystem(F.client_conf(short_circuit=False, read_chunk_size="64KB")) as fs:
            fs.load_namespace(man2)
            r = fs.open("/ha")
            got = r.read_full((1 << 20) + 5000)
            serving = w1 if w1.metrics()["read_blocks_remote"] else w2
            assert (w1.metrics()["read_blocks_remote"] + w2.metrics()["read_blocks_remote"]) == 1
            serving.stop()
            got += r.read_full(n)
            assert got == want and r.pos() == n
            other = w2 if serving is w1 else w1
            assert other.metrics()["read_blocks_remote"] == 1  # reopened at pos on the surviving replica
            r.complete()
    finally:
        w1.stop()
        w2.stop()


def test_hung_worker_times_out_with_an_io_error(cluster):
    """client_conf.rs:361-363 + block_client.rs:56,88-95: every block RPC runs under data_timeout_ms; an elapsed timer
    is io::ErrorKind::TimedOut -> FsError::IO (orpc/src/io/io_error.rs:148-153).  A worker that accepts the connection
    and never answers must therefore surface as kind IO after about data_timeout_ms, not hang the reader; a worker
    address nothing listens on fails the connect.  The hung connection must not go back to the pool."""
    import socket
    import threading
    import time
    w, _ = cluster
    man = w.create_file("/hung", 4650, 1 << 20, 1 << 20)
    srv = socket.socket()
    srv.bind(("127.0.0.1", 0))
    srv.listen(8)
    held = []
    stop = threading.Event()

    def black_hole():
        srv.settimeout(0.1)
        while not stop.is_set():
            try:
                held.append(srv.accept()[0])  # accept, read nothing, answer nothing
            except OSError:
                pass

    t = threading.Thread(target=black_hole, daemon=True)
    t.start()
    try:
        man2 = man.replace(":%d:" % w.port, ":%d:" % srv.getsockname()[1])
        for sc in (True, False):
            with F.CurvineFileSystem(F.client_conf(short_circuit=sc, extra_client="data_timeout_ms = 300\nconn_timeout_ms = 1000")) as fs:
                fs.load_namespace(man2)
                r = fs.open("/hung")
                t0 = time.time()
                with pytest.raises(F.FsError) as ei:
                    r.read(10)
                dt = time.time() - t0
                assert ei.value.kind == 1 and "timed out" in ei.value.msg, (ei.value.kind, ei.value.msg)
                assert 0.25 <= dt < 5.0, dt
                with pytest.raises(F.FsError):  # the broken connection was dropped: a second attempt times out again, it does not
                    r.read(10)                  # read a stale answer off a pooled socket
        # the same file through the real worker still reads fine with the short timeouts
        with F.CurvineFileSystem(F.client_conf(short_circuit=False, extra_client="data_timeout_ms = 300")) as fs:
            fs.load_namespace(man)
            assert fs.open("/hung").read_full(1 << 20) == synth.file_bytes(4650, 1 << 20, 1 << 20)
    finally:
        stop.set()
        t.join()
        for c in held:
            c.close()
        srv.close()


def test_empty_and_ragged_files(cluster):
    """Edge shapes: empty file; file shorter than a chunk; block size that is not a multiple of the chunk size
    (chunks restart at every block: local_file.rs:103-117, fs_reader_base.rs:181-204)."""
    w, _ = cluster
    man = w.create_file("/edge/empty", 4700, 0, 1 << 20) + w.create_file("/edge/tiny", 4701, 5, 1 << 20) \
        + w.create_file("/edge/ragged", 4702, 3 * ((1 << 20) + 4096) + 777, (1 << 20) + 4096)
    for sc in (True, False):
        with F.CurvineFileSystem(F.client_conf(short_circuit=sc)) as fs:
            fs.load_namespace(man)
            with fs.open("/edge/empty") as r:
                assert r.len() == 0 and r.read(10) == b"" and r.read_full(10) == b"" and r.read_chunk() == b"" and r.pos() == 0
                r.seek(0)
                assert r.fuse_read(0, 100) == []
            with fs.open("/edge/tiny") as r:
                assert r.read_full(100) == synth.block_bytes(4701, 0, 5) and r.pos() == 5 and r.read(1) == b""
            bs, n = (1 << 20) + 4096, 3 * ((1 << 20) + 4096) + 777
            model, data = _model_for(4702, n, bs, RM.ClientConf(short_circuit=sc))
            with fs.open("/edge/ragged") as r:
                while True:
                    c = r.read_chunk()
                    assert c == model.blocking_read()
                    if not c:
                        break
                assert r.pos() == n
                # the last chunk of every block is short (4096 bytes past 8 x 128 KiB)
                r.seek(bs - 4096)
                assert len(r.read_chunk()) == 4096


def test_write_path_hand_built_messages_then_read_back(cluster):
    """worker_test.rs:49-176, write half: WriteBlock Open -> Running x N -> Complete built with the oracle codec against
    the product worker; the block file lands in the reference layout; read back, write-side sum == read-side sum."""
    w, d = cluster
    chunk, count = 1024, 100
    bid = layout.create_block_id(4800, 0)
    s = socket.create_connection(("127.0.0.1", w.port))
    rid, wsum, blob = 0x5566, 0, bytearray()
    o = _rpc(s, W.request(80, W.REQ_OPEN, rid, 0, W.BlockWriteRequest(bid, 0, W.STORAGE_MEM, 1, 0, 1 << 20, False, "t", chunk).encode()))
    assert o.is_success()
    r = W.BlockWriteResponse.decode(o.header)
    assert (r.id, r.path, r.off, r.block_size, r.storage_type) == (bid, None, 0, 1 << 20, W.STORAGE_MEM)
    rng = np.random.default_rng(4)
    for i in range(count):
        data = rng.bytes(chunk)
        m = _rpc(s, W.request(80, W.REQ_RUNNING, rid, i + 1, b"", data))
        assert m.is_success() and m.seq_id == i + 1 and m.data == b""
        wsum += zlib.crc32(data)
        blob += data
    # a flush header must not seek; a seek header rewrites in place; out-of-range writes are error responses
    assert _rpc(s, W.request(80, W.REQ_RUNNING, rid, count + 1, W.DataHeaderProto(5, True, False).encode())).is_success()
    patch = b"PATCHED!"
    assert _rpc(s, W.request(80, W.REQ_RUNNING, rid, count + 2, W.DataHeaderProto(10, False, False).encode(), patch)).is_success()
    blob[10:18] = patch
    e = _rpc(s, W.request(80, W.REQ_RUNNING, rid, count + 3, W.DataHeaderProto((1 << 20) - 4, False, False).encode(), b"12345678"))
    assert e.resp_status == W.RESP_ERROR and "exceeds block size" in W.decode_error(e.data)[1]
    e = _rpc(s, W.request(80, W.REQ_RUNNING, rid + 1, count + 4, b"", b"x"))
    assert "Request id mismatch" in W.decode_error(e.data)[1]
    c = _rpc(s, W.request(80, W.REQ_COMPLETE, rid, count + 5, W.BlockWriteRequest(bid, len(blob), W.STORAGE_MEM, 1, len(blob), 1 << 20, False, "t", 0).encode()))
    assert c.is_success()
    path = layout.block_path(str(d / "mem" / "curvine"), bid)
    assert open(path, "rb").read() == bytes(blob)
    # read it back through ReadBlock
    o = _rpc(s, W.request(81, W.REQ_OPEN, 9, 0, W.BlockReadRequest(bid, 0, len(blob), chunk).encode()))
    assert W.BlockReadResponse.decode(o.header).len == len(blob)
    got = bytearray()
    for i in range(count):
        got += _rpc(s, W.request(81, W.REQ_RUNNING, 9, i + 1)).data
    assert bytes(got) == bytes(blob)
    # cancel removes the block
    bid2 = layout.create_block_id(4800, 1)
    assert _rpc(s, W.request(80, W.REQ_OPEN, 77, 0, W.BlockWriteRequest(bid2, 0, 0, 1, 0, 4096, False, "t", 1024).encode())).is_success()
    assert _rpc(s, W.request(80, W.REQ_RUNNING, 77, 1, b"", b"abc")).is_success()
    assert _rpc(s, W.request(80, W.REQ_CANCEL, 77, 2, W.BlockWriteRequest(bid2, 3, 0, 1, 3, 4096, False, "t", 0).encode())).is_success()
    e = _rpc(s, W.request(81, W.REQ_OPEN, 9, 0, W.BlockReadRequest(bid2, 0, 3, 1024).encode()))
    assert e.resp_status == W.RESP_ERROR
    e = _rpc(s, W.request(80, W.REQ_OPEN, 78, 0, W.BlockWriteRequest(bid2, 0, 0, 1, 8192, 4096, False, "t", 1024).encode()))
    assert "Invalid write offset" in W.decode_error(e.data)[1]
    s.close()


def test_writer_then_reader_checksums_agree(cluster):
    """block_test.rs:209-226 discipline through the product's own writer: write 10240 x 1 KiB + a tail with 1 MiB blocks,
    read back in 1 KiB calls; lengths and sum-crc equal; the manifest carries the write-time per-block CRCs."""
    w, _ = cluster
    rng = np.random.default_rng(9)
    with F.CurvineFileSystem(F.client_conf(short_circuit=False, read_chunk_size="64KB")) as fs:
        wr = fs.create("/w/f1", 4900, 1 << 20, w.port, chunk_size=65536)
        data, wsum = bytearray(), 0
        for _ in range(10240):
            rec = rng.bytes(1024)
            wr.write(rec)
            wsum += zlib.crc32(rec)
            data += rec
        tail = b"timestamp-1234567"
        wr.write(tail)
        data += tail
        man = wr.complete()
        blocks = [l.split() for l in man.splitlines() if l.startswith("block ")]
        assert len(blocks) == 11 and int(blocks[-1][2]) == len(tail)
        assert [int(b[4], 16) for b in blocks] == [zlib.crc32(bytes(data[i << 20:(i + 1) << 20])) for i in range(11)]
        assert [int(b[5], 16) for b in blocks] == [clib.crc(1, bytes(data[i << 20:(i + 1) << 20])) for i in range(11)]
        r = fs.open("/w/f1")  # registered in the namespace by complete()
        assert r.len() == len(data)
        rsum, total = 0, 0
        while True:
            b = r.read(1024)
            if not b:
                break
            total += len(b)
            if total <= 10240 * 1024:
                rsum += zlib.crc32(b)
        assert total == len(data) and rsum == wsum
        r.seek(0)
        assert r.read_full(len(data)) == bytes(data)
        r.complete()
        # cancel: nothing registered
        wr = fs.create("/w/f2", 4901, 1 << 20, w.port)
        wr.write(b"abc")
        wr.complete(cancel=True)
        with pytest.raises(F.FsError):
            fs.open("/w/f2")


def test_random_op_sequences_match_reader_model(cluster):
    """Property test (hypothesis): arbitrary interleavings of read / read_full / read_chunk / seek / fuse_read give the
    same bytes, the same short reads and the same pos() as the oracle's model of the reference reader stack, for
    striped (read_parallel 3) and plain readers, short-circuit and framed."""
    from hypothesis import given, settings, strategies as st
    w, _ = cluster
    bs, n, ino = 1 << 20, (6 << 20) + 4097, 5000
    man = w.create_file("/prop", ino, n, bs)
    op = st.one_of(
        st.tuples(st.just("read"), st.integers(0, 300000)),
        st.tuples(st.just("read_full"), st.integers(0, 700000)),
        st.tuples(st.just("chunk"), st.just(0)),
        st.tuples(st.just("seek"), st.integers(0, n + 10)),
        st.tuples(st.just("fuse"), st.integers(0, n), st.integers(0, 400000)),
    )

    @settings(max_examples=25, deadline=None)
    @given(st.lists(op, min_size=1, max_size=25), st.booleans(), st.sampled_from([(64, 4, 1), (64, 2, 3), (128, 8, 1)]))
    def run(ops, sc, shape):
        chunk_kb, chunk_num, parallel = shape
        conf = F.client_conf(short_circuit=sc, read_chunk_size="%dKB" % chunk_kb, read_chunk_num=chunk_num, read_parallel=parallel)
        model, data = _model_for(ino, n, bs, RM.ClientConf(read_chunk_size=chunk_kb * 1024, read_chunk_num=chunk_num, read_parallel=parallel, short_circuit=sc))
        with F.CurvineFileSystem(conf) as fs:
            fs.load_namespace(man)
            r = fs.open("/prop")
            for o in ops:
                if o[0] == "read":
                    assert r.read(o[1]) == model.read(o[1])
                elif o[0] == "read_full":
                    assert r.read_full(o[1]) == model.read_full(o[1])
                elif o[0] == "chunk":
                    assert r.read_chunk() == model.blocking_read()
                elif o[0] == "seek":
                    r.seek(o[1])
                    model.seek(o[1])
                else:
                    assert r.fuse_read(o[1], o[2]) == model.fuse_read(o[1], o[2])
                assert r.pos() == model.pos
            r.complete()

    run()


@pytest.mark.parametrize("sc", [True, False])
def test_config_c1_shape_cpu_reader_end_to_end(cluster, sc):
    """BASELINE config C1: single 64 MiB file, 1 MiB blocks, mem-tier local worker, CPU reader end to end (plumbing, no
    GPU): bytes == generator, curvine-bench checksum (sum of crc32 over 128 KiB read_full buffers) == oracle."""
    w, _ = cluster
    n, bs, ino = 64 << 20, 1 << 20, 5100
    man = w.create_file("/c1cpu", ino, n, bs)
    want = b"".join(clib.synth_block(ino, b, bs).tobytes() for b in range(n // bs))  # C oracle generator (fast)
    with F.CurvineFileSystem(F.client_conf(short_circuit=sc)) as fs:
        fs.load_namespace(man)
        with fs.open("/c1cpu") as r:
            cks, total = 0, 0
            while True:
                b = r.read_full(128 * 1024)
                if not b:
                    break
                assert b == want[total:total + len(b)]
                cks += zlib.crc32(b)
                total += len(b)
            assert total == n and r.pos() == n
    assert cks == clib.bench_checksum(want, 128 * 1024)
    m = w.metrics()
    assert (m["read_blocks_local"] if sc else m["read_blocks_remote"]) >= 64


@pytest.mark.parametrize("chunk_num,ahead", [(8, True), (1, False)])
def test_host_reader_prefetches_read_chunk_num_chunks_ahead(cluster, chunk_num, ahead):
    """fs_reader_buffer.rs:147-222,332-406: with read_chunk_num > 1 every striped sub-reader is a prefetch task that keeps a
    bounded channel of read_chunk_num chunks filled; with read_chunk_num == 1 the sub-reader is read inline (ReaderAdapter::Base).
    Observed at the worker: after ONE chunk was consumed, the prefetching reader has already pulled the next ones."""
    import time
    w, _ = cluster
    n, bs, ino = 4 << 20, 4 << 20, 2600 + chunk_num
    man = w.create_file("/pf%d" % chunk_num, ino, n, bs)
    before = w.metrics()["read_count"]
    with F.CurvineFileSystem(F.client_conf(short_circuit=False, read_chunk_size="64KB", read_chunk_num=chunk_num)) as fs:
        fs.load_namespace(man)
        r = fs.open("/pf%d" % chunk_num)
        first = r.read_chunk()
        assert first == synth.file_bytes(ino, n, bs)[:65536]
        time.sleep(0.3)
        pulled = w.metrics()["read_count"] - before
        assert (pulled >= 8 and pulled <= 10) if ahead else pulled == 1, pulled
        # a seek drops what was prefetched and the stream continues bit-exact from the new position
        r.seek(1 << 20)
        rest = r.read_full(n)
        assert rest == synth.file_bytes(ino, n, bs)[1 << 20:] and r.pos() == n
        r.complete()


def test_failed_worker_list_has_a_ttl_and_shows_in_the_no_worker_error(tmp_path):
    """fs_context.rs:83-86,182-205 + block_reader.rs:209-213: a worker the write path could not reach is excluded for
    failed_worker_ttl; the read path's "There is no available worker" error lists the block's locations and the excluded ids."""
    import socket
    import time
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    dead_port = s.getsockname()[1]
    s.close()  # nobody listens here
    man = "file /gone 4501 1048576 1048576 0\nblock %d 1048576 0 - - - localhost:%d:7\n" % (layout.create_block_id(4501, 0), dead_port)
    with F.CurvineFileSystem(F.client_conf(short_circuit=False, extra_client='failed_worker_ttl = "400ms"\n')) as fs:
        fs.load_namespace(man)
        with pytest.raises(F.FsError):
            fs.create("/w", 4502, 1 << 20, dead_port)  # connect fails: worker id 1 (the writer's fixture id) goes on the list
        r = fs.open("/gone")
        with pytest.raises(F.FsError) as ei:
            r.read(10)
        assert ei.value.kind == 1  # the connect error itself (IO): open-time errors are not failed over (block_reader.rs:168-215)
        time.sleep(0.5)
    with F.CurvineFileSystem(F.client_conf(short_circuit=False, extra_client='failed_worker_ttl = "1h"\n')) as fs:
        with pytest.raises(F.FsError):
            fs.create("/w", 4502, 1 << 20, dead_port)
        fs.load_namespace("file /noloc 4503 1048576 1048576 0\nblock %d 1048576 0 - - - -\n" % layout.create_block_id(4503, 0))
        r = fs.open("/noloc")
        with pytest.raises(F.FsError) as ei:
            r.read(10)
        assert "There is no available worker, locs: [], failed workers: [1]" in ei.value.msg


def test_reader_and_writer_outlive_their_filesystem_handle():
    """FFI ownership as in the reference (FsReader / FsWriter hold an Arc<FsContext>; closeFilesystem drops only the handle's reference,
    lib_filesystem.rs:25-40): closing the filesystem handle first leaves open readers and writers valid."""
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
        with F.MiniWorker(["[MEM]" + d + "/m"]) as w:
            n, bs, ino = (3 << 20) + 5, 1 << 20, 4411
            man = w.create_file("/late", ino, n, bs)
            want = synth.file_bytes(ino, n, bs)
            for sc in (True, False):
                fs = F.CurvineFileSystem(F.client_conf(short_circuit=sc))
                fs.load_namespace(man)
                r = fs.open("/late")
                head = r.read_full(1000)
                fs.close()                      # the handle goes first
                assert head + r.read_full(n) == want and r.read_full(10) == b""
                r.seek(bs - 3)
                assert r.read_full(7) == want[bs - 3:bs + 4]
                r.complete()
            fs = F.CurvineFileSystem(F.client_conf())
            wr = fs.create("/late_w", 4412, bs, w.port)
            wr.write(want[:bs + 17])
            fs.close()
            wr.write(want[bs + 17:])
            man2 = wr.complete()
            with F.CurvineFileSystem(F.client_conf()) as fs2:
                fs2.load_namespace(man2)
                with fs2.open("/late_w") as r2:
                    assert r2.read_full(n + 1) == want


def test_environment_overrides_like_cluster_conf_from():
    """ClusterConf::from (cluster_conf.rs:78-110): CURVINE_CLIENT_HOSTNAME beats the file's [client] hostname; entry points without a
    path fall back to $CURVINE_CONF_FILE (cluster_conf.rs:76, curvine-cli/src/main.rs:62).  Run in a subprocess: the environment is process-wide."""
    code = r'''
import ctypes, os, sys, tempfile
sys.path.insert(0, %r)
from curvine_b200 import _lib, fs as F
with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
    with F.MiniWorker(["[MEM]" + d + "/m"], hostname="worker-host") as w:
        man = w.create_file("/e", 4601, 3 << 20, 1 << 20)
        open(d + "/ns", "w").write(man)
        # the file says the client sits on another host: reads go framed ...
        open(d + "/conf.toml", "w").write('namespace_manifest = "%%s/ns"\n' %% d + F.client_conf(hostname="elsewhere"))
        os.environ["CURVINE_CONF_FILE"] = d + "/conf.toml"
        h = ctypes.c_void_p()
        assert _lib.lib().cv_fs_new(None, ctypes.byref(h)) == 0          # no path: $CURVINE_CONF_FILE
        fs = F.CurvineFileSystem.__new__(F.CurvineFileSystem); fs._h = h
        with fs.open("/e") as r:
            assert len(r.read_full(3 << 20)) == 3 << 20
        fs.close()
        m0 = w.metrics()
        assert m0["read_blocks_remote"] == 3 and m0["read_blocks_local"] == 0, m0
        # ... unless the environment says it is the worker's host: short-circuit
        os.environ["CURVINE_CLIENT_HOSTNAME"] = "worker-host"
        with F.CurvineFileSystem(conf_path=d + "/conf.toml") as fs:
            with fs.open("/e") as r:
                assert len(r.read_full(3 << 20)) == 3 << 20
        m1 = w.metrics()
        assert m1["read_blocks_local"] == 3 and m1["read_blocks_remote"] == 3, m1
print("env ok")
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert r.returncode == 0 and "env ok" in r.stdout, r.stdout[-2000:]


def test_headers_are_plain_c_and_the_c_example_links_against_the_library_alone():
    """include/*.h compile as C99 (-pedantic -Werror: no C++ or torch types in the boundary) and examples/c_host.c links against
    libcurvine_b200.so with no CUDA headers or libraries on the command line (the GPU suite runs it)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with tempfile.TemporaryDirectory() as d:
        libdir = os.path.join(root, "curvine_b200")
        r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(root, "include"), os.path.join(root, "examples", "c_host.c"),
                            "-o", os.path.join(d, "c_host"), "-L", libdir, "-l:libcurvine_b200.so", "-Wl,-rpath," + libdir],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 0, r.stdout
        u = subprocess.run([os.path.join(d, "c_host")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert u.returncode == 2 and "usage" in u.stdout
        # without a GPU the example fails loudly at its first CUDA call, with the library's message -- no fallback
        open(os.path.join(d, "conf.toml"), "w").write(F.client_conf())
        e = subprocess.run([os.path.join(d, "c_host"), os.path.join(d, "conf.toml"), "/nope"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert e.returncode == 1 and "cv_open" in e.stdout, e.stdout

def test_gds_probe_does_not_open_cufile_without_nvidia_fs(tmp_path):
    """gds.h: without the nvidia-fs module cuFile is never read through, so the probe neither loads libcufile nor opens its driver (on a
    B200 without nvidia-fs that stalled the first short-circuit read of a process for more than three minutes, observed in one test run):
    {available: False, compat: True}, and no cufile.log appears in the working directory.  Run in a subprocess: the probe is once per process."""
    if os.path.exists("/proc/driver/nvidia-fs/stats"):
        pytest.skip("nvidia-fs is loaded: the probe opens cuFile here by design")
    code = r'''
import sys
sys.path.insert(0, %r)
from curvine_b200 import fs as F
i = F.gds_info()
print(i["available"], i["compat"], any("libcufile" in l for l in open("/proc/self/maps")))
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120, cwd=str(tmp_path))
    assert r.returncode == 0 and r.stdout.split()[-3:] == ["False", "True", "False"], r.stdout[-2000:]
    assert not os.path.exists(str(tmp_path / "cufile.log"))


@pytest.mark.parametrize("mode", ["on", "true", "sometimes"])
def test_gds_accepts_only_off_and_auto(mode):
    """[b200] gds: "off" and "auto" (the default) parse; "on" -- cuFile's compatibility mode, which is not used -- and anything else are refused
    by name instead of being read as another mode."""
    for ok in ("off", "auto"):
        F.CurvineFileSystem(F.client_conf(b200='gds = "%s"\n' % ok)).close()
    with pytest.raises(F.FsError) as e:
        F.CurvineFileSystem(F.client_conf(b200='gds = "%s"\n' % mode))
    assert "gds" in str(e.value) and mode in str(e.value), str(e.value)
