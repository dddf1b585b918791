"""Python mirror of the reference reader surface over the C ABI (include/curvine_b200.h).

Names and behaviour follow the reference traits so tests read like the reference's own:
  CurvineFileSystem.open(path) -> Reader          curvine-common/src/fs/filesystem.rs:35
  Reader.{read_chunk, read, read_full, fuse_read, seek, pos, len, complete}
                                                   curvine-common/src/fs/reader.rs:23-156
plus the CUDA counterpart (read_device / read_device_sharded / verify) on the same handle.
Errors raise FsError carrying the reference's ErrorKind (fs_error.rs:35-66).
"""
import ctypes
from typing import List, Optional

from . import _lib


class FsError(Exception):
    def __init__(self, kind: int, msg: str):
        super().__init__("[kind %d] %s" % (kind, msg))
        self.kind = kind
        self.msg = msg


def _check(rc: int):
    if rc != 0:
        raise FsError(-rc, _lib.lib().cv_last_error().decode(errors="replace"))


def gds_info() -> dict:
    """GPUDirect Storage probe (gds.h): {available, compat (no nvidia-fs: cuFile not opened), detail}."""
    a = (ctypes.c_int64 * 2)()
    _check(_lib.lib().cv_gds_info(a))
    return {"available": bool(a[0]), "compat": bool(a[1]), "detail": _lib.lib().cv_last_error().decode(errors="replace")}


class MiniWorker:
    """In-process worker over a BlockStore directory tree (fixture; worker_test.rs:35-48 analogue)."""

    def __init__(self, data_dirs: List[str], cluster_id: str = "curvine", hostname: str = "localhost",
                 enable_send_file: bool = True, port: int = 0, extra_worker: str = ""):
        conf = 'cluster_id = "%s"\n[worker]\ndata_dir = [%s]\nhostname = "%s"\nrpc_port = %d\nenable_send_file = %s\n%s\n' % (
            cluster_id, ", ".join('"%s"' % d for d in data_dirs), hostname, port, "true" if enable_send_file else "false", extra_worker)
        self.hostname = hostname
        self._h = ctypes.c_void_p()
        p = ctypes.c_int32()
        _check(_lib.lib().cv_worker_start(conf.encode(), ctypes.byref(self._h), ctypes.byref(p)))
        self.port = p.value

    def create_file(self, path: str, inode_id: int, length: int, block_size: int, storage_type: int = 0, mode: int = 0,
                    hole_every: int = 0, threads: int = 8, worker_hostname: Optional[str] = None) -> str:
        """Writes synthetic blocks in the reference layout; returns the namespace manifest text."""
        out = ctypes.c_void_p()
        _check(_lib.lib().cv_synth_create_file(self._h, path.encode(), inode_id, length, block_size, storage_type, mode,
                                               hole_every, threads, (worker_hostname or self.hostname).encode(),
                                               ctypes.byref(out)))
        text = ctypes.string_at(out).decode()
        _lib.lib().cv_free(out)
        return text

    def delete_file(self, inode_id: int, n_blocks: int):
        """Drop the blocks of a synthetic file from the BlockStore (block files unlinked / arena extents freed)."""
        _check(_lib.lib().cv_synth_delete_file(self._h, inode_id, n_blocks))

    def arena_stats(self) -> dict:
        a = (ctypes.c_int64 * 5)()
        _check(_lib.lib().cv_worker_arena_stats(self._h, a))
        return dict(zip(["arenas", "segments", "segment_bytes", "used_bytes", "populate_us"], a))

    def hbm_load(self, block_id: int, device: int = 0):
        """HBM tier: make a finalized block resident in device memory; remote reads are then served from HBM (K4-packed frames)."""
        _check(_lib.lib().cv_worker_hbm_load(self._h, block_id, device))

    def hbm_drain(self):
        """Wait until the HBM tier's promoter thread has nothing queued or running (promotion is asynchronous)."""
        _check(_lib.lib().cv_worker_hbm_drain(self._h))

    def hbm_stats(self) -> dict:
        a = (ctypes.c_int64 * 3)()
        _check(_lib.lib().cv_worker_hbm_stats(self._h, a))
        return dict(zip(["resident_blocks", "reads_from_hbm", "packed_bytes"], a))

    def hbm_tier(self) -> dict:
        """HBM tier occupancy and policy counters ([worker] hbm_capacity / hbm_promote_after / hbm_device)."""
        a = (ctypes.c_int64 * 6)()
        _check(_lib.lib().cv_worker_hbm_tier(self._h, a))
        return dict(zip(["resident_blocks", "resident_bytes", "capacity", "evictions", "promotions", "refused"], a))

    def metrics(self) -> dict:
        a = (ctypes.c_int64 * 6)()
        _check(_lib.lib().cv_worker_metrics(self._h, a))
        return dict(zip(["read_bytes", "read_time_us", "read_count", "read_blocks_local", "read_blocks_remote", "num_blocks"], a))

    def stop(self):
        if self._h:
            _check(_lib.lib().cv_worker_stop(self._h))
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.stop()


class Reader:
    def __init__(self, h):
        self._h = h

    def len(self) -> int:
        return _lib.lib().cv_len(self._h)

    def pos(self) -> int:
        return _lib.lib().cv_pos(self._h)

    def chunk_size(self) -> int:
        return _lib.lib().cv_chunk_size(self._h)

    def remaining(self) -> int:
        return self.len() - self.pos()

    def read_chunk(self) -> bytes:
        """blocking_read: the whole current chunk (copied out of the reader-owned buffer)."""
        p, n = ctypes.c_void_p(), ctypes.c_int64()
        _check(_lib.lib().cv_read(self._h, ctypes.byref(p), ctypes.byref(n)))
        return ctypes.string_at(p, n.value) if n.value else b""

    def read(self, size: int) -> bytes:
        buf = ctypes.create_string_buffer(max(size, 1))
        n = ctypes.c_int64()
        _check(_lib.lib().cv_read_buf(self._h, buf, size, ctypes.byref(n)))
        return buf.raw[:n.value]

    def read_full(self, size: int) -> bytes:
        buf = ctypes.create_string_buffer(max(size, 1))
        n = ctypes.c_int64()
        _check(_lib.lib().cv_read_full(self._h, buf, size, ctypes.byref(n)))
        return buf.raw[:n.value]

    def read_full_into(self, ptr: int, size: int) -> int:
        n = ctypes.c_int64()
        _check(_lib.lib().cv_read_full(self._h, ctypes.c_void_p(ptr), size, ctypes.byref(n)))
        return n.value

    def fuse_read(self, pos: int, size: int) -> List[bytes]:
        buf = ctypes.create_string_buffer(max(size, 1))
        n, ns = ctypes.c_int64(), ctypes.c_int32()
        segs = (ctypes.c_int64 * 4096)()
        _check(_lib.lib().cv_fuse_read(self._h, pos, size, buf, ctypes.byref(n), segs, 4096, ctypes.byref(ns)))
        out, off = [], 0
        for i in range(ns.value):
            out.append(buf.raw[off:off + segs[i]])
            off += segs[i]
        return out

    def seek(self, pos: int):
        _check(_lib.lib().cv_seek(self._h, pos))

    # ---- CUDA counterpart
    def read_device(self, d_ptr: int, cap: int, stream: int = 0) -> int:
        n = ctypes.c_int64()
        _check(_lib.lib().cv_read_device(self._h, ctypes.c_void_p(d_ptr), cap, ctypes.c_void_p(stream), ctypes.byref(n)))
        return n.value

    def read_device_sharded(self, rank: int, world: int, d_ptr: int, cap: int, stream: int = 0) -> int:
        n = ctypes.c_int64()
        _check(_lib.lib().cv_read_device_sharded(self._h, rank, world, ctypes.c_void_p(d_ptr), cap, ctypes.c_void_p(stream),
                                                 ctypes.byref(n)))
        return n.value

    def shard_plan(self, rank: int, world: int):
        """-> list of (block_index, file_off, len, dst_off): what read_device_sharded(rank, world) executes."""
        n, tot = ctypes.c_int32(), ctypes.c_int64()
        _check(_lib.lib().cv_shard_plan(self._h, rank, world, None, None, None, None, 0, ctypes.byref(n), ctypes.byref(tot)))
        arrs = [(ctypes.c_int64 * max(1, n.value))() for _ in range(4)]
        _check(_lib.lib().cv_shard_plan(self._h, rank, world, arrs[0], arrs[1], arrs[2], arrs[3], n.value, ctypes.byref(n), ctypes.byref(tot)))
        return [tuple(a[i] for a in arrs) for i in range(n.value)]

    def fuse_read_device(self, pos: int, size: int, d_scratch: int, d_page_base: int, page_offsets, page_size: int,
                         stream: int = 0) -> int:
        arr = (ctypes.c_uint64 * len(page_offsets))(*page_offsets)
        n = ctypes.c_int64()
        _check(_lib.lib().cv_fuse_read_device(self._h, pos, size, ctypes.c_void_p(d_scratch), ctypes.c_void_p(d_page_base), arr,
                                              len(page_offsets), page_size, ctypes.c_void_p(stream), ctypes.byref(n)))
        return n.value

    def verify(self):
        """-> (sum_crc, n_bad, n_verified); blocks until outstanding device reads finished."""
        s, b, v = ctypes.c_uint64(), ctypes.c_uint32(), ctypes.c_uint64()
        _check(_lib.lib().cv_verify(self._h, ctypes.byref(s), ctypes.byref(b), ctypes.byref(v)))
        return s.value, b.value, v.value

    def device_stats(self) -> dict:
        st = _lib.CvReadStats()
        _check(_lib.lib().cv_device_stats(self._h, ctypes.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_}

    def complete(self):
        if self._h:
            h, self._h = self._h, None
            _check(_lib.lib().cv_close_reader(h))

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.complete()

    def __del__(self):  # a handle that was never closed still releases its connections and prefetch threads
        try:
            if self._h:
                h, self._h = self._h, None
                _lib.lib().cv_close_reader(h)
        except Exception:
            pass


class Writer:
    """Write-side mirror: Writer::{write, complete, cancel} (curvine-common/src/fs/writer.rs) + write_device."""

    def __init__(self, h):
        self._h = h

    def write(self, data: bytes):
        _check(_lib.lib().cv_write(self._h, data, len(data)))

    def write_device(self, d_ptr: int, n: int, stream: int = 0):
        _check(_lib.lib().cv_write_device(self._h, ctypes.c_void_p(d_ptr), n, ctypes.c_void_p(stream)))

    def complete(self, cancel: bool = False) -> str:
        out = ctypes.c_void_p()
        h, self._h = self._h, None
        _check(_lib.lib().cv_writer_close(h, 1 if cancel else 0, ctypes.byref(out)))
        text = ctypes.string_at(out).decode() if out else ""
        if out:
            _lib.lib().cv_free(out)
        return text


class CurvineFileSystem:
    def __init__(self, conf_toml: str = "", conf_path: Optional[str] = None):
        self._h = ctypes.c_void_p()
        if conf_path:
            _check(_lib.lib().cv_fs_new(conf_path.encode(), ctypes.byref(self._h)))
        else:
            _check(_lib.lib().cv_fs_new_from_string(conf_toml.encode(), ctypes.byref(self._h)))

    def load_namespace(self, text: Optional[str] = None, path: Optional[str] = None):
        if text is not None:
            _check(_lib.lib().cv_fs_load_namespace_string(self._h, text.encode()))
        if path is not None:
            _check(_lib.lib().cv_fs_load_namespace(self._h, path.encode()))

    def open(self, path: str) -> Reader:
        h, n = ctypes.c_void_p(), ctypes.c_int64()
        _check(_lib.lib().cv_open(self._h, path.encode(), ctypes.byref(h), ctypes.byref(n)))
        return Reader(h)

    def preregister(self):
        """Mem-arena tier: start mapping + pinning the `[b200] arena_preregister` dirs now (mount time), in the background."""
        _check(_lib.lib().cv_fs_preregister(self._h))

    def arena_stats(self) -> dict:
        a = (ctypes.c_uint64 * 5)()
        _check(_lib.lib().cv_fs_arena_stats(self._h, a))
        return dict(zip(["segments", "pinned_bytes", "register_us", "dma_jobs", "dma_bytes"], a))

    def wait_registered(self):
        """Block until the background registrar of the zero-copy mem tier is idle (optional; reads never wait for it)."""
        _check(_lib.lib().cv_fs_wait_registered(self._h))

    def read_to_tensor(self, path: str, device=None, verify: bool = True):
        """Binding convenience (SURVEY 8f-4): the whole file as a uint8 CUDA tensor (DLPack-exportable), CRC-verified
        on the GPU.  Replaces curvinefs' copy-and-decode read (curvine-libsdk/python/curvinefs/curvineReader.py:17-49)."""
        import torch
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        r = self.open(path)
        try:
            out = torch.empty(r.len(), dtype=torch.uint8, device=dev)
            if r.len():
                got = r.read_device(out.data_ptr(), r.len(), torch.cuda.current_stream(dev).cuda_stream)
                assert got == r.len()
            _, bad, _ = r.verify()
            if verify and bad:
                raise FsError(12, "%d blocks of %s failed CRC verification" % (bad, path))  # AbnormalData
            return out
        finally:
            r.complete()

    def fuse_read_file_device(self, path: str, size: int, d_scratch: int, d_page_base: int, page_offsets, page_size: int, stream: int = 0):
        """One small file in one call: open -> FUSE-shaped device read -> verify -> close.  `page_offsets` may be a prepared
        ctypes c_uint64 array (reused across calls).  -> (bytes, n_bad)."""
        arr = page_offsets if isinstance(page_offsets, ctypes.Array) else (ctypes.c_uint64 * len(page_offsets))(*page_offsets)
        n, bad = ctypes.c_int64(), ctypes.c_uint32()
        _check(_lib.lib().cv_fuse_read_file_device(self._h, path.encode(), size, ctypes.c_void_p(d_scratch), ctypes.c_void_p(d_page_base), arr, len(arr),
                                                   page_size, ctypes.c_void_p(stream), ctypes.byref(n), ctypes.byref(bad)))
        return n.value, bad.value

    def read_many_device(self, paths, d_ptr: int, dst_offs, cap: int, stream: int = 0):
        """Small-file batching: every file of ``paths`` lands at d_ptr + dst_offs[i] in one pipelined pass.
        -> (total_bytes, sum_crc, n_bad, n_verified)."""
        arr = (ctypes.c_char_p * len(paths))(*[p.encode() for p in paths])
        offs = (ctypes.c_int64 * len(paths))(*dst_offs)
        s, b, v, t = ctypes.c_uint64(), ctypes.c_uint32(), ctypes.c_uint64(), ctypes.c_int64()
        _check(_lib.lib().cv_read_many_device(self._h, arr, len(paths), ctypes.c_void_p(d_ptr), offs, cap, ctypes.c_void_p(stream),
                                              ctypes.byref(s), ctypes.byref(b), ctypes.byref(v), ctypes.byref(t)))
        return t.value, s.value, b.value, v.value

    def create(self, path: str, inode_id: int, block_size: int, worker_port: int, worker_host: str = "localhost", storage_type: int = 0,
               chunk_size: int = 0) -> Writer:
        h = ctypes.c_void_p()
        _check(_lib.lib().cv_writer_open(self._h, path.encode(), inode_id, block_size, storage_type, worker_host.encode(), worker_port, chunk_size,
                                         ctypes.byref(h)))
        return Writer(h)

    def metrics(self) -> dict:
        a = (ctypes.c_int64 * 2)()
        _check(_lib.lib().cv_fs_metrics(self._h, a))
        return {"read_bytes": a[0], "read_time_us": a[1]}

    def pool_stats(self) -> dict:
        """Block connection pool: idle connections now, connections opened so far, pooled connections dropped as expired."""
        a = (ctypes.c_int64 * 3)()
        _check(_lib.lib().cv_fs_pool_stats(self._h, a))
        return {"idle": a[0], "opened": a[1], "expired": a[2]}

    def close(self):
        if self._h:
            h, self._h = self._h, None
            _check(_lib.lib().cv_fs_close(h))

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def client_conf(hostname: str = "localhost", short_circuit: bool = True, read_chunk_size: str = "128KB", read_chunk_num: int = 8,
                read_parallel: int = 1, extra_client: str = "", b200: str = "") -> str:
    return ('[client]\nhostname = "%s"\nshort_circuit = %s\nread_chunk_size = "%s"\nread_chunk_num = %d\nread_parallel = %d\n%s\n[b200]\n%s\n'
            % (hostname, "true" if short_circuit else "false", read_chunk_size, read_chunk_num, read_parallel, extra_client, b200))
