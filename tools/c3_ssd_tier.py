"""Config C3's tier at the size the box holds: a synthetic file on an [SSD] BlockStore directory (the box's disk, not tmpfs),
4 MiB blocks, 1 GPU, CRC-32C verify on the GPU.  Reports end-to-end GB/s into HBM for
  cold   page cache dropped before every pass (fsync + posix_fadvise(DONTNEED) on every block file): the disk is the source
  warm   page cache holds the file (what a second pass over a recently written/read file sees)
and the same two cases for the reference-shaped CPU reader (oracle/cpu_reader.c), host cores stated; beside them
  disk   the disk's own ceiling for this access pattern: the same block files read cold with O_DIRECT by 16 threads (a dd/fio stand-in)
  gds    [b200] gds = off|auto: cuFileRead straight into HBM (curvine_b200/csrc/host/gds.h) vs the pinned ring
  hbm    (--hbm) the worker's HBM tier over the SSD tier: framed reads cold from the disk, then -- after asynchronous promotion
         (hbm_promote_after = 1) -- served out of HBM as K4-packed frames; hit rate and GB/s per pass.
BASELINE.json names 128 GiB over 8 GPUs; the GPU box has a 79 GB overlay disk, so the size is a parameter (default 16 GiB)."""
import argparse
import glob
import json
import os
import shutil
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
BLOCK = 4 << 20


def drop_cache(root):
    n = 0
    for p in glob.glob(os.path.join(root, "**", "blk_*"), recursive=True):
        fd = os.open(p, os.O_RDONLY)
        try:
            os.fsync(fd)
            os.posix_fadvise(fd, 0, 0, os.POSIX_FADV_DONTNEED)
        finally:
            os.close(fd)
        n += 1
    return n


def disk_ceiling(root, threads=16, limit_bytes=8 << 30):
    """Cold sequential read of the block files with O_DIRECT (no page cache on either side), `threads` files at a time."""
    import mmap
    import threading
    files = sorted(glob.glob(os.path.join(root, "**", "blk_*"), recursive=True))
    files = files[:max(1, limit_bytes // BLOCK)]
    nxt, lock, total = [0], threading.Lock(), [0]

    def work():
        buf = mmap.mmap(-1, BLOCK)  # page-aligned
        while True:
            with lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= len(files):
                return
            try:
                fd = os.open(files[i], os.O_RDONLY | os.O_DIRECT)
            except OSError:
                fd = os.open(files[i], os.O_RDONLY)
            got = 0
            while True:
                n = os.preadv(fd, [buf], got)
                if n <= 0:
                    break
                got += n
            os.close(fd)
            with lock:
                total[0] += got

    t0 = time.perf_counter()
    ts = [threading.Thread(target=work) for _ in range(threads)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return total[0] / (time.perf_counter() - t0) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=16.0)
    ap.add_argument("--dir", default="/tmp")
    ap.add_argument("--passes", type=int, default=2)
    ap.add_argument("--zero-copy", type=int, default=1)
    ap.add_argument("--gds", default="auto")
    ap.add_argument("--hbm", type=float, default=0.0, help="GiB of the file's head to run the HBM-tier leg over (0 = skip)")
    a = ap.parse_args()
    import torch
    from curvine_b200 import fs as F
    from oracle import clib, layout
    torch.cuda.set_device(0)
    n = int(a.gib * (1 << 30)) // BLOCK * BLOCK
    d = tempfile.mkdtemp(prefix="cvc3_", dir=a.dir)
    st = os.statvfs(d)
    res = {"file_bytes": n, "dir": d, "fs_free_GB": st.f_bavail * st.f_frsize / 1e9, "host_cpus": os.cpu_count()}
    try:
        with F.MiniWorker(["[SSD]" + d], hostname="localhost") as w:
            t0 = time.time()
            man = w.create_file("/c3/file", 5151, n, BLOCK, storage_type=1, threads=32)
            res["file_gen_sec"] = time.time() - t0
            conf = F.client_conf(hostname="localhost", short_circuit=True,
                                 b200='zero_copy = %s\nregister_cache = "%dGB"\nfetch_threads = 16\nverify_batch = 16\ncopy_group = 8\ngds = "%s"\n'
                                      % ("true" if a.zero_copy else "false", int(a.gib * 1.5) + 1, a.gds))
            res["gds"] = dict(F.gds_info(), mode=a.gds)
            with F.CurvineFileSystem(conf) as fs:
                fs.load_namespace(man)
                dst = torch.empty(n, dtype=torch.uint8, device="cuda")
                stream = torch.cuda.current_stream().cuda_stream

                def one_pass():
                    t1 = time.perf_counter()
                    r = fs.open("/c3/file")
                    got = r.read_device(dst.data_ptr(), n, stream)
                    s, bad, ver = r.verify()
                    stats = r.device_stats()
                    r.complete()
                    dt = time.perf_counter() - t1
                    assert got == n and bad == 0 and ver == n // BLOCK
                    return n / dt / 1e9, dt, stats

                cold, warm = [], []
                for _ in range(a.passes):
                    res["blocks_dropped"] = drop_cache(d)
                    cold.append(one_pass()[:2])
                for _ in range(a.passes + 1):
                    v, dt, stats = one_pass()
                    warm.append((v, dt))
                fs.wait_registered()
                v, dt, stats = one_pass()
                res["gds_bytes_last_pass"] = stats["gds_bytes"]
                res["gds_after"] = F.gds_info()
                res["gpu_cold_GBps"] = [round(x[0], 2) for x in cold]
                res["gpu_warm_GBps"] = [round(x[0], 2) for x in warm]
                res["gpu_warm_after_registration_GBps"] = round(v, 2)
                res["registered_mapping_cache"] = {"hits": stats["reg_hits"], "misses": stats["reg_misses"]}
            ids = [layout.create_block_id(5151, i) for i in range(n // BLOCK)]
            par = clib.reference_read_parallel(n)

            def cpu_pass():
                t1 = time.time()
                got, cks, threads = clib.cpu_read_file(w.port, True, n, BLOCK, ids, 131072, 8, par, 131072, n, 1)
                return got / (time.time() - t1) / 1e9, threads

            drop_cache(d)
            res["cpu_cold_GBps"], res["cpu_threads"] = cpu_pass()
            res["cpu_warm_GBps"], _ = cpu_pass()
            drop_cache(d)
            res["disk_cold_o_direct_16thr_GBps"] = round(disk_ceiling(d), 2)
        if a.hbm > 0:
            nh = int(a.hbm * (1 << 30)) // BLOCK * BLOCK
            with F.MiniWorker(["[SSD]" + d], hostname="localhost", extra_worker='hbm_capacity = "%dGB"\nhbm_promote_after = 1\nhbm_device = 0\n' % (int(a.hbm) + 1)) as w2:
                man2 = w2.create_file("/c3/hot", 5252, nh, BLOCK, storage_type=1, threads=32)
                conf = F.client_conf(hostname="localhost", short_circuit=False,
                                     b200='fetch_threads = 16\nverify_batch = 16\ncopy_group = 1\npinned_slots = 72\ngpu_chunk_size = "4MB"\nlocal_unix_socket = true\n')
                with F.CurvineFileSystem(conf) as fs:
                    fs.load_namespace(man2)
                    dst = torch.empty(nh, dtype=torch.uint8, device="cuda")
                    legs = []
                    for name, cold in (("cold_from_ssd", True), ("second_read_queues_promotion", True), ("from_hbm", True), ("from_hbm_again", True)):
                        if cold:
                            drop_cache(d)
                        before = w2.hbm_stats()["reads_from_hbm"]
                        t1 = time.perf_counter()
                        r = fs.open("/c3/hot")
                        got = r.read_device(dst.data_ptr(), nh, torch.cuda.current_stream().cuda_stream)
                        s, bad, ver = r.verify()
                        r.complete()
                        dt = time.perf_counter() - t1
                        assert got == nh and bad == 0
                        t2 = time.perf_counter()
                        w2.hbm_drain()
                        tier = w2.hbm_tier()
                        legs.append({"pass": name, "GBps": round(nh / dt / 1e9, 2), "served_from_hbm": (w2.hbm_stats()["reads_from_hbm"] - before) / (nh // BLOCK),
                                     "promoter_drain_ms_after_pass": round((time.perf_counter() - t2) * 1e3, 1), "resident_blocks": tier["resident_blocks"],
                                     "promotions": tier["promotions"]})
                    res["hbm_tier_over_ssd"] = {"file_bytes": nh, "page_cache_dropped_before_every_pass": True, "passes": legs}
    finally:
        shutil.rmtree(d, ignore_errors=True)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
