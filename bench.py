#!/usr/bin/env python
"""bench.py -- sequential read GB/s into HBM (CRC-verified), the metric BASELINE.json names.

    python bench.py --gpus N --steps K --warmup W                      # this implementation
    python bench.py --impl reference --gpus N --steps K --warmup W     # the reference's CPU read path (oracle port)
    python bench.py --config c4 --gpus N                               # model distribution: every GPU ends up with the whole file
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR   # also write the last step's outputs to DIR/*.npy (seeded inputs)
    (N > 1: launched by torchrun, one rank per GPU)

Workload (config C2 of BASELINE.json per GPU, scaled weakly: C3's shape at N=8): synthetic files of N x 16 GiB in 4 MiB
blocks in the worker's mem tier; GPU g reads the blocks b % N == g (16 GiB per GPU).  EVERY step reads a file that no client
has read before: rank 0 drops the previous step's file and writes a fresh one (new inode, new bytes) before the step, all
outside the timed region.  A step = one full pass through the public C ABI:
    cv_open -> cv_read_device[_sharded] -> cv_verify -> cv_close_reader
block locations -> worker Open/Complete RPCs per block -> DMA of the block bytes from host memory into HBM -> on-GPU CRC-32C
(K1) -> compare with the manifest on the GPU -> D2H of the per-block CRCs and the mismatch count.  Host bytes in, HBM out.
    value   the ingest rate of those steps, timed on the device from the first H2D copy to the verified result (CUDA events on the
            calling stream around cv_read_device .. cv_verify), max over ranks
    e2e     the same steps timed around the whole reader life cycle (cv_open .. cv_close_reader): what a caller sees
Beside the headline (mem-ARENA tier: blocks are extents of segments the client pinned once at mount, arena.h) the line reports
the same read over the reference's one-file-per-block mem tier through the pinned ring (`e2e_pread`), over TCP frames unpacked by
K2 on the GPU (`e2e_framed`), a re-read of an already-read file (`e2e_reread`), the HBM-resident K1 verify rate (`resident_verify`,
`roofline`) and the reference's CPU reader on the host cores (`cpu_baseline`).
Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.  Inputs (16 GiB per GPU per
step, never the same bytes twice) are >> L2 (126 MB): no L2 flush needed.
"""
import argparse
import ctypes
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sequential read GB/s into HBM (CRC-verified)"
UNIT = "GB/s"
BLOCK = 4 << 20
PCIE_RAW = 63.0  # PCIe Gen5 x16 per direction, GB/s (SURVEY.md 8d)
SEG = 256 << 20  # arena segment size


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c4", "c5"])
    ap.add_argument("--gib-per-gpu", type=float, default=16.0)
    ap.add_argument("--mode", default="short_circuit", choices=["short_circuit", "framed"], help="read path of the headline steps")
    ap.add_argument("--tier", default="arena", choices=["arena", "files"], help="mem tier of the headline steps: pinned-once arena (arena.h) or the reference's one file per block")
    ap.add_argument("--pool", type=int, default=0, help="files kept alive BESIDE the one a step reads (0: the previous step's file is dropped before the next is written)")
    ap.add_argument("--fetch-threads", type=int, default=0)
    ap.add_argument("--slots", type=int, default=0)
    ap.add_argument("--verify-batch", type=int, default=16)
    ap.add_argument("--copy-group", type=int, default=8)
    ap.add_argument("--copy-streams", type=int, default=1)
    ap.add_argument("--register-threads", type=int, default=16)
    ap.add_argument("--register-slice", default="256MB")
    ap.add_argument("--numa-node", type=int, default=-1, help="-1 bind fetch threads to the GPU's node, -2 no binding")
    ap.add_argument("--gpu-chunk", default="4MB")
    ap.add_argument("--framed-threads", type=int, default=0)
    ap.add_argument("--poly", type=int, default=1)
    ap.add_argument("--settle-ms", type=int, default=0, help="pause between writing a step's file and reading it (diagnostic)")
    ap.add_argument("--legs", default="reread,pread,framed,framed_unix,resident,cpu", help="side legs to run besides the headline (comma list)")
    ap.add_argument("--side-steps", type=int, default=2, help="timed steps of each side leg (reread / pread / framed); 0 skips them")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dir", default="")
    ap.add_argument("--no-memory-guard", action="store_true", help="do not shrink --gib-per-gpu when the stores would not fit into the container's memory")
    ap.add_argument("--ref-materialize-gib", type=float, default=64.0, help="reference arm: how much of the file's head is written to the store (the CPU reader never reads past its sample)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="after the timed steps, write what the last headline step returned as DIR/<name>.npy (see dump_outputs); "
                                                                     "refused when the memory guard would shrink --gib-per-gpu, so the same arguments always read the same files")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config != "c2"):
        ap.error("--dump-outputs applies to the headline read (--impl ours --config c2)")
    return args


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.p, self.index = [], None, index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.p = None

    def _pump(self):
        for line in self.p.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.p:
            self.p.terminate()

    def summary(self, windows):
        sm, mx, reasons = [], 0.0, set()
        for t, r in self.rows:
            if len(r) < 8 or not any(t0 <= t <= t1 + 0.2 for t0, t1 in windows):
                continue
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def host_memory_budget(shm_dir):
    """Bytes this container can safely put into tmpfs + pinned memory: the smallest of MemAvailable, the cgroup limit (v2 or v1, minus
    what is in use) and the free space of the tmpfs the store lives on.  -> (bytes, {source: bytes})."""
    found = {}
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                found["MemAvailable"] = int(line.split()[1]) * 1024
    except OSError:
        pass
    for limit, used in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                        ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            v = open(limit).read().strip()
            if v != "max" and int(v) < (1 << 60):
                found["cgroup"] = int(v) - int(open(used).read().strip())
                break
        except (OSError, ValueError):
            pass
    try:
        st = os.statvfs(shm_dir)
        found["tmpfs_free"] = st.f_bavail * st.f_frsize
    except OSError:
        pass
    return (min(found.values()) if found else None), found


def fit_gib_per_gpu(want_gib, world, pool, budget, reserve_per_gpu=3 << 30, frac=0.7):
    """The largest power-of-two fraction of want_gib whose stores fit into `frac` of the budget.  One GPU holds the arena (pool+1 files + a
    segment) AND, for the reference-layout side leg, one more file; beyond one GPU only the arenas exist.  (SURVEY 8d: "if the box cannot
    hold a named size, run the largest power of two that fits and say so".)"""
    gib = want_gib
    while budget is not None and gib > 1.0 / 64:
        shard = int(gib * (1 << 30))
        need = world * ((pool + 1) * shard + SEG + reserve_per_gpu) + (shard if world == 1 else 0)
        if need <= frac * budget:
            break
        gib /= 2
    return gib


def claim_store_dir(base, prefix):
    """A fresh directory for this run's stores under `base`, after removing what DEAD earlier runs left there (a run that was killed keeps
    its tmpfs files -- up to 130 GiB at 8 GPUs -- and the driver starts the next run on the same box right away)."""
    for name in os.listdir(base):
        if not name.startswith(("cvbench_", "cvref_")):
            continue
        p = os.path.join(base, name)
        try:
            pid = int(open(os.path.join(p, "owner.pid")).read().strip())
            os.kill(pid, 0)  # raises if no such process
        except (OSError, ValueError):
            if time.time() - os.stat(p).st_mtime > 60:  # not a directory some process is creating right now
                log("removing the stores of a dead run:", p)
                shutil.rmtree(p, ignore_errors=True)
        except Exception:
            pass
    d = tempfile.mkdtemp(prefix=prefix, dir=base)
    with open(os.path.join(d, "owner.pid"), "w") as f:
        f.write(str(os.getpid()))
    return d


def setup_dist(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "ours":
        torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        if args.impl == "ours":
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group("gloo")
    return rank, world, local, dist


def barrier(dist, cuda=True):
    import torch
    if cuda:
        torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    if cuda:
        torch.cuda.synchronize()


_REAL_STDOUT = None


def quiet_stdout():
    """Everything incidental (NCCL's version banner, library chatter) goes to stderr: stdout carries exactly one JSON line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(obj):
    _REAL_STDOUT.write(json.dumps(obj) + "\n")
    _REAL_STDOUT.flush()


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------ cluster (rank 0 hosts the workers and writes the files)

class Cluster:
    """Two in-process workers on rank 0: `arena` ([MEM] dirs kept as pinned-once arenas, one per GPU, each on its GPU's NUMA
    node) and `files` (the reference layout: one tmpfs file per block).  Files are created on demand and dropped again."""

    def __init__(self, args, rank, world, dist, shard_bytes, need_files_tier):
        from curvine_b200 import _lib, fs as F
        self.args, self.rank, self.world, self.dist, self.F = args, rank, world, dist, F
        self.shard_bytes = shard_bytes
        self.live = {}  # path -> (worker key, inode, blocks)
        self.gen_sec = 0.0
        payload = [None]
        if rank == 0:
            base = args.dir or ("/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir())
            self.dir = claim_store_dir(base, "cvbench_")
            L = _lib.lib()
            nodes = [int(L.cv_gpu_numa_node(g)) for g in range(world)]
            # memory discipline: the arena holds the file being read (+ `pool` older ones) and one segment of slack, nothing more -- the
            # GPU boxes lose the container somewhere below 257 GiB of tmpfs (round 2 lost three boxes to a 128 GiB-per-GPU run)
            cap = (args.pool + 1) * shard_bytes + SEG
            dirs = ["[MEM:%d]%s/arena%d" % (cap, self.dir, g) for g in range(world)]
            t0 = time.time()
            self.arena = F.MiniWorker(dirs, hostname="localhost",
                                      extra_worker='mem_arena = true\narena_segment = "%d"\narena_numa = [%s]\narena_reuse_delay = "0ms"\n'
                                                   % (SEG, ", ".join(str(n) for n in nodes)))
            self.arena_start_sec = time.time() - t0
            self.files = F.MiniWorker(["[MEM]%s/files%d" % (self.dir, g) for g in range(world)], hostname="localhost") if need_files_tier else None
            L.cv_synth_set_shard_world(world)  # block b -> dir b % world, first-touched on GPU (b % world)'s node
            payload = [{"dir": self.dir, "arena_port": self.arena.port, "files_port": self.files.port if self.files else 0, "nodes": nodes,
                        "arena_stats": self.arena.arena_stats(), "arena_start_sec": self.arena_start_sec}]
        if dist is not None:
            dist.broadcast_object_list(payload, src=0)
        self.info = payload[0]
        self.dir = self.info["dir"]

    def create(self, tier, path, inode, nbytes):
        """rank 0 writes the file; every rank gets the manifest text."""
        payload = [None]
        if self.rank == 0:
            w = self.arena if tier == "arena" else self.files
            t0 = time.time()
            payload = [w.create_file(path, inode, nbytes, BLOCK, storage_type=0, threads=min(64, os.cpu_count() or 8))]
            self.gen_sec += time.time() - t0
            self.live[path] = (tier, inode, (nbytes + BLOCK - 1) // BLOCK)
        if self.dist is not None:
            self.dist.broadcast_object_list(payload, src=0)
        return payload[0]

    def drop(self, path):
        if self.rank == 0 and path in self.live:
            tier, inode, nb = self.live.pop(path)
            (self.arena if tier == "arena" else self.files).delete_file(inode, nb)

    def close(self):
        if self.rank == 0:
            from curvine_b200 import _lib
            _lib.lib().cv_synth_set_shard_world(0)
            self.arena.stop()
            if self.files:
                self.files.stop()
            shutil.rmtree(self.dir, ignore_errors=True)


def client_conf(args, cluster, sc, device, threads, slots, rank, zero_copy=True, copy_group=None, chunk=None, unix=False):
    from curvine_b200 import fs as F
    b200 = ('device = %d\nfetch_threads = %d\npinned_slots = %d\nverify_poly = %d\nverify = true\nverify_batch = %d\ncopy_group = %d\ngpu_chunk_size = "%s"\n'
            'zero_copy = %s\nregister_threads = %d\nregister_cache = "%dGB"\ncopy_streams = %d\nnuma_node = %d\narena_preregister = ["%s/arena%d"]\n'
            'arena_register_slice = "%s"\nlocal_unix_socket = %s\n'
            % (device, threads, slots, args.poly, args.verify_batch, args.copy_group if copy_group is None else copy_group, chunk or args.gpu_chunk,
               "true" if zero_copy else "false", args.register_threads, int(args.gib_per_gpu * 1.5) + 1, args.copy_streams, args.numa_node, cluster.dir, rank, args.register_slice, "true" if unix else "false"))
    return F.client_conf(hostname="localhost", short_circuit=sc, b200=b200)


def timed_read(fs, path, rank, world, dst, shard_bytes, stream):
    """One step through the C ABI.  -> (e2e_ms, ingest_ms, sum_crc, stats).  CUDA events on the calling stream; cv_verify blocks
    until the CRCs and the mismatch count are back on the host, so the closing events are complete when they are read."""
    import torch
    a, a2, b2, b = (torch.cuda.Event(enable_timing=True) for _ in range(4))
    a.record()
    r = fs.open(path)
    a2.record()
    if world == 1:
        got = r.read_device(dst.data_ptr(), shard_bytes, stream)
    else:
        got = r.read_device_sharded(rank, world, dst.data_ptr(), shard_bytes, stream)
    s, bad, ver = r.verify()
    b2.record()
    stats = r.device_stats()
    r.complete()
    b.record()
    b.synchronize()
    assert bad == 0, "CRC mismatch in %d blocks of %s" % (bad, path)
    assert got == shard_bytes and ver == shard_bytes // BLOCK, (got, ver, shard_bytes)
    return a.elapsed_time(b), a2.elapsed_time(b2), s, stats


DUMP_SAMPLE = 4 << 20  # bytes of HBM output --dump-outputs keeps, over all ranks (16 MiB as float32)


def dump_positions(shard_bytes, world):
    """Offsets into a rank's shard that --dump-outputs samples: seeded, sorted, the same for every run and build at this size."""
    import numpy as np
    return np.sort(np.random.default_rng(0).integers(0, shard_bytes, min(shard_bytes, DUMP_SAMPLE // world)))


def dump_outputs(out_dir, rank, world, dst, sum_crc):
    """What a caller of the timed path holds after the last headline step, as .npy files two builds can be compared by:
         bytes_sample     float32  the HBM bytes at dump_positions()
         block_byte_sums  float64  the sum of the bytes of every 4 MiB block of the shard (every byte counts, exact in float64)
         crc_sum          float64  the sum of the per-block CRCs cv_verify returned (its mismatch count was asserted to be 0)
    Several ranks: one set per rank, names suffixed _rank<r>."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    pos = torch.from_numpy(dump_positions(dst.numel(), world)).to(dst.device)
    chunk = 64 * BLOCK  # the reduction may widen its input first: 256 MiB at a time; a block sums to < 2**31
    sums = torch.cat([dst[i:i + chunk].view(-1, BLOCK).sum(dim=1, dtype=torch.int32) for i in range(0, dst.numel(), chunk)])
    arrays = {"bytes_sample": dst[pos].cpu().numpy().astype(np.float32),
              "block_byte_sums": sums.cpu().numpy().astype(np.float64),
              "crc_sum": np.array([sum_crc], dtype=np.float64)}
    suffix = "_rank%d" % rank if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def run_leg(name, cluster, fs, tier, args, rank, world, dist, dst, shard_bytes, steps, warmup, fresh, inode0, pool=None):
    """steps+warmup passes; fresh=True: every pass reads a file written just before it (never read by anyone), and the file of
    `pool` passes ago is dropped; fresh=False: one file, read again and again.  -> dict(e2e_ms[], ingest_ms[], warm_ms[], stats)."""
    import torch
    stream = torch.cuda.current_stream().cuda_stream
    out = {"e2e_ms": [], "ingest_ms": [], "warm_e2e_ms": [], "windows": []}
    paths = []
    n_total = shard_bytes * world
    for it in range(warmup + steps):
        if fresh or it == 0:
            # the file read `pool`+1 steps ago goes first (its read was verified and is complete: no DMA can be in flight, which is
            # why this bench runs the arena with arena_reuse_delay = 0), then the new one is written -- possibly into the same pages
            while len(paths) > (args.pool if pool is None else pool):
                cluster.drop(paths.pop(0))
            path = "/bench/%s_%d" % (name, it)
            fs.load_namespace(cluster.create(tier, path, inode0 + it, n_total))
            paths.append(path)
        if args.settle_ms:
            time.sleep(args.settle_ms / 1e3)
        barrier(dist)
        t0 = time.time()
        e2e_ms, ing_ms, s, stats = timed_read(fs, paths[-1], rank, world, dst, shard_bytes, stream)
        barrier(dist)
        if it >= warmup:
            out["e2e_ms"].append(e2e_ms)
            out["ingest_ms"].append(ing_ms)
            out["windows"].append((t0, time.time()))
        else:
            out["warm_e2e_ms"].append(e2e_ms)
        out["stats"], out["sum_crc"] = stats, s
    for p in paths:
        cluster.drop(p)
    return out


def main():
    args = parse()
    quiet_stdout()
    if args.impl == "reference":
        return main_reference(args)
    if args.config == "c4":
        from tools import c4_allgather
        return c4_allgather.main_bench(args, emit)
    if args.config == "c5":
        from tools import c5_smallfiles
        return c5_smallfiles.main_bench(args, emit)
    import numpy as np
    import torch
    from curvine_b200 import _lib, fs as F, kernels as K

    rank, world, local, dist = setup_dist(args)
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d" % args.gpus
    L = _lib.lib()
    _lib.check(L.cvk_init(local), "cvk_init")
    # memory guard (round 2 lost three boxes to a run that outgrew its container): shrink the per-GPU size if the stores would not fit
    budget, budget_sources = host_memory_budget(args.dir or ("/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()))
    asked_gib = args.gib_per_gpu
    if not args.no_memory_guard:
        pick = [fit_gib_per_gpu(asked_gib, world, args.pool, budget)]
        if dist is not None:  # one decision for all ranks (MemAvailable moves between two reads of it)
            dist.broadcast_object_list(pick, src=0)
        args.gib_per_gpu = pick[0]
        if args.gib_per_gpu != asked_gib and rank == 0:
            log("memory guard: %g GiB per GPU does not fit into 70%% of %s; running %g GiB per GPU" % (asked_gib, budget_sources, args.gib_per_gpu))
        if args.dump_outputs and args.gib_per_gpu != asked_gib:  # a dump of another size cannot be compared with one taken at the asked size
            raise SystemExit("--dump-outputs: the memory guard cut --gib-per-gpu %g to %g; ask for a size this host holds" % (asked_gib, args.gib_per_gpu))
    shard_bytes = int(args.gib_per_gpu * (1 << 30)) // BLOCK * BLOCK
    n_total = shard_bytes * world
    my_blocks = shard_bytes // BLOCK
    ncpu = os.cpu_count() or 8
    threads = args.fetch_threads or max(4, min(16, ncpu // (2 * world)))
    # loopback TCP stops scaling at ~16 connections on this box (profiles/r02_loopback_probe.txt: 46 GB/s at 16, 35 at 24, 28 at 32)
    fthreads = args.framed_threads or max(4, min(16, ncpu // (2 * world)))
    slots = args.slots or (2 * args.verify_batch + threads + 8)
    side = args.side_steps
    # side legs report a rate: beyond one GPU they read 2 GiB per GPU per step and skip the reference-layout leg (no tmpfs beside the arena)
    side_bytes = shard_bytes if world == 1 else min(shard_bytes, (2 << 30) // BLOCK * BLOCK)
    cluster = Cluster(args, rank, world, dist, shard_bytes, need_files_tier=True)
    dst = torch.empty(shard_bytes, dtype=torch.uint8, device="cuda")
    sampler = ClockSampler(local)
    sampler.start()
    out = {}
    try:
        sc = args.mode == "short_circuit"
        fs = F.CurvineFileSystem(client_conf(args, cluster, sc, local, threads, slots, rank))
        # ---- mount: map + pin this rank's arena (off every read path), then one small read so the process is warm
        t0 = time.time()
        fs.preregister()
        fs.wait_registered()
        mount_ms = (time.time() - t0) * 1e3
        arena0 = fs.arena_stats()
        t0 = time.time()
        fs.load_namespace(cluster.create(args.tier, "/bench/ctxwarm", 4100, 16 * world * BLOCK))
        timed_read(fs, "/bench/ctxwarm", rank, world, dst, 16 * BLOCK, torch.cuda.current_stream().cuda_stream)
        cluster.drop("/bench/ctxwarm")
        ctx_warm_ms = (time.time() - t0) * 1e3
        # ---- headline: every step reads a never-read file
        launches0 = K.launch_count()
        head = run_leg("fresh", cluster, fs, args.tier, args, rank, world, dist, dst, shard_bytes, args.steps, args.warmup, True, 5000)
        launches = (K.launch_count() - launches0) * args.steps // max(1, args.steps + args.warmup)
        arena1 = fs.arena_stats()
        if args.dump_outputs:  # before the side legs overwrite dst
            dump_outputs(args.dump_outputs, rank, world, dst, head["sum_crc"])
        # ---- side legs
        legs = set(x for x in args.legs.split(",") if x) if side > 0 else set()
        if world > 1:  # beyond one GPU the side legs are the re-read and the kernel-only pass; the transport legs are one-GPU numbers
            legs -= {"pread", "framed", "framed_unix"}
        side_errors = {}

        def guarded(leg_name, fn):
            """A side leg must never cost the headline its JSON line (one GPU only: with several ranks a leg that fails on one rank
            would leave the others in a barrier, which is why those legs do not run there)."""
            try:
                return fn()
            except Exception as e:  # noqa: BLE001
                side_errors[leg_name] = "%s: %s" % (type(e).__name__, e)
                log("side leg %s failed: %s" % (leg_name, side_errors[leg_name]))
                for p in [p for p in list(cluster.live) if p.startswith("/bench/%s_" % leg_name)]:
                    cluster.drop(p)  # whatever it left in the store must not starve the legs behind it
                return None
        reread = pread = framed = framed_unix = None
        if "reread" in legs:
            reread = run_leg("reread", cluster, fs, args.tier, args, rank, world, dist, dst, side_bytes, side, 1, False, 6000)  # the headline's own path: not guarded
        # ---- resident verify (K1 over what the last step left in HBM) + roofline of K1
        fs.load_namespace(cluster.create(args.tier, "/bench/resident", 4200, n_total))
        _, _, sum_crc, _ = timed_read(fs, "/bench/resident", rank, world, dst, shard_bytes, torch.cuda.current_stream().cuda_stream)
        
        d_off = torch.arange(my_blocks, dtype=torch.int64, device="cuda") * BLOCK
        d_len = torch.full((my_blocks,), BLOCK, dtype=torch.int64, device="cuda")
        d_crc = torch.empty(my_blocks, dtype=torch.int32, device="cuda")
        stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

        def resident_step():
            _lib.check(L.cvk_crc_blocks(ctypes.c_void_p(dst.data_ptr()), ctypes.c_void_p(d_off.data_ptr()), ctypes.c_void_p(d_len.data_ptr()),
                                        my_blocks, args.poly, shard_bytes, ctypes.c_void_p(d_crc.data_ptr()), stream), "cvk_crc_blocks")

        for _ in range(3):
            resident_step()
        barrier(dist)
        L.cvk_profile_enable(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_c = time.time()
        a.record()
        for _ in range(5):
            resident_step()
        b.record()
        barrier(dist)
        t_d = time.time()
        res_ms = a.elapsed_time(b) / 5
        walk_ms, walk_n = ctypes.c_double(), ctypes.c_uint32()
        _lib.check(L.cvk_profile_collect(ctypes.byref(walk_ms), ctypes.byref(walk_n)), "cvk_profile_collect")
        L.cvk_profile_enable(0)
        assert int(d_crc.cpu().numpy().view(np.uint32).astype(np.uint64).sum()) == sum_crc, "resident K1 pass disagrees with the ingest's CRCs"
        cluster.drop("/bench/resident")
        fs.close()
        if "pread" in legs:
            # reference layout (one tmpfs file per block), never-read files, through the pinned ring
            def leg_pread():
                fs3 = F.CurvineFileSystem(client_conf(args, cluster, True, local, threads, slots, rank, zero_copy=False, copy_group=1))
                try:
                    return run_leg("pread", cluster, fs3, "files", args, rank, world, dist, dst, side_bytes, side, 1, True, 7000, pool=0)
                finally:
                    fs3.close()
            pread = guarded("pread", leg_pread)
        for leg_name, unix in (("framed", False), ("framed_unix", True)):
            if leg_name not in legs:
                continue
            # frames from the arena worker (sendfile out of the segment file), received verbatim, unpacked + CRC'd by K2; one block per
            # ring slot (copy_group 1): every connection fills its own slot, the verifier frees slots 16 blocks at a time
            def leg_framed(leg_name=leg_name, unix=unix):
                fs2 = F.CurvineFileSystem(client_conf(args, cluster, False, local, fthreads, 2 * args.verify_batch + 2 * fthreads + 8, rank, copy_group=1, unix=unix))
                try:
                    return run_leg(leg_name, cluster, fs2, "arena", args, rank, world, dist, dst, side_bytes, side, 1, True, 8000 + 500 * unix, pool=0)
                finally:
                    fs2.close()
            res_leg = guarded(leg_name, leg_framed)
            if unix:
                framed_unix = res_leg
            else:
                framed = res_leg

        # ---- max over ranks
        def maxr(x):
            if dist is None or x is None:
                return x
            t = torch.tensor([x], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        def mean(v):
            return sum(v) / len(v) if v else None

        e2e_ms = maxr(mean(head["e2e_ms"]))
        ing_ms = maxr(mean(head["ingest_ms"]))
        res_ms = maxr(res_ms)
        walk_avg_ms = maxr(walk_ms.value / max(1, walk_n.value))
        side_ms = {k: maxr(mean(v["e2e_ms"])) if v else None for k, v in (("reread", reread), ("pread", pread), ("framed", framed), ("framed_unix", framed_unix))}
        side_total = side_bytes * world
        per_step_e2e = [maxr(x) for x in head["e2e_ms"]]

        if rank == 0:
            peaks = {}
            try:
                peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            except Exception:
                pass
            hbm_peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
            gbps = lambda ms: n_total / ms / 1e6 if ms else None
            e2e_val, ing_val = gbps(e2e_ms), gbps(ing_ms)
            stats = head["stats"]
            out = {
                "metric": METRIC, "value": ing_val, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ing_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "value_is": "device-timed ingest of never-read files: first H2D copy .. CRCs verified and back on the host (cv_read_device + cv_verify), max over ranks",
                "config": {"workload": "C2 per GPU: %g GiB synthetic file per GPU per step, 4 MiB blocks, mem tier = %s, blocks round-robin across GPUs "
                                       "(C3 shape at N=8), on-GPU CRC-%s verify; every step reads a file nobody has read before"
                                       % (args.gib_per_gpu, "pinned-once arena (arena.h)" if args.tier == "arena" else "one tmpfs file per block", "32C" if args.poly else "32"),
                           "file_bytes": n_total, "block_bytes": BLOCK, "blocks_per_gpu": my_blocks, "read_path": args.mode, "mem_tier": args.tier,
                           "fresh_file_every_step": True, "files_kept_beside_the_current": args.pool, "arena_reuse_delay_ms": 0, "fetch_threads": threads, "pinned_slots": slots, "verify_batch": args.verify_batch,
                           "copy_group": args.copy_group, "arena_segment_bytes": SEG, "arena_register_slice": args.register_slice,
                           "l2": "inputs (%g GiB per GPU per step, new bytes every step) are larger than L2; no flush needed" % args.gib_per_gpu, "host_cpus": ncpu,
                           "gib_per_gpu_asked": asked_gib, "host_memory_budget": budget_sources,
                           "size_note": None if args.gib_per_gpu == asked_gib else "the box cannot hold %g GiB per GPU (stores must fit into 70%% of the smallest of %s): ran %g GiB per GPU" % (asked_gib, budget_sources, args.gib_per_gpu)},
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(stats["h2d_bytes"]) * world, "d2h_bytes_per_step": 4 * (my_blocks + 4) * world,
                        "ms_per_step": e2e_ms, "timed_steps_ms": per_step_e2e, "warmup_steps_ms": head["warm_e2e_ms"],
                        "what": "cv_open -> cv_read_device[_sharded] -> cv_verify -> cv_close_reader on a file written just before the step (never read), "
                                "host memory in, HBM + CRCs out",
                        "per_gpu_GBps": e2e_val / world, "frac_of_pcie_gen5_x16_raw_63GBps": e2e_val / world / PCIE_RAW,
                        "last_step_fetch_thread_sec": stats["fetch_sec"], "last_step_wall_sec": stats["wall_sec"]},
                "mount": {"arena_map_and_pin_ms": mount_ms, "pinned_bytes": arena0["pinned_bytes"], "segments": arena0["segments"],
                          "pin_GBps": arena0["pinned_bytes"] / max(arena0["register_us"], 1) / 1e3, "context_warmup_ms": ctx_warm_ms,
                          "worker_arena_create_populate_sec": cluster.info["arena_start_sec"],
                          "note": "paid once per client context, before any read; segments pinned after the headline steps: %d (unchanged = no per-file registration)" % arena1["segments"]},
                "arena_dma": {"block_jobs": arena1["dma_jobs"] - arena0["dma_jobs"], "bytes": arena1["dma_bytes"] - arena0["dma_bytes"],
                              "registered_mapping_cache_hits": stats["reg_hits"], "pinned_ring_allocated": stats["ring_alloc_sec"] > 0},
                "gpu_launches": int(launches),
                "resident_verify": {"value": gbps(res_ms), "unit": UNIT, "ms": res_ms, "what": "K1 + fold over the bytes already in HBM (no ingest): an HBM-bound kernel rate, not a read rate"},
                "roofline": {"bound": "hbm", "kernel": "walk_kernel<CRC,!DST> (K1 CRC verify)", "achieved": shard_bytes / walk_avg_ms / 1e6, "peak": hbm_peak,
                             "unit": "GB/s", "frac": shard_bytes / walk_avg_ms / 1e6 / hbm_peak, "traffic": ncu_traffic(shard_bytes), "peak_source": peak_src,
                             "note": "K1 only reads (N bytes in, 4 bytes per block out) while the peak is a read+write copy rate, so frac can exceed 1. The metric itself "
                                     "is bound by PCIe ingest (e2e.frac_of_pcie_gen5_x16_raw_63GBps), under which K1 hides completely.",
                             "algorithmic_bytes_per_launch": shard_bytes, "avg_launch_ms": walk_avg_ms, "launches_timed": int(walk_n.value)},
                "clocks": sampler.summary(head["windows"]),
                "clocks_resident": sampler.summary([(t_c, t_d)]),
                "setup": {"file_gen_sec_total": cluster.gen_sec, "sum_crc_last": head["sum_crc"]},
            }
            for k, what in (("reread", "the same (already read) arena file again: same path as the headline, nothing is cached per file"),
                            ("pread", "reference layout (one tmpfs file per block), never-read files: pread into the pinned ring, then H2D"),
                            ("framed", "short_circuit = false: frames from the arena worker over loopback TCP received verbatim, H2D of the wire image, K2 validates "
                                       "every prefix, gathers and CRCs (gpu_chunk %s, %d connections)" % (args.gpu_chunk, fthreads)),
                            ("framed_unix", "the same over the worker's same-host abstract unix socket ([b200] local_unix_socket)")):
                if side_ms[k]:
                    v = side_total / side_ms[k] / 1e6
                    leg = {"reread": reread, "pread": pread, "framed": framed, "framed_unix": framed_unix}[k]
                    out["e2e_" + k] = {"value": v, "unit": UNIT, "ms_per_step": side_ms[k], "per_gpu_GBps": v / world,
                                       "frac_of_pcie_gen5_x16_raw_63GBps": v / world / PCIE_RAW, "steps": side, "bytes_per_step": side_total, "what": what,
                                       "timed_steps_ms": leg["e2e_ms"], "last_step_fetch_thread_sec": leg["stats"]["fetch_sec"],
                                       "last_step_wall_sec": leg["stats"]["wall_sec"], "h2d_bytes_last_step": int(leg["stats"]["h2d_bytes"])}
            if side_errors:
                out["side_leg_errors"] = side_errors
            if world == 1 and not args.no_cpu_baseline and "cpu" in (legs or {"cpu"}):
                try:
                    out["cpu_baseline"] = cpu_baseline(cluster, args)
                except Exception as e:  # noqa: BLE001  (the reference arm reports the CPU number too; the headline line must still go out)
                    out["cpu_baseline_error"] = "%s: %s" % (type(e).__name__, e)
    finally:
        sampler.stop()
        cluster.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(out)


def ncu_traffic(shard_bytes):
    """dram bytes per K1 launch from the committed `ncu --set full` capture -- only when that capture was taken from THIS kernels.cu
    at this launch size; anything else reports null rather than a stale constant."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "k1_ncu_traffic.json")))
        sha = hashlib.sha256(open(os.path.join(ROOT, "curvine_b200", "csrc", "kernels.cu"), "rb").read()).hexdigest()
        if rec.get("kernels_cu_sha256") == sha and rec.get("launch_bytes") == shard_bytes:
            return rec.get("dram_bytes_per_launch")
    except Exception:
        pass
    return None


# ------------------------------------------------------------------ the reference's CPU read path (oracle port)

def cpu_run(port, n_total, sc, parallel, limit, inode, checksum=1):
    from oracle import clib, layout
    ids = [layout.create_block_id(inode, i) for i in range(n_total // BLOCK)]
    t0 = time.time()
    got, cks, threads = clib.cpu_read_file(port, sc, n_total, BLOCK, ids, 131072, 8, parallel, 131072, limit, checksum)
    dt = time.time() - t0
    return got / dt / 1e9, threads, got, cks, dt


def reference_policy(n_total):
    """The reference stripes one file over min(max_read_parallel = 8, ceil(len / large_file_size = 10 GiB)) sub-readers
    (read_detector.rs:130-135); both arms use this one policy."""
    from oracle import clib
    return clib.reference_read_parallel(n_total)


def cpu_baseline(cluster, args):
    """The reference's CPU read path (oracle port: per-chunk pread / ping-pong, memcpy, PCLMUL crc32 on the caller thread) on a
    bounded sample of the same workload in the reference's own layout (one tmpfs file per block), with the reference's
    read_parallel for this file size; whole-file passes repeated for about 12 s of CPU work."""
    n_total = int(args.gib_per_gpu * (1 << 30)) // BLOCK * BLOCK
    cluster.create("files", "/bench/cpu", 9100, n_total)
    port = cluster.info["files_port"]
    sc = args.mode == "short_circuit"
    par = reference_policy(n_total)
    pilot, _, _, _, _ = cpu_run(port, n_total, sc, par, 1 << 30, 9100)  # also the warm-up pass
    sample = int(min(n_total, max(1 << 30, pilot * 1e9 * 12))) // BLOCK * BLOCK
    passes, got_total, dt_total, threads = 0, 0, 0.0, 0
    while dt_total < 12.0 and passes < 16:
        v, threads, got, cks, dt = cpu_run(port, n_total, sc, par, sample, 9100)
        passes, got_total, dt_total = passes + 1, got_total + got, dt_total + dt
    cluster.drop("/bench/cpu")
    return {"value": got_total / dt_total / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d pass(es) over the first %.1f GiB of a %g GiB file in the reference layout, read_parallel=%d (reference default for this size), "
                      "128 KiB chunks and buffers, %s, crc32 (PCLMUL) on the caller thread; %.1f s of wall time"
                      % (passes, sample / 2 ** 30, n_total / 2 ** 30, par, "short-circuit pread" if sc else "framed over loopback TCP", dt_total)}


def main_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  It is Rust and cannot be built in this image
    (no cargo/rustc), so this times the oracle port (oracle/cpu_reader.c) on the host cores, against a worker emulator that is
    test infrastructure too (oracle/ref_worker.c: Open/Running/Complete over a reference-layout BlockStore written by the
    oracle's own generator) -- nothing of the product library is on this path."""
    rank, world, local, dist = setup_dist(args)
    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return
    from oracle import clib, refworker
    gib = args.gib_per_gpu * args.gpus
    n_total = int(gib * (1 << 30)) // BLOCK * BLOCK
    sc = args.mode == "short_circuit"
    base = args.dir or ("/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir())
    d = claim_store_dir(base, "cvref_")
    w = None
    try:
        w = refworker.RefWorker(d)
        # the file is n_total long for the reader (its striping policy depends on the length); only the head a step can reach is
        # written to the store -- the sub-readers stop at the sample's end, so the blocks behind it are never opened
        gen_total = min(n_total, int(args.ref_materialize_gib * (1 << 30)) // BLOCK * BLOCK)
        budget, _ = host_memory_budget(base)
        if budget is not None and not args.no_memory_guard:
            gen_total = max(BLOCK, min(gen_total, int(0.5 * budget) // BLOCK * BLOCK))
        w.create_file(9200, gen_total, BLOCK, threads=min(64, os.cpu_count() or 8))
        par = reference_policy(n_total)
        pilot, _, _, _, _ = cpu_run(w.port, n_total, sc, par, min(1 << 30, gen_total), 9200)
        sample = int(min(gen_total, max(1 << 30, pilot * 1e9 * 6))) // BLOCK * BLOCK
        times = []
        for it in range(args.warmup + args.steps):
            v, threads, got, cks, dt = cpu_run(w.port, n_total, sc, par, sample, 9200)
            if it >= args.warmup:
                times.append(dt)
        ms = 1e3 * sum(times) / len(times)
        val = sample / ms / 1e6
        # beside the stock policy: the same sample with the most sub-readers the reference ever uses (max_read_parallel = 8, client_conf.rs), for
        # a reader who wants to know what the CPU path does when it is given every thread it can take
        v8, threads8, _, _, _ = cpu_run(w.port, n_total, sc, 8, sample, 9200)
        out = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
               "config": {"workload": "C2 per GPU: %g GiB synthetic file, 4 MiB blocks, mem-tier (tmpfs, one file per block) BlockStore; CPU reader, bytes land in host memory" % gib,
                          "file_bytes": n_total, "materialized_bytes": gen_total, "block_bytes": BLOCK, "read_path": args.mode, "host_cpus": os.cpu_count()},
               "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": "each step reads the first %.1f GiB; read_parallel=%d (reference default for this size), 128 KiB chunks/buffers, "
                                          "crc32 (PCLMUL) on the caller thread; worker = oracle/ref_worker.c" % (sample / 2 ** 30, par)},
               "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
               "at_max_read_parallel": {"read_parallel": 8, "threads": threads8, "value": v8, "unit": UNIT, "note": "one pass over the same sample; not the stock policy for this file size"},
               "gpu_launches": 0}
    finally:
        if w is not None:
            w.stop()
        shutil.rmtree(d, ignore_errors=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    emit(out)


if __name__ == "__main__":
    main()
