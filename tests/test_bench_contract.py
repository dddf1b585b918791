"""bench.py's output contract, exercised on CPU through the reference arm (no GPU): exactly one JSON line on stdout with the
keys the driver reads."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gib-per-gpu", "0.125", "--steps", "1", "--warmup", "1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"] == "sequential read GB/s into HBM (CRC-verified)"
    for k in ("n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 2 and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def _shim_env():
    """The library the bench runs against here: the product's host side AND kernel source on the SIMT shim (tests/simt_emu), the runtime
    stand-in's streams asynchronous -- so the bench's own assertions (no CRC mismatch, the HBM-resident K1 pass agreeing with the ingest's
    CRCs) are checked by the real kernels, and its stream usage by the stream-order check."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("simt_emu_build", os.path.join(ROOT, "tests", "simt_emu", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return dict(os.environ, CV_TEST_MOCK_CUDA_LIB=mod.build(), MOCK_CUDA_ASYNC="1", MOCK_CUDA_JITTER_US="300", CV_SIMT_EMU_THREADS="4")


def test_own_arm_control_flow_and_json_line_on_the_mock_runtime():
    """bench.py's own arm (arena mount, context warm-up read, fresh-file steps, re-read / pread / framed side legs, HBM-resident K1
    steps, roofline, cpu_baseline) executed end to end without a GPU: tests/mock_cuda/run_bench_on_mock.py swaps in the mock library and
    tells torch that "cuda" tensors are CPU tensors.  Checks the control flow and the contract of the printed line; every number
    in it is meaningless here and is looked at only for type and bookkeeping (bytes per step, launch counts, DMA counters)."""
    env = _shim_env()
    gib, steps, warmup = 0.25, 2, 2
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "mock_cuda", "run_bench_on_mock.py"), "--gib-per-gpu", str(gib), "--steps", str(steps),
                        "--warmup", str(warmup)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    n = int(gib * (1 << 30))
    blocks = n // (4 << 20)
    assert "impl" not in d and d["metric"] == "sequential read GB/s into HBM (CRC-verified)" and d["unit"] == "GB/s"
    assert d["n_gpus"] == 1 and d["steps"] == steps and d["warmup"] == warmup and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "u8" and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"] and "model" not in d["config"]
    assert d["config"]["fresh_file_every_step"] is True and d["config"]["mem_tier"] == "arena"
    e = d["e2e"]
    assert e["unit"] == "GB/s" and e["value"] > 0 and e["h2d_bytes_per_step"] == n and e["d2h_bytes_per_step"] == 4 * (blocks + 4)
    assert len(e["timed_steps_ms"]) == steps and len(e["warmup_steps_ms"]) == warmup
    # `value` is an ingest rate of the same steps (device-timed region inside the e2e region), never the HBM-resident kernel rate
    assert d["value"] >= e["value"] * 0.999 and d["value"] < e["value"] * 1.5
    # every headline block was DMA'd out of the arena pinned at mount: nothing registered per file, no pinned ring
    a = d["arena_dma"]
    assert a["block_jobs"] == blocks * (steps + warmup) + 16 and a["registered_mapping_cache_hits"] == 0 and a["pinned_ring_allocated"] is False
    assert d["mount"]["segments"] >= 1 and d["mount"]["pinned_bytes"] == d["mount"]["segments"] * (256 << 20)
    assert d["gpu_launches"] > 0
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["algorithmic_bytes_per_launch"] == n and r["launches_timed"] == 5
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and "note" in r and r["traffic"] is None
    assert d["resident_verify"]["value"] > 0
    for leg in ("e2e_reread", "e2e_pread", "e2e_framed"):
        assert d[leg]["unit"] == "GB/s" and d[leg]["value"] > 0 and d[leg]["steps"] == 2, leg
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["unit"] == "GB/s" and c["value"] > 0 and c["cores"] >= 2 and "pass" in c["sample"]


def test_dump_outputs_are_the_last_steps_bytes_and_repeat_run_to_run(tmp_path):
    """--dump-outputs DIR: after the timed steps the bench writes what the last headline step put into HBM (a seeded byte sample and
    per-block byte sums) and the CRC sum cv_verify returned, as float .npy files.  Two runs with the same arguments write the same
    arrays, and they are the oracle's bytes of the file the last timed step read."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from oracle import clib, synth
    env = _shim_env()
    gib, steps, warmup, block = 1.0 / 16, 2, 1, 4 << 20
    dumps = []
    for k in range(2):
        d = tmp_path / str(k)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "mock_cuda", "run_bench_on_mock.py"), "--gib-per-gpu", str(gib), "--steps", str(steps),
                            "--warmup", str(warmup), "--side-steps", "0", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, env=env, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-3000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps.append({f: np.load(str(d / f)) for f in os.listdir(str(d))})
    assert set(dumps[0]) == {"bytes_sample.npy", "block_byte_sums.npy", "crc_sum.npy"}
    assert sum(a.nbytes for a in dumps[0].values()) <= 64 << 20
    for name, a in dumps[0].items():
        assert a.dtype in (np.float32, np.float64), name
        np.testing.assert_array_equal(a, dumps[1][name], err_msg=name)
    n = int(gib * (1 << 30))
    want = np.frombuffer(synth.file_bytes(5000 + warmup + steps - 1, n, block), dtype=np.uint8)  # run_leg's inode of the last timed step
    pos = bench.dump_positions(n, 1)
    assert pos.size == bench.DUMP_SAMPLE
    np.testing.assert_array_equal(dumps[0]["bytes_sample.npy"], want[pos].astype(np.float32))
    np.testing.assert_array_equal(dumps[0]["block_byte_sums.npy"], want.reshape(-1, block).sum(axis=1, dtype=np.int64).astype(np.float64))
    assert dumps[0]["crc_sum.npy"].tolist() == [float(clib.crc_blocks(1, want, block).astype(np.uint64).sum())]


def test_own_arm_two_ranks_on_the_mock_runtime():
    """The N>1 launch the driver uses (torch.distributed.run, one rank per GPU) with world_size 2 on CPU: gloo stands in for NCCL, the
    mock runtime for the GPUs.  Rank 0 hosts the worker and generates the 2 x 0.25 GiB file, the manifest is broadcast, every rank
    reads its round-robin shard out of ITS arena dir, timings are max-reduced, rank 0 prints the one line."""
    import socket
    env = dict(_shim_env(), OMP_NUM_THREADS="1", CV_SIMT_EMU_THREADS="2")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "tests", "mock_cuda", "run_bench_on_mock.py"), "--gpus", "2", "--gib-per-gpu", "0.25", "--steps", "2", "--warmup", "1", "--side-steps", "1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [l for l in p.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    d = json.loads(lines[0])
    n = 2 * int(0.25 * (1 << 30))
    assert d["n_gpus"] == 2 and d["scaling"] == "weak" and d["config"]["file_bytes"] == n and d["config"]["blocks_per_gpu"] == n // (4 << 20) // 2
    assert d["e2e"]["h2d_bytes_per_step"] == n and d["e2e"]["value"] > 0 and d["value"] > 0
    assert "cpu_baseline" not in d  # rank 0 at N=1 only


def test_smoke_control_flow_on_the_mock_runtime():
    """__graft_entry__.smoke() end to end without a GPU (mock runtime): the three passes it makes on the B200 -- files tier short-circuit,
    files tier framed, arena tier DMA -- each land the oracle's bytes and CRC sums."""
    env = _shim_env()
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "mock_cuda", "run_smoke_on_mock.py")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0 and "smoke ok" in p.stdout, p.stdout[-3000:]


def test_memory_guard_shrinks_a_size_the_container_cannot_hold():
    """bench.py's guard: stores must fit into 70 % of the smallest of MemAvailable / cgroup limit / tmpfs free space, else the per-GPU size
    is halved until they do (and the JSON line says so).  The run that cost round 2 its GPU access (128 GiB per GPU, one file kept beside
    the current one, on a ~250 GiB container) would have been cut down; the default sizes are untouched on the 2 TB boxes."""
    sys.path.insert(0, ROOT)
    import bench
    budget, src = bench.host_memory_budget("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp")
    assert budget and budget == min(src.values()) and "MemAvailable" in src
    G = 1 << 30
    assert bench.fit_gib_per_gpu(16, 1, 0, 2000 * G) == 16 and bench.fit_gib_per_gpu(16, 8, 0, 2000 * G) == 16
    assert bench.fit_gib_per_gpu(16, 8, 0, 250 * G) == 16          # round 1's 8-GPU footprint fits a 250 GiB container
    assert bench.fit_gib_per_gpu(128, 1, 1, 250 * G) == 32          # the lost-box run: 257 GiB asked of ~250
    assert bench.fit_gib_per_gpu(128, 1, 0, 2000 * G) == 128
    assert bench.fit_gib_per_gpu(16, 8, 0, 120 * G) == 4
    assert bench.fit_gib_per_gpu(16, 1, 0, None) == 16              # nothing known about the host: no change


def test_config_c5_line_on_the_shim():
    """bench.py --config c5 (small files, FUSE-shaped: tools/c5_smallfiles.py) end to end with 64 files: per-file path, batched path and the CPU
    port beside them, CRC checks inside the tool done by the real kernel source."""
    env = dict(_shim_env(), CV_C5_FILES="64")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "mock_cuda", "run_bench_on_mock.py"), "--config", "c5"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [l for l in p.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["unit"] == "files/s" and d["value"] > 0 and d["n_gpus"] == 1 and d["higher_is_better"] is True and "workload" in d["config"]
    assert d["e2e"]["value"] > 0 and d["gpu_launches"] > 0
