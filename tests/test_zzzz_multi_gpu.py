"""Real multi-GPU checks (need >= 2 visible devices; skipped on a one-GPU box): the sharded read lands each rank's blocks on ITS
device, and cvk_gather_shards_p2p pulls every block straight out of its owner's HBM over NVLink (true peer pointers, not
same-device stand-ins) into file order -- config C4's exchange.  Bytes and CRCs against the oracle."""
import os
import shutil
import tempfile

import numpy as np
import pytest

from curvine_b200 import _lib, fs as F, kernels as K
from oracle import clib, synth

pytestmark = pytest.mark.gpu


MOCK = bool(os.environ.get("CV_TEST_MOCK_CUDA_LIB"))  # host-side stand-ins (tests/mock_cuda, tests/simt_emu): eight pretend devices in host memory


def _need_two():
    import torch
    if not MOCK and torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    return torch


def _on(torch, g):
    """(context that makes device g current, torch device string)"""
    import contextlib
    return (contextlib.nullcontext(), "cpu") if MOCK else (torch.cuda.device(g), "cuda:%d" % g)


@pytest.mark.parametrize("arena", [True, False])
def test_sharded_read_on_two_devices_then_p2p_gather_from_real_peer_memory(cuda, arena):
    torch = _need_two()
    world = 2 if MOCK else min(torch.cuda.device_count(), 4)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    d = tempfile.mkdtemp(prefix="cvmg", dir=base)
    bs, nb = 1 << 20, 37
    n, ino = bs * nb - 1000, 8101
    want = synth.file_bytes(ino, n, bs)
    per = (nb + world - 1) // world
    try:
        extra = 'mem_arena = true\narena_segment = "16MB"\narena_numa = [%s]\n' % ", ".join(str(_lib.lib().cv_gpu_numa_node(g)) for g in range(world)) if arena else ""
        dirs = ["[MEM:64MB]%s/m%d" % (d, g) for g in range(world)]
        with F.MiniWorker(dirs, extra_worker=extra) as w:
            _lib.lib().cv_synth_set_shard_world(world)
            try:
                man = w.create_file("/ckpt", ino, n, bs, threads=4)
            finally:
                _lib.lib().cv_synth_set_shard_world(0)
            shards, total = [], 0
            for g in range(world):
                conf = F.client_conf(b200='device = %d\nfetch_threads = 4\nverify_batch = 4\npinned_slots = 12\nzero_copy = true\ncopy_group = 2\n'
                                          'register_threads = 2\narena_register_slice = "4MB"\narena_preregister = ["%s/m%d"]\n' % (g, d, g))
                with F.CurvineFileSystem(conf) as fs:
                    fs.load_namespace(man)
                    ctx, dev = _on(torch, g)
                    with ctx:
                        shard = torch.zeros(per * bs, dtype=torch.uint8, device=dev)
                        r = fs.open("/ckpt")
                        got = r.read_device_sharded(g, world, shard.data_ptr(), per * bs, torch.cuda.current_stream().cuda_stream)
                        s, bad, ver = r.verify()
                        torch.cuda.synchronize()
                        plan = r.shard_plan(g, world)
                        r.complete()
                    assert bad == 0 and ver == len(plan) and got == sum(p[2] for p in plan)
                    if arena:
                        assert fs.arena_stats()["dma_jobs"] == len(plan)
                    host = shard.cpu().numpy().tobytes()
                    for (b, foff, ln, doff) in plan:
                        assert host[doff:doff + ln] == want[foff:foff + ln]
                    total += s
                    shards.append(shard)
            assert total == int(clib.crc_blocks(1, np.frombuffer(want, dtype=np.uint8), bs).astype(np.uint64).sum())
            # every device pulls the whole file out of the owners' HBM
            ptrs = [int(t.data_ptr()) for t in shards]
            for g in range(world):
                ctx, dev = _on(torch, g)
                with ctx:
                    final = torch.full((n + 64,), 0x77, dtype=torch.uint8, device=dev)
                    K.gather_shards_p2p(ptrs, bs, nb, n, final)
                    torch.cuda.synchronize()
                    out = final.cpu().numpy().tobytes()
                    assert out[:n] == want and out[n:] == b"\x77" * 64
                    # whole-file re-verify with K1 on the gathering device
                    offs = [b * bs for b in range(nb)]
                    lens = [min(bs, n - o) for o in offs]
                    crc = K.u32(K.crc_blocks(final, offs, lens, 1))
                    assert crc.tolist() == clib.crc_blocks(1, np.frombuffer(want, dtype=np.uint8), bs).tolist()
    finally:
        shutil.rmtree(d, ignore_errors=True)
