"""SSD-tier blocks into HBM: GPUDirect Storage (cuFileRead, curvine_b200/csrc/host/gds.h) where the box offers it (nvidia-fs loaded)
and the pinned ring otherwise.  Whatever path runs, bytes and CRCs must equal the
oracle's (SURVEY.md 8f-2; tier model: storage_info.rs:36-49, local_file.rs:202-213)."""
import os
import shutil
import tempfile

import numpy as np
import pytest

from curvine_b200 import fs as F
from oracle import clib, synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("gds", ["off", "auto"])
def test_ssd_tier_file_lands_bit_exact_whichever_path_serves_it(cuda, gds):
    import torch
    d = tempfile.mkdtemp(prefix="cvssd", dir=os.environ.get("CV_SSD_DIR", "/tmp"))  # a disk-backed directory, not tmpfs
    try:
        with F.MiniWorker(["[SSD]" + d]) as w:
            n, bs, ino = (24 << 20) + 4097, 4 << 20, 8801
            man = w.create_file("/ssd", ino, n, bs, storage_type=1)
            assert " 1 " in man.splitlines()[2]  # storage type SSD in the manifest
            want = synth.file_bytes(ino, n, bs)
            conf = F.client_conf(b200='fetch_threads = 4\nverify_batch = 4\npinned_slots = 12\nzero_copy = true\ncopy_group = 2\ngds = "%s"\n' % gds)
            with F.CurvineFileSystem(conf) as fs:
                fs.load_namespace(man)
                info = F.gds_info()
                r = fs.open("/ssd")
                r.seek(12345)
                dst = torch.full((n,), 0x11, dtype=torch.uint8, device=cuda)
                got = r.read_device(dst.data_ptr(), n, torch.cuda.current_stream().cuda_stream)
                s, bad, ver = r.verify()
                torch.cuda.synchronize()
                assert got == n - 12345 and bad == 0 and ver == 6  # block 0 is partial
                assert dst[:got].cpu().numpy().tobytes() == want[12345:]
                st = r.device_stats()
                may_gds = info["available"] and gds == "auto"
                # either every byte went through cuFileRead, or cuFile turned the files away and every byte took the pinned ring
                assert st["gds_bytes"] in ((0, got) if may_gds else (0,)), (st["gds_bytes"], F.gds_info(), gds)
                r.complete()
                # whole file again from the start: every block comparable
                r = fs.open("/ssd")
                got = r.read_device(dst.data_ptr(), n, torch.cuda.current_stream().cuda_stream)
                s, bad, ver = r.verify()
                torch.cuda.synchronize()
                assert got == n and bad == 0 and ver == 7
                assert s == int(clib.crc_blocks(1, np.frombuffer(want, dtype=np.uint8), bs).astype(np.uint64).sum())
                assert dst.cpu().numpy().tobytes() == want
                r.complete()
    finally:
        shutil.rmtree(d, ignore_errors=True)


def test_ssd_tier_file_lands_bit_exact_over_frames(cuda):
    """short_circuit = false: the worker reads the SSD-tier block files and sends them as frames, which K2 unpacks and CRCs on the GPU.
    cuFile never serves a framed read, whatever [b200] gds says."""
    import torch
    d = tempfile.mkdtemp(prefix="cvssdf", dir=os.environ.get("CV_SSD_DIR", "/tmp"))  # a disk-backed directory, not tmpfs
    try:
        with F.MiniWorker(["[SSD]" + d]) as w:
            n, bs, ino = (24 << 20) + 4097, 4 << 20, 8802
            man = w.create_file("/ssdf", ino, n, bs, storage_type=1)
            want = synth.file_bytes(ino, n, bs)
            conf = F.client_conf(short_circuit=False, b200='fetch_threads = 4\nverify_batch = 4\npinned_slots = 16\ncopy_group = 1\ngds = "auto"\n')
            with F.CurvineFileSystem(conf) as fs:
                fs.load_namespace(man)
                dst = torch.full((n,), 0x11, dtype=torch.uint8, device=cuda)
                r = fs.open("/ssdf")
                got = r.read_device(dst.data_ptr(), n, torch.cuda.current_stream().cuda_stream)
                s, bad, ver = r.verify()
                torch.cuda.synchronize()
                assert got == n and bad == 0 and ver == 7
                assert s == int(clib.crc_blocks(1, np.frombuffer(want, dtype=np.uint8), bs).astype(np.uint64).sum())
                assert dst.cpu().numpy().tobytes() == want
                assert r.device_stats()["gds_bytes"] == 0
                r.complete()
    finally:
        shutil.rmtree(d, ignore_errors=True)
