"""Multi-GPU result return on hardware (SURVEY.md §4: "N ranks each reproduce the single-GPU result on their shard; gathered list ==
single-GPU list"): the device compaction kernel against its host restatement on one GPU, and — when the box has two GPUs — two NCCL
ranks that shard a ragged batch of the shipped images, detect on their own GPU and return their lists to rank 0, which must hold
exactly what one GPU computes for the whole batch."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import yolo_fastest_b200 as yf
from yolo_fastest_b200 import _lib
from yolo_fastest_b200.dist import gather_compact, pack_host, shard_range, split_records

from conftest import GOLD

pytestmark = pytest.mark.gpu


def _batch(n):
    g = np.load(os.path.join(GOLD, "golden_256x320.npz"))
    base = g["u8"]
    return np.stack([np.roll(base[i % len(base)], (5 * (i // len(base)), 9 * (i // len(base))), axis=(0, 1)) for i in range(n)])


def test_compact_kernel_equals_host_packer():
    det = yf.Detect_YOLO(torch.device("cuda:0"), os.path.join(GOLD, "weights", "yolo_fastest_256x320.pth"), yf.config_for("256x320"), None)
    u8 = _batch(300)                                     # more images than the 256 threads of the scan block
    x = ((torch.from_numpy(u8).cuda().float().unsqueeze(1) - 128.0) / 255.0).contiguous()
    out, counts, _ = det.detect_device(x, max_det=4)     # a small capacity, so some images overflow it and are clipped
    torch.cuda.synchronize()
    assert int(counts.max()) >= 2 and int(counts.min()) == 0
    for cap in (300 * 4, 97):                            # roomy, and too small (records beyond cap are dropped, total stays)
        hdr_slots = 302
        packed = torch.zeros(4 * hdr_slots + 56 * cap, dtype=torch.uint8, device="cuda")
        ctx = det.model._ctx
        _lib.check(_lib.lib().yf_compact_dets(ctx.handle, out.data_ptr(), counts.data_ptr(), 300, 4, packed.data_ptr(), hdr_slots, cap,
                                              C.c_void_p(torch.cuda.current_stream().cuda_stream)), ctx.handle)
        want = pack_host(out.cpu(), counts.cpu(), hdr_slots, cap)
        assert torch.equal(packed.cpu(), want)


def _worker(rank, world, port, n_total, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    det = yf.Detect_YOLO(dev, os.path.join(GOLD, "weights", "yolo_fastest_256x320.pth"), yf.config_for("256x320"), None)
    u8 = _batch(n_total)
    lo, hi = shard_range(n_total, rank, world)
    ok = True
    for step in range(3):                                 # three steps: both buffer sets of the gather and their reuse
        mine = torch.from_numpy(np.roll(u8[lo:hi], step, axis=2).copy()).pin_memory()
        out, cnt = det.submit_batch_device(mine, step & 1, max_det=16)
        det.wait(step & 1)
        h = gather_compact(out, cnt, n_total, dst=0, ctx=det.model._ctx)
        recs, cnts = h.result()
        if rank == 0:
            got = split_records(recs, cnts)
            want = det.detect_batch(np.roll(u8, step, axis=2), max_det=16, raw=True)       # the whole batch on ONE GPU
            ok = ok and len(got) == n_total and sum(len(w) for w in want) > n_total // 2
            ok = ok and all(g.tobytes() == w.tobytes() for g, w in zip(got, want))
        else:
            ok = ok and recs is None
    if rank == 0:
        q.put(bool(ok))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_nccl_gather_equals_single_gpu():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    n_total, world = 41, 2                                # ragged: 21 + 20 images
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_total, q)) for r in range(world)]
    for p in procs:
        p.start()
    ok = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert ok is True
