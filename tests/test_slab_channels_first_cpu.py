"""CPU suite — host logic of depth-slab inference for channels_first models: their public tensors are NCDHW, so the
drivers cut the volume and gather the slabs along dim 2 (the slab arithmetic is covered by
tests/test_gpu_slab_channels_first.py)."""
import importlib
import os
import sys
import threading

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "3d-brain-tumor-segmentation_b200"


def test_depth_axis_follows_data_format(b3d):
    assert b3d.slab.depth_axis(b3d.Model()) == 1
    assert b3d.slab.depth_axis(b3d.Model(data_format='channels_first')) == 2


def _gather_ncdhw(b3d, comm, x):
    bounds = b3d.slab_bounds(x.shape[2], comm.world)
    d0, d1 = bounds[comm.rank]
    return torch.equal(comm.all_gather_cat(x[:, :, d0:d1].contiguous(), [b - a for a, b in bounds], dim=2), x)


def test_thread_comm_gathers_along_depth_of_ncdhw(b3d):
    x = torch.randn(1, 3, 48, 5, 4)
    for world in (1, 2, 3):
        comms = b3d.ThreadComm.make(world)
        res = [None] * world

        def work(r):
            res[r] = _gather_ncdhw(b3d, comms[r], x)

        ts = [threading.Thread(target=work, args=(r,)) for r in range(world)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert res == [True] * world


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    b3d = importlib.import_module(PKG)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, 3, 32, 5, 4, generator=g)
    q.put((rank, _gather_ncdhw(b3d, b3d.DistComm(), x)))
    dist.destroy_process_group()


def test_dist_comm_gathers_along_depth_of_ncdhw_gloo(b3d):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert res == [(0, True), (1, True)]
