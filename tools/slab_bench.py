"""Whole-volume inference (BASELINE config 4: 155x190x147 padded to 160x192x160, VAE off) on N GPUs, depth-slab
sharded (3d-brain-tumor-segmentation_b200/slab.py).  Launch: python -m torch.distributed.run --nproc-per-node N
tools/slab_bench.py [reps] [eager|graph|both] [nccl|peer] [--data-format F] [--base-filters N] [--reduction R]
[--unsharded].  Prints per-mode ms (max over ranks), Mvoxel/s and the error against the un-sharded forward.
The model options select another model (e.g. the reference CLI's channels_first / 32 filters / reduction 8; its
input and output are NCDHW, the slabs are cut along D all the same); --unsharded also times the un-sharded forward.
Either adds the model configuration and the device name to the JSON line."""
import argparse
import importlib
import json
import os
import statistics
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
b3d = importlib.import_module("3d-brain-tumor-segmentation_b200")

ap = argparse.ArgumentParser()
ap.add_argument("reps", nargs="?", type=int, default=5)
ap.add_argument("mode", nargs="?", default="both")            # eager | graph | both
ap.add_argument("backend", nargs="?", default="nccl")         # nccl | peer (NVLink peer-memory kernels)
ap.add_argument("--data-format", default=None, choices=("channels_last", "channels_first"))
ap.add_argument("--base-filters", type=int, default=None)
ap.add_argument("--reduction", type=int, default=None)
ap.add_argument("--unsharded", action="store_true")
args = ap.parse_args()
reps, mode, backend = args.reps, args.mode, args.backend
model_kw = {k: v for k, v in (("data_format", args.data_format), ("base_filters", args.base_filters),
                              ("reduction", args.reduction)) if v is not None}
rank, local, world = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("LOCAL_RANK", 0), ("WORLD_SIZE", 1)))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
os.environ.setdefault("MASTER_PORT", "29533")
dist.init_process_group("nccl", device_id=dev, rank=rank, world_size=world)

shape = (160, 192, 160)
b3d.keras_compat.set_seed(99)                     # identical random-init weights on every rank
model = b3d.Model(**model_kw)
ax = b3d.slab.depth_axis(model)                   # 2: NCDHW public tensors (channels_first), else 1
with torch.no_grad():
    model(torch.zeros(1, 16, 16, 16, 2, device=dev).movedim(4, 1) if ax == 2 else
          torch.zeros(1, 16, 16, 16, 2, device=dev), training=False, inference=True)
g = torch.Generator().manual_seed(7)
for v in model.variables():                       # non-trivial GN affine parameters (gamma2 is zero-initialised)
    if v.name in ("gamma", "beta", "bias"):
        v.tensor.data.add_(0.1 * torch.randn(v.tensor.shape, generator=g).to(dev))
g = torch.Generator().manual_seed(123)
x = torch.randn((1,) + shape + (2,), generator=g)
x[:, 155:], x[:, :, 190:], x[:, :, :, 147:] = 0, 0, 0
x = x.to(dev)
if ax == 2:
    x = x.movedim(4, 1).contiguous()
comm = b3d.PeerComm() if (backend == "peer" and world > 1) else b3d.DistComm()
bounds = b3d.slab_bounds(shape[0], world)
d0, d1 = bounds[rank]
with torch.no_grad():
    whole = model(x, training=False, inference=True)[0].narrow(ax, d0, d1 - d0).clone()


def timed(fn):
    ts = []
    for i in range(reps + 2):
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); y = fn(); e1.record(); e1.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if i >= 2:
            ts.append(float(ms))
    err = ((y - whole).double().norm() / whole.double().norm()).reshape(1).float()
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    return statistics.median(ts), float(err)


res = {"n_gpus": world, "backend": backend, "slabs": [b - a for a, b in bounds]}
if model_kw or args.unsharded:
    res["model"] = {k: model.encoder.config[k] for k in ("data_format", "base_filters", "reduction")}
    res["device"] = torch.cuda.get_device_name(dev)
if args.unsharded:
    def unsharded():
        with torch.no_grad():
            return model(x, training=False, inference=True)[0].narrow(ax, d0, d1 - d0)
    ms, err = timed(unsharded)
    res["unsharded"] = {"ms": ms, "mvoxel_per_s": 155 * 190 * 147 / ms / 1e3, "rel_l2_vs_unsharded": err}
if mode in ("eager", "both"):
    ms, err = timed(lambda: b3d.sharded_inference(model, x, comm, gather=False)[0])
    res["eager"] = {"ms": ms, "mvoxel_per_s": 155 * 190 * 147 / ms / 1e3, "rel_l2_vs_unsharded": err}
if mode in ("graph", "both"):
    gi = b3d.GraphedInference(model, x.narrow(ax, d0, d1 - d0).contiguous(), comm if world > 1 else None,
                              depth=shape[0])
    ms, err = timed(lambda: gi())
    res["graph"] = {"ms": ms, "mvoxel_per_s": 155 * 190 * 147 / ms / 1e3, "rel_l2_vs_unsharded": err}
if rank == 0:
    print(json.dumps(res), flush=True)
dist.barrier(); torch.cuda.synchronize(); sys.stdout.flush()
os._exit(0)
