"""GPU suite — depth-slab sharded whole-volume inference (BASELINE config 4, SURVEY §8e): the halo form of the
conv kernels, the slab form of GroupNormalization, and the whole model run as N virtual ranks on one device must
reproduce the un-sharded forward (which tests/test_gpu_model.py pins to the oracle)."""
import pytest
import torch

from oracle import ref_model as R

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def t32(*shape, seed=0, scale=1.0, dev=None):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dev)


HALO_CASES = [
    # (D, H, W), Cin, Cout, k, stride, transposed
    ((16, 16, 8), 16, 16, 3, 1, False),
    ((16, 20, 12), 32, 16, 3, 1, False),
    ((16, 8, 8), 2, 16, 3, 1, False),          # CUDA-core path
    ((16, 16, 16), 16, 16, 3, 2, False),
    ((16, 8, 24), 64, 32, 3, 2, False),
    ((16, 8, 8), 12, 8, 3, 2, False),          # CUDA-core path
    ((8, 8, 8), 32, 16, 3, 2, True),
    ((8, 6, 10), 64, 32, 3, 2, True),
    ((8, 4, 4), 1, 128, 3, 2, True),           # CUDA-core path
]


@pytest.mark.parametrize("case", HALO_CASES)
@pytest.mark.parametrize("tc", [False, True])
def test_conv_halo_equals_whole_volume(b3d, dev, case, tc):
    sp, cin, cout, k, stride, tr = case
    ops = b3d.ops
    ops.USE_TC["on"] = tc
    try:
        x = t32(1, *sp, cin, seed=1, dev=dev)
        w = t32(k, k, k, *((cout, cin) if tr else (cin, cout)), seed=2, scale=0.2, dev=dev)
        bias = t32(cout, seed=3, dev=dev)
        with torch.no_grad():
            whole = ops.conv3d(x, w, bias, stride, tr)[0]
        D = sp[0]
        cuts = [0, D // 4, D // 2, D] if D >= 8 else [0, D // 2, D]
        before, after = (1, 0) if tr else ((0, 1) if stride == 2 else (1, 1))
        parts = []
        for a, b in zip(cuts, cuts[1:]):
            lo, hi = a - before, b + after
            xin = torch.zeros((1, hi - lo) + tuple(x.shape[2:]), device=dev)
            l2, h2 = max(lo, 0), min(hi, D)
            xin[:, l2 - lo:h2 - lo] = x[:, l2:h2]
            od = 2 * (b - a) if tr else (b - a) // stride
            oh, ow = (2 * sp[1], 2 * sp[2]) if tr else (sp[1] // stride, sp[2] // stride)
            y = torch.empty(1, od, oh, ow, cout, device=dev)
            wp = None
            if tc and ops.tc_supported(w, stride, tr, False):
                wp = ops.pack_weights(w, False, stride, tr)
            ops._call("b3d_conv3d_fwd_halo", xin, w, bias, y, stride, int(tr), 0, before, after, None, wp)
            parts.append(y)
        got = torch.cat(parts, dim=1)
        assert got.shape == whole.shape
        assert rel(got, whole) < 1e-6, rel(got, whole)
    finally:
        ops.USE_TC["on"] = True


@pytest.mark.parametrize("shape", [(1, 16, 6, 4, 16), (1, 20, 24, 20, 128), (1, 40, 6, 6, 8)])
@pytest.mark.parametrize("relu", [False, True])
def test_group_norm_slab_equals_whole(b3d, dev, shape, relu):
    """Chunks (1/8 of the flat volume) do not line up with the slabs (20 slices / 8 chunks = 2.5 slices each)."""
    ops = b3d.ops
    x = t32(*shape, seed=4, dev=dev)
    ga, be = 1 + 0.3 * t32(shape[-1], seed=5, dev=dev), 0.3 * t32(shape[-1], seed=6, dev=dev)
    with torch.no_grad():
        whole = ops.group_norm(x, ga, be, None, 8, 1e-5, relu)
    D = shape[1]
    cuts = [0, D // 4, D // 4 * 3, D]
    per = shape[2] * shape[3]
    total = D * per
    stats = torch.zeros(1, 8, 2, dtype=torch.float64, device=dev)
    for a, b in zip(cuts, cuts[1:]):
        part = torch.empty_like(stats)
        ops._call("b3d_gn_stats", x[:, a:b].contiguous(), part, 8, a * per, total)
        stats += part
    ch = x.double().reshape(1, 8, -1)
    assert rel(stats, torch.stack([ch.sum(-1), (ch ** 2).sum(-1)], dim=-1)) < 1e-6
    parts = []
    for a, b in zip(cuts, cuts[1:]):
        xs = x[:, a:b].contiguous()
        y = torch.empty_like(xs)
        ops._call("b3d_gn_apply", xs, stats, ga, be, y, None, None, 8, 1e-5, int(relu), a * per, total)
        parts.append(y)
    assert rel(torch.cat(parts, dim=1), whole) < 1e-6
    yr = R.group_norm(x.double().cpu(), ga.double().cpu(), be.double().cpu())
    yr = torch.relu(yr) if relu else yr
    assert rel(torch.cat(parts, dim=1), yr) < 2e-5


def _built_model(b3d, dev, seed=0):
    b3d.keras_compat.set_seed(1234 + seed)
    model = b3d.Model()
    with torch.no_grad():
        model(torch.zeros(1, 16, 16, 16, 2, device=dev), training=False, inference=True)
    # non-trivial GroupNorm affine parameters / biases (gamma2 is zero-initialised in the reference)
    g = torch.Generator().manual_seed(7)
    for v in model.variables():
        if v.name in ("gamma", "beta", "bias"):
            v.tensor.data.add_(0.1 * torch.randn(v.tensor.shape, generator=g).to(dev))
    return model


@pytest.mark.parametrize("world,shape", [(2, (32, 16, 16)), (3, (48, 32, 16)), (4, (64, 16, 32))])
@pytest.mark.parametrize("tc", [False, True])
def test_virtual_rank_slab_inference_equals_whole_volume(b3d, dev, world, shape, tc):
    ops = b3d.ops
    ops.USE_TC["on"] = tc
    try:
        model = _built_model(b3d, dev)
        x = t32(1, *shape, 2, seed=11, dev=dev)
        with torch.no_grad():
            whole = model(x, training=False, inference=True)[0]
        got, stats = b3d.slab.run_virtual_ranks(model, x, world)
        assert got.shape == whole.shape
        # same kernels, same per-voxel accumulation order; only the summation order of the statistics differs.
        # With tf32 operands those last-bit differences move some conv inputs across a tf32 rounding boundary
        # (2^-11), so the sharded result is compared at half the north_star per-layer TF32 tolerance.
        assert rel(got, whole) < (1e-3 if tc else 5e-5), rel(got, whole)
        agree = (got.argmax(-1) == whole.argmax(-1)).float().mean()
        assert float(agree) >= 0.999
        # one exchange per 3x3x3 conv of the inference forward: 26 stride-1 (13 blocks x 2), 3 strided, 3 transposed.
        # P16 form (tensor cores on): a conv reading a virtual concat exchanges every source that has not been
        # exchanged yet — one more per decoder level (encoder residual + upsampled tensor), none for the dense
        # connections of the encoder (their older sources were exchanged by earlier blocks)
        assert stats[0]["halo_exchanges"] == (35 if tc else 32)
        # statistics / pooling sums: 2 exchanges per ResnetBlock + 1 per resampling layer in the P16 form
        if tc:
            assert stats[0]["all_reduces"] <= 13 * 2 + 6 + 2
    finally:
        ops.USE_TC["on"] = True


def test_slab_inference_matches_oracle(b3d, dev):
    """End to end against the fp64 oracle (fp32 CUDA-core mode, tight tolerance)."""
    crop = (32, 32, 16)
    p = R.init_params(R.param_shapes(crop=crop))
    x, _, eps, _ = R.synth_batch((1,) + crop)
    yr = R.model_forward(p, x, eps, inference=True)[0]
    ops = b3d.ops
    ops.USE_TC["on"] = False
    try:
        model = b3d.Model()
        xd = x.float().to(dev)
        with torch.no_grad():
            model(xd, training=False, inference=False, eps=eps.float().to(dev))
        model.load_named_weights(p)
        got, _ = b3d.slab.run_virtual_ranks(model, xd, 2)
        assert rel(got, yr) < 2e-5, rel(got, yr)
    finally:
        ops.USE_TC["on"] = True


def _peer_worker(rank, world, port, q):
    import importlib
    import os
    import sys
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    b3d = importlib.import_module("3d-brain-tumor-segmentation_b200")
    try:
        model = _built_model(b3d, dev)                     # same seed => same weights on every rank
        x = t32(1, 32, 32, 16, 2, seed=11, dev=dev)
        with torch.no_grad():
            whole = model(x, training=False, inference=True)[0]
        res = {}
        for name, comm in (("peer", b3d.PeerComm(mailbox_bytes=1 << 20)), ("nccl", b3d.DistComm())):
            y, (d0, d1) = b3d.sharded_inference(model, x, comm, gather=False)
            res[name] = rel(y, whole[:, d0:d1])
            # twice more through one CUDA graph (epoch counter / sequence numbers advance on replay)
            if name == "peer":
                gi = b3d.GraphedInference(model, x[:, d0:d1].contiguous(), comm, depth=x.shape[1])
                gi(); res["peer_graph"] = rel(gi(), whole[:, d0:d1])
        q.put((rank, res))
    except BaseException as e:      # noqa: BLE001
        q.put((rank, repr(e)))
    dist.barrier()
    torch.cuda.synchronize()
    os._exit(0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_peer_memory_comm_two_gpus():
    """PeerComm (NVLink peer-memory halo exchange + small all-reduces, csrc/slab_comm.cu) and DistComm (NCCL) on two
    real GPUs against the un-sharded forward, eagerly and through a replayed CUDA graph."""
    import os
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 30500 + os.getpid() % 2000
    procs = [ctx.Process(target=_peer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for r in (0, 1):
        assert isinstance(out[r], dict), out[r]
        assert all(v < 1e-3 for v in out[r].values()), out
