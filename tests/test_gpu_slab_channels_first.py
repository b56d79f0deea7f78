"""GPU suite — depth-slab sharded inference of channels_first models (true channel GroupNorm, NCDHW public tensors):
the slab form of the channel GroupNorm (`b3d_gn_channel_apply_slab` over the summed `b3d_gn_channel_stats` of the
slabs) and the whole model run as N ranks must reproduce the un-sharded channels_first forward, which
tests/test_gpu_model.py pins to the oracle."""
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


cf = lambda t: t.permute(0, 4, 1, 2, 3).contiguous()        # NDHWC -> NCDHW


@pytest.mark.parametrize("shape", [(1, 16, 6, 4, 16), (1, 20, 24, 20, 128), (1, 24, 8, 8, 256)])
@pytest.mark.parametrize("relu", [False, True])
def test_channel_group_norm_slab_equals_whole(b3d, dev, shape, relu):
    ops, G = b3d.ops, 8
    C = shape[-1]
    x = t32(*shape, seed=4, dev=dev) + 0.5
    ga, be = 1 + 0.3 * t32(C, seed=5, dev=dev), 0.3 * t32(C, seed=6, dev=dev)
    D, S = shape[1], shape[1] * shape[2] * shape[3]
    cuts = [0, D // 4, D // 4 * 3, D]
    stats = torch.zeros(1, G, 2, dtype=torch.float64, device=dev)
    for a, b in zip(cuts, cuts[1:]):
        part = torch.empty_like(stats)
        ops._call("b3d_gn_channel_stats", x[:, a:b].contiguous(), part, G)
        stats += part
    grp = x.double().reshape(S, G, C // G)
    assert rel(stats[0], torch.stack([grp.sum((0, 2)), (grp ** 2).sum((0, 2))], dim=-1)) < 1e-6

    whole_stats = torch.empty_like(stats)
    ops._call("b3d_gn_channel_stats", x, whole_stats, G)
    whole = torch.empty_like(x)
    ops._call("b3d_gn_channel_apply", x, whole_stats, ga, be, whole, G, 1e-5, int(relu))
    parts = []
    for a, b in zip(cuts, cuts[1:]):
        xs = x[:, a:b].contiguous()
        y = torch.empty_like(xs)
        y16 = ops.p16_empty(xs.shape, xs, torch.float16)
        ops._call("b3d_gn_channel_apply_slab", xs, stats, ga, be, y, y16, G, 1e-5, int(relu), S)
        assert torch.equal(y16, ops.to_p16(y, torch.float16))
        only16 = ops.p16_empty(xs.shape, xs, torch.float16)          # twin-only call: the same twin
        ops._call("b3d_gn_channel_apply_slab", xs, stats, ga, be, None, only16, G, 1e-5, int(relu), S)
        assert torch.equal(only16, y16)
        parts.append(y)
    got = torch.cat(parts, dim=1)
    assert rel(got, whole) < 1e-6, rel(got, whole)
    with R.channels_first_semantics():
        yr = R.group_norm(x.double().cpu(), ga.double().cpu(), be.double().cpu())
    yr = torch.relu(yr) if relu else yr
    assert rel(got, yr) < 2e-5, rel(got, yr)

    # total_voxels = the tensor's own voxel count: the un-sharded apply
    y1 = torch.empty_like(x)
    ops._call("b3d_gn_channel_apply_slab", x, whole_stats, ga, be, y1, None, G, 1e-5, int(relu), S)
    assert rel(y1, whole) < 1e-6


def test_channel_group_norm_slab_rejects_bad_arguments(b3d, dev):
    ops = b3d.ops
    x = t32(1, 4, 4, 4, 16, dev=dev)
    ga, be = torch.ones(16, device=dev), torch.zeros(16, device=dev)
    st = torch.zeros(1, 8, 2, dtype=torch.float64, device=dev)
    y = torch.empty_like(x)
    with pytest.raises(b3d._lib.B3DError, match="neither y nor y16"):
        ops._call("b3d_gn_channel_apply_slab", x, st, ga, be, None, None, 8, 1e-5, 0, 64)
    with pytest.raises(b3d._lib.B3DError, match="stats"):
        ops._call("b3d_gn_channel_apply_slab", x, st[:, :4], ga, be, y, None, 8, 1e-5, 0, 64)
    with pytest.raises(b3d._lib.B3DError, match="total_voxels"):
        ops._call("b3d_gn_channel_apply_slab", x, st, ga, be, y, None, 8, 1e-5, 0, 32)
    with pytest.raises(b3d._lib.B3DError, match="twin"):
        ops._call("b3d_gn_channel_apply_slab", x, st, ga, be, y, ops.p16_empty((1, 4, 4, 4, 32), x, torch.float16),
                  8, 1e-5, 0, 64)


def _built_model(b3d, dev, seed=0, **kw):
    b3d.keras_compat.set_seed(1234 + seed)
    model = b3d.Model(data_format='channels_first', **kw)
    with torch.no_grad():
        model(torch.zeros(1, 2, 16, 16, 16, device=dev), training=False, inference=True)
    # non-trivial GroupNorm affine parameters / biases (gamma2 is zero-initialised in the reference)
    g = torch.Generator().manual_seed(7)
    for v in model.variables():
        if v.name in ("gamma", "beta", "bias"):
            v.tensor.data.add_(0.1 * torch.randn(v.tensor.shape, generator=g).to(dev))
    return model


def _check_virtual_ranks(b3d, model, x, world, tc):
    with torch.no_grad():
        whole = model(x, training=False, inference=True)[0]
    got, stats = b3d.slab.run_virtual_ranks(model, x, world)
    assert got.shape == whole.shape == (1, 3) + tuple(x.shape[2:])          # NCDHW in, NCDHW out
    assert rel(got, whole) < (1e-3 if tc else 5e-5), rel(got, whole)
    agree = (got.argmax(1) == whole.argmax(1)).float().mean()
    assert float(agree) >= 0.999
    # one exchange per 3x3x3 conv (26 stride-1, 3 strided, 3 transposed); P16 form: one more per decoder level, as in
    # the channels_last model (every GroupNorm output reaches its convs as a twin)
    assert stats[0]["halo_exchanges"] == (35 if tc else 32)
    # statistics / pooling sums: 2 exchanges per ResnetBlock (GN1 statistics paired with the pooling sums, GN2
    # statistics) + 1 per resampling layer in the P16 form
    if tc:
        assert stats[0]["all_reduces"] <= 13 * 2 + 6 + 2


@pytest.mark.parametrize("world,shape", [(2, (32, 16, 16)), (3, (48, 32, 16)), (4, (64, 16, 32))])
@pytest.mark.parametrize("tc", [False, True])
def test_channels_first_virtual_rank_slab_inference_equals_whole_volume(b3d, dev, world, shape, tc):
    ops = b3d.ops
    ops.USE_TC["on"] = tc
    try:
        model = _built_model(b3d, dev)
        _check_virtual_ranks(b3d, model, t32(1, 2, *shape, seed=11, dev=dev), world, tc)
    finally:
        ops.USE_TC["on"] = True


@pytest.mark.parametrize("tc", [False, True])
def test_channels_first_cli_defaults_slab_inference(b3d, dev, tc):
    """The reference CLI's model on a GPU: channels_first, base_filters=32, reduction=8."""
    ops = b3d.ops
    ops.USE_TC["on"] = tc
    try:
        model = _built_model(b3d, dev, base_filters=32, reduction=8)
        _check_virtual_ranks(b3d, model, t32(1, 2, 32, 16, 16, seed=12, dev=dev), 2, tc)
    finally:
        ops.USE_TC["on"] = True


def test_channels_first_slab_inference_matches_oracle(b3d, dev):
    """End to end against the fp64 oracle under its channels_first semantics (fp32 CUDA-core mode)."""
    crop = (32, 32, 16)
    p = R.init_params(R.param_shapes(crop=crop))
    x, _, eps, _ = R.synth_batch((1,) + crop)
    with R.channels_first_semantics():
        yr = R.model_forward(p, x, eps, inference=True)[0]
    ops = b3d.ops
    ops.USE_TC["on"] = False
    try:
        model = b3d.Model(data_format='channels_first')
        with torch.no_grad():
            model(torch.zeros((1, 2) + crop, device=dev), training=False, inference=False)
        model.load_named_weights(p)
        got, _ = b3d.slab.run_virtual_ranks(model, cf(x).float().to(dev), 2)
        assert rel(got, cf(yr)) < 2e-5, rel(got, cf(yr))
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
        x = t32(1, 2, 32, 32, 16, seed=11, dev=dev)
        with torch.no_grad():
            whole = model(x, training=False, inference=True)[0]
        res = {}
        for name, comm in (("peer", b3d.PeerComm(mailbox_bytes=1 << 20)), ("nccl", b3d.DistComm())):
            y, (d0, d1) = b3d.sharded_inference(model, x, comm, gather=False)
            res[name] = rel(y, whole[:, :, d0:d1])
            if name == "peer":
                # twice through one replayed CUDA graph; the depth of the whole volume from the NCDHW example
                gi = b3d.GraphedInference(model, x[:, :, d0:d1].contiguous(), comm)
                res["peer_graph_1"] = rel(gi(), whole[:, :, d0:d1])
                res["peer_graph_2"] = rel(gi(), whole[:, :, d0:d1])
        full = b3d.sharded_inference(model, x, b3d.DistComm())           # gathered along D of NCDHW
        res["gathered"] = rel(full, whole)
        q.put((rank, res))
    except BaseException as e:      # noqa: BLE001
        q.put((rank, repr(e)))
    dist.barrier()
    torch.cuda.synchronize()
    os._exit(0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_channels_first_peer_memory_comm_two_gpus():
    """A channels_first model through PeerComm and DistComm on two real GPUs, eagerly and through a replayed CUDA
    graph, against the un-sharded forward's slab."""
    import os
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 32500 + os.getpid() % 2000
    procs = [ctx.Process(target=_peer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for r in (0, 1):
        assert isinstance(out[r], dict), out[r]
        assert all(v < 1e-3 for v in out[r].values()), out
