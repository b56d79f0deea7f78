"""GPU suite (needs 2 GPUs) — data-parallel training step == single-GPU step on the concatenated batch
(SURVEY section 4 item 5, VERDICT r01 "missing" 3), for both objectives of train.DataParallel:

  global_batch   the reference's `--batch_size N` objective (util.py:11,18-20: I, P, T summed over the batch axis): the
                 3C+2 loss sums are all-reduced in the forward, gradients are SUMMED  ==  one GPU fed both crops (B = 2)
  replica_mean   gradients of the per-crop losses averaged  ==  mean of two single-crop gradients

Every rank computes the single-GPU reference itself (identical weights), runs the 2-rank step eagerly and through the
CUDA graph, and compares the all-reduced flat gradient buffer and the loss.  The L2 penalties are added once (inside the
Adam kernel), never averaged."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, q):
    import importlib
    import sys
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    sys.path.insert(0, ROOT)
    b3d = importlib.import_module("3d-brain-tumor-segmentation_b200")
    import synthdata as R
    res = {}
    try:
        # depth 3 at 64^3: the bottleneck is 16^3 and the VAE normalises groups of 64 values — at the default depth a
        # 32^3 / 64^3 crop ends in GroupNorm groups of 8 values, which amplify last-bit differences (summation order of
        # B = 2 vs two B = 1 runs) to O(1) in the gradients and would make the comparison meaningless
        crop, depth = (64, 64, 64), 3
        p = R.init_params(R.param_shapes(crop=crop, depth=depth), dtype=torch.float32)
        data = [R.synth_batch((1,) + crop, seed=100 * r, latent=32, dtype=torch.float32) for r in range(world)]
        f = lambda t: t.to(dev)
        rel = lambda a, b: float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))

        def fresh():
            m = b3d.Model(depth=depth)
            with torch.no_grad():
                m(torch.zeros((1,) + crop + (2,), device=dev), training=False, inference=False)
            m.load_named_weights(p)
            o = b3d.ScheduledOptim(learning_rate=1e-4)
            o(epoch=0)
            return m, o

        def grads_of(model, x, y, eps, mask):
            with b3d.GradientTape() as tape:
                outs = model(f(x), training=True, inference=False, dropout_mask=f(mask), eps=f(eps))
                loss = b3d.DiceVAELoss()(f(x), f(y), *outs)
            tape.gradient(loss, model.trainable_variables, direct=True)
            return float(loss), model.flat.grad.clone()

        # ---- single-GPU references
        model, _ = fresh()
        cat = [torch.cat([d[i] for d in data], dim=0) for i in range(4)]
        loss_b2, g_b2 = grads_of(model, *cat)                                   # one GPU fed both crops
        per = [grads_of(model, *d) for d in data]
        loss_mean, g_mean = sum(l for l, _ in per) / world, sum(g for _, g in per) / world

        x, y, eps, mask = data[rank]
        for objective, loss_ref, g_ref in (("global_batch", loss_b2, g_b2), ("replica_mean", loss_mean, g_mean)):
            model, opt = fresh()
            loss_fn = b3d.DiceVAELoss()
            dp = b3d.DataParallel(model, opt, world, objective=objective, loss_fn=loss_fn)
            theta0 = model.flat.theta.clone()
            loss, _, _ = b3d.train_step(model, opt, loss_fn, b3d.DiceCoefficient(), f(x), f(y), dropout_mask=f(mask),
                                        eps=f(eps), dp=dp)
            torch.cuda.synchronize()
            g = model.flat.grad * opt.grad_scale                              # what Adam consumed (before the L2 term)
            l = torch.tensor([float(loss)], device=dev)
            if objective == "replica_mean":                                   # each rank reports its own crop's loss
                dist.all_reduce(l); l /= world
            reg = float(b3d.reduce_sum(model.losses))
            res[objective] = {"grad_rel": rel(g, g_ref), "loss_rel": abs(float(l) - reg - loss_ref) / abs(loss_ref),
                              "moved": float((model.flat.theta - theta0).abs().max())}
            # replicas stay identical after the step
            th = model.flat.theta.clone()
            dist.all_reduce(th, op=dist.ReduceOp.MAX)
            res[objective]["replicas_equal"] = bool(torch.equal(th, model.flat.theta))
            # the same step through a CUDA graph (NCCL all-reduces captured on the side stream)
            model2, opt2 = fresh()
            loss_fn2 = b3d.DiceVAELoss()
            dp2 = b3d.DataParallel(model2, opt2, world, objective=objective, loss_fn=loss_fn2)
            step = b3d.GraphedTrainStep(model2, opt2, loss_fn2, b3d.DiceCoefficient(), f(x), f(y), warmup=1, dp=dp2)
            res[objective]["graph_unchanged_by_warmup"] = bool(torch.equal(model2.flat.theta, theta0))
            step()
            torch.cuda.synchronize()
            res[objective]["graph_moved"] = float((model2.flat.theta - theta0).abs().max())
            del step
        q.put((rank, res))
    except BaseException as e:      # noqa: BLE001
        import traceback
        q.put((rank, repr(e) + traceback.format_exc()))
    dist.barrier()
    torch.cuda.synchronize()
    try:
        dist.destroy_process_group()
    except BaseException:           # noqa: BLE001
        pass
    os._exit(0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_dp_step_equals_single_gpu_step():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    print(out)
    for r in (0, 1):
        assert isinstance(out[r], dict), out[r]
        for objective, v in out[r].items():
            # same kernels, same rounding points; the difference is the summation order of the all-reduce and of the
            # per-sample partial sums (fp32), amplified by the network's conditioning at 32^3
            assert v["loss_rel"] < 5e-5, (objective, v)
            # two runs of the SAME single-GPU step differ by 4-6e-3 here (tools/dp_debug2.py: atomics order decides
            # 16-bit rounding ties); a missed or doubled bucket all-reduce shows as 0.5-1.0
            assert v["grad_rel"] < 2e-2, (objective, v)
            assert v["replicas_equal"] and v["graph_unchanged_by_warmup"], (objective, v)
            assert 0.0 < v["moved"] < 1e-3 and 0.0 < v["graph_moved"] < 1e-3, (objective, v)
