#!/usr/bin/env python
"""bench.py — headline metric of BASELINE.json: 128^3 train crops/sec (fwd + loss + bwd + Adam).

    python bench.py --gpus N --steps K --warmup W                 (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K --warmup W  (reference math on the host cores)
    python bench.py ... --dump-outputs DIR                          (also save what the last timed step computed)

One "step" = one pass of the hot path (reference train.py:140-152) over one synthetic 128^3 crop per GPU
with the default Model() (in 2, out 3, base_filters 16).  Prints ONE JSON line (rank 0).  See DESIGN.md §4.

The benchmark writes nothing into the source tree (no bytecode caches either): the tree may be read-only.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "3d-brain-tumor-segmentation_b200"
CROP = (128, 128, 128)
FWD_GFLOP = 550.7            # SURVEY App. A (default model, 128^3, VAE on); train step ~ 3x
METRIC = "128^3 train crops/sec (fwd+bwd+Adam)"


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v == "Active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
def cpu_reference_step_fn(crop, threads=None):
    """The reference's math (oracle restatement, fp32, oneDNN convs via torch-CPU) as one training step:
    fwd + DiceVAELoss + L2 + backward + TF-form Adam.  The real TF-2.0-alpha path is not installable."""
    import torch
    from oracle import ref_model as R
    if threads:
        torch.set_num_threads(threads)
    dt = torch.float32
    p = R.init_params(R.param_shapes(crop=crop), dtype=dt)
    x, y, eps, mask = R.synth_batch((1,) + crop, dtype=dt)
    m = {k: torch.zeros_like(v) for k, v in p.items()}
    v = {k: torch.zeros_like(v) for k, v in p.items()}
    state = {"t": 0}

    def step():
        pg = {k: t.requires_grad_(True) for k, t in p.items()}
        outs = R.model_forward(pg, x, eps, dropout_mask=mask)
        loss = R.dice_vae_loss(x, y, *outs) + R.l2_reg(pg)
        grads = torch.autograd.grad(loss, list(pg.values()))
        state["t"] += 1
        with torch.no_grad():
            for (k, t), g in zip(p.items(), grads):
                t.requires_grad_(False)
                R.adam_step_tf(t, m[k], v[k], g, state["t"], 1e-4)
        return float(loss)

    return step, torch.get_num_threads()


def run_reference(args):
    """--impl reference: the reference's own CPU math for the path on this box's host cores, ALWAYS on the stated
    configuration (full 128^3 crop).  When the host is too slow for `--steps K --warmup W` full crops within the time
    budget, fewer steps are timed (never a smaller crop): `steps` in the line is what was actually timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, threads = cpu_reference_step_fn(CROP)
    t0 = time.time(); step(); t1 = time.time() - t0          # first step: also the probe (untimed warm-up)
    budget = float(os.environ.get("B3D_REF_BUDGET_S", "200"))
    warm = max(0, min(args.warmup - 1, int(0.2 * budget / t1)))
    steps = max(1, min(args.steps, int((budget - (1 + warm) * t1) / t1)))
    for _ in range(warm):
        step()
    t0 = time.time()
    for _ in range(steps):
        step()
    dt = time.time() - t0
    val = steps / dt
    sample = (f"{steps} full 128^3 crops (fwd+loss+bwd+Adam), fp32 torch-CPU oracle"
              + ("" if steps == args.steps else f"; {args.steps} requested, bounded by a {budget:.0f} s budget"))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "crops/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1 + warm, "ms_per_step": 1e3 * dt / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "train_128cube_b1_default_model", "crop": list(CROP), "in_ch": 2, "out_ch": 3,
                       "base_filters": 16, "note": "reference math on host cores; TF 2.0-alpha itself is not "
                                                   "installable (SURVEY §8c)"},
            "cpu_baseline": {"value": val, "unit": "crops/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "crops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
def measure_conv_roofline(b3d, torch, dev, steps=20):
    """Dominant kernel: the tcgen05 3x3x3 conv.  Timed in isolation on the largest layer of the default
    model (dec L0 conv1: 128^3, Cin 32 -> Cout 16, 58.0 GFLOP) with CUDA events on the launching stream, fed the way
    the training step feeds it: the input as two 16-channel fp16 P16 twins (decoder.py:75 concat as a source list)."""
    ops = b3d.ops
    cin, cout = 32, 16
    x = torch.randn((1,) + CROP + (cin,), device=dev)
    w = torch.randn(3, 3, 3, cin, cout, device=dev) * 0.05
    bias = torch.zeros(cout, device=dev)
    y = torch.empty((1,) + CROP + (cout,), device=dev)
    stats = torch.empty(1, 8, 2, dtype=torch.float64, device=dev)
    wp = ops.pack_weights(w, False)
    tw = [ops.to_p16(x[..., :16].contiguous(), torch.float16), ops.to_p16(x[..., 16:].contiguous(), torch.float16)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    call = lambda: ops._call("b3d_conv3d_fwd_p16", tw[0], tw[1], None, None, w, bias, y, 1, 0, 0, stats, 8, None, 0, wp)
    for _ in range(3):
        call()
    times = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); call(); e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = statistics.median(times)
    vox = CROP[0] * CROP[1] * CROP[2]
    flops = 2.0 * vox * 27 * cin * cout
    alg_bytes = vox * (2.0 * cin + 4.0 * cout)          # fp16 operand read once + fp32 result written once
    return ms, flops, alg_bytes


def roofline_capture():
    """ncu evidence of the kernel `roofline` reports (committed under profiles/, produced by tools/ncu_summary.py from
    the `ncu --set full` capture of the SAME kernel variant on the same layer): dram traffic and both tensor-pipe
    readings.  None when the file is missing."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "roofline_kernel.json")))
    except Exception:
        return None


def measure_step_classes(b3d, torch, model, opt, xd, yd, pk):
    """In-step aggregates (VERDICT r01 item 2): one EAGER training step with CUDA events around every C-ABI call
    (ops.profile_calls), summed per kernel class.  Conv classes carry their algorithmic FLOPs -> achieved TF/s inside
    the step, next to the tensor peak measured for a kernel inside a long step (bf16_tflops_sustained)."""
    ops = b3d.ops
    args = (model, opt, b3d.DiceVAELoss(), b3d.DiceCoefficient())
    b3d.train_step(*args, xd, yd)
    torch.cuda.synchronize()
    with ops.profile_calls() as rows:
        # the host needs ~30 ms to issue the ~400 calls of an eager step, the GPU ~15 ms to run them: without a head
        # start the GPU idles between calls and every event pair also measures launch latency (round-2 numbers were
        # 1.7x the ncu durations).  A spin kernel of ~80 ms lets the host run ahead, so the calls execute back to back.
        torch.cuda._sleep(int(1.6e8))
        b3d.train_step(*args, xd, yd)
        torch.cuda.synchronize()
    agg = {}
    for name, tag, e0, e1 in rows:
        ms = e0.elapsed_time(e1)
        key = name.replace("b3d_", "")
        if tag is not None:
            pas = "wgrad" if "wgrad" in name else ("dgrad" if "dgrad" in name else "fwd")
            key = f"conv_{tag[0]}_{pas}"
        a = agg.setdefault(key, [0, 0.0, 0.0])
        a[0] += 1; a[1] += ms; a[2] += tag[1] if tag is not None else 0.0
    tot = sum(v[1] for v in agg.values())
    conv = {k: v for k, v in agg.items() if k.startswith("conv_")}
    cls = lambda pre: [v for k, v in conv.items() if k.startswith(pre)]
    tf = lambda vs: (sum(v[2] for v in vs) / 1e12) / (sum(v[1] for v in vs) / 1e3) if vs and sum(v[1] for v in vs) > 0 else None
    k3 = [v for k, v in conv.items() if k.startswith("conv_k3_") and not k.endswith("wgrad")]
    out = {"how": "one eager step queued behind an 80 ms spin kernel (the host runs ahead, calls execute back to back), "
                  "CUDA events around every C-ABI call (includes the call's memsets / helper kernels)",
           "abi_calls": len(rows), "sum_ms": tot,
           "k3_fwd_dgrad_tflops": tf(k3), "k3_wgrad_tflops": tf(cls("conv_k3_wgrad")),
           "all_conv_tflops": tf(list(conv.values())),
           "conv_ms": sum(v[1] for v in conv.values()), "conv_gflop": sum(v[2] for v in conv.values()) / 1e9,
           "peak_tflops_sustained": pk.get("bf16_tflops_sustained"),
           "top": [{"call": k, "n": v[0], "ms": round(v[1], 3)} for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])[:14]]}
    if out["all_conv_tflops"] and pk.get("bf16_tflops_sustained"):
        out["all_conv_frac_of_sustained"] = out["all_conv_tflops"] / pk["bf16_tflops_sustained"]
    return out


def measure_config(b3d, torch, dev, name, crop, steps=5, **kw):
    """A further BASELINE configuration as an extra entry: graphed training step (+ inference forward) of a model built
    with **kw at `crop` (cfg 5: skull-strip 256x256x192; the CLI-default bf=32 / r=8 model of the README's V100 run)."""
    import synthdata as R
    in_ch, out_ch = kw.get("in_ch", 2), kw.get("out_ch", 3)
    bf, red = kw.get("base_filters", 16), kw.get("reduction", 2)
    p = R.init_params(R.param_shapes(in_ch=in_ch, out_ch=out_ch, base_filters=bf, reduction=red, crop=crop),
                      dtype=torch.float32)
    x, y, _, _ = R.synth_batch((1,) + crop, in_ch=in_ch, out_ch=out_ch, latent=bf * 4, dtype=torch.float32)
    xd, yd = x.to(dev), y.to(dev)
    torch.cuda.reset_peak_memory_stats()
    model = b3d.Model(**kw)
    with torch.no_grad():
        model(xd, training=False, inference=False)
    model.load_named_weights(p)
    opt = b3d.ScheduledOptim(learning_rate=1e-4)
    opt(epoch=0)
    step = b3d.GraphedTrainStep(model, opt, b3d.DiceVAELoss(), b3d.DiceCoefficient(), xd, yd, warmup=2)
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = step()
    e1.record(); e1.synchronize()
    ms = e0.elapsed_time(e1) / steps
    gi = b3d.GraphedInference(model, xd)
    gi()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(3):
        gi()
    f1.record(); f1.synchronize()
    msi = f0.elapsed_time(f1) / 3
    vox = crop[0] * crop[1] * crop[2]
    res = {"config": name, "crop": list(crop), "model": kw, "params": int(model.flat.total),
           "train_ms_per_step": ms, "train_crops_per_s": 1e3 / ms, "loss": float(out[0]),
           "inference_ms_per_forward": msi, "inference_mvoxel_per_s": vox / msi / 1e3,
           "peak_gpu_mem_gib": torch.cuda.max_memory_allocated() / 2 ** 30}
    del step, gi, model
    torch.cuda.empty_cache()
    return res


def measure_inference(b3d, torch, dev, model, reps=3):
    """BASELINE config 4 (single GPU): one `inference=True` forward (reference test.py:133) of a 155x190x147
    volume padded to 160x192x160; Mvoxel/s counts ORIGINAL voxels (SURVEY §8d).  VAE branch skipped."""
    shape = (160, 192, 160)
    x = torch.randn((1,) + shape + (2,), device=dev)
    x[:, 155:], x[:, :, 190:], x[:, :, :, 147:] = 0, 0, 0
    times = []
    with torch.no_grad():
        for i in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            y = model(x, training=False, inference=True)[0]
            e1.record(); e1.synchronize()
            if i:
                times.append(e0.elapsed_time(e1))
    ms_eager = statistics.median(times)
    gi = b3d.GraphedInference(model, x)
    times = []
    for i in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); gi(); e1.record(); e1.synchronize()
        if i:
            times.append(e0.elapsed_time(e1))
    ms = statistics.median(times)
    return {"shape_padded": list(shape), "ms_per_forward": ms, "mvoxel_per_s": 155 * 190 * 147 / ms / 1e3,
            "ms_per_forward_eager": ms_eager, "gflop_per_forward": 1006.8,
            "note": "CUDA-graph replay of model(x, inference=True), 1 GPU; 8-flip TTA = 8 such forwards"}


def measure_inference_sharded(b3d, torch, dist, dev, model, world, reps=3):
    """BASELINE config 4 at N GPUs: the padded 160x192x160 volume cut into depth slabs, one per GPU, halo
    exchange (NCCL P2P over NVLink) before every 3x3x3 conv, all-reduced GroupNorm chunk statistics and SE
    pooling sums (3d-brain-tumor-segmentation_b200/slab.py).  Time = max over ranks of the slab forward."""
    shape = (160, 192, 160)
    g = torch.Generator().manual_seed(123)
    x = torch.randn((1,) + shape + (2,), generator=g)
    x[:, 155:], x[:, :, 190:], x[:, :, :, 147:] = 0, 0, 0
    x = x.to(dev)
    try:
        comm, backend = b3d.PeerComm(), "NVLink peer-memory kernels (csrc/slab_comm.cu)"
    except Exception as e:                      # noqa: BLE001 — symmetric memory unavailable: NCCL P2P / all-reduce
        comm, backend = b3d.DistComm(), f"NCCL (peer memory unavailable: {type(e).__name__})"
    d0, d1 = b3d.slab_bounds(shape[0], world)[comm.rank]
    gi = b3d.GraphedInference(model, x[:, d0:d1].contiguous(), comm, depth=shape[0])   # halo exchanges captured too
    times, err = [], None
    for i in range(reps + 1):
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        y = gi()
        e1.record(); e1.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if i:
            times.append(float(ms))
    with torch.no_grad():
        whole = model(x, training=False, inference=True)[0][:, d0:d1]
    e = ((y - whole).double().norm() / whole.double().norm()).reshape(1).float()
    dist.all_reduce(e, op=dist.ReduceOp.MAX)
    ms = statistics.median(times)
    return {"shape_padded": list(shape), "n_gpus": world, "ms_per_forward": ms,
            "mvoxel_per_s": 155 * 190 * 147 / ms / 1e3, "max_rel_l2_vs_unsharded": float(e),
            "slabs": [b - a for a, b in b3d.slab_bounds(shape[0], world)],
            "comm": backend,
            "note": "depth-slab sharded, one CUDA graph per rank incl. the halo exchanges and GN/SE all-reduces"}


def measure_tta(b3d, torch, dist, dev, model, world, reps=2):
    """8-flip test-time augmentation of one padded volume (reference test.py:105-161).  N GPUs: replica mode — the
    flips are dealt to the ranks (whole-volume forwards, no halo exchange), one all-reduce of the class maps."""
    shape = (160, 192, 160)
    g = torch.Generator().manual_seed(321)
    x = torch.randn(shape + (2,), generator=g).to(dev)
    mask = torch.ones(shape + (1,), device=dev)
    tta = b3d.TestTimeAugmentor(0.0, 1.0, model, "channels_last", group=dist.group.WORLD if world > 1 else None)
    times = []
    for i in range(reps + 1):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); tta(x, mask); e1.record(); e1.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if i:
            times.append(float(ms))
    ms = statistics.median(times)
    return {"ms_per_volume": ms, "mvoxel_per_s": 155 * 190 * 147 / ms / 1e3, "flips": 8,
            "mode": "replicas: flips dealt to ranks + 1 all-reduce" if world > 1 else "8 sequential forwards"}


def dump_step_outputs(out_dir, out):
    """What a caller of the timed training step receives from its last step, as DIR/<name>.npy: the loss, macro Dice
    and micro Dice that train_step returns.  Weights and crops are seeded (synthdata), dropout hashes a fixed seed
    with a step counter and run_b3d seeds the generator the VAE draws eps from: runs with the same arguments see the
    same inputs, so two builds can be compared array by array.
    The weights the step updates are not saved: the step is not bit-reproducible (float atomics in the pooling and
    parameter-gradient reductions change 16-bit roundings), and Adam turns the resulting noise in near-zero gradients
    into learning-rate-sized weight differences between runs of one build.  The returned values stay close: three
    runs of one build with --steps 20 --warmup 5 on a B200 (1000 W limit) spread by 5e-5 relative in the loss and
    2e-3 relative in both Dice scores."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in zip(("loss", "macro_dice", "micro_dice"), out):
        t = t.detach().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (t.double() if t.dtype == torch.float64 else t.float()).numpy())


def run_b3d(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    b3d = importlib.import_module(PKG)
    import synthdata as R               # seeded synthetic weights / inputs (neutral module: nothing under oracle/)

    # ---- model, synthetic data (rank r uses seed + 100 r), optimizer.  The VAE draws eps from torch's default
    # generators inside the step, and torch seeds those at random in every process: seed them like the crops.
    torch.manual_seed(100 * rank)
    p = R.init_params(R.param_shapes(crop=CROP), dtype=torch.float32)
    x, y, _, _ = R.synth_batch((1,) + CROP, seed=100 * rank, dtype=torch.float32)
    xh, yh = x.pin_memory(), y.pin_memory()
    xd, yd = xh.to(dev), yh.to(dev)
    model = b3d.Model()
    model(xd, training=False, inference=False)
    model.load_named_weights(p)
    opt = b3d.ScheduledOptim(learning_rate=1e-4)
    opt(epoch=0)
    # data parallel: the reference's `--batch_size N` objective (Dice sums over the batch axis, util.py:11,18-20): the
    # 3C+2 loss sums are all-reduced in the forward, parameter gradients are summed (train.DataParallel docstring)
    loss_fn = b3d.DiceVAELoss()
    dp = b3d.DataParallel(model, opt, world, objective="global_batch", loss_fn=loss_fn) if world > 1 else None
    step = b3d.GraphedTrainStep(model, opt, loss_fn, b3d.DiceCoefficient(), xd, yd, warmup=2, dp=dp)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    # ---- device-resident throughput
    for _ in range(max(args.warmup, 3)):
        step()
    with ClockSampler(local) as cs:
        ms = timed(lambda: step(), args.steps)
    clocks = cs.summary()
    value = world * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:        # before the end-to-end pass below trains the model further
        dump_step_outputs(args.dump_outputs, step.out)

    # ---- end to end through the public API: pinned host inputs -> H2D -> step -> D2H of the loss
    loss_host = torch.empty(1).pin_memory()

    # every step: H2D of that step's inputs from pinned host memory (issued one step ahead on a copy stream, as a
    # data loader would, so it overlaps the previous step's compute), the step, D2H of the loss, host sync
    def e2e_step():
        out = step.step_prefetched()             # consumes the batch whose H2D copy was started a step earlier
        step.prefetch(xh, yh)                    # next step's inputs: pinned host -> device staging
        loss_host.copy_(out[0].reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    step.prefetch(xh, yh)
    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    e2e_val = world * args.steps / (ms_e2e / 1e3)

    inf_sharded = measure_inference_sharded(b3d, torch, dist, dev, model, world) if world > 1 else None
    tta = measure_tta(b3d, torch, dist, dev, model, world)

    def finish():
        # Orderly teardown: the CUDA graphs that captured NCCL collectives are destroyed BEFORE the process group (the
        # other order deadlocks inside ncclCommDestroy), then the group.  A watchdog ends the process should a
        # communicator still refuse to go down, so that a finished measurement is never turned into a hung job.
        if world > 1:
            import gc
            nonlocal step, dp
            sys.stdout.flush()
            dist.barrier()
            torch.cuda.synchronize()
            step = dp = None
            gc.collect()
            torch.cuda.synchronize()
            guard = threading.Timer(30.0, lambda: os._exit(0))
            guard.daemon = True
            guard.start()
            dist.destroy_process_group()
            guard.cancel()

    if rank != 0:
        finish()
        return
    pk, pk_src = peaks()
    conv_ms, conv_flops, conv_alg_bytes = measure_conv_roofline(b3d, torch, dev)
    ach = conv_flops / (conv_ms * 1e-3) / 1e12
    cap = roofline_capture()
    roof = {"bound": "tensor",
            "kernel": "conv_tc_kernel<TcCfg<16,8,1,3,1,OP_F16,FOLD>> (tcgen05 kind::f16, kd-folded, fp16 P16 operand fetched "
                      "by TMA, fp32 accumulate in TMEM, fused bias + GroupNorm statistics) on dec.L0 conv1 128^3 32->16",
            "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"],
            "peak_source": f"{pk_src} dense bf16 burst (cuBLAS 8192^3); 16-bit operands, same tensor-pipe rate",
            "ms_per_launch": conv_ms, "algorithmic_flops": conv_flops, "algorithmic_bytes": conv_alg_bytes,
            "traffic": (cap or {}).get("dram_bytes"),
            "traffic_source": (cap or {}).get("source", "no ncu capture committed for this build"),
            "tensor_pipe": {k: (cap or {}).get(k) for k in ("pipe_tensor_cycles_active_pct_of_peak_sustained_elapsed",
                                                             "hmma_cycles_active_realtime_sum_over_subpipes",
                                                             "sm_cycles_elapsed", "duration_us_under_ncu")}}
    classes = measure_step_classes(b3d, torch, model, opt, xd, yd, pk)
    step_tflop = 3 * FWD_GFLOP / 1e3
    mfu = {"step_tflop": step_tflop, "achieved_tflops": step_tflop / (ms / args.steps / 1e3),
           "peak_tflops_sustained": pk.get("bf16_tflops_sustained"),
           "frac_of_sustained": step_tflop / (ms / args.steps / 1e3) / pk["bf16_tflops_sustained"]
           if pk.get("bf16_tflops_sustained") else None}
    # CPU baseline on a bounded sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        stepc, threads = cpu_reference_step_fn(CROP, os.cpu_count())
        t0 = time.time(); stepc(); t1 = time.time() - t0
        cpu = {"value": 1.0 / t1, "unit": "crops/s", "cores": threads, "kind": "port",
               "sample": "1 full 128^3 crop (fwd+loss+bwd+Adam), fp32 torch-CPU restatement of the reference "
                         "(oracle/ref_model.py); TF 2.0-alpha not installable"}
    line = {"metric": METRIC, "value": value, "unit": "crops/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp16 forward / bf16 backward operands, fp32 accumulate and storage", "data": "synthetic",
            "config": {"workload": "train_128cube_b1_default_model", "crop": list(CROP), "per_gpu_batch": 1,
                       "global_batch": world, "in_ch": 2, "out_ch": 3, "base_filters": 16,
                       "parallelism": f"dp{world}",
                       "dp_objective": "global_batch: batch-global Dice as in the reference's --batch_size N (3C+2 loss "
                                       "sums all-reduced in the forward, gradients summed)" if world > 1 else None,
                       "l2_flush": "working set (4.6 GiB of activations per step) "
                                                              "exceeds the 126 MB L2",
                       "train_tflop_per_step": 3 * FWD_GFLOP / 1e3, "cuda_graph": True},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "crops/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int(xh.numel() * 4 + yh.numel() * 4), "d2h_bytes_per_step": 4},
            "gpu_launches": int(step.launches_per_step * args.steps),
            "roofline": roof, "step_mfu": mfu, "step_classes": classes, "cpu_baseline": cpu,
            "inference": measure_inference(b3d, torch, dev, model) if world == 1 else inf_sharded,
            "inference_tta": tta}
    if world == 1 and not args.no_extra_configs:
        del step
        torch.cuda.empty_cache()
        line["extra_configs"] = [
            measure_config(b3d, torch, dev, "cfg5 skull-strip (in 1 / out 1) 256x256x192", (256, 256, 192), steps=3,
                           in_ch=1, out_ch=1),
            measure_config(b3d, torch, dev, "CLI defaults base_filters=32 reduction=8 (README V100 configuration), 128^3",
                           CROP, steps=5, base_filters=32, reduction=8)]
    print(json.dumps(line), flush=True)
    finish()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps; --impl reference times fewer when its B3D_REF_BUDGET_S budget (200 s) runs out, "
                         "and its JSON line reports the number it timed")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b3d", choices=["b3d", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, save the loss and Dice scores the last step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b3d":
        ap.error("--dump-outputs saves the CUDA path's step (--impl b3d)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b3d(args)


if __name__ == "__main__":
    main()
