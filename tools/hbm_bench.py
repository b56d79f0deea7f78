"""Achieved HBM bandwidth of the bandwidth-bound kernels on the path (GroupNorm, ResnetBlock epilogue / scSE, loss,
Dice, Adam, bf16 casts) at the shapes of the default model's 128^3 level: algorithmic bytes (DESIGN.md §4) /
CUDA-event time, L2 flushed between launches.  Usage: python tools/hbm_bench.py [reps] [json-out]"""
import importlib
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
b3d = importlib.import_module("3d-brain-tumor-segmentation_b200")
ops = b3d.ops
dev = torch.device("cuda:0")
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
try:
    PEAK = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
except Exception:
    PEAK = 6650.0
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timeit(fn):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


rows = []


def report(name, bytes_, fn):
    ms = timeit(fn)
    gbs = bytes_ / ms / 1e6
    rows.append({"kernel": name, "us": ms * 1e3, "alg_MB": bytes_ / 1e6, "GBps": gbs, "frac_of_measured_peak": gbs / PEAK})
    print(f"{name:44s} {ms * 1e3:9.1f} us  {bytes_ / 1e6:8.1f} MB  {gbs:7.0f} GB/s  {100 * gbs / PEAK:5.1f} % of {PEAK:.0f}",
          flush=True)


for n, C in ((128, 16), (64, 32), (32, 64)):
    shp = (1, n, n, n, C)
    E = n ** 3 * C
    x, dy = torch.randn(shp, device=dev), torch.randn(shp, device=dev)
    y, dx = torch.empty_like(x), torch.empty_like(x)
    ga, be = torch.rand(C, device=dev) + 0.5, torch.randn(C, device=dev) * 0.1
    dga, dbe = torch.empty_like(ga), torch.empty_like(be)
    st = torch.empty(1, 8, 2, dtype=torch.float64, device=dev)
    cs = torch.empty_like(st)
    tag = f"{n}^3x{C}"
    report(f"gn_stats {tag}", 4 * E, lambda: ops._call("b3d_gn_stats", x, st, 8, 0, 0))
    report(f"gn_apply+relu {tag}", 8 * E, lambda: ops._call("b3d_gn_apply", x, st, ga, be, y, None, None, 8, 1e-5, 1, 0, 0))
    report(f"gn_bwd_reduce {tag}", 8 * E,
           lambda: ops._call("b3d_gn_bwd_reduce", dy, x, st, ga, be, dga, dbe, cs, 8, 1e-5, 1))
    report(f"gn_bwd_apply {tag}", 12 * E,
           lambda: ops._call("b3d_gn_bwd_apply", dy, x, st, ga, be, cs, dx, None, None, 8, 1e-5, 1))
    # ResnetBlock epilogue (GN2 + ReLU + scSE + add)
    F, R = C, C // 2
    res, h2, out = torch.randn(shp, device=dev), torch.randn(shp, device=dev), torch.empty(shp, device=dev)
    wsp = torch.randn(F, device=dev) * 0.1
    chse = torch.rand(1, F, device=dev)
    ops._call("b3d_gn_stats", h2, st, 8, 0, 0)
    report(f"block_epilogue_fwd {tag}", 12 * E,
           lambda: ops._call("b3d_block_epilogue_fwd", res, h2, st, ga, be, wsp, chse, out, None, None, 8, 1e-5, 1,
                             0, 0))
    dchse, dwsp, dgap = torch.empty(1, F, device=dev), torch.empty(F, device=dev), torch.randn(1, F, device=dev) * 1e-3
    dres, dh2 = torch.empty(shp, device=dev), torch.empty(shp, device=dev)
    report(f"block_epilogue_bwd_reduce {tag}", 12 * E,
           lambda: ops._call("b3d_block_epilogue_bwd_reduce", dy, res, h2, st, ga, be, wsp, dchse, dwsp, dga, dbe, cs,
                             8, 1e-5, 1))
    report(f"block_epilogue_bwd_apply {tag}", 20 * E,
           lambda: ops._call("b3d_block_epilogue_bwd_apply", dy, res, h2, st, ga, be, wsp, chse, dgap, cs, dres, dh2,
                             None, None, None, None, 8, 1e-5, 1))
    # ---- the P16 twin forms the training step actually runs (fp32 outputs not materialised)
    t16, t16b = ops.p16_empty(shp, x, torch.float16), ops.p16_empty(shp, x, torch.bfloat16)
    u16b = ops.p16_empty(shp, x, torch.bfloat16)
    dbias, dbias2 = torch.empty(C, device=dev), torch.empty(C, device=dev)
    report(f"gn_apply fp16 twin only (inference) {tag}", 6 * E,
           lambda: ops._call("b3d_gn_apply", x, st, ga, be, None, t16, None, 8, 1e-5, 1, 0, 0))
    report(f"gn_apply fp16+bf16 twins (training) {tag}", 8 * E,
           lambda: ops._call("b3d_gn_apply", x, st, ga, be, None, t16, t16b, 8, 1e-5, 1, 0, 0))
    report(f"gn_apply fp32 + both twins {tag}", 12 * E,
           lambda: ops._call("b3d_gn_apply", x, st, ga, be, y, t16, t16b, 8, 1e-5, 1, 0, 0))
    report(f"gn_bwd_apply bf16 twin + dbias {tag}", 10 * E,
           lambda: ops._call("b3d_gn_bwd_apply", dy, x, st, ga, be, cs, None, t16b, dbias, 8, 1e-5, 1))
    report(f"gn_bwd_apply bf16 twin, no dbias {tag}", 10 * E,
           lambda: ops._call("b3d_gn_bwd_apply", dy, x, st, ga, be, cs, None, t16b, None, 8, 1e-5, 1))
    report(f"block_epilogue_fwd twins only {tag}", 12 * E,
           lambda: ops._call("b3d_block_epilogue_fwd", res, h2, st, ga, be, wsp, chse, None, t16, t16b, 8, 1e-5, 1,
                             0, 0))
    report(f"block_epilogue_bwd_apply twins + dbias {tag}", 16 * E,
           lambda: ops._call("b3d_block_epilogue_bwd_apply", dy, res, h2, st, ga, be, wsp, chse, dgap, cs, None, None,
                             t16b, u16b, dbias, dbias2, 8, 1e-5, 1))
    report(f"block_epilogue_bwd_apply twins, no dbias {tag}", 16 * E,
           lambda: ops._call("b3d_block_epilogue_bwd_apply", dy, res, h2, st, ga, be, wsp, chse, dgap, cs, None, None,
                             t16b, u16b, None, None, 8, 1e-5, 1))
    del res, h2, out, dres, dh2, t16, t16b, u16b

# loss / dice at 128^3 (out_ch 3, in_ch 2)
n = 128
yp, yt = torch.rand(1, n, n, n, 3, device=dev), (torch.rand(1, n, n, n, 3, device=dev) > 0.9).float()
xin, yv = torch.randn(1, n, n, n, 2, device=dev), torch.randn(1, n, n, n, 2, device=dev)
mu, lv = torch.randn(1, 64, device=dev), torch.randn(1, 64, device=dev) * 0.1
sums, out4 = torch.empty(11, dtype=torch.float64, device=dev), torch.empty(4, device=dev)
S = n ** 3
report("loss_fwd (dice+l2+kl) 128^3", 4 * (2 * S * 3 + 2 * S * 2),
       lambda: ops._call("b3d_loss_fwd", xin, yt, yp, yv, mu, lv, sums, out4))
g1 = torch.ones(1, device=dev)
dyp, dyv, dmu, dlv = torch.empty_like(yp), torch.empty_like(yv), torch.empty_like(mu), torch.empty_like(lv)
report("loss_bwd 128^3", 4 * (3 * S * 3 + 3 * S * 2),
       lambda: ops._call("b3d_loss_bwd", xin, yt, yp, yv, mu, lv, sums, g1, dyp, dyv, dmu, dlv))
acc, out2 = torch.empty(n * 3 * 3, device=dev), torch.empty(2, device=dev)
report("dice_coeff 128^3", 4 * (2 * S * 3), lambda: ops._call("b3d_dice_coeff", yt, yp, acc, out2, 0))
report("loss_fwd + dice_coeff in one pass 128^3", 4 * (2 * S * 3 + 2 * S * 2),
       lambda: ops._call("b3d_loss_dice_fwd", xin, yt, yp, yv, mu, lv, sums, out4, acc, out2, 0))
# Adam over the flat parameter buffer (10.6 M params; 28 B/param)
P = 10_636_064
th, m, v, g = (torch.randn(P, device=dev) * 0.01 for _ in range(4))
v.abs_()
state = torch.tensor([0.0, 1e-4], dtype=torch.float64, device=dev)
report("adam 10.6M params", 28 * P,
       lambda: ops._call("b3d_adam_step", th, m, v, g, state, 0.9, 0.999, 1e-7, 1.0, 2e-5, P // 2, 1))
if len(sys.argv) > 2:
    json.dump({"peak_gbs": PEAK, "rows": rows}, open(sys.argv[2], "w"), indent=1)
