"""Per-layer timing of the narrow-layer weight gradients at the model's 128^3 shapes: the fp32 entry point
b3d_conv3d_wgrad (staged stacked + plain bf16 copies, then the KS = 1 GEMM; its bias gradient from the copy or a
column-sum pass) against b3d_conv3d_wgrad_narrow (stacked operand built in shared memory from the fp32 tensor, wide
operand the bf16 P16 twin that the training step already holds).  CUDA events around each call, L2 overwritten
(256 MB write) before every timed call; median over `reps`.  Prints one line per layer and the device it ran on.

    python tools/wgrad_narrow_bench.py [reps]"""
import ctypes
import importlib
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
b3d = importlib.import_module("3d-brain-tumor-segmentation_b200")
ops, lib = b3d.ops, b3d._lib.lib

LAYERS = [
    # (name, Cin, Cout, k, pair)
    ("block1 3x3x3 2->16 + pointwise 2->16", 2, 16, 3, True),
    ("decoder out 1x1x1 16->3", 16, 3, 1, False),
    ("vae out 3x3x3 16->2", 16, 2, 3, False),
]


def timed(fn, flush, reps):
    ts = []
    for _ in range(reps):
        flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return statistics.median(ts)


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
    dev = torch.device("cuda:0")
    p = torch.cuda.get_device_properties(0)
    print(f"device: {p.name}, {p.multi_processor_count} SMs")
    flush = torch.empty(64 * 2 ** 20, device=dev)
    sp = (1, 128, 128, 128)
    g = torch.Generator().manual_seed(5)
    for name, cin, cout, k, pair in LAYERS:
        x = torch.randn(*sp, cin, generator=g).to(dev)
        dy = torch.randn(*sp, cout, generator=g).to(dev)
        dres = torch.randn(*sp, cout, generator=g).to(dev) if pair else None
        dw = torch.empty(k, k, k, cin, cout, device=dev)
        db = torch.empty(cout, device=dev)
        xc, yc = ctypes.c_longlong(), ctypes.c_longlong()
        lib.b3d_conv3d_wgrad_plan(k, 1, 0, cin, cout, ctypes.byref(xc), ctypes.byref(yc))
        xb = torch.empty(x.numel() // cin * xc.value, device=dev, dtype=torch.bfloat16)
        yb = torch.empty(dy.numel() // cout * yc.value, device=dev, dtype=torch.bfloat16)

        if pair:     # the pointwise layer on the fp32 entry point: its own staging copies and a second GEMM
            xc1, yc1 = ctypes.c_longlong(), ctypes.c_longlong()
            lib.b3d_conv3d_wgrad_plan(1, 1, 0, cin, cout, ctypes.byref(xc1), ctypes.byref(yc1))
            xb1 = torch.empty(x.numel() // cin * xc1.value, device=dev, dtype=torch.bfloat16)
            dwp_old = torch.empty(1, 1, 1, cin, cout, device=dev)

        def old():
            ops._call("b3d_conv3d_wgrad", x, dy, dw, None if cin < 8 else db, 1, 0, xb, yb, 0)
            if pair:
                ops._call("b3d_conv3d_wgrad", x, dres, dwp_old, None, 1, 0, xb1, yb, 0)

        if cin < 8:
            dy16 = ops.to_p16(dy, torch.bfloat16)
            dres16 = ops.to_p16(dres, torch.bfloat16) if pair else None
            dwp = torch.empty(1, 1, 1, cin, cout, device=dev) if pair else None
            new = lambda: ops._call("b3d_conv3d_wgrad_narrow", x, dy16, dres16, dw, dwp, None)
        else:
            x16 = ops.to_p16(x, torch.bfloat16)
            new = lambda: ops._call("b3d_conv3d_wgrad_narrow", dy, x16, None, dw, None, db)
        for _ in range(3):
            old(); new()
        torch.cuda.synchronize()
        t_old, t_new = timed(old, flush, reps), timed(new, flush, reps)
        print(f"{name:40s} fp32 entry {t_old:8.1f} us   narrow {t_new:8.1f} us   ({t_old / t_new:.2f}x)", flush=True)


if __name__ == "__main__":
    main()
