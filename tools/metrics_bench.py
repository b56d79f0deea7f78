"""Time the device evaluation of one BraTS-sized case (155x240x240, three regions WT/TC/ET): predict_labels +
segmentation_metrics with CUDA events (warm-up, then the median of --reps runs), and the fp64 scipy oracle
(oracle/metrics_ref.py) on the host for the same case.  Reports achieved bytes/s against the algorithmic bytes
computed from the shapes, the card and its power limit, and the largest difference from the oracle.
Usage: tools/metrics_bench.py [--reps N] [--out FILE.json]"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
b3d = importlib.import_module("3d-brain-tumor-segmentation_b200")
from oracle import metrics_ref as M  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=30)
ap.add_argument("--out", default=None)
args = ap.parse_args()
assert torch.cuda.is_available(), "metrics_bench.py measures the GPU path and needs a CUDA device"
dev = torch.device("cuda:0")

SHAPE, C, SPACING = (155, 240, 240), 3, (1.0, 1.0, 1.0)
R = len(M.BRATS_REGIONS)
N = SHAPE[0] * SHAPE[1] * SHAPE[2]


def phantom(seed, perturb):
    """Nested ellipsoids (2 = ED shell, 1 = NCR/NET shell, 3 = ET core) of a tumour-sized lesion."""
    rng = np.random.default_rng(seed)
    z, y, x = np.meshgrid(*[np.arange(n, dtype=np.float32) for n in SHAPE], indexing="ij")
    c = np.array([80.0, 120.0, 110.0]) + (rng.normal(0, 2.0, 3) if perturb else 0)
    rad = np.array([30.0, 40.0, 36.0]) * (rng.uniform(0.9, 1.1, 3) if perturb else 1)
    r2 = ((z - c[0]) / rad[0]) ** 2 + ((y - c[1]) / rad[1]) ** 2 + ((x - c[2]) / rad[2]) ** 2
    lab = np.zeros(SHAPE, np.uint8)
    lab[r2 < 1.0], lab[r2 < 0.45], lab[r2 < 0.15] = 2, 1, 3
    return lab


true = phantom(0, False)
# class probabilities whose hard decision is a perturbed phantom: one-hot of it, blurred by noise
rng = np.random.default_rng(1)
onehot = np.eye(4, dtype=np.float32)[phantom(2, True)][..., 1:]
probs_h = np.clip(onehot * 0.8 + rng.random(SHAPE + (C,), dtype=np.float32) * 0.35, 0, 1).astype(np.float32)
probs = torch.from_numpy(probs_h).to(dev)
true_d = torch.from_numpy(true).to(dev)


def run():
    pred = b3d.predict_labels(probs)
    return b3d.segmentation_metrics(pred, true_d, spacing=SPACING)


for _ in range(3):
    got = run()
torch.cuda.synchronize()
times = []
for _ in range(args.reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    got = run()                       # ends in the device-to-host copy of the scores
    e1.record()
    e1.synchronize()
    times.append(e0.elapsed_time(e1))
gpu_ms = statistics.median(times)

t0 = time.perf_counter()
pred_h = M.label_map(probs_h)
ref = M.segmentation_metrics(pred_h, true, SPACING)
host_s = time.perf_counter() - t0

# algorithmic bytes: every tensor read and written once per pass
surf_entries = sum(int(M.surface(M.region_mask(a, reg)).sum()) for reg in M.BRATS_REGIONS.values()
                   for a in (pred_h, true))
bytes_ = {
    "label_map": N * C * 4 + N,
    "region_surface": 2 * N + 2 * N,
    "surface_edt": 2 * R * (N + 4 * N + 4 * 4 * N),     # pass 1: bits in, fp32 out; passes 2, 3: fp32 in and out
    "hd95": 2 * N + 4 * surf_entries * (2 + 4 + 1),     # gather, four radix histogram passes, one min pass
}
total = sum(bytes_.values())
err = max(abs(got[k][m] - ref[k][m]) / max(abs(ref[k][m]), 1e-300) for k in ref for m in ref[k])
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
res = {
    "case": "155x240x240, C=3, regions WT/TC/ET, spacing 1 mm",
    "device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi,
    "gpu_ms_per_case_median": round(gpu_ms, 4), "gpu_ms_min": round(min(times), 4),
    "gpu_ms_max": round(max(times), 4), "reps": args.reps,
    "host_oracle_s_per_case": round(host_s, 3), "speedup": round(host_s * 1e3 / gpu_ms, 1),
    "algorithmic_bytes": bytes_, "algorithmic_bytes_total": total,
    "achieved_GBps": round(total / (gpu_ms * 1e-3) / 1e9, 1),
    "surface_entries": surf_entries, "max_rel_diff_vs_oracle": err,
    "scores": got, "scores_oracle": ref,
}
line = json.dumps(res)
print(line)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
