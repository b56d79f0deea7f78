"""Evaluation of one whole-volume segmentation on the device: the label map of averaged class probabilities, and per
region Dice, sensitivity, specificity and the 95th-percentile Hausdorff distance (csrc/metrics.cu).

    probs = tta(x, bmask)                                   # [D, H, W, C] class probabilities
    pred = predict_labels(probs, shape=orig_shape)          # uint8 [D, H, W]: 0 background, c + 1 for class c
    scores = segmentation_metrics(pred, true, spacing=(1.0, 1.0, 1.0))
    scores["ET"]["hd95"]

Label c + 1 is class channel c, the preprocessed BraTS convention (1 = NCR/NET, 2 = ED, 3 = ET), so
`predict_labels` also turns a one-hot target back into labels.
"""
from __future__ import annotations

import math

import torch

from . import ops

BRATS_REGIONS = {"WT": (1, 2, 3), "TC": (1, 3), "ET": (3,)}
MAX_REGIONS = 8
_NAMES = ("dice", "sensitivity", "specificity", "hd95")


def predict_labels(y_pred, threshold=0.5, data_format='channels_last', shape=None):
    """Label map of class probabilities: first argmax + 1 where the maximum is > `threshold`, else 0.

    y_pred: fp32 CUDA [D,H,W,C] or [1,D,H,W,C]; with data_format='channels_first', [C,D,H,W] or [1,C,D,H,W].
    shape: the `orig_shape` returned by pad_to_spatial_res; the result is then the leading [d,h,w] corner.
    Returns uint8 [D,H,W] (or `shape`)."""
    ops._check(y_pred, "y_pred")
    if data_format == 'channels_first':
        if y_pred.dim() == 4:
            y_pred = y_pred.unsqueeze(0)
        if y_pred.dim() != 5 or y_pred.shape[0] != 1:
            raise ValueError(f"predict_labels: channels_first y_pred must be [C,D,H,W] or [1,C,D,H,W], got "
                             f"{tuple(y_pred.shape)}")
        y_pred = ops.to_channels_last(y_pred)
    elif data_format != 'channels_last':
        raise ValueError(f"predict_labels: unknown data_format {data_format!r}")
    if y_pred.dim() == 5 and y_pred.shape[0] == 1:
        y_pred = y_pred[0]
    if y_pred.dim() != 4:
        raise ValueError(f"predict_labels: y_pred must be [D,H,W,C] or [1,D,H,W,C], got {tuple(y_pred.shape)}")
    full = tuple(y_pred.shape[:3])
    out_shape = full if shape is None else tuple(int(s) for s in shape)
    if len(out_shape) != 3 or any(s < 1 or s > f for s, f in zip(out_shape, full)):
        raise ValueError(f"predict_labels: shape {out_shape} is not within the volume {full}")
    labels = torch.empty(out_shape, dtype=torch.uint8, device=y_pred.device)
    ops._call("b3d_label_map", y_pred.contiguous(), labels, float(threshold))
    return labels


def _region_lut(regions):
    if not 1 <= len(regions) <= MAX_REGIONS:
        raise ValueError(f"segmentation_metrics: 1..{MAX_REGIONS} regions, got {len(regions)}")
    lut = [0] * 256
    for r, (name, labels) in enumerate(regions.items()):
        for lab in labels:
            if not isinstance(lab, int) or not 1 <= lab <= 255:
                raise ValueError(f"segmentation_metrics: region {name!r} has label {lab!r} outside 1..255")
            lut[lab] |= 1 << r
    return lut


def segmentation_metrics(pred, true, spacing=(1.0, 1.0, 1.0), regions=BRATS_REGIONS):
    """Scores of the label map `pred` against `true` (uint8 CUDA [D,H,W] of one shape) per region.

    regions: {name: labels}; a voxel belongs to a region when its label is in that region's set.
    spacing: voxel size (sd, sh, sw) in the arrays' axis order.
    Returns {name: {"dice", "sensitivity", "specificity", "hd95"}}.  A ratio with a zero denominator is 1.0;
    hd95 (medpy's definition, numpy 'linear' percentile of both directed surface distances) is 0.0 when both
    surfaces are empty and inf when exactly one is.  One device-to-host copy per call.

    Device memory per call: two fp32 distance fields of [R, D, H, W] and a workspace of 8 * R * D*H*W bytes (room for
    every voxel being on both surfaces, so that no count has to reach the host first): for 155x240x240 and three
    regions about 214 MB each, handed back to the caching allocator when the call returns."""
    for name, t in (("pred", pred), ("true", true)):
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != torch.uint8 or t.dim() != 3:
            raise ValueError(f"segmentation_metrics: {name} must be a uint8 CUDA [D,H,W] label map")
    if pred.shape != true.shape or pred.device != true.device:
        raise ValueError(f"segmentation_metrics: pred {tuple(pred.shape)} and true {tuple(true.shape)} differ "
                         "in shape or device")
    sp = tuple(float(s) for s in spacing)
    if len(sp) != 3 or not all(s > 0 and math.isfinite(s) for s in sp):
        raise ValueError(f"segmentation_metrics: spacing must be three positive numbers, got {spacing!r}")
    lut = torch.tensor(_region_lut(regions), dtype=torch.uint8).to(pred.device, non_blocking=True)
    R, n = len(regions), pred.numel()
    pred, true = pred.contiguous(), true.contiguous()
    dev = pred.device
    counts = torch.empty((R, 4), dtype=torch.int64, device=dev)
    surf_pred, surf_true = torch.empty_like(pred), torch.empty_like(true)
    edt_pred = torch.empty((R,) + tuple(pred.shape), dtype=torch.float32, device=dev)
    edt_true = torch.empty_like(edt_pred)
    work = torch.empty(4 * R * (264 + 2 * n), dtype=torch.uint8, device=dev)
    out = torch.empty((R, 4), dtype=torch.float64, device=dev)
    ops._call("b3d_region_surface", pred, true, lut, counts, surf_pred, surf_true)
    ops._call("b3d_surface_edt", surf_pred, edt_pred, R, *sp)
    ops._call("b3d_surface_edt", surf_true, edt_true, R, *sp)
    ops._call("b3d_hd95", edt_true, surf_pred, edt_pred, surf_true, counts, out, work)
    vals = out.cpu().tolist()
    return {name: dict(zip(_NAMES, row)) for name, row in zip(regions, vals)}
