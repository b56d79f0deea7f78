"""ORACLE — fp64 numpy / scipy reference of the segmentation metrics (3d-brain-tumor-segmentation_b200/metrics.py,
csrc/metrics.cu).  Test infrastructure only.

    label      = argmax_c p[c] + 1 (first maximum) where max_c p[c] > threshold, else 0
    region     = a set of labels; TP, FP, FN, TN over the volume
    dice       = 2TP / (2TP + FP + FN), sensitivity = TP / (TP + FN), specificity = TN / (TN + FP); 0/0 -> 1.0
    surface(A) = A & ~binary_erosion(A, 6-connectivity, border_value=0)
    hd95       = percentile(concat(d_AB, d_BA), 95, 'linear'): distances (with spacing) from each surface voxel of the
                 prediction to the nearest truth surface voxel and back; 0.0 if both surfaces are empty, inf if one is
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

BRATS_REGIONS = {"WT": (1, 2, 3), "TC": (1, 3), "ET": (3,)}
_STRUCT = ndimage.generate_binary_structure(3, 1)


def label_map(p, threshold=0.5, shape=None):
    """p: [D,H,W,C] probabilities -> uint8 labels of the leading `shape` corner."""
    p = np.asarray(p)
    if shape is not None:
        p = p[:shape[0], :shape[1], :shape[2]]
    lab = np.argmax(p, axis=-1) + 1
    return np.where(p.max(axis=-1) > threshold, lab, 0).astype(np.uint8)


def region_mask(labels, region):
    return np.isin(labels, np.asarray(region))


def surface(mask):
    mask = np.asarray(mask, dtype=bool)
    return mask & ~ndimage.binary_erosion(mask, _STRUCT, border_value=0)


def counts(pred_mask, true_mask):
    p, t = np.asarray(pred_mask, bool), np.asarray(true_mask, bool)
    return (int(np.sum(p & t)), int(np.sum(p & ~t)), int(np.sum(~p & t)), int(np.sum(~p & ~t)))


def edt_sq(surf, spacing=(1.0, 1.0, 1.0)):
    """Squared distance from every voxel to the nearest set voxel of `surf`; inf everywhere when it is empty."""
    surf = np.asarray(surf, bool)
    if not surf.any():
        return np.full(surf.shape, np.inf)
    return ndimage.distance_transform_edt(~surf, sampling=spacing) ** 2


def surface_distances(pred_mask, true_mask, spacing=(1.0, 1.0, 1.0)):
    """(d_AB, d_BA): distances from the prediction's surface voxels to the truth's surface and back (both surfaces
    non-empty)."""
    sp, st = surface(pred_mask), surface(true_mask)
    d_ab = ndimage.distance_transform_edt(~st, sampling=spacing)[sp]
    d_ba = ndimage.distance_transform_edt(~sp, sampling=spacing)[st]
    return d_ab, d_ba


def hd95(pred_mask, true_mask, spacing=(1.0, 1.0, 1.0)):
    sp, st = surface(pred_mask).any(), surface(true_mask).any()
    if not sp and not st:
        return 0.0
    if not sp or not st:
        return float("inf")
    d_ab, d_ba = surface_distances(pred_mask, true_mask, spacing)
    return float(np.percentile(np.concatenate([d_ab, d_ba]), 95))


def _ratio(a, b):
    return 1.0 if b == 0 else a / b


def segmentation_metrics(pred, true, spacing=(1.0, 1.0, 1.0), regions=BRATS_REGIONS):
    out = {}
    for name, region in regions.items():
        pm, tm = region_mask(pred, region), region_mask(true, region)
        tp, fp, fn, tn = counts(pm, tm)
        out[name] = {"dice": _ratio(2 * tp, 2 * tp + fp + fn), "sensitivity": _ratio(tp, tp + fn),
                     "specificity": _ratio(tn, tn + fp), "hd95": hd95(pm, tm, spacing)}
    return out
