"""CPU suite — the fp64 segmentation-metric oracle (oracle/metrics_ref.py) against brute force, its edge rules, and the
argument checks of metrics.py that run before any device work."""
import numpy as np
import pytest
import torch

from oracle import metrics_ref as M


def _surface_brute(mask):
    D, H, W = mask.shape
    out = np.zeros_like(mask)
    for z, y, x in zip(*np.nonzero(mask)):
        for dz, dy, dx in ((1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)):
            a, b, c = z + dz, y + dy, x + dx
            if not (0 <= a < D and 0 <= b < H and 0 <= c < W) or not mask[a, b, c]:
                out[z, y, x] = True
                break
    return out


def _hd95_brute(pm, tm, spacing):
    sp, st = _surface_brute(pm), _surface_brute(tm)
    if not sp.any() and not st.any():
        return 0.0
    if not sp.any() or not st.any():
        return float("inf")
    s = np.asarray(spacing)
    a, b = np.argwhere(sp) * s, np.argwhere(st) * s
    d = np.sqrt(((a[:, None, :] - b[None, :, :]) ** 2).sum(-1))
    return float(np.percentile(np.concatenate([d.min(1), d.min(0)]), 95))


@pytest.mark.parametrize("seed", range(6))
def test_oracle_hd95_is_brute_force(seed):
    rng = np.random.default_rng(seed)
    shape = tuple(rng.integers(1, 13, size=3))
    spacing = tuple(rng.uniform(0.5, 3.0, size=3))
    pred = rng.integers(0, 4, size=shape).astype(np.uint8)
    true = rng.integers(0, 4, size=shape).astype(np.uint8)
    for region in M.BRATS_REGIONS.values():
        pm, tm = M.region_mask(pred, region), M.region_mask(true, region)
        assert np.array_equal(M.surface(pm), _surface_brute(pm))
        ref = _hd95_brute(pm, tm, spacing)
        got = M.hd95(pm, tm, spacing)
        assert got == pytest.approx(ref, rel=1e-12, abs=0.0) or (got == ref == 0.0)
        st = _surface_brute(tm)
        if st.any():
            pts = np.argwhere(st) * np.asarray(spacing)
            grid = np.stack(np.meshgrid(*[np.arange(n) for n in shape], indexing="ij"), -1) * np.asarray(spacing)
            brute = ((grid[..., None, :] - pts) ** 2).sum(-1).min(-1)
            np.testing.assert_allclose(M.edt_sq(st, spacing), brute, rtol=1e-12)


def test_oracle_edge_rules():
    z = np.zeros((5, 6, 7), bool)
    full = np.ones((5, 6, 7), bool)
    one = z.copy()
    one[2, 3, 4] = True
    assert M.hd95(z, z) == 0.0
    assert M.hd95(one, z) == float("inf") and M.hd95(z, one) == float("inf")
    assert M.hd95(full, full) == 0.0
    assert M.hd95(one, one) == 0.0
    # a region filling the volume: its surface is the volume's border
    s = M.surface(full)
    assert s.sum() == full.size - 3 * 4 * 5 and not s[1:-1, 1:-1, 1:-1].any()
    r = M.segmentation_metrics(np.zeros((4, 4, 4), np.uint8), np.zeros((4, 4, 4), np.uint8))
    assert all(v == {"dice": 1.0, "sensitivity": 1.0, "specificity": 1.0, "hd95": 0.0} for v in r.values())
    r = M.segmentation_metrics(np.full((4, 4, 4), 3, np.uint8), np.full((4, 4, 4), 3, np.uint8))
    assert r["ET"] == {"dice": 1.0, "sensitivity": 1.0, "specificity": 1.0, "hd95": 0.0}


def test_oracle_label_rule_ties_and_threshold():
    p = np.zeros((1, 1, 6, 3), np.float32)
    p[0, 0, 0] = [0.7, 0.7, 0.1]      # tie: first maximum
    p[0, 0, 1] = [0.2, 0.9, 0.9]      # tie: first maximum
    p[0, 0, 2] = [0.5, 0.5, 0.5]      # exactly at the threshold: background
    p[0, 0, 3] = [0.1, 0.2, np.nextafter(np.float32(0.5), np.float32(1))]
    p[0, 0, 4] = [0.0, 0.0, 0.0]
    p[0, 0, 5] = [0.3, 0.1, 0.2]      # below the threshold
    assert M.label_map(p).tolist() == [[[1, 2, 0, 3, 0, 0]]]
    assert M.label_map(p, threshold=0.25).tolist() == [[[1, 2, 1, 3, 0, 1]]]
    assert M.label_map(p, shape=(1, 1, 2)).tolist() == [[[1, 2]]]


def test_metrics_reject_bad_arguments(b3d):
    m = b3d.metrics
    cpu = torch.zeros(4, 4, 4, dtype=torch.uint8)
    with pytest.raises(ValueError, match="uint8 CUDA"):
        m.segmentation_metrics(cpu, cpu)
    with pytest.raises(ValueError, match="regions"):
        m._region_lut({str(i): (1,) for i in range(9)})
    for bad in ((0,), (256,), (1.5,)):
        with pytest.raises(ValueError, match="outside 1..255"):
            m._region_lut({"x": bad})
    lut = m._region_lut(m.BRATS_REGIONS)
    assert lut[0] == 0 and lut[1] == 0b011 and lut[2] == 0b001 and lut[3] == 0b111 and not any(lut[4:])
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.predict_labels(torch.zeros(2, 2, 2, 3))
    assert m.BRATS_REGIONS == M.BRATS_REGIONS
