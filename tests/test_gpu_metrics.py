"""GPU suite — whole-volume segmentation metrics (csrc/metrics.cu, metrics.py) against the fp64 scipy oracle
(oracle/metrics_ref.py): label maps, confusion counts, region surfaces, squared distance transforms, HD95, graph
capture, and TTA -> labels -> scores end to end."""
import numpy as np
import pytest
import torch
from scipy import ndimage

from oracle import metrics_ref as M

pytestmark = pytest.mark.gpu

ANISO = (2.0, 0.9375, 0.9375)


def phantom(shape, seed, perturb=False):
    """Nested ellipsoids: label 2 (ED) shell of WT, 1 (NCR/NET) shell of TC, 3 (ET) core.  `perturb`: moved, resized
    and with salt-and-pepper noise near the boundaries, as a prediction of the same case."""
    rng = np.random.default_rng(seed)
    D, H, W = shape
    z, y, x = np.meshgrid(np.arange(D), np.arange(H), np.arange(W), indexing="ij")
    c = np.array([D, H, W]) * rng.uniform(0.4, 0.6, size=3)
    rad = np.array([D, H, W]) * rng.uniform(0.22, 0.3, size=3)
    if perturb:
        c = c + rng.normal(0, 1.5, size=3)
        rad = rad * rng.uniform(0.92, 1.08, size=3)
    r2 = ((z - c[0]) / rad[0]) ** 2 + ((y - c[1]) / rad[1]) ** 2 + ((x - c[2]) / rad[2]) ** 2
    lab = np.zeros(shape, np.uint8)
    lab[r2 < 1.0] = 2
    lab[r2 < 0.45] = 1
    lab[r2 < 0.15] = 3
    if perturb:
        noise = (rng.random(shape) < 0.02) & (np.abs(r2 - 0.45) < 0.2)
        lab[noise] = rng.integers(0, 4, size=int(noise.sum()))
    return lab


def cuda_u8(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def lut_of(b3d, regions, dev):
    return torch.tensor(b3d.metrics._region_lut(regions), dtype=torch.uint8, device=dev)


def surfaces_and_counts(b3d, dev, pred, true, regions=M.BRATS_REGIONS):
    R = len(regions)
    p, t = cuda_u8(pred, dev), cuda_u8(true, dev)
    counts = torch.full((R, 4), -7, dtype=torch.int64, device=dev)       # the call must clear it
    sp, st = torch.full_like(p, 0xAA), torch.full_like(t, 0xAA)
    b3d._lib.call("b3d_region_surface", p, t, lut_of(b3d, regions, dev), counts, sp, st)
    return counts.cpu().numpy(), sp.cpu().numpy(), st.cpu().numpy()


def surface_bits(labels, regions=M.BRATS_REGIONS):
    out = np.zeros(labels.shape, np.uint8)
    for r, region in enumerate(regions.values()):
        out |= M.surface(M.region_mask(labels, region)).astype(np.uint8) << r
    return out


def edt_gpu(b3d, dev, bits, R, spacing=(1.0, 1.0, 1.0)):
    e = torch.full((R,) + bits.shape, -1.0, dtype=torch.float32, device=dev)
    b3d._lib.call("b3d_surface_edt", cuda_u8(bits, dev), e, R, *spacing)
    return e.cpu().numpy()


# ---- label maps ----------------------------------------------------------------------------------------------------

def torch_labels(p, threshold=0.5):
    """Torch restatement of the label rule on [D,H,W,C]: first argmax + 1 where the maximum is > threshold."""
    mx, am = p.max(dim=-1)
    return torch.where(mx > threshold, am + 1, torch.zeros_like(am)).to(torch.uint8)


def test_label_map_matches_torch(b3d, dev):
    g = torch.Generator(device=dev).manual_seed(1)
    p = torch.rand(160, 192, 160, 3, generator=g, device=dev)
    got = b3d.predict_labels(p, shape=[155, 190, 147])
    assert got.dtype == torch.uint8 and tuple(got.shape) == (155, 190, 147)
    assert torch.equal(got, torch_labels(p)[:155, :190, :147])
    assert torch.equal(b3d.predict_labels(p.unsqueeze(0), threshold=0.7), torch_labels(p, 0.7))
    # channels_first, with and without the batch axis
    pcf = p.permute(3, 0, 1, 2).contiguous()
    assert torch.equal(b3d.predict_labels(pcf, data_format='channels_first', shape=(155, 190, 147)),
                       torch_labels(p)[:155, :190, :147])
    assert torch.equal(b3d.predict_labels(pcf.unsqueeze(0), data_format='channels_first'), torch_labels(p))
    # a skull-strip model: one channel
    p1 = torch.rand(33, 17, 9, 1, generator=g, device=dev)
    assert torch.equal(b3d.predict_labels(p1), torch_labels(p1))
    # ties go to the first maximum; a maximum equal to the threshold is background
    above = float(np.nextafter(np.float32(0.5), np.float32(1.0)))       # the next fp32 after the threshold
    q = torch.tensor([[0.7, 0.7, 0.1], [0.2, 0.9, 0.9], [0.5, 0.5, 0.5], [0.1, 0.2, above],
                      [0.0, 0.0, 0.0], [0.3, 0.1, 0.2], [0.6, 0.6, 0.6], [0.1, 0.5, 0.5]],
                     dtype=torch.float32, device=dev).reshape(2, 2, 2, 3)
    got = b3d.predict_labels(q)
    assert got.flatten().tolist() == [1, 2, 0, 3, 0, 0, 1, 0]
    assert torch.equal(got, torch_labels(q))
    assert torch.equal(got.cpu(), torch.from_numpy(M.label_map(q.cpu().numpy())))
    # one-hot targets turn back into labels
    lab = torch.from_numpy(phantom((20, 24, 22), 3)).to(dev).long()
    onehot = torch.nn.functional.one_hot(lab, 4)[..., 1:].float()
    assert torch.equal(b3d.predict_labels(onehot), lab.to(torch.uint8))
    with pytest.raises(ValueError):
        b3d.predict_labels(p, shape=(161, 1, 1))


# ---- counts and surfaces -------------------------------------------------------------------------------------------

def border_cases():
    a = np.zeros((12, 10, 14), np.uint8)
    a[0:5, :, 9:] = 3                    # touches five faces
    a[7:, 0:3, 0:2] = 2
    b = np.zeros_like(a)
    b[0:4, 2:, 8:] = 3
    b[6:, 0:4, 0:3] = 1
    return a, b


@pytest.mark.parametrize("shape", [(155, 240, 240), (1, 1, 1), (1, 7, 1), (3, 5, 7), (33, 17, 9)])
def test_counts_and_surfaces_match_oracle(b3d, dev, shape):
    true = phantom(shape, 10)
    pred = phantom(shape, 10, perturb=True)
    if shape == (1, 7, 1):
        true, pred = np.array([0, 3, 3, 1, 2, 0, 3], np.uint8).reshape(shape), \
            np.array([3, 3, 0, 1, 1, 2, 3], np.uint8).reshape(shape)
    if shape == (1, 1, 1):
        true, pred = np.full(shape, 3, np.uint8), np.full(shape, 1, np.uint8)
    counts, sp, st = surfaces_and_counts(b3d, dev, pred, true)
    assert np.array_equal(sp, surface_bits(pred)) and np.array_equal(st, surface_bits(true))
    for r, region in enumerate(M.BRATS_REGIONS.values()):
        assert tuple(counts[r]) == M.counts(M.region_mask(pred, region), M.region_mask(true, region))


def test_counts_and_surfaces_border_and_full(b3d, dev):
    a, b = border_cases()
    for pred, true in ((a, b), (np.full(a.shape, 2, np.uint8), b), (np.full(a.shape, 3, np.uint8), a)):
        counts, sp, st = surfaces_and_counts(b3d, dev, pred, true)
        assert np.array_equal(sp, surface_bits(pred)) and np.array_equal(st, surface_bits(true))
        for r, region in enumerate(M.BRATS_REGIONS.values()):
            assert tuple(counts[r]) == M.counts(M.region_mask(pred, region), M.region_mask(true, region))
    # eight regions, labels up to 255, a region that no label reaches
    rng = np.random.default_rng(4)
    regions = {str(i): (i + 1, 255 - i) for i in range(7)}
    regions["none"] = (200,)
    pred = rng.choice(np.array([0, 1, 2, 3, 4, 5, 6, 7, 249, 250, 255], np.uint8), size=(9, 11, 13))
    true = rng.choice(np.array([0, 1, 3, 5, 7, 251, 254], np.uint8), size=(9, 11, 13))
    counts, sp, st = surfaces_and_counts(b3d, dev, pred, true, regions)
    assert np.array_equal(sp, surface_bits(pred, regions)) and np.array_equal(st, surface_bits(true, regions))
    for r, region in enumerate(regions.values()):
        assert tuple(counts[r]) == M.counts(M.region_mask(pred, region), M.region_mask(true, region))


# ---- distance transforms -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape", [(155, 240, 240), (33, 17, 9), (1, 7, 1), (3, 5, 7), (4, 512, 3), (4, 600, 3),
                                   (2, 3, 1024), (1030, 2, 2)])
def test_edt(b3d, dev, shape):
    bits = surface_bits(phantom(shape, 20)) if min(shape) > 2 else \
        (np.random.default_rng(5).random(shape) < 0.01).astype(np.uint8) * 5
    bits.flat[0] |= 2                       # region 1 always has a voxel; region 2 may have none
    R = 3
    if max(shape) > 1024:
        with pytest.raises(b3d._lib.B3DError, match="1024"):
            edt_gpu(b3d, dev, bits, R)
        return
    got = edt_gpu(b3d, dev, bits, R)
    got_a = edt_gpu(b3d, dev, bits, R, ANISO)
    for r in range(R):
        m = ((bits >> r) & 1).astype(bool)
        if not m.any():
            assert np.all(np.isinf(got[r])) and np.all(np.isinf(got_a[r]))
            continue
        ref = np.round(ndimage.distance_transform_edt(~m) ** 2).astype(np.float32)
        assert np.array_equal(got[r], ref), np.abs(got[r] - ref).max()
        ref_a = ndimage.distance_transform_edt(~m, sampling=ANISO) ** 2
        nz = ref_a > 0
        assert np.all(got_a[r][~nz] == 0)
        assert np.max(np.abs(got_a[r][nz] - ref_a[nz]) / ref_a[nz]) <= 1e-6


# ---- HD95 ----------------------------------------------------------------------------------------------------------

def check_scores(got, ref, spacing):
    tol = 1e-9 if tuple(spacing) == (1.0, 1.0, 1.0) else 1e-6
    assert got.keys() == ref.keys()
    for name in ref:
        for k in ("dice", "sensitivity", "specificity"):
            assert got[name][k] == pytest.approx(ref[name][k], rel=1e-15, abs=0.0), (name, k)
        a, b = got[name]["hd95"], ref[name]["hd95"]
        if np.isinf(b) or b == 0.0:
            assert a == b, (name, a, b)
        else:
            assert abs(a - b) <= tol * b, (name, a, b)


@pytest.mark.parametrize("spacing", [(1.0, 1.0, 1.0), ANISO])
@pytest.mark.parametrize("shape", [(155, 240, 240), (33, 17, 9), (3, 5, 7)])
def test_hd95_matches_oracle(b3d, dev, shape, spacing):
    for seed in (30, 31):
        true = phantom(shape, seed)
        pred = phantom(shape, seed, perturb=True)
        got = b3d.segmentation_metrics(cuda_u8(pred, dev), cuda_u8(true, dev), spacing=spacing)
        check_scores(got, M.segmentation_metrics(pred, true, spacing), spacing)


@pytest.mark.parametrize("spacing", [(1.0, 1.0, 1.0), ANISO])
def test_hd95_edge_rules(b3d, dev, spacing):
    shape = (9, 10, 11)
    z = np.zeros(shape, np.uint8)
    one_a, one_b = z.copy(), z.copy()
    one_a[2, 3, 4] = 3
    one_b[7, 1, 9] = 3
    a, b = border_cases()
    cases = [(z, z), (one_a, z), (z, one_a), (one_a, one_a), (one_a, one_b), (np.full(shape, 2, np.uint8), z),
             (np.full(shape, 3, np.uint8), np.full(shape, 1, np.uint8)), (a[:9, :10, :11], b[:9, :10, :11])]
    for pred, true in cases:
        got = b3d.segmentation_metrics(cuda_u8(pred, dev), cuda_u8(true, dev), spacing=spacing)
        check_scores(got, M.segmentation_metrics(pred, true, spacing), spacing)
    got = b3d.segmentation_metrics(cuda_u8(one_a, dev), cuda_u8(one_b, dev), spacing=spacing)
    d = np.sqrt(sum(((p - q) * s) ** 2 for p, q, s in zip((2, 3, 4), (7, 1, 9), spacing)))
    assert got["ET"]["hd95"] == pytest.approx(d, rel=1e-12)
    assert got["ET"]["dice"] == 0.0 and got["WT"]["dice"] == 0.0
    # skull-strip form: one region
    brain = {"brain": (1,)}
    pm, tm = (phantom(shape, 8, perturb=True) > 0).astype(np.uint8), (phantom(shape, 8) > 0).astype(np.uint8)
    got = b3d.segmentation_metrics(cuda_u8(pm, dev), cuda_u8(tm, dev), spacing=spacing, regions=brain)
    check_scores(got, M.segmentation_metrics(pm, tm, spacing, brain), spacing)


def test_metrics_reject_bad_arguments(b3d, dev):
    a = cuda_u8(np.zeros((4, 5, 6), np.uint8), dev)
    with pytest.raises(ValueError, match="differ"):
        b3d.segmentation_metrics(a, a[:, :, :5])
    with pytest.raises(ValueError, match="uint8"):
        b3d.segmentation_metrics(a.float(), a)
    with pytest.raises(ValueError, match="spacing"):
        b3d.segmentation_metrics(a, a, spacing=(1.0, 0.0, 1.0))
    with pytest.raises(ValueError, match="regions"):
        b3d.segmentation_metrics(a, a, regions={str(i): (1,) for i in range(9)})
    with pytest.raises(ValueError, match="outside 1..255"):
        b3d.segmentation_metrics(a, a, regions={"x": (0, 1)})
    work = torch.empty(16, dtype=torch.uint8, device=dev)
    e = torch.empty((1, 4, 5, 6), device=dev)
    counts = torch.zeros((1, 4), dtype=torch.int64, device=dev)
    out = torch.empty((1, 4), dtype=torch.float64, device=dev)
    with pytest.raises(b3d._lib.B3DError, match="workspace"):
        b3d._lib.call("b3d_hd95", e, a, e, a, counts, out, work)


# ---- graph capture -------------------------------------------------------------------------------------------------

def test_graph_capture_replays(b3d, dev):
    shape = (40, 48, 36)
    true, pred = phantom(shape, 50), phantom(shape, 50, perturb=True)
    p, t = cuda_u8(pred, dev), cuda_u8(true, dev)
    R, n = 3, p.numel()
    lut = lut_of(b3d, M.BRATS_REGIONS, dev)
    counts = torch.empty((R, 4), dtype=torch.int64, device=dev)
    sp, st = torch.empty_like(p), torch.empty_like(t)
    ep, et = torch.empty((R,) + shape, device=dev), torch.empty((R,) + shape, device=dev)
    work = torch.empty(4 * R * (264 + 2 * n), dtype=torch.uint8, device=dev)
    out = torch.empty((R, 4), dtype=torch.float64, device=dev)

    def run():
        b3d._lib.call("b3d_region_surface", p, t, lut, counts, sp, st)
        b3d._lib.call("b3d_surface_edt", sp, ep, R, *ANISO)
        b3d._lib.call("b3d_surface_edt", st, et, R, *ANISO)
        b3d._lib.call("b3d_hd95", et, sp, ep, st, counts, out, work)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run()                                                   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    eager = out.clone()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    out.fill_(-1.0)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
    ref = M.segmentation_metrics(pred, true, ANISO)
    check_scores({k: dict(zip(("dice", "sensitivity", "specificity", "hd95"), row))
                  for k, row in zip(M.BRATS_REGIONS, out.cpu().tolist())}, ref, ANISO)
    # the replay reads the current inputs
    p.copy_(t)
    g.replay()
    torch.cuda.synchronize()
    assert torch.all(out[:, :3] == 1.0) and torch.all(out[:, 3] == 0.0)


# ---- end to end ----------------------------------------------------------------------------------------------------

def test_tta_labels_scores_end_to_end(b3d, dev):
    torch.manual_seed(0)
    shape = (37, 45, 33)
    g = torch.Generator().manual_seed(6)
    vol = torch.randn(*shape, 2, generator=g) * 40 + 100
    mask = (vol.max(dim=-1, keepdim=True).values > 80).float()
    xp, mp, orig = b3d.pad_to_spatial_res(8, vol.to(dev), mask.to(dev))
    model = b3d.Model()
    with torch.no_grad():
        model(torch.zeros(1, 16, 16, 16, 2, device=dev), training=False, inference=True)      # build
    tta = b3d.TestTimeAugmentor([100.0, 98.0], [40.0, 42.0], model, 'channels_last')
    probs = tta(xp, mp)
    true = phantom(tuple(orig), 60)
    for thr in (0.5, float(probs.float().median())):
        pred = b3d.predict_labels(probs, threshold=thr, shape=orig)
        pred_ref = M.label_map(probs.cpu().numpy(), thr, orig)
        assert np.array_equal(pred.cpu().numpy(), pred_ref)
        for spacing in ((1.0, 1.0, 1.0), ANISO):
            got = b3d.segmentation_metrics(pred, cuda_u8(true, dev), spacing=spacing)
            check_scores(got, M.segmentation_metrics(pred_ref, true, spacing), spacing)
