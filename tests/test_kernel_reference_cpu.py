"""CPU suite — the fp64 references of tests/test_gpu_kernel_paths.py (oracle/kernel_ref.py) and the checker they feed.

1. The tap-sum conv references (forward, data gradient, weight gradient; k = 1 and 3; with and without the operand
   rounding of the tensor-core kernels) equal the oracle's `conv3d_same` and its autograd to 1e-12.
2. Sensitivity: the checker accepts an fp32 computation of the same rounded operands (what a correct kernel returns)
   and rejects it once a realistic bug is applied to it — one 16-channel K chunk of one tap missing inside one edge
   patch, one CTA's voxel range missing from a dgamma, one warp's statistics flush missing."""
import pytest
import torch

from oracle import kernel_ref as K
from oracle import ref_model as R


def r64(*shape, seed=0, scale=1.0, mean=0.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g, dtype=torch.float64) * scale + mean


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("op", [None, "fp16", "bf16", "tf32"])
@pytest.mark.parametrize("shape", [(2, 3, 4, 5, 6, 7), (1, 5, 2, 9, 16, 3)])
def test_tap_references_equal_oracle_conv(k, op, shape):
    B, D, H, W, ci, co = shape
    x = K.round_act(r64(B, D, H, W, ci, seed=1, mean=0.5), op)
    w = K.round_weight(r64(k, k, k, ci, co, seed=2, scale=0.3), op)
    dy = K.round_act(r64(B, D, H, W, co, seed=3), op)
    xr, wr = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    y = R.conv3d_same(xr, wr, None, 1)
    dx, dw = torch.autograd.grad(y, (xr, wr), dy)
    assert K.rel_l2(K.conv_taps(x, w), y) < 1e-12
    assert K.rel_l2(K.dgrad_taps(dy, w), dx) < 1e-12
    assert K.rel_l2(K.wgrad_taps(x, dy, k), dw) < 1e-12


def test_operand_roundings():
    t = torch.tensor([1.0 + 2.0 ** -11, -(1.0 + 2.0 ** -11), 1.0 + 3 * 2.0 ** -11, 1.0 + 2.0 ** -11 + 2.0 ** -20,
                      1.0 + 2.0 ** -10 - 2.0 ** -23], dtype=torch.float32)
    # ties away from zero (cvt.rna) | toward zero (fp32 bits fed to a kind::tf32 MMA) | ties to even (round_operand)
    assert K.round_tf32_rna(t).tolist() == [1.0 + 2.0 ** -10, -(1.0 + 2.0 ** -10), 1.0 + 2 * 2.0 ** -10,
                                            1.0 + 2.0 ** -10, 1.0 + 2.0 ** -10]
    assert K.round_tf32_tz(t).tolist() == [1.0, -1.0, 1.0 + 2.0 ** -10, 1.0, 1.0]
    assert R.round_operand(t, "tf32").tolist()[:3] == [1.0, -1.0, 1.0 + 2 * 2.0 ** -10]
    assert torch.equal(K.round_act(t, "fp16"), t.half().float())


# ------------------------------------------------------------------------------------------------- sensitivity
def _conv_fp32(x, w):
    """A correct kernel's result: the same rounded operands, fp32 accumulation over taps and channel chunks."""
    k = w.shape[0]
    B, D, H, W, ci = x.shape
    xp = torch.nn.functional.pad(x.float(), (0, 0, 1, 1, 1, 1, 1, 1)) if k == 3 else x.float()
    y = torch.zeros(B, D, H, W, w.shape[4])
    for c0 in range(0, ci, 16):
        for kd, kh, kw in K._taps(k):
            y += xp[:, kd:kd + D, kh:kh + H, kw:kw + W, c0:c0 + 16] @ w[kd, kh, kw, c0:c0 + 16].float()
    return y


def test_checker_catches_a_dropped_k_chunk_in_an_edge_patch():
    B, D, H, W, ci, co = 1, 20, 24, 20, 32, 16
    x = K.round_act(r64(B, D, H, W, ci, seed=4, mean=1.0), "bf16")
    w = K.round_weight(r64(3, 3, 3, ci, co, seed=5, scale=0.1), "bf16")
    ref, A = K.conv_taps(x, w), K.conv_taps(x.abs(), w.abs())
    n_acc = 27 * ci // 16
    good = _conv_fp32(x, w)
    c = K.check("fp32 accumulation", good, ref, A, n_acc, 1e-5, tile=(4, 16, 16, 16))
    assert c.ok, c
    # the last (partial) patch of the volume: d 16..19, h 16..23, w 16..19; K chunk 1 (channels 16..31) of the centre tap
    bad = good.clone()
    patch = (slice(None), slice(16, 20), slice(16, 24), slice(16, 20))
    bad[patch] -= (x[patch][..., 16:32] @ w[1, 1, 1, 16:32]).float()
    c = K.check("dropped chunk", bad, ref, A, n_acc, 1e-5, tile=(4, 16, 16, 16))
    assert not c.ok and c.ratio > 1.0, c
    assert c.where["d"] >= 16 and c.where["h"] >= 16 and c.where["w"] >= 16
    assert "tile (b, d/4, h/16, w/16, c/16) = (0, 4, 1, 1" in c.msg


def test_checker_catches_a_dropped_cta_range_in_dgamma():
    B, D, H, W, C = 1, 16, 16, 16, 32
    x, dy = r64(B, D, H, W, C, seed=6, mean=3.0), r64(B, D, H, W, C, seed=7)
    ga, be = 1 + 0.3 * r64(C, seed=8), 0.3 * r64(C, seed=9)
    gr, br = ga.clone().requires_grad_(True), be.clone().requires_grad_(True)
    y = torch.relu(R.group_norm(x, gr, br))
    dga, dbe = torch.autograd.grad(y, (gr, br), dy)
    # fp32 evaluation of the same sums (a correct kernel)
    x32, dy32 = x.float(), dy.float()
    with torch.enable_grad():
        g32, b32 = ga.float().requires_grad_(True), be.float().requires_grad_(True)
        d32 = torch.autograd.grad(torch.relu(R.group_norm(x32, g32, b32)), (g32, b32), dy32)
    assert K.check("dgamma fp32", d32[0], dga, None, None, 1e-5).ok
    assert K.check("dbeta fp32", d32[1], dbe, None, None, 1e-5).ok
    # one CTA of the reduction grid owns a contiguous voxel range of one chunk: drop 1/74 of chunk 3 (128^3 spreads a
    # 16-channel chunk over ~74 CTAs)
    L = D * H * W // 8
    v0, v1 = 3 * L + 10 * (L // 74), 3 * L + 11 * (L // 74)
    xh = ((x.reshape(B, 8, -1) - x.reshape(B, 8, -1).mean(-1, keepdim=True)) /
          torch.sqrt(x.reshape(B, 8, -1).var(-1, unbiased=False, keepdim=True) + 1e-5)).reshape(B, -1, C)
    mask = (y.reshape(B, -1, C) > 0).double()
    lost = (dy.reshape(B, -1, C) * mask * xh)[:, v0 // 1:v1].sum(dim=(0, 1))
    bad = d32[0].double() - lost
    c = K.check("dgamma, one CTA dropped", bad, dga, None, None, 1e-5)
    assert not c.ok, c


def test_checker_catches_a_dropped_warp_statistics_flush():
    B, D, H, W, co = 2, 16, 24, 16, 16
    y = r64(B, D, H, W, co, seed=10, mean=0.7).float()
    # a correct epilogue: fp32 partial sums over 32-row warp slices, added in fp64
    rows = y.reshape(B, 8, -1, 32 * co)
    part = torch.stack([rows.sum(-1), (rows * rows).sum(-1)], dim=-1).double()
    good = part.sum(2)
    ref, scale = K.gn_chunk_sums(y), K.gn_chunk_scale(y)
    c = K.check_sums("stats", good, ref, scale)
    assert c.ok, c
    bad = good.clone()
    bad[1, 5] -= part[1, 5, 7]                 # sample 1, chunk 5: the flush of one warp (32 voxels) is lost
    c = K.check_sums("stats, one warp dropped", bad, ref, scale)
    assert not c.ok and c.where[0] == 1 and c.where[1] == 5, c
