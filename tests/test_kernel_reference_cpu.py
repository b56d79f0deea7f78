"""CPU suite — the fp64 references of tests/test_gpu_kernel_paths.py (oracle/kernel_ref.py) and the checker they feed.

1. The tap-sum conv references (forward, data gradient, weight gradient; k = 1 and 3; with and without the operand
   rounding of the tensor-core kernels) equal the oracle's `conv3d_same` and its autograd to 1e-12.
2. Sensitivity: the checker accepts an fp32 computation of the same rounded operands (what a correct kernel returns)
   and rejects it once a realistic bug is applied to it — one 16-channel K chunk of one tap missing inside one edge
   patch, one CTA's voxel range missing from a dgamma (chunk and channel GroupNorm), one warp's statistics flush
   missing, a depth-slab window normalising the cells past a chunk boundary with the neighbouring chunk's statistics,
   a P16 twin whose start is one cell off."""
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


def test_checker_catches_a_dropped_cta_range_in_channel_group_dgamma():
    """True channel groups (norm_channel.cu): a CTA of gnc_bwd_reduce_kernel owns a contiguous voxel range of every
    channel; at 128^3 x 16 cgeom cuts a sample into ~1,184 such ranges."""
    B, D, H, W, C, G = 1, 16, 16, 16, 32, 8
    x, dy = r64(B, D, H, W, C, seed=12, mean=3.0), r64(B, D, H, W, C, seed=13)
    ga, be = 1 + 0.3 * r64(C, seed=14), 0.3 * r64(C, seed=15)
    gr, br = ga.clone().requires_grad_(True), be.clone().requires_grad_(True)
    with R.channels_first_semantics():
        y = torch.relu(R.group_norm(x, gr, br, G))
        dga, dbe = torch.autograd.grad(y, (gr, br), dy)
        with torch.enable_grad():
            g32, b32 = ga.float().requires_grad_(True), be.float().requires_grad_(True)
            d32 = torch.autograd.grad(torch.relu(R.group_norm(x.float(), g32, b32, G)), (g32, b32), dy.float())
    assert K.check("dgamma fp32", d32[0], dga, None, None, 1e-5).ok
    assert K.check("dbeta fp32", d32[1], dbe, None, None, 1e-5).ok
    S = D * H * W
    per_cta = -(-S // 1184)
    v0, v1 = 10 * per_cta, 11 * per_cta
    grp = x.reshape(B, S, G, C // G)
    xh = ((grp - grp.mean((1, 3), keepdim=True)) / torch.sqrt(grp.var((1, 3), unbiased=False, keepdim=True) + 1e-5))
    xh = xh.reshape(B, S, C)
    mask = (y.reshape(B, S, C) > 0).double()
    lost = (dy.reshape(B, S, C) * mask * xh)[:, v0:v1].sum(dim=(0, 1))
    c = K.check("channel dgamma, one CTA dropped", d32[0].double() - lost, dga, None, None, 1e-5)
    assert not c.ok, c


def _slab_x(D, H, W, C, seed):
    """A volume whose mean and scale change with depth (as in test_slab_window_kernels): neighbouring GroupNorm chunks
    have different statistics."""
    t = (torch.arange(D, dtype=torch.float64) / D).view(1, D, 1, 1, 1)
    return r64(1, D, H, W, C, seed=seed) * (0.5 + t) + (2 * t - 1)


def _gn_apply_slab_fp32(x, stats, ga, be, d0, d1, relu, chunk_of=None):
    """fp32 evaluation of the slab apply (gn_apply16_kernel): window [d0, d1) of the volume x, chunk statistics of the
    whole volume (fp64 sums -> fp32 mean, rstd), y = (x - mean) * (rstd * gamma_j) + beta_j.  chunk_of(e): the chunk
    whose statistics flat element e is normalised with (default e // L)."""
    _, D, H, W, C = x.shape
    L, cg = x.numel() // 8, C // 8
    xs = x[:, d0:d1].reshape(-1).float()
    e = d0 * H * W * C + torch.arange(xs.numel())
    chunk = e // L if chunk_of is None else chunk_of(e)
    m = stats[0, :, 0] / L
    mean = m.float()
    rstd = (1.0 / torch.sqrt(stats[0, :, 1] / L - m * m + 1e-5)).float()
    j = (e // L) * cg + (e % C) % cg
    y = (xs - mean[chunk]) * (rstd[chunk] * ga.float()[j]) + be.float()[j]
    y = torch.relu(y) if relu else y
    return y.reshape(1, d1 - d0, H, W, C)


def test_checker_catches_a_slab_window_with_the_neighbouring_chunks_statistics():
    D, H, W, C = 20, 6, 8, 16                  # a chunk holds 2.5 slices
    x = _slab_x(D, H, W, C, seed=16)
    ga, be = 1 + 0.3 * r64(C, seed=17), 0.3 * r64(C, seed=18)
    ref = torch.relu(R.group_norm(x, ga, be))
    stats, L = K.gn_chunk_sums(x), x.numel() // 8
    d0, d1 = 1, 9                              # chunks 0..3
    good = _gn_apply_slab_fp32(x, stats, ga, be, d0, d1, True)
    c = K.check("fp32 slab apply", good, ref[:, d0:d1], None, None, 1e-5)
    assert c.ok, c
    # the cells of chunk 1 (past the window's first chunk boundary) normalised with chunk 0's statistics
    bad = _gn_apply_slab_fp32(x, stats, ga, be, d0, d1, True, chunk_of=lambda e: torch.where(e // L == 1, 0, e // L))
    c = K.check("neighbouring chunk's statistics", bad, ref[:, d0:d1], None, None, 1e-5)
    assert not c.ok, c
    assert L <= (d0 + c.where["d"]) * H * W * C + (c.where["h"] * W + c.where["w"]) * C + c.where["c"] < 2 * L, c


def test_checker_catches_a_twin_shifted_by_one_cell():
    """A P16 twin written alone (no fp32 output next to it) is checked against the rounded fp64 reference; a twin whose
    start is one 8-channel cell off fails, in fp16 and bf16."""
    D, H, W, C = 20, 6, 8, 16
    x = _slab_x(D, H, W, C, seed=19)
    ga, be = 1 + 0.3 * r64(C, seed=20), 0.3 * r64(C, seed=21)
    ref = R.group_norm(x, ga, be)[:, 3:11]
    y32 = _gn_apply_slab_fp32(x, K.gn_chunk_sums(x), ga, be, 3, 11, False)
    for dt in (torch.float16, torch.bfloat16):
        twin = y32.to(dt).float()
        c = K.check_rounded("twin", twin, ref, dt)
        assert c.ok, c
        shifted = twin.clone().reshape(-1)
        shifted[8:] = twin.reshape(-1)[:-8].clone()
        c = K.check_rounded("twin one cell off", shifted.reshape(twin.shape), ref, dt)
        assert not c.ok and c.ratio > 10, c
