"""ORACLE — test infrastructure only (never imported by the product path).

fp64 references of the conv passes written as a sum over taps, and the bound they are checked with
(tests/test_gpu_kernel_paths.py, pinned to `ref_model.conv3d_same` by tests/test_kernel_reference_cpu.py).

    y[v]      = sum_tap  pad(x)[v + tap] @ w[tap]                     (forward, stride 1, TF 'SAME')
    dx[v]     = sum_tap  pad(dy)[v + tap] @ w[flip(tap)]^T            (data gradient)
    dw[tap]   = sum_v    pad(x)[v + tap]^T dy[v]                      (weight gradient)

A tap sum holds only x and y in memory (plus one shifted view at a time), so it runs at 128^3 where the oracle's
vol2col path would need more than 14 GB of columns.  The operands are rounded first exactly as the tensor-core kernels
round them (`round_act`, `round_weight`), so the only difference left to a correct kernel is fp32 summation order; the
same sums over |x|, |w| give the per-element magnitude A of that difference.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

from oracle import ref_model as R

U32 = 2.0 ** -23          # fp32 unit of the last place at 1.0 (twice the unit roundoff)

# c of the per-element bound |got - ref| <= c*(n_acc + 4)*2^-23*A + 2^-23*|ref|.  One sequential fp32 accumulation
# (an MMA's K step added into the TMEM accumulator, a split-K slice, the bias) errs by at most one rounding of the
# running sum, 2^-24*A; the tensor core aligns the products of a K step to the largest one before adding them and
# drops the bits shifted out (truncation, not rounding), which costs up to one more 2^-24*A per step.  Together that is
# 2^-23*A per step, i.e. c = 1 is the worst case; c = 2 leaves a factor 2 for the fp32 rounding of the stored output
# and of the slices written to the split-K workspace.  The "+ 4" covers the epilogue (bias, finish, sigmoid input).
C_BOUND = 2.0


def round_tf32_rna(t: torch.Tensor) -> torch.Tensor:
    """cvt.rna.tf32.f32: round to 10 explicit significand bits, ties AWAY from zero (how the pack kernels round the
    tf32 weights; `ref_model.round_operand('tf32')` rounds ties to even)."""
    i = t.to(torch.float32).contiguous().view(torch.int32)
    i = (i + 0x1000) & ~0x1FFF                      # sign-magnitude: adding half an ulp to the bits rounds |t| up
    return i.view(torch.float32).to(t.dtype)


def round_tf32_tz(t: torch.Tensor) -> torch.Tensor:
    """The low 13 significand bits dropped (round toward zero): what kind::tf32 MMAs do with fp32 activations that the
    loader stores to shared memory unconverted (csrc/conv_tc.cu operand loaders)."""
    i = t.to(torch.float32).contiguous().view(torch.int32) & ~0x1FFF
    return i.view(torch.float32).to(t.dtype)


def round_act(t: torch.Tensor, op: Optional[str]) -> torch.Tensor:
    """Rounding of an activation / gradient operand on its way to the MMA (op: 'fp16' | 'bf16' | 'tf32' | None)."""
    if op == "tf32":
        return round_tf32_tz(t)
    return R.round_operand(t, op)


def round_weight(t: torch.Tensor, op: Optional[str]) -> torch.Tensor:
    """Rounding of a packed weight operand (tc_pack_kernel / pack_s2_kernel: cvt.rn for 16-bit, cvt.rna for tf32)."""
    if op == "tf32":
        return round_tf32_rna(t)
    return R.round_operand(t, op)


def _taps(k: int):
    for kd in range(k):
        for kh in range(k):
            for kw in range(k):
                yield kd, kh, kw


def _pad(x: torch.Tensor, p: int) -> torch.Tensor:
    return F.pad(x, (0, 0, p, p, p, p, p, p)) if p else x


def conv_taps(x: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """Stride-1 'SAME' Conv3D, x [B,D,H,W,Ci], w [k,k,k,Ci,Co] (k odd) -> [B,D,H,W,Co], as fp64 GEMMs over taps."""
    k = w.shape[0]
    B, D, H, W, _ = x.shape
    xp = _pad(x.double(), k // 2)
    wd = w.double()
    y = torch.zeros(B, D, H, W, w.shape[4], dtype=torch.float64, device=x.device)
    for kd, kh, kw in _taps(k):
        y += xp[:, kd:kd + D, kh:kh + H, kw:kw + W, :] @ wd[kd, kh, kw]
    return y


def dgrad_taps(dy: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """Data gradient of the stride-1 conv: the conv of dy with the tap-reversed, channel-transposed kernel."""
    return conv_taps(dy, w.flip(0, 1, 2).transpose(3, 4))


def wgrad_taps(x: torch.Tensor, dy: torch.Tensor, k: int) -> torch.Tensor:
    """Weight gradient of the stride-1 conv: dw[tap] = pad(x)[. + tap]^T dy -> [k,k,k,Ci,Co] fp64."""
    B, D, H, W, ci = x.shape
    xp = _pad(x.double(), k // 2)
    d2 = dy.double().reshape(-1, dy.shape[-1])
    dw = torch.zeros(k, k, k, ci, dy.shape[-1], dtype=torch.float64, device=x.device)
    for kd, kh, kw in _taps(k):
        dw[kd, kh, kw] = xp[:, kd:kd + D, kh:kh + H, kw:kw + W, :].reshape(-1, ci).T @ d2
    return dw


def conv_s2_ref(x: torch.Tensor, w: torch.Tensor, transposed: bool) -> torch.Tensor:
    """Stride-2 family through the oracle's own restatement (small sizes only: vol2col)."""
    x, w = x.double().cpu(), w.double().cpu()
    return R.conv3d_transpose_same(x, w, None) if transposed else R.conv3d_same(x, w, None, 2)


def gn_chunk_sums(y: torch.Tensor, groups: int = 8) -> torch.Tensor:
    """fp64 (sum, sum of squares) per GroupNorm chunk (the g-th contiguous 1/G of a sample) -> [B, G, 2]."""
    c = y.double().reshape(y.shape[0], groups, -1)
    return torch.stack([c.sum(-1), (c * c).sum(-1)], dim=-1)


def gn_chunk_scale(y: torch.Tensor, groups: int = 8) -> torch.Tensor:
    """Scale of each chunk's sums: (sum |y|, sum y^2) — the bound of a correct fp32 reduction of them is relative to
    this, not to the (possibly cancelling) sum itself."""
    c = y.double().reshape(y.shape[0], groups, -1)
    return torch.stack([c.abs().sum(-1), (c * c).sum(-1)], dim=-1)


# --------------------------------------------------------------------------------------------------------- checker
def rel_l2(got: torch.Tensor, ref: torch.Tensor) -> float:
    r = ref.detach().double()
    g = got.detach().double().to(r.device)
    return float((g - r).norm() / (r.norm() + 1e-300))


class Check:
    """Result of `check`: rel-L2, the worst per-element error ratio (error / bound) and where it sits."""

    def __init__(self, what, rel, ratio, where, ok, msg):
        self.what, self.rel, self.ratio, self.where, self.ok, self.msg = what, rel, ratio, where, ok, msg

    def __repr__(self):
        return self.msg


def check(what: str, got: torch.Tensor, ref: torch.Tensor, A: Optional[torch.Tensor], n_acc: Optional[int],
          rel_tol: float, tile: Optional[Sequence[int]] = None, labels: str = "bdhwc") -> Check:
    """rel-L2(got, ref) <= rel_tol and, when A is given, every element within
    C_BOUND*(n_acc + 4)*2^-23*A + 2^-23*|ref|.  `tile` (TD, TH, TW, N): extent of one CTA output tile, to name the tile
    of the worst element in the message.  Evaluated on ref's device (a GPU reference is compared on the GPU)."""
    r = ref.detach().double()
    g = got.detach().double().to(r.device)
    assert g.shape == r.shape, (what, tuple(g.shape), tuple(r.shape))
    rel = rel_l2(g, r)
    err = (g - r).abs()
    if A is not None:
        bound = C_BOUND * (n_acc + 4) * U32 * A.detach().double().to(r.device) + U32 * r.abs() + 1e-300
        q = err / bound
    else:
        q = err / (r.abs().max() + 1e-300)
    finite = bool(torch.isfinite(g).all())
    flat = int(torch.argmax(torch.nan_to_num(q, nan=float("inf"))).item())
    idx = np.unravel_index(flat, tuple(g.shape))
    ratio = float(q.reshape(-1)[flat])
    where = dict(zip(labels, (int(i) for i in idx)))
    loc = ", ".join(f"{k}={v}" for k, v in where.items())
    if tile is not None and len(idx) == 5:
        td, th, tw, n = tile
        loc += f"; tile (b, d/{td}, h/{th}, w/{tw}, c/{n}) = ({idx[0]}, {idx[1] // td}, {idx[2] // th}, {idx[3] // tw}, " \
               f"{idx[4] // n})"
    ok = finite and rel <= rel_tol and (A is None or ratio <= 1.0)
    msg = (f"{what}: rel-L2 {rel:.2e} (<= {rel_tol:.0e}), worst element error/bound {ratio:.3f} at {loc} "
           f"(got {float(g.reshape(-1)[flat]):.8g}, ref {float(r.reshape(-1)[flat]):.8g})"
           + ("" if finite else "; NON-FINITE output"))
    return Check(what, rel, ratio, where, ok, msg)


def check_sums(what: str, got: torch.Tensor, ref: torch.Tensor, scale: torch.Tensor, tol: float = 1e-6) -> Check:
    """Reductions (GroupNorm chunk sums, pooling sums) against fp64 sums of the kernel's OWN output: every entry
    |got - ref| <= tol * scale (scale = the sum of magnitudes of the entry's terms)."""
    g, r, s = (t.detach().double().cpu() for t in (got, ref, scale))
    err = (g - r).abs() / (tol * s + 1e-300)
    flat = int(torch.argmax(torch.nan_to_num(err, nan=float("inf"))).item())
    idx = np.unravel_index(flat, tuple(g.shape))
    ratio = float(err.reshape(-1)[flat])
    ok = bool(torch.isfinite(g).all()) and ratio <= 1.0
    msg = (f"{what}: worst |got - ref| / ({tol:.0e} * sum|terms|) = {ratio:.3f} at index {tuple(int(i) for i in idx)} "
           f"(got {float(g.reshape(-1)[flat]):.10g}, ref {float(r.reshape(-1)[flat]):.10g})")
    return Check(what, rel_l2(g, r), ratio, dict(enumerate(int(i) for i in idx)), ok, msg)


def half_ulp(v: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """Half the spacing of `dtype` (torch.float16 | torch.bfloat16) numbers at |v|: the largest error of rounding v to
    nearest (subnormals included)."""
    mant, tiny = {torch.float16: (10, 2.0 ** -24), torch.bfloat16: (7, 2.0 ** -133)}[dtype]
    _, e = torch.frexp(v.double().abs())                   # |v| = m * 2^e, m in [0.5, 1)
    return torch.clamp(torch.ldexp(torch.ones_like(v, dtype=torch.float64), e - 1 - mant), min=tiny) * 0.5


def check_rounded(what: str, got: torch.Tensor, ref: torch.Tensor, dtype: torch.dtype, tol32: float = 1e-5,
                  labels: str = "bdhwc") -> Check:
    """A 16-bit output that exists only in its rounded form (a P16 twin written without its fp32 tensor), unpacked to
    fp32, against the fp64 reference: every element within half a `dtype` ulp (at the larger of |got|, |ref|) plus
    tol32 * max|ref| for the fp32 evaluation that was rounded.  A value taken from a neighbouring cell or chunk misses
    this bound by orders of magnitude."""
    r = ref.detach().double()
    g = got.detach().double().to(r.device)
    assert g.shape == r.shape, (what, tuple(g.shape), tuple(r.shape))
    bound = half_ulp(torch.maximum(g.abs(), r.abs()), dtype) + tol32 * float(r.abs().max()) + 1e-300
    q = (g - r).abs() / bound
    flat = int(torch.argmax(torch.nan_to_num(q, nan=float("inf"))).item())
    idx = np.unravel_index(flat, tuple(g.shape))
    ratio = float(q.reshape(-1)[flat])
    where = dict(zip(labels, (int(i) for i in idx)))
    ok = bool(torch.isfinite(g).all()) and ratio <= 1.0
    msg = (f"{what}: worst |got - ref| / (half {str(dtype)[6:]} ulp + {tol32:.0e} max|ref|) = {ratio:.3f} at "
           + ", ".join(f"{k}={v}" for k, v in where.items())
           + f" (got {float(g.reshape(-1)[flat]):.8g}, ref {float(r.reshape(-1)[flat]):.8g})")
    return Check(what, rel_l2(g, r), ratio, where, ok, msg)
