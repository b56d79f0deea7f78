"""GPU suite — the P16 operand-twin path (csrc/p16.cu, DESIGN.md section 3): 16-bit [B, D, H, C/8, W, 8] copies of conv
operands written by their producers and consumed by the tcgen05 convs through TMA, with channel concatenation as a
list of sources.  Every P16 entry point must reproduce its fp32-operand twin: the rounding points are identical (the
fp32 entry points convert the same values to the same 16-bit type inside their loaders / cast passes), so the
comparisons are tight (summation order only)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def rnd(*shape, seed=0, scale=1.0, dev=None):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dev)


def to_p16_ref(x, dtype):
    """[B,D,H,W,C] fp32 -> [B,D,H,C/8,W,8] by torch ops (reference for the layout)."""
    B, D, H, W, C = x.shape
    return x.reshape(B, D, H, W, C // 8, 8).permute(0, 1, 2, 4, 3, 5).contiguous().to(dtype)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("shape", [(1, 4, 6, 8, 16), (2, 3, 5, 7, 64), (1, 2, 2, 9, 8)])
def test_pack_unpack_layout(b3d, dev, dtype, shape):
    ops = b3d.ops
    x = rnd(*shape, seed=1, dev=dev)
    cs = torch.empty(shape[-1], device=dev)
    t = ops.p16_empty(shape, x, dtype)
    ops._call("b3d_p16_pack", x, t, cs)
    assert torch.equal(t, to_p16_ref(x, dtype))
    assert rel(cs, x.sum(dim=(0, 1, 2, 3))) < 1e-5
    y = torch.empty_like(x)
    ops._call("b3d_p16_unpack", t, y)
    assert torch.equal(y, x.to(dtype).float())
    # channel-sliced source / destination (pitch)
    wide = rnd(*shape[:-1], shape[-1] + 16, seed=2, dev=dev)
    ops._call("b3d_p16_pack", wide[..., 8:8 + shape[-1]], t, None)
    assert torch.equal(t, to_p16_ref(wide[..., 8:8 + shape[-1]].contiguous(), dtype))
    out = torch.zeros_like(wide)
    ops._call("b3d_p16_unpack", t, out[..., 8:8 + shape[-1]])
    assert torch.equal(out[..., 8:8 + shape[-1]], wide[..., 8:8 + shape[-1]].to(dtype).float())
    assert float(out[..., :8].abs().max()) == 0 and float(out[..., 8 + shape[-1]:].abs().max()) == 0


CONV_CASES = [
    # spatial, source channels, Cout, k, stride, transposed
    ((8, 16, 8), [16], 16, 3, 1, False),
    ((9, 17, 11), [32], 16, 3, 1, False),            # partial tiles, kd-folded N=16
    ((8, 16, 16), [16, 16], 32, 3, 1, False),        # virtual concat, kd-folded N=32
    ((4, 16, 16), [32, 64], 64, 3, 1, False),
    ((4, 8, 8), [64, 64, 128, 128], 128, 3, 1, False),
    ((6, 10, 12), [32, 16], 16, 1, 1, False),        # pointwise
    ((8, 16, 16), [16], 16, 3, 2, False),            # strided: space-to-depth loader reads P16 cells
    ((8, 8, 16), [32, 32], 32, 3, 2, False),
    ((4, 8, 8), [32], 16, 3, 2, True),               # transposed
    ((4, 4, 8), [64, 64], 32, 3, 2, True),
    # weight gradients over several channel tiles and sources: Cin 48 on the per-tap kernel (conv3_wgrad_tc_kernel),
    # Cin 16 / 64 / 96 with the depth taps folded into M
    ((8, 16, 8), [16], 32, 3, 1, False),
    ((6, 10, 24), [48], 16, 3, 1, False),            # 432 accumulator columns, partial tiles in d and h
    ((8, 8, 16), [64], 32, 3, 1, False),             # N' = 192, one pair per CTA
    ((4, 8, 16), [32, 32, 32], 32, 3, 1, False),     # three sources, 288 columns
    ((4, 6, 8), [16, 32], 16, 3, 1, False),          # unequal sources
    # weight gradient with the depth taps folded into M (conv3_wgrad_kdf_kernel): Cin 16 (M = 64) | 32 (M = 128),
    # Cout 16 | 32; the 64-channel cases stay on the per-tap kernel
    ((5, 6, 24), [16], 32, 3, 1, False),             # M = 64, partial tiles
    ((9, 10, 8), [16], 16, 3, 1, False),             # M = 64, partial tiles in d and h
    ((8, 16, 16), [32], 32, 3, 1, False),
    ((5, 6, 24), [16, 16], 16, 3, 1, False),         # two sources inside one channel tile, partial tiles
    ((4, 8, 8), [32, 32], 32, 3, 1, False),          # two channel tiles
    ((6, 10, 16), [16, 32, 16], 16, 3, 1, False),    # a source straddling the tiles
]


@pytest.mark.parametrize("case", CONV_CASES)
@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_conv_forward_p16_equals_fp32_operand_path(b3d, dev, case, prec):
    sp, cs, cout, k, stride, tr = case
    ops = b3d.ops
    ops.set_conv_precision(prec, "bf16")
    try:
        dt = torch.float16 if prec == "fp16" else torch.bfloat16
        xs = [rnd(2, *sp, c, seed=10 + i, dev=dev) for i, c in enumerate(cs)]
        x = torch.cat(xs, dim=-1).contiguous()
        cin = sum(cs)
        w = rnd(k, k, k, *((cout, cin) if tr else (cin, cout)), seed=3, scale=0.1, dev=dev)
        bias = rnd(cout, seed=4, dev=dev)
        od = tuple(2 * n for n in sp) if tr else tuple(n // stride for n in sp)
        S = od[0] * od[1] * od[2]
        want_stats = S % 8 == 0
        wp = ops.pack_weights(w, False, stride, tr)
        res = []
        for p16 in (False, True):
            y = torch.empty(2, *od, cout, device=dev)
            stats = torch.empty(2, 8, 2, dtype=torch.float64, device=dev) if want_stats else None
            gap = torch.empty(2, cout, device=dev) if stride == 1 else None
            if p16:
                tw = [ops.to_p16(t, dt) for t in xs]
                ops._call("b3d_conv3d_fwd_p16", *(tw + [None] * (4 - len(tw))), w, bias, y, stride, int(tr), 0, stats, 8,
                          gap, 0, wp)
            else:
                ops._call("b3d_conv3d_fwd", x, w, bias, y, stride, int(tr), 0, stats, 8, gap, 0, wp)
            res.append((y, stats, gap))
        torch.cuda.synchronize()
        assert rel(res[1][0], res[0][0]) < 2e-6, rel(res[1][0], res[0][0])
        if want_stats:
            assert rel(res[1][1], res[0][1]) < 1e-6
        if stride == 1:
            assert rel(res[1][2], res[0][2]) < 1e-5
    finally:
        ops.set_conv_precision("fp16", "bf16")


@pytest.mark.parametrize("case", [c for c in CONV_CASES if len(c[1]) == 1 or True])
def test_conv_backward_p16_equals_fp32_operand_path(b3d, dev, case):
    """Data gradient from a bf16 twin of dy, weight gradient from bf16 twins of x (one or several sources) and dy —
    against the fp32 entry points (which cast to bf16 themselves) and a fp64 reference with the same roundings.
    (tcgen05 kind::f16 takes ONE operand type for A and B: feeding the fp16 forward twin next to a bf16 dy is an illegal
    instruction on sm_100a, which is why forward activations carry a second, bf16 twin.)"""
    sp, cs, cout, k, stride, tr = case
    ops = b3d.ops
    lib = b3d._lib.lib
    xs = [rnd(2, *sp, c, seed=20 + i, dev=dev) for i, c in enumerate(cs)]
    x = torch.cat(xs, dim=-1).contiguous()
    cin = sum(cs)
    w = rnd(k, k, k, *((cout, cin) if tr else (cin, cout)), seed=5, scale=0.1, dev=dev)
    od = tuple(2 * n for n in sp) if tr else tuple(n // stride for n in sp)
    dy = rnd(2, *od, cout, seed=6, dev=dev)
    wpd = ops.pack_weights(w, True, stride, tr)
    dx0, dx1 = torch.empty_like(x), torch.empty_like(x)
    ops._call("b3d_conv3d_dgrad", dy, w, dx0, stride, int(tr), 0, wpd)
    db = torch.empty(cout, device=dev)
    dy16 = ops.to_p16(dy, torch.bfloat16, db)
    ops._call("b3d_conv3d_dgrad_p16", dy16, w, dx1, stride, int(tr), 0, wpd)
    assert rel(dx1, dx0) < 2e-6, rel(dx1, dx0)
    assert rel(db, dy.sum(dim=(0, 1, 2, 3))) < 1e-5
    # weight gradient
    import ctypes
    xc, yc = ctypes.c_longlong(), ctypes.c_longlong()
    kind = lib.b3d_conv3d_wgrad_plan(k, stride, int(tr), cin, cout, ctypes.byref(xc), ctypes.byref(yc))
    assert kind == 1
    nvx, nvy = x.numel() // cin, dy.numel() // cout
    xb = torch.empty(nvx * xc.value, device=dev, dtype=torch.bfloat16)
    yb = torch.empty(nvy * yc.value, device=dev, dtype=torch.bfloat16)
    dw0, dw1 = torch.empty_like(w), torch.empty_like(w)
    ops._call("b3d_conv3d_wgrad", x, dy, dw0, None, stride, int(tr), xb, yb, 0)
    plan = lib.b3d_conv3d_wgrad_p16_plan(k, stride, int(tr), cin, cout, od[2])
    assert plan in (1, 2, 3)
    tw = [ops.to_p16(t, torch.bfloat16) for t in xs]
    if tr:
        tw = [ops._p16_cat(tw)]
    scratch = None
    if plan == 2:
        scratch = torch.empty(dy16.numel() if tr else sum(t.numel() for t in tw), device=dev, dtype=torch.bfloat16)
    elif plan == 3:
        scratch = torch.empty(dy16.numel(), device=dev, dtype=torch.bfloat16)
    ops._call("b3d_conv3d_wgrad_p16", *(tw + [None] * (4 - len(tw))), dy16, dw1, stride, int(tr), scratch)
    torch.cuda.synchronize()
    # exact reference with the same roundings (x, dy -> bf16) in fp64
    xr, dyr = x.bfloat16().double(), dy.bfloat16().double()
    e_legacy, e = rel(dw0, _dw_ref(xr, dyr, k, stride, tr)), rel(dw1, _dw_ref(xr, dyr, k, stride, tr))
    print(f"wgrad {case}: plan {plan}, P16 vs rounded fp64 reference {e:.2e} (fp32-operand path: {e_legacy:.2e})")
    assert e < 2e-5 and rel(dw1, dw0) < 2e-5, (e, rel(dw1, dw0))


@pytest.mark.parametrize("case", [((8, 16, 8), [16], 16), ((9, 17, 11), [32], 16), ((8, 16, 16), [16, 16], 32),
                                  ((4, 16, 16), [32, 64], 64), ((4, 8, 8), [64, 64, 128], 128), ((6, 10, 12), [48], 32)])
def test_block_input_data_gradient_in_one_kernel(b3d, dev, case):
    """b3d_conv3d_dgrad_p16_block: d/dx of conv3x3x3(x, w) and of conv1x1x1(x, w_pw) in ONE launch — the pointwise conv's
    incoming gradient is a further K segment used at the centre tap only — written as one compact tensor per piece of a
    virtually concatenated input; against the two separate data gradients (same operand roundings) and their split form."""
    sp, pieces, cb = case
    ops = b3d.ops
    cin = sum(pieces)
    w = rnd(3, 3, 3, cin, cb, seed=5, scale=0.1, dev=dev)
    wpw = rnd(1, 1, 1, cin, cb, seed=6, scale=0.3, dev=dev)
    dy, dres = rnd(2, *sp, cb, seed=7, dev=dev), rnd(2, *sp, cb, seed=8, dev=dev)
    dy16, dres16 = ops.to_p16(dy, torch.bfloat16), ops.to_p16(dres, torch.bfloat16)
    wp, wpp = ops.pack_weights(w, True, 1, False), ops.pack_weights(wpw, True, 1, False)
    ref = torch.empty(2, *sp, cin, device=dev)
    ops._call("b3d_conv3d_dgrad_p16", dy16, w, ref, 1, 0, 0, wp)
    ops._call("b3d_conv3d_dgrad_p16", dres16, wpw, ref, 1, 0, 1, wpp)            # accumulate = 1
    outs = [torch.full((2,) + tuple(sp) + (c,), float("nan"), device=dev) for c in pieces]
    ops._call("b3d_conv3d_dgrad_p16_block", dy16, dres16, w, wpw, *(outs + [None] * (4 - len(outs))), wp, wpp)
    got = torch.cat(outs, dim=-1)
    assert rel(got, ref) < 2e-6, rel(got, ref)
    # the split form of the plain data gradient (no pointwise part)
    ref3 = torch.empty(2, *sp, cin, device=dev)
    ops._call("b3d_conv3d_dgrad_p16", dy16, w, ref3, 1, 0, 0, wp)
    outs3 = [torch.full((2,) + tuple(sp) + (c,), float("nan"), device=dev) for c in pieces]
    ops._call("b3d_conv3d_dgrad_p16_split", dy16, w, *(outs3 + [None] * (4 - len(outs3))), 0, wp)
    assert rel(torch.cat(outs3, dim=-1), ref3) < 2e-6


@pytest.mark.parametrize("case", [((8, 16, 8), [16], 16), ((9, 10, 24), [32], 16), ((8, 16, 16), [16, 16], 32),
                                  ((4, 16, 16), [32, 64], 32), ((5, 6, 16), [16], 32), ((4, 8, 8), [64, 32, 32], 16)])
def test_block_weight_gradients_in_one_kernel(b3d, dev, case):
    """b3d_conv3d_wgrad_p16_block: dw of conv3x3x3(x, .) and of conv1x1x1(x, .) in ONE launch of the kd-in-M kernel (the
    pointwise layer is one more MMA per K step over the x tile in shared memory) against the two separate weight
    gradients from the same bf16 operands (same products, different summation order) and against fp64."""
    sp, pieces, cb = case
    ops = b3d.ops
    cin = sum(pieces)
    assert b3d._lib.lib.b3d_conv3d_wgrad_p16_block_ok(cin, cb, sp[1], sp[2]) == 1
    xs = [rnd(2, *sp, c, seed=11 + i, dev=dev) for i, c in enumerate(pieces)]
    xs16 = [ops.to_p16(t, torch.bfloat16) for t in xs]
    dy, dres = rnd(2, *sp, cb, seed=7, dev=dev), rnd(2, *sp, cb, seed=8, dev=dev)
    dy16, dres16 = ops.to_p16(dy, torch.bfloat16), ops.to_p16(dres, torch.bfloat16)
    pad = xs16 + [None] * (4 - len(xs16))
    ref3, ref1 = torch.empty(3, 3, 3, cin, cb, device=dev), torch.empty(1, 1, 1, cin, cb, device=dev)
    plan = b3d._lib.lib.b3d_conv3d_wgrad_p16_plan(3, 1, 0, cin, cb, sp[2])
    scratch = torch.empty(dy16.numel(), device=dev, dtype=torch.bfloat16) if plan == 3 else None
    ops._call("b3d_conv3d_wgrad_p16", *pad, dy16, ref3, 1, 0, scratch)
    ops._call("b3d_conv3d_wgrad_p16", *pad, dres16, ref1, 1, 0, None)
    dw3 = torch.full_like(ref3, float("nan"))
    dw1 = torch.full_like(ref1, float("nan"))
    ops._call("b3d_conv3d_wgrad_p16_block", *pad, dy16, dres16, dw3, dw1)
    assert rel(dw3, ref3) < 2e-6, rel(dw3, ref3)
    assert rel(dw1, ref1) < 2e-6, rel(dw1, ref1)
    # fp64 reference from the bf16-rounded operands
    xr = torch.cat([t.bfloat16().float() for t in xs], dim=-1)
    e1 = torch.einsum("bdhwi,bdhwo->io", xr.double(), dres.bfloat16().double())
    assert rel(dw1[0, 0, 0].double(), e1) < 1e-5
    assert rel(dw3.double().cpu(), _dw_ref(xr.double(), dy.bfloat16().double(), 3, 1, False)) < 1e-5
    # a layer off the kd-in-M path is refused, not mis-computed
    assert b3d._lib.lib.b3d_conv3d_wgrad_p16_block_ok(256, 64, 32, 32) == 0


def _dw_ref(x, dy, k, stride, tr):
    """fp64 weight gradient by autograd of the oracle's conv restatement."""
    from oracle import ref_model as R
    cin, cout = x.shape[-1], dy.shape[-1]
    w = torch.zeros(k, k, k, *((cout, cin) if tr else (cin, cout)), dtype=torch.float64, requires_grad=True)
    xc = x.cpu()
    y = R.conv3d_transpose_same(xc, w, None) if tr else R.conv3d_same(xc, w, None, stride)
    return torch.autograd.grad(y, w, dy.cpu())[0]


@pytest.mark.parametrize("shape", [(2, 8, 8, 8, 16), (1, 4, 6, 10, 32), (1, 8, 4, 4, 128)])
@pytest.mark.parametrize("relu", [False, True])
def test_group_norm_twin_outputs(b3d, dev, shape, relu):
    ops = b3d.ops
    x = rnd(*shape, seed=1, dev=dev)
    ga, be = 1 + 0.3 * rnd(shape[-1], seed=2, dev=dev), 0.3 * rnd(shape[-1], seed=3, dev=dev)
    stats = torch.empty(shape[0], 8, 2, dtype=torch.float64, device=dev)
    ops._call("b3d_gn_stats", x, stats, 8, 0, 0)
    y0, y1 = torch.empty_like(x), torch.empty_like(x)
    ops._call("b3d_gn_apply", x, stats, ga, be, y0, None, None, 8, 1e-5, int(relu), 0, 0)
    y16 = ops.p16_empty(shape, x, torch.float16)
    yw = ops.p16_empty(shape, x, torch.bfloat16)
    ops._call("b3d_gn_apply", x, stats, ga, be, y1, y16, yw, 8, 1e-5, int(relu), 0, 0)
    # separate kernels (one 16-byte cell per thread): same formula, fused-multiply-add grouping may differ in the last bit
    assert rel(y1, y0) < 1e-6 and torch.equal(y16, to_p16_ref(y1, torch.float16))
    assert torch.equal(yw, to_p16_ref(y1, torch.bfloat16))
    y16b = ops.p16_empty(shape, x, torch.float16)
    ops._call("b3d_gn_apply", x, stats, ga, be, None, y16b, None, 8, 1e-5, int(relu), 0, 0)     # one twin only
    assert torch.equal(y16b, y16)
    # backward
    dy = rnd(*shape, seed=4, dev=dev)
    dga, dbe, csum = torch.empty_like(ga), torch.empty_like(be), torch.empty_like(stats)
    ops._call("b3d_gn_bwd_reduce", dy, x, stats, ga, be, dga, dbe, csum, 8, 1e-5, int(relu))
    dx0, dx1 = torch.empty_like(x), torch.empty_like(x)
    ops._call("b3d_gn_bwd_apply", dy, x, stats, ga, be, csum, dx0, None, None, 8, 1e-5, int(relu))
    dx16 = ops.p16_empty(shape, x, torch.bfloat16)
    db = torch.empty(shape[-1], device=dev)
    ops._call("b3d_gn_bwd_apply", dy, x, stats, ga, be, csum, dx1, dx16, db, 8, 1e-5, int(relu))
    assert rel(dx1, dx0) < 1e-6 and torch.equal(dx16, to_p16_ref(dx1, torch.bfloat16))
    ref = dx0.double().sum(dim=(0, 1, 2, 3))
    assert float((db.double() - ref).abs().max()) < 1e-4 * float(dx0.abs().sum(dim=(0, 1, 2, 3)).max()) + 1e-6


@pytest.mark.parametrize("shape", [(2, 8, 8, 8, 16), (1, 4, 6, 8, 32), (1, 4, 4, 4, 128)])
def test_block_epilogue_twin_outputs(b3d, dev, shape):
    ops = b3d.ops
    F = shape[-1]
    res, h2 = rnd(*shape, seed=1, dev=dev), rnd(*shape, seed=2, dev=dev)
    ga, be = 1 + 0.3 * rnd(F, seed=3, dev=dev), 0.3 * rnd(F, seed=4, dev=dev)
    wsp, chse = 0.3 * rnd(F, seed=5, dev=dev), torch.sigmoid(rnd(shape[0], F, seed=6, dev=dev))
    stats = torch.empty(shape[0], 8, 2, dtype=torch.float64, device=dev)
    ops._call("b3d_gn_stats", h2, stats, 8, 0, 0)
    o0, o1 = torch.empty_like(res), torch.empty_like(res)
    ops._call("b3d_block_epilogue_fwd", res, h2, stats, ga, be, wsp, chse, o0, None, None, 8, 1e-5, 1, 0, 0)
    o16 = ops.p16_empty(shape, res, torch.float16)
    ow = ops.p16_empty(shape, res, torch.bfloat16)
    ops._call("b3d_block_epilogue_fwd", res, h2, stats, ga, be, wsp, chse, o1, o16, ow, 8, 1e-5, 1, 0, 0)
    assert rel(o1, o0) < 1e-6 and torch.equal(o16, to_p16_ref(o1, torch.float16))
    assert torch.equal(ow, to_p16_ref(o1, torch.bfloat16))
    o16b = ops.p16_empty(shape, res, torch.float16)
    ops._call("b3d_block_epilogue_fwd", res, h2, stats, ga, be, wsp, chse, None, o16b, None, 8, 1e-5, 1, 0, 0)
    assert torch.equal(o16b, o16)
    # backward apply
    dout = rnd(*shape, seed=7, dev=dev)
    dgap = 0.01 * rnd(shape[0], F, seed=8, dev=dev)
    dch, dws = torch.empty(shape[0], F, device=dev), torch.empty(F, device=dev)
    dga, dbe, csum = torch.empty_like(ga), torch.empty_like(be), torch.empty_like(stats)
    ops._call("b3d_block_epilogue_bwd_reduce", dout, res, h2, stats, ga, be, wsp, dch, dws, dga, dbe, csum, 8, 1e-5, 1)
    dr0, dh0 = torch.empty_like(res), torch.empty_like(res)
    ops._call("b3d_block_epilogue_bwd_apply", dout, res, h2, stats, ga, be, wsp, chse, dgap, csum, dr0, dh0, None, None,
              None, None, 8, 1e-5, 1)
    dr16, dh16 = ops.p16_empty(shape, res, torch.bfloat16), ops.p16_empty(shape, res, torch.bfloat16)
    dbr, dbh = torch.empty(F, device=dev), torch.empty(F, device=dev)
    dr1, dh1 = torch.empty_like(res), torch.empty_like(res)
    ops._call("b3d_block_epilogue_bwd_apply", dout, res, h2, stats, ga, be, wsp, chse, dgap, csum, dr1, dh1, dr16,
              dh16, dbr, dbh, 8, 1e-5, 1)
    assert rel(dr1, dr0) < 1e-6 and rel(dh1, dh0) < 1e-6
    assert torch.equal(dr16, to_p16_ref(dr1, torch.bfloat16)) and torch.equal(dh16, to_p16_ref(dh1, torch.bfloat16))
    dr16b, dh16b = ops.p16_empty(shape, res, torch.bfloat16), ops.p16_empty(shape, res, torch.bfloat16)
    ops._call("b3d_block_epilogue_bwd_apply", dout, res, h2, stats, ga, be, wsp, chse, dgap, csum, None, None, dr16b,
              dh16b, None, None, 8, 1e-5, 1)                                        # twins only, no bias gradients
    assert torch.equal(dr16b, dr16) and torch.equal(dh16b, dh16)
    for got, full in ((dbr, dr0), (dbh, dh0)):
        ref = full.double().sum(dim=(0, 1, 2, 3))
        assert float((got.double() - ref).abs().max()) < 1e-4 * float(full.abs().sum(dim=(0, 1, 2, 3)).max()) + 1e-6


def test_train_step_with_and_without_twins(b3d, dev):
    """The whole training step with operand twins (default) against the fp32-operand path (ops.P16 off): the rounding
    points are the same (fp16 forward operands, bf16 gradient operands), so losses, outputs and gradients agree to
    summation order — except the few bias gradients that are now column sums taken in the producing kernel."""
    from oracle import ref_model as R
    crop = (64, 64, 64)          # at 32^3 the VAE bottleneck normalises groups of 8 values: any last-bit change is amplified
    p = R.init_params(R.param_shapes(crop=crop), dtype=torch.float32)
    x, y, eps, mask = R.synth_batch((1,) + crop, dtype=torch.float32)
    f = lambda t: t.to(dev)
    out = []
    for on in (False, True):
        b3d.ops.P16["on"] = on
        try:
            model = b3d.Model()
            with torch.no_grad():
                model(torch.zeros((1,) + crop + (2,), device=dev), training=False, inference=False)
            model.load_named_weights(p)
            n0 = b3d.ops.LAUNCHES["n"]
            with b3d.GradientTape() as tape:
                outs = model(f(x), training=True, inference=False, dropout_mask=f(mask), eps=f(eps))
                loss = b3d.DiceVAELoss()(f(x), f(y), *outs) + b3d.reduce_sum(model.losses)
            tape.gradient(loss, model.trainable_variables, direct=True)
            torch.cuda.synchronize()
            out.append((float(loss), [o.clone() for o in outs], model.flat.grad.clone(), b3d.ops.LAUNCHES["n"] - n0))
        finally:
            b3d.ops.P16["on"] = True
    (l0, o0, g0, n0), (l1, o1, g1, n1) = out
    print(f"loss {l0:.6f} / {l1:.6f}; ABI calls per step {n0} -> {n1}; flat gradient rel {rel(g1, g0):.2e}")
    # same rounding points, different summation order of the GroupNorm statistics: values next to a rounding boundary
    # flip, so agreement is at the operand-rounding level divided by sqrt(#terms), not at fp32 epsilon
    a, b = g1.double().flatten(), g0.double().flatten()
    cosine = float((a @ b) / (a.norm() * b.norm()))
    print(f"outputs rel {[f'{rel(u, v):.1e}' for u, v in zip(o1, o0)]}; flat-gradient cosine {cosine:.5f}")
    # (north_star's loss tolerance against the reference is 1e-3; between the two operand paths 0.3-1.1e-4 is measured,
    # the same size as the run-to-run spread of ONE path: profiles/r02e_parity_spread.txt)
    assert abs(l1 - l0) / abs(l0) < 3e-4
    assert rel(o1[0], o0[0]) < 1e-3 and rel(o1[1], o0[1]) < 4e-3
    assert cosine > 0.995
    assert n1 < n0                       # no cast passes, no concat copies
