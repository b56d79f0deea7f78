"""GPU suite — every conv kernel path and the GroupNorm / block reductions at the model's shapes, against fp64
references that round the operands the way the kernels do (oracle/kernel_ref.py).

Tolerance rule.  With the operands rounded as the MMAs see them, a correct kernel differs from the fp64 reference only by
its fp32 summation order, so each output is held to
  * rel-L2 <= 1e-5 (weight gradients, which sum over every voxel: 2e-5), and
  * per element |got - ref| <= c*(n_acc + 4)*2^-23*A + 2^-23*|ref|, with A the same sum over |operands| and n_acc the
    sequential fp32 accumulations of one output (K steps of the MMA, split-K slices, bias); c: kernel_ref.C_BOUND.
A localised fault (a tile, a K chunk, a tap) fails the second bound even where it hardly moves the first.  Reductions
fused into a kernel (GroupNorm chunk statistics, pooling sums) are checked against fp64 sums of the kernel's OWN output
at 1e-6 of the sum of magnitudes, which separates them from the conv's rounding.

Every case names the kernel it is meant to reach, and the profiler confirms it: `expect_conv` / `expect_wgrad` restate
the host heuristics (N tile, kd folding, operand type, split-K, weight-gradient plan), so a changed heuristic fails here
instead of silently moving a case onto another path.  The quick forward / data-gradient cases run once more with kd
folding off (`ops.set_kd_fold(False)`, ids ending in `-kd_fold_off`).  Ids containing `large` are the real-size cases;
`-k "not large"` is the quick subset.

GroupNorm (chunk and channel form) and the block epilogue are checked output by output against fp64 at the model's
shapes; the depth-slab forms on the windows sharded inference produces, against fp64 of the whole volume sliced, with
their P16 twins held to the rounding of the fp32 values they were stored from (`test_slab_window_kernels`)."""
import contextlib
import math
import re

import pytest
import torch

from oracle import kernel_ref as K
from oracle import ref_model as R

pytestmark = pytest.mark.gpu

OPCODE = {"tf32": 0, "bf16": 1, "fp16": 2}
TWIN = {"fp16": torch.float16, "bf16": torch.bfloat16}
SEEN = []          # (case id, kernel names, worst per-element ratio, worst rel-L2): printed with -s


# ------------------------------------------------------------------------------------------------ fixtures / helpers
@pytest.fixture(scope="module")
def env(b3d, dev):
    b3d.ops.set_conv_precision("fp16", "bf16")
    yield b3d
    b3d.ops.set_conv_precision("fp16", "bf16")
    b3d._lib.lib.b3d_set_wgrad_ts(1)


@pytest.fixture
def kd_fold(env, request):
    """The kd-folding setting of the case (indirect parameter); the previous one is restored afterwards."""
    prev = env.ops.set_kd_fold(request.param)
    yield request.param
    env.ops.set_kd_fold(prev)


def with_fold_off(cases):
    """(case, kd_fold) parameters: every case with kd folding on, the quick ones once more with it off."""
    return ([pytest.param(c, True, id=c[0]) for c in cases] +
            [pytest.param(c, False, id=c[0] + "-kd_fold_off") for c in cases if "large" not in c[0]])


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def rnd(*shape, seed=0, scale=1.0, mean=0.0, dev="cuda"):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale + mean).to(dev)


def run_profiled(fn, repeatable=True):
    """Run fn under torch.profiler (CUDA activities) and return (its result, the names of the CUDA kernels it ran).
    On a shared device CUPTI occasionally delivers no activity at all for a short profiled region; a trace without a
    single CUDA event is then taken once more, if fn may run twice (`repeatable`: False for calls that accumulate into
    their outputs)."""
    from torch.profiler import ProfilerActivity, profile
    for attempt in range(2 if repeatable else 1):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        names = []
        try:
            for e in prof.profiler.kineto_results.events():
                if "cuda" in str(e.device_type()).lower():
                    names.append(e.name())
        except AttributeError:
            names = [e.name for e in prof.events() if "cuda" in str(e.device_type).lower()]
        if names:
            break
        print("    torch.profiler recorded no CUDA activity" + ("; profiling the call again" if repeatable and not attempt
                                                               else ""))
    kernels = [n for n in names if "kernel" in n]
    assert kernels, ("torch.profiler recorded no CUDA kernel for this case (CUPTI unavailable?): the kernel path "
                     f"cannot be verified; events seen: {names[:10]}")
    return out, kernels


TCFG = re.compile(r"TcCfg<(\d+), ?(\d+), ?(\d+), ?(\d+), ?(\d+), ?(\d+)(?:, ?(\d+))?\s*>")


def tc_cfgs(kernels):
    """(N, TD, NW, KS, HB, OP, FOLD) of every conv_tc_kernel launch in the list."""
    out = []
    for n in kernels:
        m = TCFG.search(n)
        if m and "conv_tc_kernel" in n:
            out.append(tuple(int(v) if v is not None else 0 for v in m.groups()))
    return out


def has(kernels, name):
    return any(name in n for n in kernels)


def record(case, kernels, checks):
    ratios = [c.ratio for c in checks if c.ratio is not None]
    SEEN.append((case, sorted(set(kernels)), max(ratios) if ratios else None, max(c.rel for c in checks)))
    print(f"[path] {case}: {sorted(set(kernels))} worst ratio {max(ratios) if ratios else float('nan'):.3f} "
          f"worst rel {max(c.rel for c in checks):.2e}")
    for c in checks:
        print("   ", c)
        assert c.ok, c


# ------------------------------------------------------------------------------------------- the host heuristics
def pick_n(c):
    return 128 if c % 128 == 0 else 64 if c % 64 == 0 else 32 if c % 32 == 0 else 16


def pad(c, m):
    return (c + m - 1) // m * m


def expect_conv(mode, k, gcin, gcout, op, B, out_sp, *, act=0, accumulate=0, contiguous=True, nyd=1, stats=False,
                stat_total=0, fold=True):
    """Kernel configuration the host picks (csrc/conv_tc.cu operand_type / pick_n / use_fold / dispatch_n and the
    split-K rule of launch_cfg) for a conv pass in gather terms: gcin = channels read, gcout = channels written.
    mode: 's1' | 'down' (space-to-depth) | 'up' (depth-to-space); fold = ops.set_kd_fold.  Returns (TcCfg tuple,
    split-K?, operand type)."""
    if not (op != "tf32" and (gcin % 16 == 0 or (mode == "s1" and gcin < 8))):
        op = "tf32"
    ck = 8 if op == "tf32" else 16
    Do, Ho, Wo = out_sp
    if mode == "s1":
        ks, hb, qcin, qcout, qd = k, k // 2, pad(gcin, ck), pad(gcout, 16), (Do, Ho, Wo)
    elif mode == "down":
        ks, hb, qcin, qcout, qd = 2, 0, 8 * gcin, pad(gcout, 16), (Do, Ho, Wo)
    else:
        ks, hb, qcin, qcout, qd = 2, 1, gcin, 8 * gcout, (Do // 2, Ho // 2, Wo // 2)
    n = pick_n(qcout)
    fold = fold and mode == "s1" and k == 3 and op != "tf32" and n in (16, 32)
    if fold:
        cfg = (n, 8 if n == 16 else 4, 1, 3, 1, OPCODE[op], 1)
    else:
        td, nw = {128: (2, 1), 64: (2, 2), 32: (4, 2), 16: (4, 2)}[n]
        cfg = (n, td, nw, ks, hb, OPCODE[op], 0)
    N, TD, NW = cfg[0], cfg[1], cfg[2]
    ntiles = B * -(-qd[0] // TD) * -(-qd[1] // 16) * -(-qd[2] // (8 * NW))
    SM = sm_count()
    nsplit = qcout // N
    gx = min(ntiles, SM)
    if nsplit > 1:
        gx = -(-gx // nsplit)
    ctas, nchunks = gx * nsplit, qcin // ck
    S = Do * Ho * Wo
    out_elems = B * S * gcout
    split = False
    if (ctas * 2 <= SM and nchunks >= 8 and act == 0 and not accumulate and gcout % 16 == 0 and contiguous and nyd <= 1
            and (S * gcout) % 32 == 0 and (not stats or S % 8 == 0)
            and (not stats or stat_total == 0 or (B == 1 and (stat_total * gcout) % 32 == 0))):
        ks_ = min(SM // ctas, nchunks // 4, 8)
        while ks_ >= 2 and ks_ * out_elems > (16 << 20):
            ks_ -= 1
        split = ks_ >= 2
    return cfg, split, op


def expect_wgrad(pieces, cout, H, W, ts=True):
    """Weight-gradient kernel of a stride-1 3x3x3 layer on the P16 path (conv_abi.cu b3d_conv3d_wgrad_p16,
    conv_tc_wgrad.cu tc_wgrad_kdf_supported, conv_tc_wgrad_ts.cu; ts = b3d_set_wgrad_ts): 'kdf' | 'ts' | 'tc',
    and the plan b3d_conv3d_wgrad_p16_plan reports (3: a scratch for the TS kernel, else 1)."""
    cin = sum(pieces)
    ts_ok = ts and cin == 16 and cout in (16, 32) and W % 8 == 0
    plan = 3 if ts_ok else 1
    if cin in (16, 32, 64, 96, 128) and cout in (16, 32) and W % 8 == 0 and H % 2 == 0:
        return "kdf", plan
    if ts_ok and len(pieces) == 1:
        return "ts", plan
    return "tc", plan


WGRAD_KERNEL = {"kdf": "conv3_wgrad_kdf_kernel", "ts": "conv3_wgrad_ts_kernel", "tc": "conv3_wgrad_tc_kernel"}


# ------------------------------------------------------------------------------------------------ forward, stride 1
# (id, B, spatial, source channels, Cout, k, op, P16 sources, act, accumulate, output pitch extra, stats, gap, mean)
FWD = [
    ("k3_n16_fold_fp16", 2, (9, 17, 11), [16], 16, 3, "fp16", True, 0, 0, 0, True, True, 0.0),
    ("k3_n32_fold_bf16", 1, (6, 18, 20), [32], 32, 3, "bf16", True, 0, 0, 0, True, True, 1.5),
    ("k3_n64_fp16", 3, (5, 17, 12), [32], 64, 3, "fp16", True, 0, 0, 0, True, True, 0.5),
    ("k3_n128_fp16", 2, (3, 18, 9), [64], 128, 3, "fp16", True, 0, 0, 0, False, True, 0.0),
    ("k3_n16_fp32entry_fp16", 2, (7, 9, 13), [32], 16, 3, "fp16", False, 0, 0, 0, True, True, 2.0),
    ("k3_tf32_cin24", 2, (6, 10, 12), [24], 16, 3, "fp16", False, 0, 0, 0, True, True, 1.0),
    ("k3_tf32_op", 1, (5, 17, 9), [16], 32, 3, "tf32", False, 0, 0, 0, True, True, 0.0),
    ("k3_concat3", 2, (6, 10, 16), [16, 48, 32], 32, 3, "fp16", True, 0, 0, 0, True, True, 0.3),
    ("k3_concat4", 1, (4, 16, 8), [32, 16, 64, 16], 64, 3, "bf16", True, 0, 0, 0, True, True, 0.0),
    ("k3_cin2_narrow", 2, (8, 8, 16), [2], 16, 3, "fp16", False, 0, 0, 0, True, True, 0.5),
    ("k1_wide", 2, (6, 10, 12), [32, 16], 32, 1, "fp16", True, 0, 0, 0, True, True, 0.0),
    ("k1_cout3_sigmoid", 2, (6, 10, 16), [16], 3, 1, "fp16", True, 1, 0, 0, False, False, 0.0),
    ("k1_accumulate_slice", 1, (4, 9, 16), [32], 16, 1, "fp16", True, 0, 1, 24, False, False, 0.0),
    ("k3_slice_pitch", 2, (4, 8, 8), [16], 16, 3, "fp16", True, 0, 0, 16, False, False, 0.0),
    ("k3_sigmoid_cout3", 1, (6, 8, 16), [16], 3, 3, "fp16", True, 1, 0, 0, False, False, 0.0),
    # GN statistics edges: 9 voxels per chunk cut a 16x8 patch row; B = 3 with tiles of one CTA crossing samples
    ("stats_chunk9", 2, (2, 3, 12), [16], 16, 3, "fp16", True, 0, 0, 0, True, True, 0.0),
    ("stats_b3", 3, (4, 6, 20), [16], 32, 3, "fp16", True, 0, 0, 0, True, True, 1.0),
    # pooling: N <= 32 persistent | N = 64, B = 1 | N = 128 per tile
    ("gap_n64_b1", 1, (8, 16, 16), [32], 64, 3, "fp16", True, 0, 0, 0, True, True, 0.5),
    ("gap_n128", 2, (4, 16, 16), [64], 128, 3, "fp16", True, 0, 0, 0, True, True, 0.5),
    # split-K + conv_finish_kernel (small volumes, long reductions)
    ("splitk_16c_512to128", 1, (16, 16, 16), [512], 128, 3, "fp16", True, 0, 0, 0, True, True, 0.5),
    ("splitk_16c_512to128_b2", 2, (16, 16, 16), [256, 256], 128, 3, "fp16", True, 0, 0, 0, True, True, 0.0),
    ("splitk_8c_256to64", 1, (8, 8, 8), [256], 64, 3, "fp16", True, 0, 0, 0, True, True, 0.0),
    ("splitk_8c_256to64_b2", 2, (8, 8, 8), [256], 64, 3, "fp16", True, 0, 0, 0, True, True, 1.0),
    # real sizes: many tiles per persistent CTA
    ("large_128c_16to16_fold", 1, (128, 128, 128), [16], 16, 3, "fp16", True, 0, 0, 0, True, True, 0.0),
    ("large_64c_32to32_fold_b2", 2, (64, 64, 64), [32], 32, 3, "fp16", True, 0, 0, 0, True, True, 3.0),
    ("large_32c_64to64", 1, (32, 32, 32), [64], 64, 3, "fp16", True, 0, 0, 0, True, True, 0.0),
]


@pytest.mark.parametrize("case,kd_fold", with_fold_off(FWD), indirect=["kd_fold"])
def test_fwd_path(env, dev, case, kd_fold):
    cid, B, sp, cins, cout, k, op, p16, act, acc, extra, want_stats, want_gap, mean = case
    ops, lib = env.ops, env._lib.lib
    cin = sum(cins)
    ops.set_conv_precision(op, "bf16")
    try:
        xs = [rnd(B, *sp, c, seed=11 + i, mean=mean) for i, c in enumerate(cins)]
        w = rnd(k, k, k, cin, cout, seed=3, scale=(k ** 3 * cin) ** -0.5)
        bias = rnd(cout, seed=4, scale=0.3)
        S = sp[0] * sp[1] * sp[2]
        want_stats = want_stats and S % 8 == 0           # fused statistics need whole chunks of voxels
        stats = torch.empty(B, 8, 2, dtype=torch.float64, device=dev) if want_stats else None
        gap = torch.empty(B, cout, device=dev) if want_gap else None
        if extra:
            ybuf = rnd(B, *sp, cout + extra, seed=5)
            y = ybuf[..., extra // 2:extra // 2 + cout]
        else:
            ybuf = y = torch.empty(B, *sp, cout, device=dev)
        y0, ybuf0 = y.clone(), ybuf.clone()
        wp = ops.pack_weights(w, False, 1, False)
        cfg_e, split_e, op_e = expect_conv("s1", k, cin, cout, op, B, sp, act=act, accumulate=acc,
                                           contiguous=not extra, stats=want_stats, fold=kd_fold)
        if p16:
            tw = [ops.to_p16(t, TWIN[op]) for t in xs]
            call = lambda: ops._call("b3d_conv3d_fwd_p16", *(tw + [None] * (4 - len(tw))), w, bias, y, 1, 0, act, stats,
                                     8, gap, acc, wp)
        else:
            x = torch.cat(xs, dim=-1).contiguous()
            call = lambda: ops._call("b3d_conv3d_fwd", x, w, bias, y, 1, 0, act, stats, 8, gap, acc, wp)
        _, kern = run_profiled(call, repeatable=not acc)
    finally:
        ops.set_conv_precision("fp16", "bf16")
    cfgs = tc_cfgs(kern)
    assert cfgs == [cfg_e], (cid, cfgs, cfg_e, kern)
    assert has(kern, "conv_finish_kernel") == split_e, (cid, split_e, kern)
    if extra:        # the channels outside the slice are untouched
        assert torch.equal(ybuf[..., :extra // 2], ybuf0[..., :extra // 2])
        assert torch.equal(ybuf[..., extra // 2 + cout:], ybuf0[..., extra // 2 + cout:])
    xc = K.round_act(torch.cat([t.double().cpu() for t in xs], dim=-1), op_e)
    wr = K.round_weight(w.double().cpu(), op_e)
    ref = K.conv_taps(xc, wr) + bias.double().cpu()
    A = K.conv_taps(xc.abs(), wr.abs()) + bias.double().cpu().abs()
    ck = 8 if op_e == "tf32" else 16
    n_acc = k ** 3 * pad(cin, ck) // ck + 8 + 1
    extra_abs = None
    if acc:
        ref, A = ref + y0.double().cpu(), A + y0.double().cpu().abs()
        n_acc += 1
    if act:
        s = torch.sigmoid(ref)
        A = A * s * (1 - s) + 4.0 / (K.C_BOUND * (n_acc + 4))     # + 4 ulps of 1.0: the fp32 sigmoid's own roundings
        ref = s
    checks = [K.check(f"{cid} y", y, ref, A, n_acc, 1e-5, tile=(cfgs[0][1], 16, 8 * cfgs[0][2], cfgs[0][0]))]
    if op_e == "tf32":
        # the other candidate roundings of the fp32 activations, for the record
        for nm, fn in (("rn", lambda t: R.round_operand(t, "tf32")), ("rna", K.round_tf32_rna)):
            alt = K.conv_taps(fn(torch.cat([t.double().cpu() for t in xs], dim=-1)), wr) + bias.double().cpu()
            print(f"    tf32 activations modelled as {nm}: rel-L2 {K.rel_l2(y, alt):.2e}")
    yk = y.double().cpu()
    if want_stats:
        checks.append(K.check_sums(f"{cid} stats", stats, K.gn_chunk_sums(yk), K.gn_chunk_scale(yk)))
    if want_gap:
        checks.append(K.check_sums(f"{cid} gap", gap, yk.sum(dim=(1, 2, 3)), yk.abs().sum(dim=(1, 2, 3))))
    record(cid, kern, checks)


# ------------------------------------------------------------------------------------------- forward, stride 2 family
S2 = [
    # (id, B, input spatial, Cin, Cout, transposed, P16)
    ("s2d_down_16to32", 2, (8, 16, 12), 16, 32, False, True),
    ("s2d_down_64to128", 1, (8, 8, 16), 64, 128, False, False),
    ("d2s_up_64to32", 2, (4, 6, 8), 64, 32, True, True),
    ("d2s_up_128to64", 1, (4, 4, 8), 128, 64, True, False),
    ("vae_512to8", 1, (16, 16, 16), 512, 8, False, False),
]


@pytest.mark.parametrize("case", S2, ids=[c[0] for c in S2])
def test_fwd_stride2_path(env, dev, case):
    cid, B, sp, cin, cout, tr, p16 = case
    ops = env.ops
    x = rnd(B, *sp, cin, seed=21, mean=0.5)
    w = rnd(3, 3, 3, *((cout, cin) if tr else (cin, cout)), seed=22, scale=(27 * cin) ** -0.5)
    bias = rnd(cout, seed=23, scale=0.3)
    od = tuple(2 * n for n in sp) if tr else tuple(n // 2 for n in sp)
    y = torch.empty(B, *od, cout, device=dev)
    tc = ops.tc_supported(w, 2, tr, False)
    wp = ops.pack_weights(w, False, 2, tr) if tc else None
    if p16:
        xt = ops.to_p16(x, torch.float16)
        call = lambda: ops._call("b3d_conv3d_fwd_p16", xt, None, None, None, w, bias, y, 2, int(tr), 0, None, 8, None, 0, wp)
    else:
        call = lambda: ops._call("b3d_conv3d_fwd", x, w, bias, y, 2, int(tr), 0, None, 8, None, 0, wp)
    _, kern = run_profiled(call)
    xd, wd = x.double().cpu(), w.double().cpu()
    if tc:
        cfg_e, split_e, op_e = expect_conv("up" if tr else "down", 3, cin, cout, "fp16", B, od)
        assert tc_cfgs(kern) == [cfg_e], (cid, tc_cfgs(kern), cfg_e)
        assert has(kern, "conv_finish_kernel") == split_e
        xd, wd = K.round_act(xd, op_e), K.round_weight(wd, op_e)
        n_acc = 8 * (cin if not tr else cin) // 16 + 8 + 1
    else:        # the two narrow bottleneck layers run on fp32 CUDA cores
        assert cid.startswith("vae") and not tc_cfgs(kern) and has(kern, "conv_gather"), kern
        n_acc = 27 * cin
    ref = K.conv_s2_ref(xd, wd, tr) + bias.double().cpu()
    A = K.conv_s2_ref(xd.abs(), wd.abs(), tr) + bias.double().cpu().abs()
    record(cid, kern, [K.check(f"{cid} y", y, ref, A, n_acc, 1e-5)])


# ------------------------------------------------------------------------------------------------ slab forward
SLAB = [
    # (id, D0, D1 of the slab inside a D-slice volume, halo before, halo after, prezeroed, spatial, Cin, Cout)
    ("slab_mid", 5, 11, 1, 1, 0, (16, 12, 16), 16, 16),
    ("slab_first_prezeroed", 0, 7, 0, 1, 1, (16, 12, 16), 32, 32),
    ("slab_last", 9, 16, 1, 0, 0, (16, 12, 16), 16, 64),
    ("slab_thin_splitk", 6, 8, 1, 1, 0, (16, 16, 16), 256, 64),
]


@pytest.mark.parametrize("case,kd_fold", with_fold_off(SLAB), indirect=["kd_fold"])
def test_slab_fwd_window(env, dev, case, kd_fold):
    cid, d0, d1, hb, ha, pz, sp, cin, cout = case
    ops = env.ops
    D, H, W = sp
    x = rnd(1, *sp, cin, seed=31, mean=0.5)
    w = rnd(3, 3, 3, cin, cout, seed=32, scale=(27 * cin) ** -0.5)
    bias = rnd(cout, seed=33, scale=0.3)
    wp = ops.pack_weights(w, False, 1, False)
    xs = x[:, d0 - hb:d1 + ha].contiguous()
    if d0 - hb < 0 or d1 + ha > D:
        raise AssertionError("bad case")
    xt = ops.to_p16(xs, torch.float16)
    y = torch.empty(1, d1 - d0, H, W, cout, device=dev)
    pre_s = rnd(1, 8, 2, seed=34).double() if pz else None
    pre_g = rnd(1, cout, seed=35) if pz else None
    stats = pre_s.clone() if pz else torch.empty(1, 8, 2, dtype=torch.float64, device=dev)
    gap = pre_g.clone() if pz else torch.empty(1, cout, device=dev)
    off = d0 * H * W
    _, kern = run_profiled(lambda: ops._call("b3d_conv3d_fwd_p16_slab", xt, None, None, None, w, bias, y, 1, 0, 0, hb, ha,
                                             stats, 8, off, D * H * W, gap, wp, pz), repeatable=not pz)
    cfg_e, split_e, op_e = expect_conv("s1", 3, cin, cout, "fp16", 1, (d1 - d0, H, W), stats=True, stat_total=D * H * W,
                                       fold=kd_fold)
    assert tc_cfgs(kern) == [cfg_e] and has(kern, "conv_finish_kernel") == split_e, (kern, cfg_e, split_e)
    xr, wr = K.round_act(x.double().cpu(), "fp16"), K.round_weight(w.double().cpu(), "fp16")
    full = K.conv_taps(xr, wr) + bias.double().cpu()
    A = K.conv_taps(xr.abs(), wr.abs()) + bias.double().cpu().abs()
    n_acc = 27 * cin // 16 + 8 + 1
    checks = [K.check(f"{cid} y", y, full[:, d0:d1], A[:, d0:d1], n_acc, 1e-5)]
    # partial chunk sums of the kernel's own y over the window [off, off + slab) of the whole volume's chunks
    yk = torch.zeros(1, D, H, W, cout, dtype=torch.float64)
    yk[:, d0:d1] = y.double().cpu()
    mag = yk.abs()
    ref_s, scale = K.gn_chunk_sums(yk), K.gn_chunk_scale(mag)
    ref_g, scale_g = yk.sum(dim=(1, 2, 3)), mag.sum(dim=(1, 2, 3))
    if pz:
        ref_s, ref_g = ref_s + pre_s.cpu(), ref_g + pre_g.double().cpu()
        scale, scale_g = scale + pre_s.cpu().abs(), scale_g + pre_g.double().cpu().abs()
    checks.append(K.check_sums(f"{cid} stats", stats, ref_s, scale + 1e-30))
    checks.append(K.check_sums(f"{cid} gap", gap, ref_g, scale_g))
    record(cid, kern, checks)


# ------------------------------------------------------------------------------------------------ data gradient
DGRAD = [
    # (id, form, B, spatial, layer Cin (pieces), layer Cout, k, mean)
    ("dgrad_k3_fp32entry", "fp32", 2, (6, 17, 12), [32], 16, 3, 0.0),
    ("dgrad_k3_p16", "p16", 2, (5, 10, 16), [64], 32, 3, 0.5),
    ("dgrad_k1_p16", "p16", 1, (6, 10, 12), [48], 32, 1, 0.0),
    ("dgrad_k1_fp32entry", "fp32", 2, (4, 8, 8), [16], 128, 1, 0.0),
    ("dgrad_tf32_cout24", "fp32", 2, (4, 9, 12), [16], 24, 3, 0.0),
    ("dgrad_split_accumulate", "split", 2, (4, 12, 16), [16, 32, 16], 32, 3, 0.5),
    ("dgrad_block", "block", 2, (6, 10, 12), [32, 16], 16, 3, 0.0),
    ("large_dgrad_128c_32to16", "p16", 1, (128, 128, 128), [32], 16, 3, 0.0),
]


@pytest.mark.parametrize("case,kd_fold", with_fold_off(DGRAD), indirect=["kd_fold"])
def test_dgrad_path(env, dev, case, kd_fold):
    cid, form, B, sp, pieces, cout, k, mean = case
    ops = env.ops
    cin = sum(pieces)
    w = rnd(k, k, k, cin, cout, seed=41, scale=(k ** 3 * cout) ** -0.5)
    dy = rnd(B, *sp, cout, seed=42, mean=mean)
    wpd = ops.pack_weights(w, True, 1, False)
    dyr = dy.double().cpu()
    dx = torch.empty(B, *sp, cin, device=dev)
    outs = None
    if form == "fp32":
        call = lambda: ops._call("b3d_conv3d_dgrad", dy, w, dx, 1, 0, 0, wpd)
    elif form == "p16":
        dy16 = ops.to_p16(dy, torch.bfloat16)
        call = lambda: ops._call("b3d_conv3d_dgrad_p16", dy16, w, dx, 1, 0, 0, wpd)
    elif form == "split":
        dy16 = ops.to_p16(dy, torch.bfloat16)
        outs = [rnd(B, *sp, c, seed=43 + i) for i, c in enumerate(pieces)]
        pre = torch.cat(outs, dim=-1).double().cpu()
        call = lambda: ops._call("b3d_conv3d_dgrad_p16_split", dy16, w, *(outs + [None] * (4 - len(outs))), 1, wpd)
    else:
        dres = rnd(B, *sp, cout, seed=44)
        wpw = rnd(1, 1, 1, cin, cout, seed=45, scale=cout ** -0.5)
        dy16, dres16 = ops.to_p16(dy, torch.bfloat16), ops.to_p16(dres, torch.bfloat16)
        wpp = ops.pack_weights(wpw, True, 1, False)
        outs = [torch.full((B, *sp, c), float("nan"), device=dev) for c in pieces]
        call = lambda: ops._call("b3d_conv3d_dgrad_p16_block", dy16, dres16, w, wpw, *(outs + [None] * (4 - len(outs))),
                                 wpd, wpp)
    _, kern = run_profiled(call, repeatable=form != "split")
    cfg_e, split_e, op_e = expect_conv("s1", k, cout, cin, "bf16", B, sp, accumulate=form == "split",
                                       nyd=len(pieces) if form in ("split", "block") else 1, fold=kd_fold)
    if form == "block":
        cfg_e = cfg_e[:3] + (3, 1) + cfg_e[5:]
    cfgs = tc_cfgs(kern)
    assert cfgs == [cfg_e] and has(kern, "conv_finish_kernel") == split_e, (cid, cfgs, cfg_e, split_e, kern)
    dyq, wq = K.round_act(dyr, op_e), K.round_weight(w.double().cpu(), op_e)
    ref, A = K.dgrad_taps(dyq, wq), K.dgrad_taps(dyq.abs(), wq.abs())
    ck = 8 if op_e == "tf32" else 16
    n_acc = k ** 3 * pad(cout, ck) // ck + 8
    if form == "split":
        ref, A, n_acc = ref + pre, A + pre.abs(), n_acc + 1
    if form == "block":
        drq, wpq = K.round_act(dres.double().cpu(), "bf16"), K.round_weight(wpw.double().cpu(), "bf16")[0, 0, 0]
        ref, A, n_acc = ref + drq @ wpq.T, A + drq.abs() @ wpq.abs().T, n_acc + cout // 16
    got = torch.cat(outs, dim=-1) if outs is not None else dx
    record(cid, kern, [K.check(f"{cid} dx", got, ref, A, n_acc, 1e-5, tile=(cfgs[0][1], 16, 8 * cfgs[0][2], cfgs[0][0]))])


DGRAD_S2 = [("dgrad_s2_down", 2, (8, 8, 16), 32, 32, False), ("dgrad_s2_up", 1, (4, 6, 8), 64, 32, True)]


@pytest.mark.parametrize("case", DGRAD_S2, ids=[c[0] for c in DGRAD_S2])
def test_dgrad_stride2_path(env, dev, case):
    cid, B, sp, cin, cout, tr = case
    ops = env.ops
    w = rnd(3, 3, 3, *((cout, cin) if tr else (cin, cout)), seed=51, scale=(27 * cout) ** -0.5)
    od = tuple(2 * n for n in sp) if tr else tuple(n // 2 for n in sp)
    dy = rnd(B, *od, cout, seed=52, mean=0.3)
    dx = torch.empty(B, *sp, cin, device=dev)
    wpd = ops.pack_weights(w, True, 2, tr)
    dy16 = ops.to_p16(dy, torch.bfloat16)
    _, kern = run_profiled(lambda: ops._call("b3d_conv3d_dgrad_p16", dy16, w, dx, 2, int(tr), 0, wpd))
    cfg_e, split_e, op_e = expect_conv("down" if tr else "up", 3, cout, cin, "bf16", B, sp)
    assert tc_cfgs(kern) == [cfg_e] and has(kern, "conv_finish_kernel") == split_e, (kern, cfg_e)

    def vjp(dyv, wv):
        xx = torch.zeros(B, *sp, cin, dtype=torch.float64, requires_grad=True)
        y = R.conv3d_transpose_same(xx, wv, None) if tr else R.conv3d_same(xx, wv, None, 2)
        return torch.autograd.grad(y, xx, dyv)[0]
    dyq, wq = K.round_act(dy.double().cpu(), "bf16"), K.round_weight(w.double().cpu(), "bf16")
    record(cid, kern, [K.check(f"{cid} dx", dx, vjp(dyq, wq), vjp(dyq.abs(), wq.abs()), 8 * cout // 16 + 8, 1e-5)])


# ------------------------------------------------------------------------------------------------ weight gradient
WGRAD = [
    # (id, B, spatial, source channels, Cout, TS on, block (pointwise output too), mean)
    ("wgrad_kdf_16to16", 2, (5, 6, 24), [16], 16, True, False, 0.5),
    ("wgrad_kdf_32to32", 1, (8, 10, 16), [32], 32, True, False, 0.0),
    ("wgrad_kdf_64to16", 2, (4, 8, 16), [32, 32], 16, True, False, 0.0),
    ("wgrad_kdf_96to32", 1, (4, 6, 8), [32, 16, 48], 32, True, False, 0.3),
    ("wgrad_kdf_128to16", 1, (4, 8, 8), [64, 64], 16, True, False, 0.0),
    ("wgrad_kdf_block_32to16", 2, (6, 10, 16), [16, 16], 16, True, True, 0.0),
    # sources of 1 and 3 channel octets: no plane count shared with the 4-plane tile but 1, so one x box per
    # (depth slice, plane)
    ("wgrad_kdf_onebox_32to16", 1, (4, 8, 16), [8, 24], 16, True, False, 0.0),
    # odd H keeps these off kd-in-M: the per-tap kernel, the TS-mode kernel for Cin = 16, and the fused block form
    # refuses
    ("wgrad_hodd_ts_16to32", 2, (4, 7, 16), [16], 32, True, False, 0.0),
    ("wgrad_hodd_ts_16to16", 2, (4, 7, 24), [16], 16, True, False, 0.5),
    ("wgrad_hodd_tc_32to32", 1, (8, 9, 16), [32], 32, True, False, 0.0),
    ("wgrad_hodd_tc_64to16", 2, (4, 7, 16), [32, 32], 16, True, False, 0.0),
    ("wgrad_hodd_tc_96to32", 1, (4, 5, 8), [32, 16, 48], 32, True, False, 0.3),
    ("wgrad_hodd_block_32to16", 2, (6, 9, 16), [16, 16], 16, True, True, 0.0),
    ("wgrad_w12_tc_16to16_ts_off", 1, (4, 8, 12), [16], 16, False, False, 0.0),
    ("wgrad_tc_ks3_64to64", 1, (6, 10, 16), [64], 64, True, False, 0.5),
    ("wgrad_tc_ks3_256to128", 1, (4, 8, 8), [256], 128, True, False, 0.0),
    ("large_wgrad_kdf_64c_32to32", 2, (64, 64, 64), [32], 32, True, False, 0.0),
]


@pytest.mark.parametrize("case", WGRAD, ids=[c[0] for c in WGRAD])
def test_wgrad_path(env, dev, case):
    cid, B, sp, pieces, cout, ts, block, mean = case
    ops, lib = env.ops, env._lib.lib
    cin = sum(pieces)
    xs = [rnd(B, *sp, c, seed=61 + i, mean=mean) for i, c in enumerate(pieces)]
    dy = rnd(B, *sp, cout, seed=65)
    tw = [ops.to_p16(t, torch.bfloat16) for t in xs]
    dy16 = ops.to_p16(dy, torch.bfloat16)
    srcs = tw + [None] * (4 - len(tw))
    dw = torch.full((3, 3, 3, cin, cout), float("nan"), device=dev)
    lib.b3d_set_wgrad_ts(int(ts))
    try:
        kind, plan_e = expect_wgrad(pieces, cout, sp[1], sp[2], ts)
        kdf_ok = bool(lib.b3d_conv3d_wgrad_p16_block_ok(cin, cout, sp[1], sp[2]))
        assert kdf_ok == (kind == "kdf"), (cid, kind, kdf_ok)
        plan = lib.b3d_conv3d_wgrad_p16_plan(3, 1, 0, cin, cout, sp[2])
        assert plan == plan_e, (cid, plan, plan_e)
        if block and kind != "kdf":      # the fused form exists on the kd-in-M kernel only, and says so
            with pytest.raises(env._lib.B3DError, match="kd-in-M"):
                ops._call("b3d_conv3d_wgrad_p16_block", *srcs, dy16, ops.to_p16(dy, torch.bfloat16), dw,
                          torch.empty(1, 1, 1, cin, cout, device=dev))
            block = False
        scratch = torch.empty(dy16.numel(), device=dev, dtype=torch.bfloat16) if plan == 3 else None
        if block:
            dres = rnd(B, *sp, cout, seed=66)
            dres16 = ops.to_p16(dres, torch.bfloat16)
            dw1 = torch.full((1, 1, 1, cin, cout), float("nan"), device=dev)
            call = lambda: ops._call("b3d_conv3d_wgrad_p16_block", *srcs, dy16, dres16, dw, dw1)
        else:
            call = lambda: ops._call("b3d_conv3d_wgrad_p16", *srcs, dy16, dw, 1, 0, scratch)
        _, kern = run_profiled(call)
    finally:
        lib.b3d_set_wgrad_ts(1)
    assert has(kern, WGRAD_KERNEL[kind]), (cid, kind, kern)
    if kind == "tc":
        assert has(kern, "conv3_wgrad_tc_kernel<3,"), kern
    xq = K.round_act(torch.cat([t.double().cpu() for t in xs], dim=-1), "bf16")
    dq = K.round_act(dy.double().cpu(), "bf16")
    vox = B * sp[0] * sp[1] * sp[2]
    n_acc = vox // 16 + sm_count()       # longest chain: one CTA's K steps over its voxels + one atomic per CTA
    checks = [K.check(f"{cid} dw", dw, K.wgrad_taps(xq, dq, 3), K.wgrad_taps(xq.abs(), dq.abs(), 3), n_acc, 2e-5,
                      labels=("kd", "kh", "kw", "ci", "co"))]
    if block:
        drq = K.round_act(dres.double().cpu(), "bf16")
        checks.append(K.check(f"{cid} dw_pw", dw1, K.wgrad_taps(xq, drq, 1), K.wgrad_taps(xq.abs(), drq.abs(), 1), n_acc,
                              2e-5, labels=("kd", "kh", "kw", "ci", "co")))
    record(cid, kern, checks)


WGRAD_OTHER = [
    # (id, B, spatial, Cin, Cout, k, stride, transposed, route)
    ("wgrad_k1_ks1", 2, (6, 10, 16), 32, 32, 1, 1, False, "p16"),
    ("wgrad_s2_ks2_scratch", 2, (8, 8, 16), 32, 32, 3, 2, False, "p16"),
    ("wgrad_up_ks2_scratch", 1, (4, 6, 8), 64, 32, 3, 2, True, "p16"),
    ("wgrad_stacked_2to16", 2, (8, 8, 16), 2, 16, 3, 1, False, "fp32"),
    ("wgrad_stacked_16to3", 2, (8, 8, 16), 16, 3, 1, 1, False, "fp32"),
    ("wgrad_cuda_cores", 2, (6, 8, 10), 16, 16, 3, 1, False, "cuda"),
]


@pytest.mark.parametrize("case", WGRAD_OTHER, ids=[c[0] for c in WGRAD_OTHER])
def test_wgrad_other_paths(env, dev, case):
    import ctypes
    cid, B, sp, cin, cout, k, stride, tr, route = case
    ops, lib = env.ops, env._lib.lib
    od = tuple(2 * n for n in sp) if tr else tuple(n // stride for n in sp)
    x = rnd(B, *sp, cin, seed=71, mean=0.5)
    dy = rnd(B, *od, cout, seed=72)
    dw = torch.full((k, k, k) + ((cout, cin) if tr else (cin, cout)), float("nan"), device=dev)
    db = torch.empty(cout, device=dev)
    if route == "p16":
        plan = lib.b3d_conv3d_wgrad_p16_plan(k, stride, int(tr), cin, cout, od[2])
        assert plan == (2 if stride == 2 else 1), plan
        xt, dyt = ops.to_p16(x, torch.bfloat16), ops.to_p16(dy, torch.bfloat16)
        scratch = torch.empty(dyt.numel() if tr else xt.numel(), device=dev, dtype=torch.bfloat16) if plan == 2 else None
        call = lambda: ops._call("b3d_conv3d_wgrad_p16", xt, None, None, None, dyt, dw, stride, int(tr), scratch)
        want = "conv3_wgrad_tc_kernel<%d," % (1 if k == 1 else 2)
    else:
        xc, yc = ctypes.c_longlong(), ctypes.c_longlong()
        kind = lib.b3d_conv3d_wgrad_plan(k, stride, int(tr), cin, cout, ctypes.byref(xc), ctypes.byref(yc))
        if route == "cuda":
            xb = yb = None
            want = "conv_wgrad"
        else:
            assert kind == (2 if cin < 8 else 3), kind
            xb = torch.empty(x.numel() // cin * xc.value, device=dev, dtype=torch.bfloat16)
            yb = torch.empty(dy.numel() // cout * yc.value, device=dev, dtype=torch.bfloat16)
            want = "conv3_wgrad_tc_kernel<1,"
        call = lambda: ops._call("b3d_conv3d_wgrad", x, dy, dw, db, stride, int(tr), xb, yb, 0)
    _, kern = run_profiled(call)
    assert has(kern, want), (cid, want, kern)
    if route == "fp32":
        assert has(kern, "cast_stack_bf16_kernel"), kern
    if route == "cuda":
        assert not any("conv3_wgrad" in n for n in kern), kern
    rq = "bf16" if route != "cuda" else None
    xq, dq = K.round_act(x.double().cpu(), rq), K.round_act(dy.double().cpu(), rq)
    vox = dy.numel() // cout if not tr else x.numel() // cin

    def dw_of(xv, dv):
        if stride == 1:
            return K.wgrad_taps(xv, dv, k)
        ww = torch.zeros(dw.shape, dtype=torch.float64, requires_grad=True)
        y = R.conv3d_transpose_same(xv, ww, None) if tr else R.conv3d_same(xv, ww, None, 2)
        return torch.autograd.grad(y, ww, dv)[0]
    n_acc = max(dy.numel() // cout, x.numel() // cin) // 16 + sm_count()
    checks = [K.check(f"{cid} dw", dw, dw_of(xq, dq), dw_of(xq.abs(), dq.abs()), n_acc, 2e-5,
                      labels=("kd", "kh", "kw", "ci", "co"))]
    if route != "p16":
        dyd = dy.double().cpu()
        checks.append(K.check_sums(f"{cid} dbias", db, dyd.sum(dim=(0, 1, 2, 3)), dyd.abs().sum(dim=(0, 1, 2, 3)), 1e-5))
    del vox
    record(cid, kern, checks)


# --------------------------------------------------------------------------- GroupNorm / block kernels at model shapes
GN_SHAPES = [("large_128c_16", (1, 128, 128, 128, 16)), ("large_64c_32_b2", (2, 64, 64, 64, 32)),
             ("32c_64", (1, 32, 32, 32, 64)), ("16c_128", (1, 16, 16, 16, 128)), ("8c_256", (1, 8, 8, 8, 256)),
             ("fallback_c24", (1, 6, 10, 12, 24))]


def _gn_layout(shape, groups, channel, device):
    """The element -> group and element -> affine-index maps of GroupNorm on NDHWC storage [B, D, H, W, C]:
      * chunk form (channels_last, norm.cu / block.cu): group g of a sample is the g-th contiguous 1/G of its flat buffer,
        and flat element e has the affine index g*C/G + (e % C) % (C/G) (SURVEY F1, ref_model.group_norm_chunk);
      * channel form (channels_first, norm_channel.cu): group g is channels [g*C/G, (g+1)*C/G) of every voxel, and the
        affine index is the channel.
    Returns (per_group: [B, ...] -> [B, G] sums over each group, expand: [B, G] -> [B, ...], the affine index of every
    element of a sample)."""
    B, C = shape[0], shape[-1]
    cg, n = C // groups, math.prod(shape[1:])
    if channel:
        per_group = lambda t: t.reshape(B, -1, groups, cg).sum((1, 3))
        expand = lambda v: v[:, None, :, None].expand(B, n // C, groups, cg).reshape(shape)
        j = torch.arange(C, device=device).expand(shape[1:])
    else:
        per_group = lambda t: t.reshape(B, groups, -1).sum(-1)
        expand = lambda v: v[:, :, None].expand(B, groups, n // groups).reshape(shape)
        e = torch.arange(n, device=device)
        j = ((e // (n // groups)) * cg + (e % C) % cg).reshape(shape[1:])
    return per_group, expand, j


def _gn_ref(x, ga, be, dy, dx_kernel, groups=8, channel=False, relu=True):
    """fp64 GroupNorm (+ ReLU) (the oracle, `channel`: under its channels_first semantics) and its gradients (autograd),
    plus csum = per group (sum h, sum h*xhat) with h = dy*[y > 0]*gamma_j.

    The ReLU decision of an element whose pre-activation lies within fp32 resolution of 0 (|xhat*gamma + beta| below
    1e-5 of the magnitude of its terms) is not determined by the fp64 value: the kernel takes it on its fp32 value.  One
    such element changes dgamma_j by dy*xhat and dx by rstd*dy*gamma at that voxel, i.e. far more than 1e-5 of the
    result at 128^3 (a handful of such elements are expected among 33M).  For those elements the reference takes the
    decision the kernel took, read off the kernel's dx (the two candidates differ by rstd*dy*gamma there)."""
    shape = tuple(x.shape)
    per_group, expand, j = _gn_layout(shape, groups, channel, x.device)
    xd = x.double()
    n = xd[0].numel() // groups
    mean = expand(per_group(xd) / n)
    rstd = expand(1.0 / torch.sqrt(per_group((xd - mean) ** 2) / n + 1e-5))
    xh = (xd - mean) * rstd
    gj, bj = ga.double()[j], be.double()[j]
    pre = xh * gj + bj
    dyd = dy.double()

    def gn(*t):
        with R.channels_first_semantics() if channel else contextlib.nullcontext():
            return R.group_norm(*t, groups)

    def grads(mask):
        xr, gr, br = (t.double().clone().requires_grad_(True) for t in (x, ga, be))
        return torch.autograd.grad(gn(xr, gr, br) * mask, (xr, gr, br), dyd)
    m = (pre > 0).double() if relu else torch.ones_like(pre)
    if relu:
        dx = grads(m)[0]
        amb = pre.abs() <= 1e-5 * ((xd.abs() + mean.abs()) * rstd * gj.abs() + bj.abs())
        t = rstd * dyd * gj
        alt = dx + torch.where(m > 0, -t, t)
        dk = dx_kernel.double()
        flip = amb & ((dk - alt).abs() < (dk - dx).abs())
        m = torch.where(flip, 1.0 - m, m)
        print(f"    ReLU decisions within fp32 resolution of 0: {int(amb.sum())}, taken as the kernel did: "
              f"{int(flip.sum())}")
    dx, dga, dbe = grads(m)
    y = gn(xd, ga.double(), be.double())
    y = torch.relu(y) if relu else y
    h = dyd * m * gj
    csum = torch.stack([per_group(h), per_group(h * xh)], dim=-1)
    return y, dx, dga, dbe, csum, m


@pytest.mark.parametrize("mean", [0.0, 3.0], ids=["zero_mean", "mean3"])
@pytest.mark.parametrize("shape", [s for _, s in GN_SHAPES], ids=[n for n, _ in GN_SHAPES])
def test_group_norm_kernels_at_model_shapes(env, dev, shape, mean):
    ops = env.ops
    B, C = shape[0], shape[-1]
    x = rnd(*shape, seed=81, mean=mean)
    ga, be = 1 + 0.3 * rnd(C, seed=82), 0.3 * rnd(C, seed=83)
    dy = rnd(*shape, seed=84)
    stats = torch.empty(B, 8, 2, dtype=torch.float64, device=dev)
    y0, y1, dga, dbe = torch.empty_like(x), torch.empty_like(x), torch.empty_like(ga), torch.empty_like(be)
    csum, dx, dbias = torch.empty_like(stats), torch.empty_like(x), torch.empty(C, device=dev)
    cells = (C // 8) & (C // 8 - 1) == 0        # power-of-two channels per group: the cell kernels (norm.cu)

    def run():
        ops._call("b3d_gn_stats", x, stats, 8)
        ops._call("b3d_gn_apply", x, stats, ga, be, y0, 8, 1e-5, 1)
        ops._call("b3d_gn_bwd_reduce", dy, x, stats, ga, be, dga, dbe, csum, 8, 1e-5, 1)
        if cells:
            y16 = ops.p16_empty(shape, x, torch.float16)
            ops._call("b3d_gn_apply_p16", x, stats, ga, be, y1, y16, None, 8, 1e-5, 1)
            dx16 = ops.p16_empty(shape, x, torch.bfloat16)
            ops._call("b3d_gn_bwd_apply_p16", dy, x, stats, ga, be, csum, dx, dx16, dbias, 8, 1e-5, 1)
        else:
            ops._call("b3d_gn_bwd_apply", dy, x, stats, ga, be, csum, dx, 8, 1e-5, 1)
    _, kern = run_profiled(run)
    assert has(kern, "gn_stats_kernel") and has(kern, "gn_apply"), kern
    assert has(kern, "gn_bwd_reduce8_kernel") == cells, kern       # the cell kernels, or the non-cell fallback
    xd = x.double()
    yr, dxr, dgar, dber, csr, _ = _gn_ref(x, ga, be, dy, dx)
    checks = [K.check_sums("stats", stats, K.gn_chunk_sums(xd), K.gn_chunk_scale(xd)),
              K.check("y (gn_apply)", y0, yr, None, None, 1e-5),
              K.check("dgamma", dga, dgar, None, None, 1e-5), K.check("dbeta", dbe, dber, None, None, 1e-5),
              K.check("csum", csum, csr, None, None, 1e-5), K.check("dx", dx, dxr, None, None, 1e-5)]
    if cells:
        checks += [K.check("y (gn_apply_p16)", y1, yr, None, None, 1e-5),
                   K.check("dbias", dbias, dxr.sum(dim=(0, 1, 2, 3)), None, None, 1e-5)]
    record(f"gn {tuple(shape)} mean {mean}", kern, checks)


def _epilogue_out(r, hh, g, b, ws, ch, mask=None):
    """fp64 restatement of the ResnetBlock epilogue (layers/resnet.py:121-137 after the pooling MLP):
    out = r*(sigmoid(r . ws) + ch) + relu(GN(hh)); `mask`: the ReLU's decisions (default: hh's fp64 ones); g = None:
    the form without GroupNorm (has_gn = 0), out = r*(sigmoid(r . ws) + ch) + hh."""
    sp = torch.sigmoid((r * ws).sum(-1, keepdim=True))
    if g is None:
        a = hh
    else:
        gn = R.group_norm(hh, g, b)
        a = torch.relu(gn) if mask is None else gn * mask
    return r * (sp + ch[:, None, None, None, :]) + a


def _epilogue_ref(res, h2, ga, be, wsp, chse, dout, dgap, mask):
    """`_epilogue_out` with the kernel's ReLU decisions at 0 (mask) and its gradients, with dgap the gradient reaching
    the pooling sums of res."""
    t = [v.double().clone().requires_grad_(True) for v in (res, h2, ga, be, wsp, chse)]
    r, hh, g, b, ws, ch = t
    out = _epilogue_out(r, hh, g, b, ws, ch, mask)
    L = (out * dout.double()).sum() + (r.sum(dim=(1, 2, 3)) * dgap.double()).sum()
    grads = torch.autograd.grad(L, t)
    return out.detach(), grads


@pytest.mark.parametrize("mean", [0.0, 3.0], ids=["zero_mean", "mean3"])
@pytest.mark.parametrize("shape", [s for _, s in GN_SHAPES[:5]], ids=[n for n, _ in GN_SHAPES[:5]])
def test_block_epilogue_kernels_at_model_shapes(env, dev, shape, mean):
    ops = env.ops
    B, F = shape[0], shape[-1]
    res, h2 = rnd(*shape, seed=91, mean=mean), rnd(*shape, seed=92, mean=mean)
    ga, be = 1 + 0.3 * rnd(F, seed=93), 0.3 * rnd(F, seed=94)
    wsp, chse = 0.3 * rnd(F, seed=95), torch.sigmoid(rnd(B, F, seed=96))
    dout, dgap = rnd(*shape, seed=97), 0.01 * rnd(B, F, seed=98)
    stats = torch.empty(B, 8, 2, dtype=torch.float64, device=dev)
    out = torch.empty_like(res)
    dch, dws, dga, dbe, csum = (torch.empty(B, F, device=dev), torch.empty(F, device=dev), torch.empty_like(ga),
                                torch.empty_like(be), torch.empty_like(stats))
    dr, dh, dbr, dbh = torch.empty_like(res), torch.empty_like(res), torch.empty(F, device=dev), torch.empty(F, device=dev)

    def run():
        ops._call("b3d_gn_stats", h2, stats, 8)
        o16 = ops.p16_empty(shape, res, torch.float16)
        ops._call("b3d_block_epilogue_fwd_p16", res, h2, stats, ga, be, wsp, chse, out, o16, None, 8, 1e-5, 1)
        ops._call("b3d_block_epilogue_bwd_reduce", dout, res, h2, stats, ga, be, wsp, dch, dws, dga, dbe, csum, 8, 1e-5, 1)
        dr16, dh16 = ops.p16_empty(shape, res, torch.bfloat16), ops.p16_empty(shape, res, torch.bfloat16)
        ops._call("b3d_block_epilogue_bwd_apply_p16", dout, res, h2, stats, ga, be, wsp, chse, dgap, csum, dr, dh, dr16,
                  dh16, dbr, dbh, 8, 1e-5, 1)
    _, kern = run_profiled(run)
    assert has(kern, "b3d::block_fwd16_kernel"), kern
    _, _, _, _, csr, mask = _gn_ref(h2, ga, be, dout, dh)
    o_r, (dres_r, dh2_r, dga_r, dbe_r, dws_r, dch_r) = _epilogue_ref(res, h2, ga, be, wsp, chse, dout, dgap, mask)
    checks = [K.check("out", out, o_r, None, None, 1e-5), K.check("dchse", dch, dch_r, None, None, 1e-5),
              K.check("dwsp", dws, dws_r, None, None, 1e-5), K.check("dgamma", dga, dga_r, None, None, 1e-5),
              K.check("dbeta", dbe, dbe_r, None, None, 1e-5), K.check("csum", csum, csr, None, None, 1e-5),
              K.check("dres", dr, dres_r, None, None, 1e-5), K.check("dh2", dh, dh2_r, None, None, 1e-5),
              K.check("dbias_res", dbr, dres_r.sum(dim=(0, 1, 2, 3)), None, None, 1e-5),
              K.check("dbias_h2", dbh, dh2_r.sum(dim=(0, 1, 2, 3)), None, None, 1e-5)]
    record(f"block epilogue {tuple(shape)} mean {mean}", kern, checks)



# ------------------------------------------------------------------------------- channel GroupNorm at model shapes
# the channels_first model's GroupNorm inputs in the NDHWC storage the kernels see: (id, shape, groups).  At 128^3 x 16
# one channel group spreads over ~1,184 CTAs (cgeom caps the segments at 8 x SM count, divided by B).  Edges: three
# channels per group; C % 4 == 0 but C % 8 != 0 (the whole-volume kernels take it, the slab kernel refuses it)
GNC_SHAPES = [("large_128c_16", (1, 128, 128, 128, 16), 8), ("large_64c_32_b2", (2, 64, 64, 64, 32), 8),
              ("32c_64", (1, 32, 32, 32, 64), 8), ("16c_128", (1, 16, 16, 16, 128), 8), ("8c_256", (1, 8, 8, 8, 256), 8),
              ("c24_cg3_b2", (2, 5, 9, 7, 24), 8), ("c12_g4", (1, 6, 10, 12, 12), 4)]


@pytest.mark.parametrize("relu", [True, False], ids=["relu", "no_relu"])
@pytest.mark.parametrize("mean", [0.0, 3.0], ids=["zero_mean", "mean3"])
@pytest.mark.parametrize("case", GNC_SHAPES, ids=[c[0] for c in GNC_SHAPES])
def test_channel_group_norm_kernels_at_model_shapes(env, dev, case, mean, relu):
    """b3d_gn_channel_stats / _apply / _bwd (csrc/norm_channel.cu) against fp64 GroupNorm over true channel groups:
    the statistics at 1e-6 of sum|terms|, y, dgamma, dbeta, csum and dx at rel-L2 <= 1e-5."""
    ops = env.ops
    _, shape, G = case
    B, C = shape[0], shape[-1]
    x = rnd(*shape, seed=101, mean=mean)
    ga, be = 1 + 0.3 * rnd(C, seed=102), 0.3 * rnd(C, seed=103)
    dy = rnd(*shape, seed=104)
    stats = torch.empty(B, G, 2, dtype=torch.float64, device=dev)
    y, dx, dga, dbe, csum = (torch.empty_like(x), torch.empty_like(x), torch.empty_like(ga), torch.empty_like(be),
                             torch.empty_like(stats))

    def run():
        ops._call("b3d_gn_channel_stats", x, stats, G)
        ops._call("b3d_gn_channel_apply", x, stats, ga, be, y, G, 1e-5, int(relu))
        ops._call("b3d_gn_channel_bwd", dy, x, stats, ga, be, dga, dbe, csum, dx, G, 1e-5, int(relu))
    _, kern = run_profiled(run)
    r = str(relu).lower()
    for k in ("gnc_stats_kernel", f"gnc_apply_kernel<{r}>", f"gnc_bwd_reduce_kernel<{r}>", f"gnc_bwd_apply_kernel<{r}>"):
        assert has(kern, k), (k, kern)
    if C % 8:
        with pytest.raises(env._lib.B3DError, match="multiple of 8"):
            ops._call("b3d_gn_channel_apply_slab", x, stats, ga, be, torch.empty_like(x), None, G, 1e-5, int(relu),
                      x[0].numel() // C)
    grp = x.double().reshape(B, -1, G, C // G)
    sums = torch.stack([grp.sum((1, 3)), (grp * grp).sum((1, 3))], dim=-1)
    scale = torch.stack([grp.abs().sum((1, 3)), (grp * grp).sum((1, 3))], dim=-1)
    yr, dxr, dgar, dber, csr, _ = _gn_ref(x, ga, be, dy, dx, groups=G, channel=True, relu=relu)
    checks = [K.check_sums("stats", stats, sums, scale), K.check("y", y, yr, None, None, 1e-5),
              K.check("dgamma", dga, dgar, None, None, 1e-5), K.check("dbeta", dbe, dber, None, None, 1e-5),
              K.check("csum", csum, csr, None, None, 1e-5), K.check("dx", dx, dxr, None, None, 1e-5)]
    record(f"gn channel {tuple(shape)} G={G} mean {mean} relu {relu}", kern, checks)


# ----------------------------------------------------------------------------------------- NCDHW <-> NDHWC re-layout
# (id, NDHWC shape): the image / output channel counts below the 32-wide tile, voxel counts that are not a multiple of
# 32, B = 2, and the inference volume with the four image channels
RELAYOUT = [("c2_odd", (1, 9, 17, 11, 2)), ("c3_odd_b2", (2, 9, 17, 11, 3)), ("c4", (1, 8, 8, 8, 4)),
            ("c16_odd", (1, 9, 17, 11, 16)), ("c256_b2", (2, 5, 6, 7, 256)), ("large_160x192x160_c4", (1, 160, 192, 160, 4))]


@pytest.mark.parametrize("case", RELAYOUT, ids=[c[0] for c in RELAYOUT])
def test_relayout(env, dev, case):
    """b3d_relayout is a permutation: bit-identical to permute().contiguous() in both directions (NaN-filled outputs,
    so an element left unwritten fails too)."""
    ops = env.ops
    cid, (B, D, H, W, C) = case
    x_cf = rnd(B, C, D, H, W, seed=111)
    z_cl = rnd(B, D, H, W, C, seed=112)          # an independent input for the inverse: not only a round trip
    x_cl = torch.full((B, D, H, W, C), float("nan"), device=dev)
    z_cf = torch.full((B, C, D, H, W), float("nan"), device=dev)

    def run():
        ops._call("b3d_relayout", x_cf, x_cl, 1)
        ops._call("b3d_relayout", z_cl, z_cf, 0)
    _, kern = run_profiled(run)
    assert has(kern, "transpose_kernel"), kern
    want_cl, want_cf = x_cf.permute(0, 2, 3, 4, 1).contiguous(), z_cl.permute(0, 4, 1, 2, 3).contiguous()
    record(cid, kern, [_same("NCDHW -> NDHWC", x_cl, want_cl), _same("NDHWC -> NCDHW", z_cf, want_cf)])


def _same(what, got, want):
    """Bit-identity (NaN counts as a difference) as a Check."""
    ok = got.shape == want.shape and torch.equal(got, want)
    nbad = 0 if ok else int((got != want).sum()) if got.shape == want.shape else -1
    return K.Check(what, 0.0 if ok else K.rel_l2(got.float(), want.float()), 0.0 if ok else float("inf"), None, ok,
                   f"{what}: " + ("bit-identical" if ok else f"{nbad} elements differ"))


# ---------------------------------------------------------------------------------------------------- slab windows
def _slab_cases():
    """(id, [D, H, W, C], windows).  The windows depth-slab inference produces: slab.slab_bounds(160, world) for 2, 4
    and 8 ranks scaled to each encoder level, as SlabContext.geometry does (8 ranks: 24,24,24,24,16,16,16,16 slices at
    160), given as (world, level) and cut in the test.  GroupNorm chunks (1/8 of the flat volume) hold 20 / 10 / 5 / 2.5
    slices, so slab and chunk boundaries do not line up.  Then hand-placed windows the 8-slice alignment never
    produces: strictly inside one chunk, across at least 3 chunks, one slice, the first and the last slice."""
    cases = []
    for lvl in range(4):
        D, H, W, C = 160 >> lvl, 192 >> lvl, 160 >> lvl, 16 << lvl
        for world in (2, 4, 8):
            # 160x192x160 and 80x96x80 (79M and 20M elements) are real-size cases; the two deeper levels are quick
            cases.append((f"{'large_' if lvl <= 1 else ''}{D}x{H}x{W}x{C}_world{world}", (D, H, W, C), (world, lvl)))
    # chunk = 2.5 slices: (3, 4) inside chunk 1 = [2.5, 5); (1, 9) across chunks 0..3
    cases.append(("hand_20x24x20x128", (20, 24, 20, 128), [(3, 4), (1, 9), (12, 13), (19, 20)]))
    # chunk = 5 slices: (11, 14) inside chunk 2 = [10, 15); (2, 33) across chunks 0..6
    cases.append(("hand_40x48x40x16", (40, 48, 40, 16), [(11, 14), (2, 33), (0, 1), (39, 40)]))
    return cases


SLAB_WINDOWS = _slab_cases()


@pytest.fixture(scope="module")
def slab_refs(dev):
    """Holds the whole-volume inputs and fp64 references of one volume at a time (the cases of a volume are adjacent;
    ~3 GB of device memory at 160x192x160), released after the module's last test."""
    cache = {}
    yield cache
    cache.clear()
    torch.cuda.empty_cache()


def _slab_volume(cache, shape, dev):
    """Inputs (batch 1) with a depth-dependent mean and scale, so that neighbouring chunks' statistics differ by O(1)
    and a value normalised with the wrong chunk's statistics is far off; and their fp64 whole-volume references."""
    if shape in cache:
        return cache[shape]
    cache.clear()
    D, H, W, C = shape
    t = torch.arange(D, device=dev, dtype=torch.float32).view(1, D, 1, 1, 1) / D
    cm = 0.5 * torch.sin(torch.arange(C, device=dev, dtype=torch.float32))
    x = rnd(1, D, H, W, C, seed=121, dev=dev) * (0.5 + t) + (2 * t - 1) + cm
    res = rnd(1, D, H, W, C, seed=122, dev=dev) * (1.5 - t) + 0.5
    ga, be = 1 + 0.3 * rnd(C, seed=123, dev=dev), 0.3 * rnd(C, seed=124, dev=dev)
    wsp, chse = 0.3 * rnd(C, seed=125, dev=dev), torch.sigmoid(rnd(1, C, seed=126, dev=dev))
    xd = x.double()
    grp = xd.reshape(-1, 8, C // 8)
    v = dict(x=x, res=res, ga=ga, be=be, wsp=wsp, chse=chse,
             st=K.gn_chunk_sums(xd), st_scale=K.gn_chunk_scale(xd),
             st_c=torch.stack([grp.sum((0, 2)), (grp * grp).sum((0, 2))], dim=-1)[None],
             y=R.group_norm(xd, ga.double(), be.double()))
    with R.channels_first_semantics():
        v["y_c"] = R.group_norm(xd, ga.double(), be.double())
    p64 = [t.double() for t in (res, x, ga, be, wsp, chse)]
    v["out"] = _epilogue_out(*p64)
    v["out_nogn"] = _epilogue_out(p64[0], p64[1], None, None, p64[4], p64[5])
    cache[shape] = v
    return v


def _unpack(ops, t, shape):
    out = torch.full(shape, float("nan"), device=t.device)
    ops._call("b3d_p16_unpack", t, out)
    return out


@pytest.mark.parametrize("case", SLAB_WINDOWS, ids=[c[0] for c in SLAB_WINDOWS])
def test_slab_window_kernels(env, dev, slab_refs, case):
    """The depth-slab GroupNorm / block-epilogue kernels on real slab windows against fp64 of the WHOLE volume, sliced:
      * b3d_gn_stats_slab: each window's partial (sum x, sum x^2) per whole-volume chunk (zero for the chunks it misses)
        at 1e-6 of sum|terms|, and their sum over a partition = the whole volume's;
      * b3d_gn_apply_slab, b3d_gn_apply_p16_slab (fp32 y + twin, and twin only), b3d_gn_channel_apply_slab (y + twin,
        y only, twin only) and b3d_block_epilogue_fwd_p16_slab (has_gn 1 with out + twin and twin only, the form
        sharded inference uses; has_gn 0), given the exact whole-volume statistics: the fp32 output at rel-L2 <= 1e-5;
      * every twin (unpacked by b3d_p16_unpack) bit-identical to the fp16 / bf16 rounding of the fp32 output stored from
        the same registers; a twin written alone within half a 16-bit ulp + 1e-5 max|ref| of the fp64 reference, and
        bit-identical to the twin written next to y.
    ReLU alternates with every window, the twin type (fp16 / bf16) with every second window, starting from the level's
    parity, so each case with 4+ windows runs all four combinations and the 2-rank cases take both twin types across the
    levels.  (The worst rel-L2 of the `[path]` line is that of a twin
    written alone: the bf16 rounding itself, ~1.7e-3.)"""
    ops = env.ops
    cid, (D, H, W, C), wins = case
    partition, lvl = isinstance(wins, tuple), 0
    if partition:
        world, lvl = wins
        wins = [(a >> lvl, b >> lvl) for a, b in env.slab.slab_bounds(160, world)]
        assert wins[0][0] == 0 and wins[-1][1] == D and all(a[1] == b[0] for a, b in zip(wins, wins[1:])), wins
    v = _slab_volume(slab_refs, (D, H, W, C), dev)
    x, res, ga, be, wsp, chse = (v[k] for k in ("x", "res", "ga", "be", "wsp", "chse"))
    per, nvox = H * W * C, D * H * W
    total, L = D * per, D * per // 8
    nan = float("nan")
    outs = []

    def run():
        outs.clear()
        for i, (d0, d1) in enumerate(wins):
            relu, td = i % 2 == 0, (torch.float16, torch.bfloat16)[(i // 2 + lvl) % 2]
            xs, rs = x[:, d0:d1].contiguous(), res[:, d0:d1].contiguous()
            f32 = lambda: torch.full_like(xs, nan)
            p16 = lambda: ops.p16_empty(xs.shape, xs, td).fill_(nan)
            o = dict(relu=relu, td=td, d0=d0, d1=d1, part=torch.full((1, 8, 2), nan, dtype=torch.float64, device=dev),
                     part_c=torch.full((1, 8, 2), nan, dtype=torch.float64, device=dev),
                     y_a=f32(), y_p=f32(), t_p=p16(), t_po=p16(), y_c=f32(), t_c=p16(), y_co=f32(), t_co=p16(),
                     o_g=f32(), t_g=p16(), t_go=p16(), o_n=f32(), t_n=p16())
            off, r = d0 * per, int(relu)
            ops._call("b3d_gn_stats_slab", xs, o["part"], 8, off, total)
            ops._call("b3d_gn_apply_slab", xs, v["st"], ga, be, o["y_a"], 8, 1e-5, r, off, total)
            ops._call("b3d_gn_apply_p16_slab", xs, v["st"], ga, be, o["y_p"], o["t_p"], 8, 1e-5, r, off, total)
            ops._call("b3d_gn_apply_p16_slab", xs, v["st"], ga, be, None, o["t_po"], 8, 1e-5, r, off, total)
            ops._call("b3d_gn_channel_stats", xs, o["part_c"], 8)
            ops._call("b3d_gn_channel_apply_slab", xs, v["st_c"], ga, be, o["y_c"], o["t_c"], 8, 1e-5, r, nvox)
            ops._call("b3d_gn_channel_apply_slab", xs, v["st_c"], ga, be, o["y_co"], None, 8, 1e-5, r, nvox)
            ops._call("b3d_gn_channel_apply_slab", xs, v["st_c"], ga, be, None, o["t_co"], 8, 1e-5, r, nvox)
            ops._call("b3d_block_epilogue_fwd_p16_slab", rs, xs, v["st"], ga, be, wsp, chse, o["o_g"], o["t_g"], 8,
                      1e-5, 1, d0 * H * W, nvox)
            ops._call("b3d_block_epilogue_fwd_p16_slab", rs, xs, v["st"], ga, be, wsp, chse, None, o["t_go"], 8,
                      1e-5, 1, d0 * H * W, nvox)
            ops._call("b3d_block_epilogue_fwd_p16_slab", rs, xs, None, None, None, wsp, chse, o["o_n"], o["t_n"], 8,
                      1e-5, 0, d0 * H * W, nvox)
            outs.append(o)
    _, kern = run_profiled(run)
    names = [n.replace(" ", "") for n in kern]
    for k in ("gn_stats_kernel<4>", "gn_apply_kernel<4,true>", "gn_apply_kernel<4,false>", "gn_apply16_kernel<true>",
              "gn_apply16_kernel<false>", "gnc_stats_kernel", "gnc_apply_slab_kernel<true>",
              "gnc_apply_slab_kernel<false>", "block_fwd16_kernel<true>", "block_fwd16_kernel<false>"):
        assert has(names, k), (cid, k, sorted(set(kern)))
    xflat = v["x"].double().reshape(-1)
    tot = torch.zeros(1, 8, 2, dtype=torch.float64, device=dev)
    checks = []
    for i, o in enumerate(outs):
        d0, d1, td = o["d0"], o["d1"], o["td"]
        w = f"w{i} [{d0},{d1})"
        act = torch.relu if o["relu"] else (lambda t: t)
        sl = lambda t: t[:, d0:d1]
        # partial chunk sums of the window's elements [d0*per, d1*per) of the flat volume
        ref_p, sc_p = torch.zeros(1, 8, 2, dtype=torch.float64, device=dev), torch.zeros(1, 8, 2, dtype=torch.float64,
                                                                                         device=dev)
        for g in range(8):
            lo, hi = max(g * L, d0 * per), min((g + 1) * L, d1 * per)
            if lo < hi:
                s = xflat[lo:hi]
                ref_p[0, g] = torch.stack([s.sum(), (s * s).sum()])
                sc_p[0, g] = torch.stack([s.abs().sum(), (s * s).sum()])
        tot += o["part"]
        grp = sl(v["x"]).double().reshape(-1, 8, C // 8)
        shp = tuple(o["y_a"].shape)
        y_r, yc_r = act(sl(v["y"])), act(sl(v["y_c"]))
        checks += [
            K.check_sums(f"{w} gn_stats_slab", o["part"], ref_p, sc_p),
            K.check_sums(f"{w} gn_channel_stats", o["part_c"], torch.stack([grp.sum((0, 2)), (grp * grp).sum((0, 2))],
                                                                           dim=-1)[None],
                         torch.stack([grp.abs().sum((0, 2)), (grp * grp).sum((0, 2))], dim=-1)[None]),
            K.check(f"{w} gn_apply_slab y", o["y_a"], y_r, None, None, 1e-5),
            K.check(f"{w} gn_apply_p16_slab y", o["y_p"], y_r, None, None, 1e-5),
            _same(f"{w} gn_apply_p16_slab twin = y rounded", _unpack(ops, o["t_p"], shp), o["y_p"].to(td).float()),
            K.check_rounded(f"{w} gn_apply_p16_slab twin only", _unpack(ops, o["t_po"], shp), y_r, td),
            _same(f"{w} gn_apply_p16_slab twin only = twin next to y", o["t_po"], o["t_p"]),
            K.check(f"{w} gn_channel_apply_slab y", o["y_c"], yc_r, None, None, 1e-5),
            _same(f"{w} gn_channel_apply_slab twin = y rounded", _unpack(ops, o["t_c"], shp), o["y_c"].to(td).float()),
            _same(f"{w} gn_channel_apply_slab y only = y next to twin", o["y_co"], o["y_c"]),
            K.check_rounded(f"{w} gn_channel_apply_slab twin only", _unpack(ops, o["t_co"], shp), yc_r, td),
            _same(f"{w} gn_channel_apply_slab twin only = twin next to y", o["t_co"], o["t_c"]),
            K.check(f"{w} block_epilogue_slab out", o["o_g"], sl(v["out"]), None, None, 1e-5),
            _same(f"{w} block_epilogue_slab twin = out rounded", _unpack(ops, o["t_g"], shp), o["o_g"].to(td).float()),
            K.check_rounded(f"{w} block_epilogue_slab twin only", _unpack(ops, o["t_go"], shp), sl(v["out"]), td),
            _same(f"{w} block_epilogue_slab twin only = twin next to out", o["t_go"], o["t_g"]),
            K.check(f"{w} block_epilogue_slab (no GN) out", o["o_n"], sl(v["out_nogn"]), None, None, 1e-5),
            _same(f"{w} block_epilogue_slab (no GN) twin = out rounded", _unpack(ops, o["t_n"], shp),
                  o["o_n"].to(td).float())]
    if partition:
        checks.append(K.check_sums("sum of the windows' gn_stats_slab = whole volume", tot, v["st"], v["st_scale"]))
    record(cid, kern, checks)
