"""Weight gradients of the narrow layers (fewer than 8 channels on one side) on b3d_conv3d_wgrad_narrow: the tap-stacked
operand of the fp32 narrow tensor is built in shared memory, the wide operand is its bf16 P16 twin.

  * every model layer of this kind at 128^3 (the first ResnetBlock's 3x3x3 + pointwise pair in one launch, the decoder's
    1x1x1 16->3 and the VAE's 3x3x3 16->2 output convs) and small odd shapes (B = 2, H / W not multiples of the tile),
    against fp64 tap sums of the bf16-rounded operands (oracle/kernel_ref.py's checker, rel-L2 <= 2e-5 plus the
    per-element bound) and the bias gradient against fp64 column sums;
  * against the fp32 entry point b3d_conv3d_wgrad (staged stacked copy) on the same inputs: the operands are the same
    bf16 values, so only the fp32 summation order differs (the bias gradient, a sum over every voxel in both, is held
    to the fp64 column sums above instead);
  * one training step launches the kernel three times and neither staging copy (the per-layer cases call the entry
    point directly, which launches that kernel only);
  * unsupported arguments return error codes."""
import pytest
import torch

from oracle import kernel_ref as K
from oracle import ref_model as R

KERNEL = "conv_wgrad_narrow_kernel"

CASES = [
    # (id, B, spatial, Cin, Cout, k, pair)
    ("block1_pair_2to16_large", 1, (128, 128, 128), 2, 16, 3, True),
    ("dec_out_16to3_k1_large", 1, (128, 128, 128), 16, 3, 1, False),
    ("vae_out_16to2_k3_large", 1, (128, 128, 128), 16, 2, 3, False),
    ("pair_2to16_odd", 2, (5, 7, 13), 2, 16, 3, True),
    ("in_2to16_k3_odd", 2, (9, 6, 11), 2, 16, 3, False),
    ("in_3to32_k1_odd", 2, (3, 10, 9), 3, 32, 1, False),
    ("out_16to3_k1_odd", 2, (7, 5, 19), 16, 3, 1, False),
    ("out_32to2_k3_odd", 2, (6, 9, 10), 32, 2, 3, False),
    ("out_16to4_k3_edge", 1, (2, 2, 8), 16, 4, 3, False),
]


@pytest.fixture(scope="module")
def env(b3d, dev):
    return b3d


def rnd(*shape, seed=0, mean=0.0, dev="cuda"):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) + mean).to(dev)


def kernels_of(fn, attempts=5):
    """Names of the CUDA kernels fn runs (fn may run more than once).  On a shared device CUPTI occasionally delivers no
    activity at all for a profiled region; such a trace is taken again."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(attempts):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        try:
            names = [e.name() for e in prof.profiler.kineto_results.events() if "cuda" in str(e.device_type()).lower()]
        except AttributeError:
            names = [e.name for e in prof.events() if "cuda" in str(e.device_type).lower()]
        if names:
            break
    kern = [n for n in names if "kernel" in n]
    assert kern, "torch.profiler recorded no CUDA kernel: the kernel path cannot be verified"
    return kern


def operands(case, dev):
    cid, B, sp, cin, cout, k, pair = case
    x = rnd(B, *sp, cin, seed=81, mean=0.5)
    dy = rnd(B, *sp, cout, seed=82)
    dres = rnd(B, *sp, cout, seed=83) if pair else None
    return x, dy, dres


def run_narrow(ops, case, x, dy, dres, dev):
    """(dw, dw_pw | None, dbias | None) of b3d_conv3d_wgrad_narrow on these operands."""
    cid, B, sp, cin, cout, k, pair = case
    dw = torch.full((k, k, k, cin, cout), float("nan"), device=dev)
    if cin < 8:
        dy16 = ops.to_p16(dy, torch.bfloat16)
        dres16 = ops.to_p16(dres, torch.bfloat16) if pair else None
        dwp = torch.full((1, 1, 1, cin, cout), float("nan"), device=dev) if pair else None
        ops._call("b3d_conv3d_wgrad_narrow", x, dy16, dres16, dw, dwp, None)
        return dw, dwp, None
    x16 = ops.to_p16(x, torch.bfloat16)
    db = torch.full((cout,), float("nan"), device=dev)
    ops._call("b3d_conv3d_wgrad_narrow", dy, x16, None, dw, None, db)
    return dw, None, db


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_wgrad_narrow_matches_taps(env, dev, case):
    cid, B, sp, cin, cout, k, pair = case
    ops = env.ops
    x, dy, dres = operands(case, dev)
    dw, dwp, db = run_narrow(ops, case, x, dy, dres, dev)
    xq, dq = K.round_act(x.double(), "bf16"), K.round_act(dy.double(), "bf16")
    vox = x.numel() // cin
    n_acc = vox // 16 + torch.cuda.get_device_properties(0).multi_processor_count
    labels = ("kd", "kh", "kw", "ci", "co")
    checks = [K.check(f"{cid} dw", dw, K.wgrad_taps(xq, dq, k), K.wgrad_taps(xq.abs(), dq.abs(), k), n_acc, 2e-5,
                      labels=labels)]
    if pair:
        rq = K.round_act(dres.double(), "bf16")
        checks.append(K.check(f"{cid} dw_pw", dwp, K.wgrad_taps(xq, rq, 1), K.wgrad_taps(xq.abs(), rq.abs(), 1), n_acc,
                              2e-5, labels=labels))
    if db is not None:
        d2 = dy.double().reshape(-1, cout)
        checks.append(K.check_sums(f"{cid} dbias", db, d2.sum(0), d2.abs().sum(0)))
    for c in checks:
        print("   ", c)
        assert c.ok, c


AB_CASES = [c for c in CASES if not c[6] and c[0] in ("dec_out_16to3_k1_large", "vae_out_16to2_k3_large",
                                                       "in_2to16_k3_odd", "out_32to2_k3_odd")]


@pytest.mark.gpu
@pytest.mark.parametrize("case", AB_CASES, ids=[c[0] for c in AB_CASES])
def test_wgrad_narrow_equals_fp32_entry(env, dev, case):
    """Same bf16 operand values as the staged path of b3d_conv3d_wgrad (plan kinds 2 / 3): the results differ by the
    fp32 summation order only."""
    import ctypes
    cid, B, sp, cin, cout, k, pair = case
    ops, lib = env.ops, env._lib.lib
    x, dy, _ = operands(case, dev)
    dw, _, _ = run_narrow(ops, case, x, dy, None, dev)
    xc, yc = ctypes.c_longlong(), ctypes.c_longlong()
    kind = lib.b3d_conv3d_wgrad_plan(k, 1, 0, cin, cout, ctypes.byref(xc), ctypes.byref(yc))
    assert kind == (2 if cin < 8 else 3), kind
    xb = torch.empty(x.numel() // cin * xc.value, device=dev, dtype=torch.bfloat16)
    yb = torch.empty(dy.numel() // cout * yc.value, device=dev, dtype=torch.bfloat16)
    dw0 = torch.empty_like(dw)
    db0 = torch.empty(cout, device=dev)
    ops._call("b3d_conv3d_wgrad", x, dy, dw0, db0, 1, 0, xb, yb, 0)
    torch.cuda.synchronize()
    rel = K.rel_l2(dw, dw0)
    print(f"    {cid}: rel-L2(narrow, fp32 entry) = {rel:.2e}")
    assert rel <= 1e-6, rel


@pytest.mark.gpu
def test_train_step_runs_narrow_wgrad(env, dev):
    """One training step: the four narrow layers take three launches of the kernel (the first block's pair shares one)
    and nothing stages a stacked or plain bf16 copy for them."""
    b3d = env
    crop = (32, 32, 32)
    p = R.init_params(R.param_shapes(crop=crop))
    x, y, eps, mask = R.synth_batch((1,) + crop)
    f = lambda t: t.to(torch.float32).to(dev)
    model = b3d.Model()
    model(f(x), training=False, inference=False, eps=f(eps))
    model.load_named_weights(p)
    opt = b3d.ScheduledOptim(learning_rate=1e-4)
    opt(epoch=0)
    args = (model, opt, b3d.DiceVAELoss(), b3d.DiceCoefficient(), f(x), f(y))
    b3d.train_step(*args, dropout_mask=f(mask), eps=f(eps))
    kern = kernels_of(lambda: b3d.train_step(*args, dropout_mask=f(mask), eps=f(eps)))
    assert sum(KERNEL in n for n in kern) == 3, [n for n in kern if "wgrad" in n]
    assert not any("cast_stack_bf16_kernel" in n or "cast_bf16_kernel" in n for n in kern), kern


@pytest.mark.gpu
def test_wgrad_narrow_rejects_unsupported(env, dev):
    ops, err = env.ops, env._lib.B3DError
    x = rnd(1, 4, 4, 8, 2, seed=1)
    dy16 = ops.to_p16(rnd(1, 4, 4, 8, 16, seed=2), torch.bfloat16)
    dw = torch.empty(3, 3, 3, 2, 16, device=dev)
    with pytest.raises(err, match="bf16 twin"):                      # fp16 wide operand
        ops._call("b3d_conv3d_wgrad_narrow", x, ops.to_p16(rnd(1, 4, 4, 8, 16, seed=2), torch.float16), None, dw,
                  None, None)
    with pytest.raises(err, match="not on this path"):               # 27 * 5 stacked rows do not fit M = 128
        ops._call("b3d_conv3d_wgrad_narrow", rnd(1, 4, 4, 8, 5, seed=3), dy16, None,
                  torch.empty(3, 3, 3, 5, 16, device=dev), None, None)
    with pytest.raises(err, match="bias gradient"):                  # dbias of the wide dy
        ops._call("b3d_conv3d_wgrad_narrow", x, dy16, None, dw, None, torch.empty(2, device=dev))
    with pytest.raises(err, match="dw channel dims"):
        ops._call("b3d_conv3d_wgrad_narrow", x, dy16, None, torch.empty(3, 3, 3, 2, 8, device=dev), None, None)
    with pytest.raises(err, match="spatial dims"):
        ops._call("b3d_conv3d_wgrad_narrow", rnd(1, 4, 4, 16, 2, seed=4), dy16, None, dw, None, None)
    with pytest.raises(err, match="dres and dw_pw"):                 # dres without dw_pw
        ops._call("b3d_conv3d_wgrad_narrow", x, dy16, dy16, dw, None, None)


def test_wgrad_narrow_ok_query(b3d):
    ok = b3d._lib.lib.b3d_conv3d_wgrad_narrow_ok
    assert ok(3, 2, 16, 1) == 1 and ok(3, 2, 16, 0) == 1        # first ResnetBlock, with and without its pointwise conv
    assert ok(1, 2, 16, 0) == 1 and ok(1, 16, 3, 0) == 1 and ok(3, 16, 2, 0) == 1
    assert ok(3, 16, 2, 1) == 0                                   # the pair form takes a narrow input
    assert ok(3, 5, 16, 0) == 0                                   # 135 stacked rows
    assert ok(3, 2, 8, 0) == 0 and ok(3, 8, 16, 0) == 0 and ok(2, 2, 16, 0) == 0
    assert ok(1, 2, 256, 1) == 0 and ok(1, 2, 256, 0) == 1        # N = 512 > 256
