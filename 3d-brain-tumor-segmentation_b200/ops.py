"""torch.autograd glue around the b3d C-ABI (include/b3d.h).  torch is only the tensor container and
the tape; every arithmetic op below is a hand-written sm_100a kernel reached through ctypes.

All activations are channels_last [B, D, H, W, C] fp32 CUDA tensors; weights are in Keras layouts.
"""
from __future__ import annotations

import torch
from torch.autograd import Function

from ctypes import byref as _byref, c_longlong as _ll

from ._lib import call, lib
from . import slab as _slab

_f32 = torch.float32

# kernel-launch accounting for bench.py ("gpu_launches"): incremented per C-ABI call that launches
LAUNCHES = {"n": 0}


# per-call device timing for bench.py's in-step aggregates (eager steps only: events cannot be read inside a graph)
_PROF = {"on": False, "rows": [], "tag": None}


class profile_calls:
    """with profile_calls() as rows: ... -> rows = [(abi name, tag, start event, end event)], tag = (class, FLOPs) set
    by the conv wrappers.  CUDA events on the launching stream around every C-ABI call."""

    def __enter__(self):
        _PROF["on"], _PROF["rows"] = True, []
        return _PROF["rows"]

    def __exit__(self, *a):
        _PROF["on"] = False
        return False


# One C-ABI call at a time per process: a call may launch several kernels that share library-owned state on ONE stream
# (split-K conv + its finish kernel and the 64 MB workspace between them).  Real ranks are separate processes; the
# virtual ranks of slab.run_virtual_ranks are THREADS on one stream, and ctypes drops the GIL during a call — without
# the lock two threads' conv + finish pairs interleaved now and then (8 slabs: rel-L2 2.2e-3 instead of 6.1e-4, 1 run in 3).
import threading as _thr
_CALL_LOCK = _thr.Lock()


def _call(name, *a):
    LAUNCHES["n"] += 1
    if not _PROF["on"]:
        with _CALL_LOCK:
            return call(name, *a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = call(name, *a)
    e1.record()
    _PROF["rows"].append((name, _PROF["tag"], e0, e1))
    _PROF["tag"] = None
    return rc


def _tag_conv(w, nvox_out, stride, transposed):
    """(kernel class, FLOPs) of one conv pass for profile_calls: 2 * output voxels * taps * Cin * Cout (transposed: input
    voxels), SURVEY section 8(d)."""
    if _PROF["on"]:
        k = w.shape[0]
        cls = "k1" if k == 1 else ("s2" if stride == 2 else "k3")
        _PROF["tag"] = (cls, 2.0 * nvox_out * k ** 3 * w.shape[3] * w.shape[4])


def _new(shape, like, dtype=_f32):
    return torch.empty(shape, device=like.device, dtype=dtype)


def _new_act(shape, like):
    """Activation that may feed a 3x3x3 conv: under depth-slab inference it is allocated between two spare depth
    slices so that the halo exchange happens in place (slab.SlabContext.new_activation)."""
    ctx = _slab.current()
    if ctx is not None and len(shape) == 5 and shape[0] == 1:
        return ctx.new_activation(shape, like)
    return torch.empty(tuple(shape), device=like.device, dtype=_f32)


def _check(x: torch.Tensor, name="input"):
    if not x.is_cuda:
        raise RuntimeError(f"b3d: {name} must be a CUDA tensor — there is no CPU path")
    if x.dtype != _f32:
        raise TypeError(f"b3d: {name} must be float32, got {x.dtype}")


def tc_supported(w, stride, transposed, dgrad) -> bool:
    """Does the tcgen05 kernel run this pass of a layer with Keras kernel `w` (k,k,k,a,b)?"""
    return bool(lib.b3d_conv3d_tc_supported(w.shape[0], stride, int(transposed), int(dgrad), w.shape[3], w.shape[4]))


def pack_weights(w: torch.Tensor, dgrad: bool, stride: int = 1, transposed: bool = False) -> torch.Tensor:
    """Operand layout of Keras kernel `w` for one pass of the tcgen05 conv.  Weights of a Model (views of its flat
    buffer) keep ONE persistent packed buffer per pass: it is refreshed for all layers together by
    `repack_all(flat)` right after the optimiser step (one launch instead of ~120 per training step, none per
    inference forward), or singly here when the stamp shows the weights were changed some other way."""
    w = getattr(w, "_b3d_base", w)          # a per-call alias of a persistent derived kernel (FoldDupFn)
    flat = getattr(w, "_b3d_flat", None)
    if flat is None:
        out = _new((lib.b3d_conv3d_packed_elems(w.shape[0], stride, w.shape[3], w.shape[4]),), w)
        _call("b3d_conv3d_pack_weights", w, out, stride, int(transposed), int(dgrad))
        return out
    e = flat.packs.get((id(w), bool(dgrad), int(stride), bool(transposed)))
    if e is None:
        e = _register_pack(flat, w, dgrad, stride, transposed)
        if not dgrad and tc_supported(w, stride, transposed, True):
            # the data-gradient operand is registered with the forward one, so that the job table is complete (and
            # can be uploaded) before anything is captured into a CUDA graph
            _register_pack(flat, w, True, stride, transposed)
    stamp = _pack_stamp(flat, w)
    if e["stamp"] != stamp:
        _call("b3d_conv3d_pack_weights", w, e["buf"], *e["cfg"])
        e["stamp"] = stamp
    return e["buf"]


def _register_pack(flat, w, dgrad, stride, transposed):
    key = (id(w), bool(dgrad), int(stride), bool(transposed))
    if key not in flat.packs:
        buf = _new((lib.b3d_conv3d_packed_elems(w.shape[0], stride, w.shape[3], w.shape[4]),), w)
        flat.packs[key] = {"w": w, "buf": buf, "cfg": (int(stride), int(transposed), int(dgrad)), "stamp": None}
        flat.pack_table = None
    return flat.packs[key]


_PREC_EPOCH = {"n": 0}       # bumped by set_conv_precision: the packed operand type depends on it


def _pack_stamp(flat, w):
    return (w._version, flat.theta._version, flat.epoch, _PREC_EPOCH["n"])


def ensure_pack_table(flat):
    """Device table of pack jobs for all registered operands of `flat` (rebuilt when a layer registers or the
    operand precision changes).  Uploading it is a host->device copy: it has to exist before graph capture."""
    if flat.pack_table is not None and flat.pack_table[3] == _PREC_EPOCH["n"]:
        return flat.pack_table
    if torch.cuda.is_current_stream_capturing():
        raise RuntimeError("b3d: a conv layer registered its packed operand during CUDA-graph capture; run the "
                           "model once (or call ops.ensure_pack_table(model.flat)) before capturing")
    import ctypes as C
    from ._lib import dl
    entries = list(flat.packs.values())
    nb = lib.b3d_conv3d_pack_job_bytes()
    host = (C.c_char * (nb * len(entries)))()
    blocks, got = 0, _ll()
    for i, e in enumerate(entries):
        pw, hw = dl(e["w"])
        pb, hb = dl(e["buf"])
        rc = lib.b3d_conv3d_pack_job(pw, pb, *e["cfg"], blocks, C.byref(host, i * nb), _byref(got))
        if rc != 0:
            raise RuntimeError("b3d_conv3d_pack_job failed: " + lib.b3d_last_error().decode())
        blocks += got.value
    tab = torch.frombuffer(bytearray(bytes(host)), dtype=torch.int64).to(flat.theta.device)
    flat.pack_table = (tab, len(entries), blocks, _PREC_EPOCH["n"], entries)
    return flat.pack_table


def repack_all(flat):
    """The weights of `flat` have just been changed by a kernel (Adam): refresh every registered packed operand with
    ONE launch (csrc/conv_tc.cu pack_many_kernel).  Captured at the end of the graphed training step."""
    flat.epoch += 1
    for w, wf, F in getattr(flat, "folds", ()):          # folded (F3) kernels follow the weights, then get packed
        _call("b3d_fold_dup", w, wf, F)
        w._b3d_fold[1] = (w._version, flat.theta._version, flat.epoch)
    if not flat.packs:
        return
    tab, n, blocks, _, entries = ensure_pack_table(flat)
    _call("b3d_conv3d_pack_many", tab, n, blocks)
    for e in entries:
        e["stamp"] = _pack_stamp(flat, e["w"])


# ---- direct parameter gradients ------------------------------------------------------------------------------
# Every trainable tensor of a Model is a view of one flat buffer and its .grad a view of the matching flat gradient
# buffer (model.FlatParams).  Inside `direct_param_grads(flat)` the backward kernels write weight / bias / affine
# gradients straight into those views and return None to autograd, which removes ~260 tiny "grad += g" launches
# per step; each parameter is used once per forward, so "write" and "accumulate" coincide (the buffer is zeroed at
# the start of the step, the L2-regulariser gradient is added afterwards by one kernel).
_DIRECT = {"flat": None}


class direct_param_grads:
    def __init__(self, flat):
        self.flat = flat

    def __enter__(self):
        self.prev = _DIRECT["flat"]
        _DIRECT["flat"] = self.flat

    def __exit__(self, *a):
        _DIRECT["flat"] = self.prev
        return False


def _grad_target(p, shape=None):
    """(tensor to write the gradient of parameter p into, direct?)"""
    flat = _DIRECT["flat"]
    if flat is not None and p is not None and getattr(p, "_b3d_flat", None) is flat and p.grad is not None:
        return (p.grad if shape is None else p.grad.reshape(shape)), True
    if p is None:
        return None, False
    return torch.empty(p.shape if shape is None else shape, device=p.device, dtype=p.dtype), False


def _grad_done(p, direct):
    if direct:
        _DIRECT["flat"].notify(p)


# set False to force the CUDA-core kernels everywhere (used by tests to cross-check the tcgen05 path)
USE_TC = {"on": True}


# ---- P16 operand twins -------------------------------------------------------------------------------------------
# Every tensor that feeds a tcgen05 conv exists as a 16-bit "P16" twin [B, D, H, C/8, W, 8] (csrc/p16.cu) written by the
# kernel that PRODUCES it (GroupNorm apply, block epilogue, their backward kernels): fp16 for forward activations, bf16
# for gradients.  The convs read the twins (TMA boxes, no conversion, channel concatenation = a list of sources) and
# the weight gradients read them directly — no cast passes.  Where every consumer of a tensor is a conv, its fp32 form
# is not materialised at all: the autograd-visible tensor is then a zero-stride placeholder of the logical shape
# (`_b3d_virtual`) that carries the twin(s); `materialize()` rebuilds fp32 for the rare consumer that needs it.
P16 = {"on": True}
# inside a Model forward (`fused_scope`) layer outputs are consumed by convs only, so blocks / resampling layers emit
# twin-only outputs and channel concatenation is virtual; outside (layers used on their own) outputs stay real fp32
import threading as _threading


class _Fused(_threading.local):
    """Per-thread flag (the virtual ranks of slab inference run the model in threads)."""
    on = False

    def __getitem__(self, k):
        return self.on

    def __setitem__(self, k, v):
        self.on = bool(v)


FUSED = _Fused()


class fused_scope:
    def __init__(self, on=True):
        self.on = on

    def __enter__(self):
        self.prev = FUSED["on"]
        FUSED["on"] = self.on

    def __exit__(self, *a):
        FUSED["on"] = self.prev
        return False


_TWIN_DT = {"fp16": torch.float16, "bf16": torch.bfloat16}


def twin_dtype(bwd: bool):
    """16-bit type of the operand twins of a pass (None: the pass does not run with 16-bit operands)."""
    if not (P16["on"] and USE_TC["on"]):
        return None
    ctx = _slab.current()
    if ctx is not None:          # depth-slab inference (forward only): the slab context's choice
        return None if bwd else ctx.p16
    return _TWIN_DT.get(get_conv_precision()[1 if bwd else 0])


def p16_empty(shape5, like, dtype):
    B, D, H, W, C = shape5
    return torch.empty((B, D, H, C // 8, W, 8), device=like.device, dtype=dtype)


def p16_ok(shape5) -> bool:
    return len(shape5) == 5 and shape5[-1] % 16 == 0 and shape5[-1] >= 16


def virtual(shape5, like, twins, wtwins=None):
    """Autograd-visible placeholder (no memory) of logical fp32 shape `shape5` carrying P16 twin(s): `twins` in the
    operand type of the pass that produced it, `wtwins` the bf16 set for weight gradients (tcgen05 kind::f16 takes one
    operand type for both operands, gradients are bf16 => forward activations carry a bf16 twin next to the fp16 one)."""
    t = torch.empty(1, device=like.device, dtype=_f32).expand(tuple(shape5))
    t._b3d_virtual = True
    t._p16_list = list(twins)
    t._p16w_list = list(wtwins) if wtwins is not None else None
    return t


def _attach(t, y16, y16b):
    """Twins of a REAL fp32 tensor."""
    t._p16 = y16
    t._p16w = y16b if y16b is not None else (y16 if y16.dtype == torch.bfloat16 else None)


def sources_w(t):
    """bf16 twins for the weight gradient of a conv reading `t` (None: not available)."""
    if is_virtual(t):
        l = t._p16w_list
        if l is None and t._p16_list and t._p16_list[0].dtype == torch.bfloat16:
            l = t._p16_list
        return l
    l = getattr(t, "_p16w_list", None)
    if l is not None:
        return l
    tw = getattr(t, "_p16w", None)
    return None if tw is None else [tw]


def want_wgrad_twin(td, grad_enabled):
    """A second (bf16) twin is written when the forward operand type is fp16 and a backward pass will follow.
    (`grad_enabled` is sampled by the caller OUTSIDE the autograd Function: inside `forward` grad mode is always off.)"""
    return td == torch.float16 and bool(grad_enabled)


_ZERO1 = {}


def _zero_placeholder(shape, device):
    """A zero gradient of `shape` without memory or a kernel per use (one cached scalar per device, zero strides): what
    autograd is handed when the real gradient travels through a gradient box; safe to be ADDED to a real gradient."""
    z = _ZERO1.get(device)
    if z is None:
        z = _ZERO1[device] = torch.zeros(1, device=device, dtype=_f32)
    return z.expand(tuple(shape))


def _grad_placeholder(like):
    """What a backward returns for an input whose gradient exists only as a twin in the producer's mailbox: a zero-stride
    tensor of the right shape (no memory, never read)."""
    return torch.empty(1, device=like.device, dtype=_f32).expand(like.shape)


def is_virtual(t) -> bool:
    return getattr(t, "_b3d_virtual", False)


def sources(t):
    """P16 twins whose channel concatenation is `t` (None: the tensor has no twin)."""
    l = getattr(t, "_p16_list", None)
    if l is not None:
        return l
    tw = getattr(t, "_p16", None)
    return None if tw is None else [tw]


def to_p16(x, dtype, colsum=None):
    out = p16_empty(x.shape, x, dtype)
    _call("b3d_p16_pack", x, out, colsum)
    return out


def materialize(t):
    """fp32 NDHWC form of a possibly-virtual tensor (conversion kernel; only legacy / narrow-layer consumers)."""
    if not is_virtual(t):
        return t.contiguous()
    srcs = t._p16_list
    out = torch.empty(tuple(t.shape), device=srcs[0].device, dtype=_f32)
    o = 0
    for sp in srcs:
        c = sp.shape[3] * 8
        _call("b3d_p16_unpack", sp, out[..., o:o + c])
        o += c
    return out


_PREC = {"tf32": 0, "bf16": 1, "fp16": 2}
_PREC_INV = {v: k for k, v in _PREC.items()}


def set_conv_precision(fwd: str = "fp16", bwd: str = "bf16"):
    """Operand type of the tcgen05 conv MMAs ('tf32' | 'bf16' | 'fp16'; fp32 accumulation in TMEM either way),
    separately for the forward pass and the data gradient.  Default: forward fp16 — TF32's 11-bit significand
    (north_star: per-layer <= 2e-3, argmax agreement >= 99.9 %) at half the operand bytes; its narrow exponent
    is safe for the forward operands (image, GroupNorm outputs, O(1) weights; conversion saturates) — and backward
    bf16 (<= 1e-2; gradients need the exponent range).  The weight-gradient kernel always uses bf16 operands.
    Packed operands are re-made at their next use; CUDA graphs captured before the change must be re-captured."""
    for v in (fwd, bwd):
        if v not in _PREC:
            raise ValueError(v)
    lib.b3d_set_conv_precision(_PREC[fwd], _PREC[bwd])
    _PREC_EPOCH["n"] += 1


def set_kd_fold(on: bool) -> bool:
    """Switch the kd-folded 3x3x3 kernel for 16 / 32-channel output tiles (csrc/conv_tc.cu header) on or off; the
    packed operands of those layers change layout, so every registered pack is marked stale (CUDA graphs captured
    before the switch keep launching the old kernel variant on the re-laid-out buffers: re-capture them).  Returns
    the previous setting."""
    prev = bool(lib.b3d_set_conv_kdfold(int(bool(on))))
    _PREC_EPOCH["n"] += 1
    return prev


def get_conv_precision():
    v = lib.b3d_get_conv_precision()
    return (_PREC_INV[v & 15], _PREC_INV[v >> 4])


class _LazyGrad:
    """A gradient that exists only as its bf16 twin: `materialize()` unpacks it for the rare fp32 consumer."""
    _b3d_virtual = True

    def __init__(self, shape, twin):
        self.shape, self._p16_list = tuple(shape), [twin]


def _materialize_from(shape, srcs):
    out = torch.empty(tuple(shape), device=srcs[0].device, dtype=_f32)
    o = 0
    for sp in srcs:
        c = sp.shape[3] * 8
        _call("b3d_p16_unpack", sp, out[..., o:o + c])
        o += c
    return out


def _pad4(l):
    return list(l) + [None] * (4 - len(l))


def _p16_cat(srcs):
    """One P16 tensor holding the channel concatenation of `srcs` (plane-range copies; only where a kernel takes a
    single source: the small operand of a transposed conv's weight gradient)."""
    if len(srcs) == 1:
        return srcs[0]
    B, D, H, _, W, _ = srcs[0].shape
    out = torch.empty((B, D, H, sum(t.shape[3] for t in srcs), W, 8), device=srcs[0].device, dtype=srcs[0].dtype)
    o = 0
    for t in srcs:
        _call("b3d_p16_copy_planes", t, out, o)
        o += t.shape[3]
    return out


class Conv3dFn(Function):
    """Conv3D / Conv3DTranspose with TF 'SAME' padding (+bias, optional sigmoid), optionally emitting
    GroupNorm chunk statistics and global-average-pool sums of its output from the epilogue.

    Operands: when the input carries P16 twins (`sources(x)`: one, or several = a virtual channel concat) and the
    layer runs on the tensor cores with 16-bit operands, the kernels read the twins (b3d_conv3d_*_p16); the incoming
    gradient likewise (twin + bias gradient attached by the kernel that produced it, else packed here once for both
    the data and the weight gradient).  Everything else takes the fp32 entry points."""

    @staticmethod
    def forward(ctx, x, w, bias, stride, transposed, act, gn_groups, want_gap, share_x=False, grad_box=None):
        ctx.set_materialize_grads(False)       # no zero tensors for the statistics / pooling outputs in backward
        ctx.share_x = bool(share_x)
        ctx.grad_box = grad_box
        B, D, H, W_, Cin = x.shape
        k = w.shape[0]
        if transposed:
            Cout, od = w.shape[3], (2 * D, 2 * H, 2 * W_)
        else:
            Cout = w.shape[4]
            od = (D, H, W_) if stride == 1 else (D // 2, H // 2, W_ // 2)
        tc = USE_TC["on"] and (not act or stride == 1) and tc_supported(w, stride, transposed, False)
        srcs = sources(x)
        td = twin_dtype(False)
        use16 = bool(tc and srcs is not None and td is not None and len(srcs) <= 4 and srcs[0].dtype == td)
        if not use16:
            x = materialize(x)
            _check(x)
        y = _new((B,) + od + (Cout,), w)
        S = od[0] * od[1] * od[2]
        stats = gap = None
        if gn_groups and Cout % gn_groups == 0 and S % gn_groups == 0:
            stats = _new((B, gn_groups, 2), w, torch.float64)
        if want_gap:
            gap = _new((B, Cout), w)
        wp = None
        if tc:
            wp = pack_weights(w, False, stride, transposed)
        elif USE_TC["on"] and getattr(getattr(w, "_b3d_base", w), "_b3d_flat", None) is not None and \
                tc_supported(w, stride, transposed, True):
            wb = getattr(w, "_b3d_base", w)
            _register_pack(wb._b3d_flat, wb, True, stride, transposed)   # forward on CUDA cores, data gradient on TC
        nv = B * (D * H * W_ if transposed else S)      # voxels the FLOP formula counts (transposed: input voxels)
        _tag_conv(w, nv, stride, transposed)
        if use16:
            _call("b3d_conv3d_fwd_p16", *_pad4(srcs), w, bias, y, stride, int(transposed), int(act), stats,
                  gn_groups or 1, gap, 0, wp)
        else:
            _call("b3d_conv3d_fwd", x, w, bias, y, stride, int(transposed), int(act), stats, gn_groups or 1, gap, 0, wp)
        ctx.save_for_backward(None if use16 and is_virtual(x) else x, w, y if act else None)
        ctx.srcs = srcs if srcs is not None and td is not None and srcs[0].dtype == td else None
        # input = a virtual concat (VirtualConcatFn): its data gradient is written piece by piece (stride-1 convs)
        ctx.pieces = getattr(x, "_b3d_pieces", None) if (stride == 1 and not transposed) else None
        ctx.gradbox = getattr(x, "_b3d_gradbox", None) if ctx.pieces is not None else None
        ctx.srcs_w = sources_w(x) if ctx.srcs is not None else None
        ctx.xshape = tuple(x.shape)
        ctx.nv = nv
        ctx.cfg = (stride, transposed, act, bias is not None)
        ctx.params = (w, bias)
        # Mailbox shared with the ONE consumer of y (GroupNorm or the block epilogue; they pick it up in their forward):
        # it tells that kernel's backward which bias to write the column sums of dy into and whether this conv's
        # backward can work from a bf16 twin of dy alone, and carries the twin / bias gradient back to this conv's
        # backward.  (Python attributes on the gradient tensors themselves do not survive the autograd engine.)
        f32_grad = not (ctx.srcs_w is not None and twin_dtype(True) == torch.bfloat16 and lib.b3d_conv3d_wgrad_p16_plan(
            k, stride, int(transposed), Cin, Cout, od[2]) != 0)
        ctx.mb = y._b3d_mb = {"bias": bias, "f32_grad": f32_grad}
        if grad_box is not None and k == 1 and stride == 1 and not transposed:
            # the block's pointwise conv: the 3x3x3 conv reading the same x may compute its dx and dw (backward below)
            grad_box["pw"] = {"mb": ctx.mb, "w": w, "srcs_w": ctx.srcs_w}
        outs = (y, stats, gap)
        ctx.mark_non_differentiable(*[t for t in (stats, gap) if t is not None])
        return outs

    @staticmethod
    def backward(ctx, dy, _ds, _dg):
        if dy is None:                         # output unused by the loss (grads are not zero-materialised)
            return (None,) * 10
        x, w, y = ctx.saved_tensors
        srcs = ctx.srcs
        stride, transposed, act, has_bias = ctx.cfg
        mb = ctx.mb
        dy16 = mb.pop("dy16", None)                  # bf16 twin of dy left by the kernel that produced dy
        dbias = mb.pop("dbias", None)                # (tensor, written directly into the flat gradient buffer?)
        dy_real = mb.pop("dy_real", True)            # False: `dy` is a placeholder, only the twin holds the gradient
        td = twin_dtype(True)
        if dy16 is not None and dy16.dtype != td:
            dy = dy if dy_real else _materialize_from(dy.shape, [dy16])
            dy16, dy_real = None, True
        if not dy_real:
            dy = _LazyGrad(dy.shape, dy16)
        if act:
            dy = materialize(dy)
            t = torch.empty_like(dy)
            _call("b3d_sigmoid_bwd", dy, y, t)
            dy, dy16, dbias = t, None, None
        k, cin, cout = w.shape[0], ctx.xshape[-1], dy.shape[-1]
        need_dx, need_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        tcd = bool(need_dx and USE_TC["on"] and tc_supported(w, stride, transposed, True))
        plan = 0
        srcs_w = ctx.srcs_w
        if need_dw and td == torch.bfloat16 and srcs_w is not None and USE_TC["on"]:
            plan = lib.b3d_conv3d_wgrad_p16_plan(k, stride, int(transposed), cin, cout, dy.shape[3])
        pw, pb = ctx.params
        db = db_direct = None
        if need_dw and has_bias:
            if dbias is not None:
                db, db_direct = dbias
            else:
                db, db_direct = _grad_target(pb)
        bias_done = dbias is not None
        if dy16 is None and td is not None and p16_ok(dy.shape) and (plan or (tcd and is_virtual(dy))):
            # no twin came with the gradient (several consumers were summed by autograd, or a fp32 producer): one packing
            # pass serves the data gradient and the weight gradient and yields the bias gradient on the way
            dy16 = to_p16(materialize(dy), td, db if (need_dw and has_bias and not bias_done) else None)
            bias_done = bias_done or (need_dw and has_bias)
        dx = dw = None
        if need_dx:
            # Two convs reading the same tensor (pointwise + first 3x3x3 of a ResnetBlock) share a `grad_box`: the first
            # data gradient to run writes a fresh buffer and hands it to autograd, the second ADDS into that buffer in
            # its epilogue (accumulate = 1) and returns no gradient — same sum, no separate add pass over the tensor.
            # Better, where both run on tcgen05 with twins, ONE kernel computes both: the pointwise conv's incoming
            # gradient joins the 3x3x3 conv's as a further K segment used at the centre tap only
            # (b3d_conv3d_dgrad_p16_block) — no pointwise data-gradient launch at all.
            box, acc = ctx.grad_box, 0
            split = ctx.pieces is not None and ctx.gradbox is not None and tcd and dy16 is not None
            fused_pw = None
            if (box is not None and "pw" in box and "dx" not in box and k == 3 and stride == 1
                    and not transposed and tcd and dy16 is not None and box["pw"]["mb"] is not mb
                    and ctx.xshape[-1] % 16 == 0):
                dres16 = box["pw"]["mb"].get("dy16")
                if dres16 is not None and dres16.dtype == dy16.dtype and tuple(dres16.shape) == tuple(dy16.shape) and \
                        tc_supported(box["pw"]["w"], 1, False, True):
                    fused_pw = (dres16, box["pw"]["w"])
            if box is not None and box.get("dx_fused"):
                dx_buf = None                      # the 3x3x3 conv's kernel has already added this conv's part
            elif box is not None and "dx" in box:
                dx_buf, acc = box.pop("dx"), 1
            elif split:
                # one compact tensor per piece of the concatenated input, handed to VirtualConcatFn.backward through
                # the input's gradient box; autograd itself only sees a zero placeholder
                dx_buf = [torch.empty(ctx.xshape[:-1] + (c,), device=w.device, dtype=_f32) for c in ctx.pieces]
                parts = ctx.gradbox.setdefault("parts", [])
                parts.append(dx_buf)
                if box is not None:
                    box["dx"] = dx_buf
                # the first depositor hands autograd a zero placeholder (so that VirtualConcatFn.backward runs); later
                # ones return nothing — two placeholders would be "summed" by a full-size torch kernel
                dx = _zero_placeholder(ctx.xshape, w.device) if len(parts) == 1 else None
            else:
                dx_buf = torch.empty(ctx.xshape, device=w.device, dtype=_f32)
                if box is not None:
                    box["dx"] = dx_buf
                dx = dx_buf
            wp = pack_weights(w, True, stride, transposed) if (tcd and dx_buf is not None) else None
            _tag_conv(w, ctx.nv, stride, transposed)
            if dx_buf is None:
                _PROF["tag"] = None
            elif fused_pw is not None:
                bufs = dx_buf if isinstance(dx_buf, list) else [dx_buf]
                _call("b3d_conv3d_dgrad_p16_block", dy16, fused_pw[0], w, fused_pw[1], *_pad4(bufs), wp,
                      pack_weights(fused_pw[1], True, 1, False))
                box.pop("dx", None)
                box["dx_fused"] = True
            elif isinstance(dx_buf, list):
                if not (tcd and dy16 is not None):
                    raise RuntimeError("b3d: a split data gradient needs the P16 tensor-core path for both convs of a block")
                _call("b3d_conv3d_dgrad_p16_split", dy16, w, *_pad4(dx_buf), acc, wp)
            elif tcd and dy16 is not None:
                _call("b3d_conv3d_dgrad_p16", dy16, w, dx_buf, stride, int(transposed), acc, wp)
            else:
                dy = materialize(dy)
                _call("b3d_conv3d_dgrad", dy, w, dx_buf, stride, int(transposed), acc, wp)
        if need_dw:
            pwbox = ctx.grad_box.get("pw") if ctx.grad_box is not None else None
            pre = pwbox.pop("dw", None) if (pwbox is not None and pwbox["mb"] is mb) else None
            if pre is not None:                    # this pointwise conv's dw came out of the 3x3x3 layer's kernel
                dw, dw_direct = pre
                if has_bias and not bias_done:
                    _call("b3d_colsum", materialize(dy), db)
                _grad_done(pw, dw_direct)
                if has_bias:
                    _grad_done(pb, db_direct)
                return (dx, None if dw_direct else dw, None if (db_direct or not has_bias) else db,
                        None, None, None, None, None, None, None)
            if pwbox is not None and pwbox["mb"] is mb:
                pwbox["done"] = True
            dw, dw_direct = _grad_target(pw)
            # the same pair shares x in the weight-gradient pass too: where the 3x3x3 layer runs on the kd-in-M kernel
            # (csrc/conv_tc_wgrad.cu) the pointwise layer's dw is one more MMA per K step over the x tile already in
            # shared memory (b3d_conv3d_wgrad_p16_block) instead of a second pass over x
            fuse_w = None
            if (plan and dy16 is not None and pwbox is not None and pwbox["mb"] is not mb
                    and not pwbox.get("done") and k == 3 and stride == 1 and not transposed
                    and pwbox["w"].requires_grad and _same_sources(pwbox.get("srcs_w"), srcs_w)):
                dres16 = pwbox["mb"].get("dy16")
                if dres16 is not None and dres16.dtype == dy16.dtype and tuple(dres16.shape) == tuple(dy16.shape) and \
                        lib.b3d_conv3d_wgrad_p16_block_ok(cin, cout, dy.shape[2], dy.shape[3]):
                    fuse_w = dres16
            if fuse_w is not None:
                dwp, dwp_direct = _grad_target(pwbox["w"])
                _tag_conv(w, ctx.nv, stride, transposed)
                _call("b3d_conv3d_wgrad_p16_block", *_pad4(srcs_w), dy16, fuse_w, dw, dwp)
                pwbox["dw"] = (dwp, dwp_direct)
                if has_bias and not bias_done:
                    _call("b3d_colsum", materialize(dy), db)
            elif plan and dy16 is not None:
                scratch = None
                if plan == 2:
                    n = dy16.numel() if transposed else sum(t.numel() for t in srcs_w)
                    scratch = torch.empty(n, device=w.device, dtype=torch.bfloat16)
                elif plan == 3:
                    scratch = torch.empty(dy16.numel(), device=w.device, dtype=torch.bfloat16)
                xs = [_p16_cat(srcs_w)] if transposed else srcs_w
                _tag_conv(w, ctx.nv, stride, transposed)
                _call("b3d_conv3d_wgrad_p16", *_pad4(xs), dy16, dw, stride, int(transposed), scratch)
                if has_bias and not bias_done:
                    _call("b3d_colsum", materialize(dy), db)
            else:
                if x is None:
                    x = _materialize_from(ctx.xshape, srcs)
                dy = materialize(dy)
                xb = yb = None
                ready = 0
                if USE_TC["on"]:
                    xc, yc = _ll(), _ll()
                    kind = lib.b3d_conv3d_wgrad_plan(k, stride, int(transposed), cin, cout, _byref(xc), _byref(yc))
                    if kind:
                        # the two convs of a ResnetBlock (pointwise + first 3x3x3) read the same input: its plain bf16
                        # copy is made by whichever weight gradient runs first and handed to the other through the
                        # block's grad_box (one dict per ResnetBlock.call: nothing outlives the forward it belongs to)
                        holder = ctx.grad_box if (kind == 1 and stride == 1 and ctx.share_x) else None
                        need = x.numel() // x.shape[-1] * xc.value
                        xb = holder.pop("xb", None) if holder is not None else None
                        if xb is not None and xb.numel() == need and holder.pop("xb_ptr", None) == x.data_ptr():
                            ready = 1
                        else:
                            xb = torch.empty(need, device=x.device, dtype=torch.bfloat16)
                            if holder is not None:
                                holder["xb"], holder["xb_ptr"] = xb, x.data_ptr()
                        yb = torch.empty(dy.numel() // dy.shape[-1] * yc.value, device=x.device, dtype=torch.bfloat16)
                _tag_conv(w, ctx.nv, stride, transposed)
                _call("b3d_conv3d_wgrad", x, dy, dw, None if bias_done else db, stride, int(transposed), xb, yb, ready)
            _grad_done(pw, dw_direct)
            if has_bias:
                _grad_done(pb, db_direct)
            dw, db = (None if dw_direct else dw), (None if (db_direct or not has_bias) else db)
        return dx, dw, db, None, None, None, None, None, None, None


def _same_sources(a, b):
    return a is not None and b is not None and len(a) == len(b) and all(
        u.data_ptr() == v.data_ptr() and u.shape == v.shape and u.dtype == v.dtype for u, v in zip(a, b))


class FoldDupFn(Function):
    """Folded form of a Keras conv kernel whose input lists one tensor twice (SURVEY F3, encoder.py:83-87):
    (k,k,k,Cf+F,Cout) -> (k,k,k,Cf,Cout), the slice of the leading duplicate added to the slice of the last source.
    The folded tensor is persistent per layer and refreshed when the weights change; backward scatters its gradient
    straight into the kernel's slot of the flat gradient buffer (both slices receive the same values)."""

    @staticmethod
    def forward(ctx, w, F):
        F = int(F)
        st = getattr(w, "_b3d_fold", None)
        flat = getattr(w, "_b3d_flat", None)
        stamp = (w._version, flat.theta._version if flat is not None else 0, flat.epoch if flat is not None else 0)
        if st is None or st[0].shape[3] != w.shape[3] - F:
            wf = torch.empty(tuple(w.shape[:3]) + (w.shape[3] - F, w.shape[4]), device=w.device, dtype=_f32)
            st = [wf, None]
            w._b3d_fold = st
        if flat is not None and getattr(st[0], "_b3d_flat", None) is not flat:
            st[0]._b3d_flat = flat           # its packed operands join the batched re-pack (ops.repack_all)
            flat.folds.append((w, st[0], F))
        if st[1] != stamp:
            _call("b3d_fold_dup", w, st[0], F)
            st[1] = stamp
        ctx.F, ctx.param = F, w
        ctx.wshape = tuple(w.shape)
        # a fresh alias per call: the persistent tensor must not carry autograd history from one step (and stream) into
        # the next — under CUDA-graph capture that is a dependency on uncaptured work
        out = st[0].detach()
        out._b3d_base = st[0]
        return out

    @staticmethod
    def backward(ctx, dwf):
        pw = ctx.param
        dw, direct = _grad_target(pw)
        _call("b3d_unfold_dup", dwf.contiguous(), dw, ctx.F)
        _grad_done(pw, direct)
        return (None if direct else dw), None


def fold_dup(w, F):
    return FoldDupFn.apply(w, F)


def conv3d(x, w, bias=None, stride=1, transposed=False, act=0, gn_groups=0, want_gap=False, share_x=False,
           grad_box=None):
    ctx = _slab.current()
    if ctx is not None:        # depth-slab sharded inference: halo exchange, partial statistics / pooling sums
        return ctx.conv3d(x, w, bias, stride, transposed, act, want_gap, gn_groups)
    return Conv3dFn.apply(x, w, bias, stride, transposed, act, gn_groups, want_gap, share_x, grad_box)


class GroupNormFn(Function):
    """GroupNormalization.call (+ optional fused ReLU) with the reference's channels_last semantics
    (layers/group_norm.py:83-124, SURVEY F1).  `stats` may come from the producing conv's epilogue.

    Returns (y, y16): y16 = fp16 P16 twin for the convs that consume y (None when the tensor cannot feed the tensor
    cores); with `operand_only` y itself is a placeholder (`ops.virtual`).  Backward emits dx likewise: a bf16 twin
    for the data / weight gradient of the conv that produced x plus that conv's bias gradient, and — x being a raw
    conv output with exactly one consumer — no fp32 dx at all when the twin can be used."""

    @staticmethod
    def forward(ctx, x, gamma, beta, stats, groups, eps, relu, operand_only=False, grad_enabled=True):
        ctx.set_materialize_grads(False)       # the twin outputs get no gradient: do not let autograd zero-fill them
        ctx.mb = getattr(x, "_b3d_mb", None)         # mailbox of the conv that produced x (see Conv3dFn.forward)
        x = materialize(x)
        _check(x)
        C = x.shape[-1]
        # reference group_norm.py:51-59
        if C < groups:
            raise ValueError(f"Number of groups ({groups}) cannot be more than the number of channels ({C}).")
        if C % groups != 0:
            raise ValueError(f"Number of groups ({groups}) must be a multiple of the number of channels ({C}).")
        if stats is None:
            stats = _new((x.shape[0], groups, 2), x, torch.float64)
            _call("b3d_gn_stats", x, stats, groups, 0, 0)
        td = twin_dtype(False)
        L = x.numel() // x.shape[0] // groups
        twin = td is not None and p16_ok(x.shape) and L % 4 == 0
        y16 = p16_empty(x.shape, x, td) if twin else None
        y16b = p16_empty(x.shape, x, torch.bfloat16) if twin and want_wgrad_twin(td, grad_enabled) else None
        y = None if (twin and operand_only) else torch.empty_like(x)
        _call("b3d_gn_apply", x, stats, gamma, beta, y, y16, y16b, groups, float(eps), int(relu), 0, 0)
        if y is None:
            y = virtual(x.shape, x, [y16], [y16b] if y16b is not None else None)
        ctx.save_for_backward(x, gamma, beta, stats)
        ctx.cfg = (groups, float(eps), int(relu))
        ctx.params = (gamma, beta)
        if y16 is None:
            return y, None, None
        ctx.mark_non_differentiable(*[t for t in (y16, y16b) if t is not None])
        return y, y16, y16b

    @staticmethod
    def backward(ctx, dy, _d16=None, _d16b=None):
        if dy is None:
            return (None,) * 9
        x, gamma, beta, stats = ctx.saved_tensors
        groups, eps, relu = ctx.cfg
        dy = materialize(dy)
        pg, pb = ctx.params
        dgamma, dg_direct = _grad_target(pg)
        dbeta, db_direct = _grad_target(pb)
        csum = torch.empty_like(stats)
        _call("b3d_gn_bwd_reduce", dy, x, stats, gamma, beta, dgamma, dbeta, csum, groups, eps, relu)
        _grad_done(pg, dg_direct)
        _grad_done(pb, db_direct)
        td = twin_dtype(True)
        C = x.shape[-1]
        L = x.numel() // x.shape[0] // groups
        mb = ctx.mb
        twin = td is not None and p16_ok(x.shape) and L % 4 == 0 and mb is not None
        dx16 = dbias = None
        if twin:
            dx16 = p16_empty(x.shape, x, td)
            bias = mb["bias"]
            fused_bias = bias is not None and 1024 % C == 0 and L % C == 0
            dbias = _grad_target(bias) if fused_bias else None
            # the producing conv takes its weight gradient through the fp32 entry point (narrow layers): keep fp32 too
            dx = torch.empty_like(x) if mb["f32_grad"] else None
        else:
            dx = torch.empty_like(x)
        _call("b3d_gn_bwd_apply", dy, x, stats, gamma, beta, csum, dx, dx16, None if dbias is None else dbias[0],
              groups, eps, relu)
        if twin:
            mb["dy16"], mb["dbias"], mb["dy_real"] = dx16, dbias, dx is not None
            if dx is None:
                dx = _grad_placeholder(x)
        return dx, (None if dg_direct else dgamma), (None if db_direct else dbeta), None, None, None, None, None, None


class GroupNormChannelFn(Function):
    """GroupNormalization with TRUE channel groups (reference data_format='channels_first': group_norm.py axis=1)
    on NDHWC storage (csrc/norm_channel.cu), optional fused ReLU."""

    @staticmethod
    def forward(ctx, x, gamma, beta, groups, eps, relu):
        _check(x)
        x = x.contiguous()
        C = x.shape[-1]
        if C < groups:
            raise ValueError(f"Number of groups ({groups}) cannot be more than the number of channels ({C}).")
        if C % groups != 0:
            raise ValueError(f"Number of groups ({groups}) must be a multiple of the number of channels ({C}).")
        stats = _new((x.shape[0], groups, 2), x, torch.float64)
        _call("b3d_gn_channel_stats", x, stats, groups)
        y = _new_act(x.shape, x)
        _call("b3d_gn_channel_apply", x, stats, gamma, beta, y, groups, float(eps), int(relu))
        ctx.save_for_backward(x, gamma, beta, stats)
        ctx.cfg = (groups, float(eps), int(relu))
        ctx.params = (gamma, beta)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, beta, stats = ctx.saved_tensors
        groups, eps, relu = ctx.cfg
        pg, pb = ctx.params
        dgamma, dg_direct = _grad_target(pg)
        dbeta, db_direct = _grad_target(pb)
        csum, dx = torch.empty_like(stats), torch.empty_like(x)
        _call("b3d_gn_channel_bwd", dy.contiguous(), x, stats, gamma, beta, dgamma, dbeta, csum, dx, groups, eps, relu)
        _grad_done(pg, dg_direct)
        _grad_done(pb, db_direct)
        return dx, (None if dg_direct else dgamma), (None if db_direct else dbeta), None, None, None


def group_norm(x, gamma, beta, stats=None, groups=8, eps=1e-5, relu=False, channel_mode=False, operand_only=False):
    ctx = _slab.current()
    if channel_mode:
        if ctx is not None:    # channel-group statistics of the WHOLE volume: partial sums + all-reduce
            return ctx.group_norm_channel(x, gamma, beta, groups, eps, relu, operand_only)
        return GroupNormChannelFn.apply(x, gamma, beta, groups, eps, relu)
    if ctx is not None:        # chunk statistics of the WHOLE volume: partial sums + all-reduce
        return ctx.group_norm(x, gamma, beta, groups, eps, relu, stats, operand_only)
    y, y16, y16b = GroupNormFn.apply(x, gamma, beta, stats, groups, eps, relu, bool(operand_only),
                                     torch.is_grad_enabled())
    if y16 is not None and not is_virtual(y):
        _attach(y, y16, y16b)
    return y


class RelayoutFn(Function):
    """NCDHW <-> NDHWC copy at the boundary of the channels_first API surface (differentiable)."""

    @staticmethod
    def forward(ctx, x, to_last):
        _check(x)
        x = x.contiguous()
        B = x.shape[0]
        shape = (B,) + tuple(x.shape[2:]) + (x.shape[1],) if to_last else (B, x.shape[4]) + tuple(x.shape[1:4])
        y = _new(shape, x)
        _call("b3d_relayout", x, y, int(to_last))
        ctx.to_last = to_last
        return y

    @staticmethod
    def backward(ctx, dy):
        return RelayoutFn.apply(dy, not ctx.to_last), None


def to_channels_last(x):
    return RelayoutFn.apply(x, True)


def to_channels_first(x):
    return RelayoutFn.apply(x, False)


class BlockEpilogueFn(Function):
    """out = res*(sigmoid(res.w_sp) + chse) + relu(GN2(h2)),  chse = sigmoid(relu(mean(res) W1) W2)
    (layers/resnet.py:121-137).  With stats2=None, `h2` is taken as already normalised+activated.
    Returns (out, out16) like GroupNormFn; backward emits dres / dh2 as bf16 twins (+ the bias gradients of the
    pointwise and the second conv) when those convs can use them."""

    @staticmethod
    def forward(ctx, res, h2, stats2, gamma2, beta2, wsp, gap_sum, w1, w2, groups, eps, operand_only=False,
                grad_enabled=True):
        ctx.set_materialize_grads(False)
        _check(res)
        ctx.mbs = (getattr(res, "_b3d_mb", None), getattr(h2, "_b3d_mb", None))
        res, h2 = res.contiguous(), materialize(h2)
        B, F = res.shape[0], res.shape[-1]
        ctx_s = _slab.current()
        S = res.numel() // (B * F) if ctx_s is None else ctx_s.global_voxels(res)   # GAP divisor: whole volume
        R = w1.shape[1]
        hidden, chse = _new((B, R), res), _new((B, F), res)
        inv = 1.0 / S
        _call("b3d_se_fc_fwd", gap_sum, w1, w2, hidden, chse, inv)
        has_gn = stats2 is not None
        wsp_v = wsp.reshape(F)
        td = twin_dtype(False)
        twin = td is not None and p16_ok(res.shape)
        if twin:
            out16 = p16_empty(res.shape, res, td)
            out16b = p16_empty(res.shape, res, torch.bfloat16) if want_wgrad_twin(td, grad_enabled) else None
            out = None if operand_only else torch.empty_like(res)
        else:
            out16 = out16b = None
            out = _new_act(res.shape, res)
        _call("b3d_block_epilogue_fwd", res, h2, stats2, gamma2 if has_gn else None, beta2 if has_gn else None,
              wsp_v, chse, out, out16, out16b, groups, float(eps), int(has_gn), 0, 0)
        if out is None:
            out = virtual(res.shape, res, [out16], [out16b] if out16b is not None else None)
        ctx.save_for_backward(res, h2, stats2, gamma2, beta2, wsp, gap_sum, w1, w2, hidden, chse)
        ctx.cfg = (groups, float(eps), has_gn, inv)
        ctx.params = (gamma2, beta2, wsp, w1, w2)
        if out16 is None:
            return out, None, None
        ctx.mark_non_differentiable(*[t for t in (out16, out16b) if t is not None])
        return out, out16, out16b

    @staticmethod
    def backward(ctx, dout, _d16=None, _d16b=None):
        if dout is None:
            return (None,) * 13
        res, h2, stats2, gamma2, beta2, wsp, gap_sum, w1, w2, hidden, chse = ctx.saved_tensors
        groups, eps, has_gn, inv = ctx.cfg
        dout = materialize(dout)
        B, F = res.shape[0], res.shape[-1]
        wsp_v = wsp.reshape(F)
        pg, pb, pwsp, pw1, pw2 = ctx.params
        dchse = _new((B, F), res)
        dwsp, dwsp_direct = _grad_target(pwsp, (F,))
        dgamma, dg_direct = _grad_target(pg) if has_gn else (None, False)
        dbeta, db_direct = _grad_target(pb) if has_gn else (None, False)
        csum = torch.empty_like(stats2) if has_gn else None
        _call("b3d_block_epilogue_bwd_reduce", dout, res, h2 if has_gn else None, stats2,
              gamma2 if has_gn else None, beta2 if has_gn else None, wsp_v, dchse, dwsp, dgamma, dbeta, csum,
              groups, eps, int(has_gn))
        (dw1, dw1_direct), (dw2, dw2_direct), dgap = _grad_target(pw1), _grad_target(pw2), _new((B, F), res)
        _call("b3d_se_fc_bwd", gap_sum, w1, w2, hidden, chse, dchse, dw1, dw2, dgap, inv)
        for p_, d_ in ((pwsp, dwsp_direct), (pg, dg_direct), (pb, db_direct), (pw1, dw1_direct), (pw2, dw2_direct)):
            _grad_done(p_, d_)
        td = twin_dtype(True)
        mb_res, mb_h2 = ctx.mbs
        twin = td is not None and p16_ok(res.shape) and has_gn and mb_res is not None and mb_h2 is not None
        dres16 = dh216 = tb_res = tb_h2 = None
        if twin:
            b_res, b_h2 = mb_res["bias"], mb_h2["bias"]
            fused_bias = b_res is not None and b_h2 is not None
            dres16, dh216 = p16_empty(res.shape, res, td), p16_empty(res.shape, res, td)
            # the first block's pointwise conv (2 input channels) takes its weight gradient through the fp32 entry point
            dres = torch.empty_like(res) if mb_res["f32_grad"] else None
            dh2 = torch.empty_like(res) if mb_h2["f32_grad"] else None
            tb_res = _grad_target(b_res) if fused_bias else None
            tb_h2 = _grad_target(b_h2) if fused_bias else None
        else:
            dres = torch.empty_like(res)
            dh2 = torch.empty_like(h2) if has_gn else None
        _call("b3d_block_epilogue_bwd_apply", dout, res, h2 if has_gn else None, stats2,
              gamma2 if has_gn else None, beta2 if has_gn else None, wsp_v, chse, dgap, csum, dres, dh2, dres16, dh216,
              None if tb_res is None else tb_res[0], None if tb_h2 is None else tb_h2[0], groups, eps, int(has_gn))
        if twin:
            mb_res["dy16"], mb_res["dbias"], mb_res["dy_real"] = dres16, tb_res, dres is not None
            mb_h2["dy16"], mb_h2["dbias"], mb_h2["dy_real"] = dh216, tb_h2, dh2 is not None
            if dres is None:
                dres = _grad_placeholder(res)
            if dh2 is None:
                dh2 = _grad_placeholder(res)
        elif not has_gn:
            dh2 = dout
        return (dres, dh2, None, None if dg_direct else dgamma, None if db_direct else dbeta,
                None if dwsp_direct else dwsp.reshape(wsp.shape), None, None if dw1_direct else dw1,
                None if dw2_direct else dw2, None, None, None, None)


def block_epilogue(res, h2, stats2, gamma2, beta2, wsp, gap_sum, w1, w2, groups=8, eps=1e-5, keep_f32=False):
    sctx = _slab.current()
    if sctx is not None and sctx.p16 is not None and p16_ok(res.shape):
        return sctx.block_epilogue(res, h2, stats2, gamma2, beta2, wsp, gap_sum, w1, w2, groups, eps,
                                   keep_f32 or not FUSED["on"])
    operand_only = FUSED["on"] and sctx is None and not keep_f32
    out, out16, out16b = BlockEpilogueFn.apply(res, h2, stats2, gamma2, beta2, wsp, gap_sum, w1, w2, groups, eps,
                                               operand_only, torch.is_grad_enabled())
    if out16 is not None and not is_virtual(out):
        _attach(out, out16, out16b)
    return out


class DenseFn(Function):
    @staticmethod
    def forward(ctx, x, w, b, act):
        _check(x)
        x = x.contiguous()
        y = _new((x.shape[0], w.shape[1]), x)
        _call("b3d_dense_fwd", x, w, b, y, int(act))
        ctx.save_for_backward(x, w, y)
        ctx.cfg = (int(act), b is not None)
        ctx.params = (w, b)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, y = ctx.saved_tensors
        act, has_b = ctx.cfg
        dy = dy.contiguous()
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        pw, pb = ctx.params
        dw, dw_direct = _grad_target(pw)
        db, db_direct = _grad_target(pb) if has_b else (None, False)
        _call("b3d_dense_bwd", x, w, y, dy, dx, dw, db, act)
        _grad_done(pw, dw_direct)
        _grad_done(pb, db_direct)
        return dx, (None if dw_direct else dw), (None if db_direct else db), None


def dense(x, w, b=None, act=0):
    return DenseFn.apply(x, w, b, act)


class VaeSampleFn(Function):
    """proj = [z_mean | z_logvar] -> (z, z_mean, z_logvar),  z = z_mean + exp(0.5 z_logvar) * eps
    (layers/vae.py:9-13, 123-125)."""

    @staticmethod
    def forward(ctx, proj, eps):
        _check(proj)
        proj, eps = proj.contiguous(), eps.contiguous()
        B, L = proj.shape[0], proj.shape[1] // 2
        z = _new((B, L), proj)
        _call("b3d_vae_sample_fwd", proj, eps, z)
        ctx.save_for_backward(proj, eps)
        return z, proj[:, :L].contiguous(), proj[:, L:].contiguous()

    @staticmethod
    def backward(ctx, dz, dmu, dlv):
        proj, eps = ctx.saved_tensors
        dproj = torch.empty_like(proj)
        c = lambda t: None if t is None else t.contiguous()
        _call("b3d_vae_sample_bwd", proj, eps, c(dz), c(dmu), c(dlv), dproj)
        return dproj, None


def vae_sample(proj, eps):
    return VaeSampleFn.apply(proj, eps)


class DiceVAELossFn(Function):
    """util.py:13-24 as one reduction pass + a scalar finalize; backward is one elementwise pass.

    `dp` = (process group, world size): the batch-global objective under data parallelism — the reference sums I, P, T
    over the batch axis (util.py:11,18-20), so with one crop per rank the 3C+2 partial sums are all-reduced before the
    loss is formed; every rank then holds the loss of the WHOLE batch and backward yields its part of that gradient."""

    @staticmethod
    def forward(ctx, x, y, y_pred, y_vae, z_mean, z_logvar, dp=None):
        _check(y_pred, "y_pred")
        C = y_pred.shape[-1]
        vae = y_vae is not None
        c = lambda t: None if t is None else t.contiguous()
        x, y, y_pred, y_vae, z_mean, z_logvar = map(c, (x, y, y_pred, y_vae, z_mean, z_logvar))
        sums = _new((3 * C + 2,), y_pred, torch.float64)
        out = _new((4,), y_pred)
        _LAST_DICE["v"] = None
        if y_pred.dim() == 5 and y_pred.shape[3] % 4 == 0:
            # the hard-Dice metric of the same (y, y_pred) comes out of the same pass (picked up by dice_coefficient)
            acc, dice = _new((y_pred.shape[3] * C * 3,), y_pred), _new((2,), y_pred)
            _call("b3d_loss_dice_fwd", x if vae else None, y, y_pred, y_vae, z_mean if vae else None,
                  z_logvar if vae else None, sums, out, acc, dice, 0)
            _LAST_DICE["v"] = dice
        else:
            _call("b3d_loss_fwd", x if vae else None, y, y_pred, y_vae, z_mean if vae else None,
                  z_logvar if vae else None, sums, out)
        ctx.replicas = 1
        if dp is not None and dp[1] > 1:
            import torch.distributed as dist
            group, world = dp
            dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
            _call("b3d_loss_finalize", sums, out, world * x.numel() if vae else 0, world * z_mean.numel() if vae else 0)
            ctx.replicas = world
        ctx.save_for_backward(x if vae else None, y, y_pred, y_vae, z_mean if vae else None,
                              z_logvar if vae else None, sums)
        ctx.parts = out
        return out[0]

    @staticmethod
    def backward(ctx, g):
        x, y, y_pred, y_vae, z_mean, z_logvar, sums = ctx.saved_tensors
        vae = y_vae is not None
        g = g.reshape(1).contiguous().to(_f32)
        dyp = torch.empty_like(y_pred)
        dyv = torch.empty_like(y_vae) if vae else None
        dmu = torch.empty_like(z_mean) if vae else None
        dlv = torch.empty_like(z_logvar) if vae else None
        if ctx.replicas > 1:
            _call("b3d_loss_bwd_dp", x, y, y_pred, y_vae, z_mean, z_logvar, sums, g, dyp, dyv, dmu, dlv, ctx.replicas)
        else:
            _call("b3d_loss_bwd", x, y, y_pred, y_vae, z_mean, z_logvar, sums, g, dyp, dyv, dmu, dlv)
        return None, None, dyp, dyv, dmu, dlv, None


_LAST_DICE = {"v": None}       # (macro, micro) left by DiceVAELossFn.forward for its wrapper


def dice_vae_loss(x, y, y_pred, y_vae=None, z_mean=None, z_logvar=None, dp=None):
    loss = DiceVAELossFn.apply(x, y, y_pred, y_vae, z_mean, z_logvar, dp)
    dice, _LAST_DICE["v"] = _LAST_DICE["v"], None
    if dice is not None and y.is_contiguous() and y_pred.is_contiguous():
        import weakref
        # the metric of exactly these tensors, for a following dice_coefficient(y, y_pred) (train.py:143,147)
        y_pred._b3d_dice = (weakref.ref(y), y._version, y_pred._version, dice)
    return loss


def dice_coefficient(y_true, y_pred, reduce_w=False):
    """util.py:35-57 -> (macro, micro) as 0-d tensors (no gradient).  reduce_w: the channels_first macro average."""
    _check(y_pred, "y_pred")
    c = getattr(y_pred, "_b3d_dice", None)
    if c is not None and not reduce_w and c[0]() is y_true and c[1] == y_true._version and c[2] == y_pred._version:
        return c[3][0], c[3][1]                # computed by the loss kernel's pass over the same tensors
    y_true, y_pred = y_true.contiguous(), y_pred.detach().contiguous()
    W, C = y_pred.shape[3], y_pred.shape[4]
    acc = _new((W * C * 3,), y_pred)
    out = _new((2,), y_pred)
    _call("b3d_dice_coeff", y_true, y_pred, acc, out, int(reduce_w))
    return out[0], out[1]


class MaxPool2Fn(Function):
    """tf.keras.layers.MaxPooling3D(pool_size=2, strides=2, padding='same') on even sizes (downsample.py:58-62);
    the gradient goes to the first maximum of each 2x2x2 window."""

    @staticmethod
    def forward(ctx, x):
        x = materialize(x)
        _check(x)
        B, D, H, W, C = x.shape
        y = _new((B, D // 2, H // 2, W // 2, C), x)
        _call("b3d_maxpool2_fwd", x, y)
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dx = torch.empty_like(x)
        _call("b3d_maxpool2_bwd", x, dy.contiguous(), dx)
        return dx


def max_pool2(x):
    return MaxPool2Fn.apply(x)


class Upsample2Fn(Function):
    """tf.keras.layers.UpSampling3D(size=2): nearest-neighbour repetition (upsample.py:71-73)."""

    @staticmethod
    def forward(ctx, x):
        x = materialize(x)
        _check(x)
        B, D, H, W, C = x.shape
        y = _new((B, 2 * D, 2 * H, 2 * W, C), x)
        _call("b3d_upsample2_fwd", x, y)
        ctx.shape = tuple(x.shape)
        return y

    @staticmethod
    def backward(ctx, dy):
        dx = _new(ctx.shape, dy)
        _call("b3d_upsample2_bwd", dy.contiguous(), dx)
        return dx


def upsample2(x):
    return Upsample2Fn.apply(x)


class ConcatFn(Function):
    """Channel concat (encoder.py:85,91; decoder.py:75) materialised by strided copies."""

    @staticmethod
    def forward(ctx, *xs):
        xs = [materialize(t) for t in xs]
        C = [t.shape[-1] for t in xs]
        out = _new_act(tuple(xs[0].shape[:-1]) + (sum(C),), xs[0])
        o = 0
        for t, c in zip(xs, C):
            _call("b3d_copy_channels", t.contiguous(), out[..., o:o + c], 0)
            o += c
        ctx.C = C
        return out

    @staticmethod
    def backward(ctx, d):
        d = materialize(d)
        outs, o = [], 0
        for i, c in enumerate(ctx.C):
            if ctx.needs_input_grad[i]:
                g = _new(tuple(d.shape[:-1]) + (c,), d)
                _call("b3d_copy_channels", d[..., o:o + c], g, 0)
                outs.append(g)
            else:
                outs.append(None)
            o += c
        return tuple(outs)


class VirtualConcatFn(Function):
    """Channel concat of tensors that carry P16 twins, without a copy: the result is a placeholder listing the sources
    (the convs take up to 4 of them as K segments); the gradient of the concatenated tensor is handed back as channel
    slices (views) of the data gradient the consuming conv wrote."""

    @staticmethod
    def forward(ctx, *xs):
        C = [t.shape[-1] for t in xs]
        twins = [tw for t in xs for tw in sources(t)]
        wl = [sources_w(t) for t in xs]
        wtwins = [tw for l in wl for tw in l] if all(l is not None for l in wl) else None
        ctx.C = C
        out = virtual(tuple(xs[0].shape[:-1]) + (sum(C),), twins[0], twins, wtwins)
        # stride-1 convs reading `out` write their data gradient as one compact tensor per piece into this box
        # (Conv3dFn.backward) instead of one tensor that would have to be sliced — and copied — here
        out._b3d_pieces = tuple(C) if (len(C) <= 4 and all(c % 16 == 0 for c in C)) else None
        out._b3d_gradbox = ctx.box = {}
        return out

    @staticmethod
    def backward(ctx, d):
        parts = ctx.box.pop("parts", None)
        real = d is not None and not (d.dim() > 0 and all(st == 0 for st in d.stride()))   # not just the zero placeholder
        if real:
            d = materialize(d)
        outs, o = [], 0
        for i, c in enumerate(ctx.C):
            g = None
            if ctx.needs_input_grad[i]:
                if parts:
                    g = parts[0][i]
                    for other in parts[1:]:
                        g = g + other[i]
                    if real:
                        g = g + d[..., o:o + c]
                elif real:
                    g = d[..., o:o + c]
            outs.append(g)
            o += c
        return tuple(outs)


def concat(xs):
    td = twin_dtype(False)
    if FUSED["on"] and td is not None:
        srcs = [sources(t) for t in xs]
        if all(l is not None and all(tw.dtype == td for tw in l) for l in srcs) and sum(len(l) for l in srcs) <= 4:
            return VirtualConcatFn.apply(*xs)
    return ConcatFn.apply(*xs)


def dropout(x, rate, training, mask=None, seed=0, counter=None):
    """tf.keras.layers.Dropout on the (non-differentiable) input volume (encoder.py:39,71).
    `mask` injects a keep-mask for deterministic parity runs."""
    if not training or rate == 0.0:
        return x
    _check(x)
    x = x.contiguous()
    y = torch.empty_like(x)
    if mask is not None:
        _call("b3d_mul_scale", x, mask.contiguous(), y, 1.0 / (1.0 - rate))
    else:
        _call("b3d_dropout", x, y, None, float(rate), int(seed), counter)
    return y
