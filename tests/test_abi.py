"""CPU suite, part 2 — the C-ABI library loads, exports every symbol include/b3d.h declares, and rejects
host tensors (there is no CPU fallback) and contradictory optional arguments loudly.  No compute is launched here."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "b3d.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b3d_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported(b3d):
    lib = ctypes.CDLL(b3d._lib.LIB_PATH)
    names = _declared()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/b3d.h but not exported"
    assert lib.b3d_abi_version() == 2


def test_python_signatures_cover_header(b3d):
    declared = set(_declared()) - {"b3d_last_error", "b3d_abi_version", "b3d_conv3d_tc_supported",
                                   "b3d_conv3d_packed_elems", "b3d_conv3d_wgrad_tc_supported", "b3d_conv3d_wgrad_plan", "b3d_slab_sym_bytes", "b3d_set_wgrad_ts", "b3d_conv3d_pack_job", "b3d_conv3d_pack_job_bytes", "b3d_set_conv_kdfold",
                                   "b3d_set_conv_precision",
                                   "b3d_get_conv_precision", "b3d_conv3d_wgrad_p16_plan",
                                   "b3d_conv3d_wgrad_p16_block_ok"}
    assert declared == set(b3d._lib.SIGNATURES), declared ^ set(b3d._lib.SIGNATURES)


def test_host_side_planning_queries(b3d):
    """Pure host logic behind the C-ABI (no device needed): which layers the fused block weight gradient and the P16
    weight-gradient plans accept."""
    lib = b3d._lib.lib
    ok = lib.b3d_conv3d_wgrad_p16_block_ok
    # kd-in-M kernel: stride-1 3x3x3, Cin = 16 or a multiple of 32 up to 128, Cout 16 | 32, W % 8 == 0, H even
    assert ok(16, 16, 128, 128) == 1 and ok(32, 16, 128, 128) == 1 and ok(96, 32, 64, 64) == 1
    assert ok(256, 64, 32, 32) == 0          # Cout = 64: 9 accumulators do not fit the tensor memory
    assert ok(48, 16, 64, 64) == 0           # channel tiles of 32
    assert ok(32, 16, 64, 12) == 0 and ok(32, 16, 7, 16) == 0
    plan = lib.b3d_conv3d_wgrad_p16_plan
    assert plan(3, 2, 0, 32, 64, 32) == 2    # stride-2 family: space-to-depth scratch
    assert plan(3, 1, 0, 2, 16, 128) == 0    # narrow input: not on the P16 path
    assert plan(3, 1, 0, 64, 64, 32) == 1


def test_cpu_tensors_are_rejected(b3d):
    x = torch.zeros(1, 4, 4, 4, 8)
    st = torch.zeros(1, 8, 2, dtype=torch.float64)
    with pytest.raises(b3d._lib.B3DError, match="CUDA device"):
        b3d._lib.call("b3d_gn_stats", x, st, 8, 0, 0)
    with pytest.raises(RuntimeError, match="no CPU path"):
        b3d.ops.group_norm(x, torch.ones(8), torch.zeros(8))
    # optional outputs that contradict each other are B3D_ERR_ARG (-1) before any tensor is looked at: a second twin
    # without the first, bias gradients without a twin (only the twin kernels sum them), a gradient without any output
    v, t = torch.ones(8), torch.zeros(1, 4, 4, 1, 4, 8, dtype=torch.bfloat16)
    for name, args in (
            ("b3d_gn_apply", (x, st, v, v, x, None, t, 8, 1e-5, 0, 0, 0)),
            ("b3d_gn_bwd_apply", (x, x, st, v, v, st, x, None, v, 8, 1e-5, 0)),
            ("b3d_gn_bwd_apply", (x, x, st, v, v, st, None, None, None, 8, 1e-5, 0)),
            ("b3d_block_epilogue_fwd", (x, x, st, v, v, v, v, x, None, t, 8, 1e-5, 1, 0, 0)),
            ("b3d_block_epilogue_bwd_apply", (x, x, x, st, v, v, v, v, v, st, x, x, None, None, v, v, 8, 1e-5, 1)),
            ("b3d_block_epilogue_bwd_apply", (x, x, x, st, v, v, v, v, v, st, x, None, None, None, None, None, 8, 1e-5,
                                              1)),
            ("b3d_block_epilogue_bwd_apply", (x, x, x, st, v, v, v, v, v, st, None, None, t, t, v, None, 8, 1e-5, 1))):
        with pytest.raises(b3d._lib.B3DError, match=r"failed \(-1\)"):
            b3d._lib.call(name, *args)


def test_dlpack_struct_matches_torch_capsule(b3d):
    """Our hand-filled DLTensor equals what torch's own DLPack exporter produces."""
    t = torch.arange(24, dtype=torch.float32).reshape(2, 3, 4)[:, 1:, :]
    cap = torch.utils.dlpack.to_dlpack(t)
    ctypes.pythonapi.PyCapsule_GetPointer.restype = ctypes.c_void_p
    ctypes.pythonapi.PyCapsule_GetPointer.argtypes = [ctypes.py_object, ctypes.c_char_p]
    ptr = ctypes.pythonapi.PyCapsule_GetPointer(cap, b"dltensor")
    theirs = ctypes.cast(ptr, ctypes.POINTER(b3d._lib.DLTensor)).contents
    p, keep = b3d._lib.dl(t)
    mine = p.contents
    assert theirs.ndim == mine.ndim == 3
    assert (theirs.dtype.code, theirs.dtype.bits, theirs.dtype.lanes) == (mine.dtype.code, mine.dtype.bits, 1)
    assert [theirs.shape[i] for i in range(3)] == [mine.shape[i] for i in range(3)]
    assert [theirs.strides[i] for i in range(3)] == [mine.strides[i] for i in range(3)]
    assert theirs.data + theirs.byte_offset == mine.data + mine.byte_offset
    assert theirs.device.device_type == mine.device.device_type == 1


def test_constructor_surface_and_errors(b3d):
    import inspect
    sig = lambda f: list(inspect.signature(f).parameters)
    assert sig(b3d.Model.__init__)[1:] == ["data_format", "groups", "reduction", "l2_scale", "dropout",
                                           "downsampling", "upsampling", "base_filters", "depth", "in_ch", "out_ch"]
    assert sig(b3d.ResnetBlock.__init__)[1:] == ["filters", "data_format", "groups", "reduction", "l2_scale"]
    assert sig(b3d.GroupNormalization.__init__)[1:6] == ["groups", "axis", "epsilon", "center", "scale"]
    assert sig(b3d.Encoder.__init__)[1:] == ["data_format", "groups", "reduction", "l2_scale", "dropout",
                                             "downsampling", "base_filters", "depth"]
    assert sig(b3d.Decoder.__init__)[1:] == ["data_format", "groups", "reduction", "l2_scale", "upsampling",
                                             "base_filters", "depth", "out_ch"]
    with pytest.raises(ValueError, match="Reduction ratio"):          # resnet.py:39-42
        b3d.ResnetBlock(filters=10, reduction=4)
    m = b3d.Model()
    with pytest.raises(AssertionError):                               # model.py:60
        m.call(torch.zeros(1), training=True, inference=True)
    cfg = b3d.ResnetBlock(16).get_config()
    assert cfg["filters"] == 16 and cfg["reduction"] == 2 and cfg["groups"] == 8
    opt = b3d.ScheduledOptim(learning_rate=1e-4)
    opt(epoch=150)
    assert abs(float(opt.learning_rate) - 1e-4 * 0.5 ** 0.9) < 1e-12   # util.py:82-84
