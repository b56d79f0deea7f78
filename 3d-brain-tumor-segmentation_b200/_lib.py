"""ctypes binding of libb3d.so — the C-ABI declared in include/b3d.h.

Tensors cross the boundary as borrowed DLPack `DLTensor` structs (include/b3d_dlpack.h) that
are filled here straight from the torch tensor's pointer / shape / strides; nothing is copied
and no torch type appears in any signature.  There is NO CPU fallback: every entry point
rejects non-CUDA tensors, and importing this module fails loudly if the library is missing.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libb3d.so")


class DLDevice(C.Structure):
    _fields_ = [("device_type", C.c_int32), ("device_id", C.c_int32)]


class DLDataType(C.Structure):
    _fields_ = [("code", C.c_uint8), ("bits", C.c_uint8), ("lanes", C.c_uint16)]


class DLTensor(C.Structure):
    _fields_ = [("data", C.c_void_p), ("device", DLDevice), ("ndim", C.c_int32), ("dtype", DLDataType),
                ("shape", C.POINTER(C.c_int64)), ("strides", C.POINTER(C.c_int64)), ("byte_offset", C.c_uint64)]


_DT = {torch.float32: (2, 32), torch.float64: (2, 64), torch.int64: (0, 64), torch.bfloat16: (4, 16),
       torch.float16: (2, 16), torch.int32: (0, 32), torch.uint8: (1, 8)}

P = C.POINTER(DLTensor)


class _Holder:
    """Keeps the ctypes arrays of one DLTensor alive for the duration of a call."""
    __slots__ = ("t", "shape", "strides", "ref")


def dl(t: torch.Tensor | None):
    """torch tensor -> (pointer to a borrowed DLTensor, keep-alive object)."""
    if t is None:
        return None, None
    nd = t.dim()
    h = _Holder()
    h.ref = t
    h.shape = (C.c_int64 * max(nd, 1))(*t.shape)
    h.strides = (C.c_int64 * max(nd, 1))(*t.stride())
    code, bits = _DT[t.dtype]
    dev = DLDevice(2 if t.is_cuda else 1, t.device.index or 0)
    h.t = DLTensor(t.data_ptr(), dev, nd, DLDataType(code, bits, 1), h.shape, h.strides, 0)
    return C.pointer(h.t), h


def _load():
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"b3d: {LIB_PATH} not found — build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU / PyTorch fallback for the hot path.")
    return C.CDLL(LIB_PATH)


lib = _load()
lib.b3d_last_error.restype = C.c_char_p
lib.b3d_conv3d_packed_elems.restype = C.c_longlong

_i, _f, _v, _ll, _ull = C.c_int, C.c_float, C.c_void_p, C.c_longlong, C.c_ulonglong

# name -> argtypes ('T' = DLTensor*)
SIGNATURES = {
    "b3d_conv3d_fwd": "TTTTiiiTiTiTv",
    "b3d_conv3d_fwd_halo": "TTTTiiiiiTTv",
    "b3d_conv3d_dgrad": "TTTiiiTv",
    "b3d_conv3d_wgrad": "TTTTiiTTiv",
    "b3d_conv3d_pack_weights": "TTiiiv",
    "b3d_conv3d_pack_many": "TiLv",
    "b3d_gn_stats": "TTiLLv",
    "b3d_gn_apply": "TTTTTTTifiLLv",
    "b3d_gn_channel_stats": "TTiv",
    "b3d_gn_channel_apply": "TTTTTifiv",
    "b3d_gn_channel_bwd": "TTTTTTTTTifiv",
    "b3d_gn_channel_apply_slab": "TTTTTTifiLv",
    "b3d_relayout": "TTiv",
    "b3d_gn_bwd_reduce": "TTTTTTTTifiv",
    "b3d_gn_bwd_apply": "TTTTTTTTTifiv",
    "b3d_se_fc_fwd": "TTTTTfv",
    "b3d_se_fc_bwd": "TTTTTTTTTfv",
    "b3d_block_epilogue_fwd": "TTTTTTTTTTifiLLv",
    "b3d_block_epilogue_bwd_reduce": "TTTTTTTTTTTTifiv",
    "b3d_block_epilogue_bwd_apply": "TTTTTTTTTTTTTTTTifiv",
    "b3d_loss_fwd": "TTTTTTTTv",
    "b3d_loss_dice_fwd": "TTTTTTTTTTiv",
    "b3d_loss_bwd": "TTTTTTTTTTTTv",
    "b3d_loss_finalize": "TTLLv",
    "b3d_loss_bwd_dp": "TTTTTTTTTTTTiv",
    "b3d_dice_coeff": "TTTTiv",
    "b3d_dense_fwd": "TTTTiv",
    "b3d_dense_bwd": "TTTTTTTiv",
    "b3d_vae_sample_fwd": "TTTv",
    "b3d_vae_sample_bwd": "TTTTTTv",
    "b3d_adam_step": "TTTTTfffffLiv",
    "b3d_l2_losses": "TTTfv",
    "b3d_l2_grad": "TTTTfv",
    "b3d_axpy": "TTLfTv",
    "b3d_sum_add": "TTTv",
    "b3d_zero": "Tv",
    "b3d_dropout": "TTTfUTv",
    "b3d_mul_scale": "TTTfv",
    "b3d_sigmoid_bwd": "TTTv",
    "b3d_copy_channels": "TTiv",
    "b3d_channel_moments": "TTv",
    "b3d_augment_crop": "TTTTTTTiiiiv",
    "b3d_maxpool2_fwd": "TTv",
    "b3d_maxpool2_bwd": "TTTv",
    "b3d_upsample2_fwd": "TTv",
    "b3d_upsample2_bwd": "TTv",
    "b3d_halo_exchange": "TTTTLLTTiLv",
    "b3d_peer_allreduce": "TTiTTiv",
    "b3d_peer_allreduce2": "TTTiTTiv",
    "b3d_conv3d_fwd_p16_slab": "TTTTTTTiiiiiTiLLTTiv",
    "b3d_epoch_tick": "Tv",
    "b3d_flip_normalize": "TTTTiv",
    "b3d_flip_accumulate": "TTTifiv",
    # evaluation of one segmented volume (csrc/metrics.cu)
    "b3d_label_map": "TTfv",
    "b3d_region_surface": "TTTTTTv",
    "b3d_surface_edt": "TTifffv",
    "b3d_hd95": "TTTTTTTv",
    # P16 operand twins (csrc/p16.cu) and the entry points that produce / consume them
    "b3d_p16_pack": "TTTv",
    "b3d_p16_unpack": "TTv",
    "b3d_p16_copy_planes": "TTiv",
    "b3d_colsum": "TTv",
    "b3d_fold_dup": "TTiv",
    "b3d_unfold_dup": "TTiv",
    "b3d_conv3d_fwd_p16": "TTTTTTTiiiTiTiTv",
    "b3d_conv3d_dgrad_p16_split": "TTTTTTiTv",
    "b3d_conv3d_dgrad_p16_block": "TTTTTTTTTTv",
    "b3d_conv3d_dgrad_p16": "TTTiiiTv",
    "b3d_conv3d_wgrad_p16": "TTTTTTiiTv",
    "b3d_conv3d_wgrad_p16_block": "TTTTTTTTv",
    "b3d_conv3d_wgrad_narrow": "TTTTTTv",
}
_CT = {"T": P, "i": _i, "f": _f, "v": _v, "L": _ll, "U": _ull}
for _name, _sig in SIGNATURES.items():
    fn = getattr(lib, _name)
    fn.argtypes = [_CT[c] for c in _sig]
    fn.restype = C.c_int
lib.b3d_conv3d_tc_supported.argtypes = [_i] * 6
lib.b3d_conv3d_tc_supported.restype = _i
lib.b3d_conv3d_packed_elems.argtypes = [_i] * 4
lib.b3d_conv3d_wgrad_tc_supported.argtypes = [_i] * 5
lib.b3d_conv3d_wgrad_tc_supported.restype = _i
lib.b3d_conv3d_wgrad_plan.argtypes = [_i] * 5 + [C.POINTER(_ll), C.POINTER(_ll)]
lib.b3d_conv3d_wgrad_plan.restype = _i
lib.b3d_set_conv_precision.argtypes = [_i, _i]
lib.b3d_set_conv_kdfold.argtypes = [_i]
lib.b3d_set_conv_kdfold.restype = _i
lib.b3d_conv3d_pack_job.argtypes = [P, P, _i, _i, _i, _ll, _v, C.POINTER(_ll)]
lib.b3d_conv3d_pack_job.restype = _i
lib.b3d_conv3d_pack_job_bytes.restype = _i
lib.b3d_slab_sym_bytes.argtypes = [_ll]
lib.b3d_slab_sym_bytes.restype = _ll
lib.b3d_get_conv_precision.restype = _i
lib.b3d_conv3d_wgrad_p16_plan.argtypes = [_i] * 6
lib.b3d_conv3d_wgrad_p16_plan.restype = _i
lib.b3d_conv3d_wgrad_p16_block_ok.argtypes = [_i] * 4
lib.b3d_conv3d_wgrad_p16_block_ok.restype = _i
lib.b3d_conv3d_wgrad_narrow_ok.argtypes = [_i] * 4
lib.b3d_conv3d_wgrad_narrow_ok.restype = _i


class B3DError(RuntimeError):
    pass


_HAS_CUDA = torch.cuda.is_available()


def stream_ptr() -> int:
    # without a GPU every entry point rejects its (host) tensors before touching the stream
    return torch.cuda.current_stream().cuda_stream if _HAS_CUDA else 0


def call(name: str, *args):
    """Invoke a C-ABI entry point.  torch tensors (or None) are converted to DLTensor*; the current
    torch CUDA stream is appended as the trailing `void* stream` argument."""
    sig = SIGNATURES[name]
    cargs, keep = [], []
    it = iter(args)
    for c in sig[:-1]:
        a = next(it)
        if c == "T":
            p, h = dl(a)
            keep.append(h)
            cargs.append(p)
        else:
            cargs.append(a)
    cargs.append(stream_ptr())
    rc = getattr(lib, name)(*cargs)
    if rc != 0:
        msg = lib.b3d_last_error().decode()
        if rc == -5 and ("Number of groups" in msg or "Reduction ratio" in msg):
            raise ValueError(msg)         # reference raises ValueError for these (group_norm.py:51-59)
        raise B3DError(f"{name} failed ({rc}): {msg}")
    return rc
