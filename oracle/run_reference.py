"""ORACLE / test infrastructure.  Imports the reference's OWN hot-path python files
({model.py,layers/*.py,util.py} of the original project) UNMODIFIED on top of oracle/tf_shim and runs
them on this repo's synthetic weights/inputs.  Only usable where a checkout of the original project is
installed: at oracle/_ref/ (kept out of git), or wherever the environment variable B3D_REFERENCE names;
elsewhere tests use the fixtures this produces (tests/golden/*.npz, written by oracle/make_golden.py).
"""
from __future__ import annotations

import importlib
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.abspath(os.environ.get("B3D_REFERENCE") or os.path.join(HERE, "_ref"))


def available() -> bool:
    return os.path.isfile(os.path.join(REF, "model.py"))


def _import_reference():
    if not available():
        raise RuntimeError(f"no checkout of the original project at {REF} (install it at oracle/_ref/ or set "
                           "B3D_REFERENCE to its directory)")
    shim = os.path.join(HERE, "tf_shim")
    for p in (REF, shim):
        if p not in sys.path:
            sys.path.insert(0, p)
    # the reference's top-level module names are generic ('model', 'util', 'layers'): import them
    # under a clean slate and hand back the module objects
    for m in ("model", "util", "layers"):
        sys.modules.pop(m, None)
    for m in [k for k in sys.modules if k.startswith("layers.")]:
        sys.modules.pop(m)
    import tensorflow as tf  # noqa: F401  (the shim)
    assert "tf_shim" in tf.__file__, "real TensorFlow found?  the shim must shadow it"
    ref_model = importlib.import_module("model")
    ref_util = importlib.import_module("util")
    assert ref_model.__file__.startswith(REF + os.sep), ref_model.__file__
    return tf, ref_model, ref_util


def _set(holder, attr, value):
    """Overwrite a shim weight in place (keeps the tensor object that the layer tracks)."""
    w = getattr(holder, attr)
    with torch.no_grad():
        assert tuple(w.shape) == tuple(value.shape), (attr, w.shape, value.shape)
        w.copy_(value)


def _load_block(blk, p, pre):
    _set(blk.conv3d_ptwise, "kernel", p[pre + "ptwise.kernel"])
    _set(blk.conv3d_ptwise, "bias", p[pre + "ptwise.bias"])
    _set(blk.dense_relu, "kernel", p[pre + "dense_relu.kernel"])
    _set(blk.dense_sigmoid, "kernel", p[pre + "dense_sigmoid.kernel"])
    _set(blk.spatial, "kernel", p[pre + "spatial.kernel"])
    for i in (0, 1):
        conv, norm, _ = blk.convs[i]
        _set(conv, "kernel", p[pre + f"conv{i+1}.kernel"])
        _set(conv, "bias", p[pre + f"conv{i+1}.bias"])
        _set(norm, "gamma", p[pre + f"gn{i+1}.gamma"])
        _set(norm, "beta", p[pre + f"gn{i+1}.beta"])


def _load_resample(layer, p, pre):
    if not hasattr(layer, "conv"):                  # MaxDownsample (no weights) / LinearUpsample (1x1x1 conv)
        if hasattr(layer, "ptwise"):
            _set(layer.ptwise, "kernel", p[pre + "ptwise.kernel"])
            _set(layer.ptwise, "bias", p[pre + "ptwise.bias"])
        return
    _set(layer.conv, "kernel", p[pre + "conv.kernel"])
    _set(layer.conv, "bias", p[pre + "conv.bias"])
    _set(layer.norm, "gamma", p[pre + "norm.gamma"])
    _set(layer.norm, "beta", p[pre + "norm.beta"])


def load_params(model, p, depth=4, with_vae=True):
    for i, (convs, _, down) in enumerate(model.encoder.levels):
        for j, (blk, _) in enumerate(convs):
            _load_block(blk, p, f"enc.L{i}.B{j}.")
        if down is not None:
            _load_resample(down, p, f"enc.L{i}.down.")
    for i, (up, _, blk) in zip(range(depth - 2, -1, -1), model.decoder.levels):
        _load_resample(up, p, f"dec.L{i}.up.")
        _load_block(blk, p, f"dec.L{i}.block.")
    _set(model.decoder.out, "kernel", p["dec.out.kernel"])
    _set(model.decoder.out, "bias", p["dec.out.bias"])
    if with_vae:
        v = model.vae
        _load_resample(v.downsample, p, "vae.down.")
        _set(v.proj, "kernel", p["vae.proj.kernel"])
        _set(v.proj, "bias", p["vae.proj.bias"])
        _set(v.unproj, "kernel", p["vae.unproj.kernel"])
        _set(v.unproj, "bias", p["vae.unproj.bias"])
        _load_resample(v.upsample, p, "vae.up.")
        for i, (up, blk) in zip(range(depth - 2, -1, -1), v.levels):
            _load_resample(up, p, f"vae.L{i}.up.")
            _load_block(blk, p, f"vae.L{i}.block.")
        _set(v.out, "kernel", p["vae.out.kernel"])
        _set(v.out, "bias", p["vae.out.bias"])


def import_reference_test_module():
    """The reference's inference script test.py (TestTimeAugmentor :75-161, pad_to_spatial_res :164-178) as a module.
    It is loaded by path (a bare `import test` would find CPython's own `test` package) with an empty stand-in for
    nibabel, which is not in this image and is only used by the NIfTI reader/writer functions."""
    import importlib.util
    import types
    _import_reference()
    sys.modules.setdefault("nibabel", types.ModuleType("nibabel"))
    spec = importlib.util.spec_from_file_location("b3d_reference_test_py", os.path.join(REF, "test.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def import_reference_train_module():
    """The reference's train.py (prepare_dataset :12-68 with its per-example map function) as a module, by path."""
    import importlib.util
    _import_reference()
    spec = importlib.util.spec_from_file_location("b3d_reference_train_py", os.path.join(REF, "train.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class ReferenceRunner:
    """Builds the reference Model(**model_args) on the shim and loads `params` (this repo's names)."""

    def __init__(self, params, in_shape, dtype=torch.float64, **model_args):
        self.tf, self.ref_model, self.ref_util = _import_reference()
        self.tf.DTYPE = dtype
        self.depth = model_args.get("depth", 4)
        self.model = self.ref_model.Model(**model_args)
        # train.py:96 / test.py:188 — weights are created by a first call on zeros
        self.tf.random.injected_normal = None
        self.model(torch.zeros(in_shape, dtype=dtype), training=False, inference=False)
        load_params(self.model, {k: v.to(dtype) for k, v in params.items()}, self.depth)

    def forward(self, x, eps=None, training=False, inference=False, dropout_mask=None):
        self.tf.random.injected_normal = eps
        self.tf.keras.layers.Dropout.injected_mask = dropout_mask
        try:
            return self.model(x, training=training, inference=inference)
        finally:
            self.tf.random.injected_normal = None
            self.tf.keras.layers.Dropout.injected_mask = None

    def loss(self, x, y, outs, data_format="channels_last"):
        """train.py:145-146"""
        loss_fn = self.ref_util.DiceVAELoss(data_format=data_format)
        l = loss_fn(x, y, *outs)
        return l + self.tf.reduce_sum(self.model.losses)

    def dice(self, y, y_pred, data_format="channels_last"):
        return self.ref_util.DiceCoefficient(data_format=data_format)(y, y_pred)

    def named_variables(self):
        """this repo's name -> reference variable tensor (for gradient comparison)"""
        out = {}

        def blk(b, pre):
            out[pre + "ptwise.kernel"] = b.conv3d_ptwise.kernel
            out[pre + "ptwise.bias"] = b.conv3d_ptwise.bias
            out[pre + "dense_relu.kernel"] = b.dense_relu.kernel
            out[pre + "dense_sigmoid.kernel"] = b.dense_sigmoid.kernel
            out[pre + "spatial.kernel"] = b.spatial.kernel
            for i in (0, 1):
                conv, norm, _ = b.convs[i]
                out[pre + f"conv{i+1}.kernel"] = conv.kernel
                out[pre + f"conv{i+1}.bias"] = conv.bias
                out[pre + f"gn{i+1}.gamma"] = norm.gamma
                out[pre + f"gn{i+1}.beta"] = norm.beta

        def rs(l, pre):
            if not hasattr(l, "conv"):
                if hasattr(l, "ptwise"):
                    out[pre + "ptwise.kernel"], out[pre + "ptwise.bias"] = l.ptwise.kernel, l.ptwise.bias
                return
            out[pre + "conv.kernel"] = l.conv.kernel
            out[pre + "conv.bias"] = l.conv.bias
            out[pre + "norm.gamma"] = l.norm.gamma
            out[pre + "norm.beta"] = l.norm.beta

        m, depth = self.model, self.depth
        for i, (convs, _, down) in enumerate(m.encoder.levels):
            for j, (b, _) in enumerate(convs):
                blk(b, f"enc.L{i}.B{j}.")
            if down is not None:
                rs(down, f"enc.L{i}.down.")
        for i, (up, _, b) in zip(range(depth - 2, -1, -1), m.decoder.levels):
            rs(up, f"dec.L{i}.up.")
            blk(b, f"dec.L{i}.block.")
        out["dec.out.kernel"], out["dec.out.bias"] = m.decoder.out.kernel, m.decoder.out.bias
        v = m.vae
        rs(v.downsample, "vae.down.")
        out["vae.proj.kernel"], out["vae.proj.bias"] = v.proj.kernel, v.proj.bias
        out["vae.unproj.kernel"], out["vae.unproj.bias"] = v.unproj.kernel, v.unproj.bias
        rs(v.upsample, "vae.up.")
        for i, (up, b) in zip(range(depth - 2, -1, -1), v.levels):
            rs(up, f"vae.L{i}.up.")
            blk(b, f"vae.L{i}.block.")
        out["vae.out.kernel"], out["vae.out.bias"] = v.out.kernel, v.out.bias
        return out
