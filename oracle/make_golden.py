"""ORACLE / test infrastructure.  Generates tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN FILES
({model.py,layers/*.py,util.py} of the original project) on oracle/tf_shim (see oracle/run_reference.py) in fp64.
Needs a checkout of the original project at oracle/_ref/ or at $B3D_REFERENCE:   python -m oracle.make_golden
Without one, tests read the committed fixtures.

Fixtures (small on purpose; weights/inputs are regenerated from seeds by oracle.ref_model):
  model_16.npz : full model, 16^3 crop, training call (dropout mask + eps injected), loss, dice,
                 gradients of 14 representative tensors (the largest one sampled) + L2 norms of all 260 gradients
  gn_cases.npz : GroupNormalization.call on odd shapes (chunk boundary mid-slice, C/G = 1, 2, 4)
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_model as R  # noqa: E402
from oracle.run_reference import REF, ReferenceRunner, _import_reference, available  # noqa: E402

GRAD_KEYS = ["enc.L0.B0.conv1.kernel", "enc.L0.B0.gn2.gamma", "enc.L0.B0.spatial.kernel",
             "enc.L1.B1.dense_relu.kernel", "enc.L2.B2.ptwise.kernel", "enc.L3.B3.conv2.kernel",
             "enc.L0.down.conv.kernel", "dec.L0.up.conv.kernel", "dec.L1.block.gn1.beta", "dec.out.kernel",
             "vae.proj.kernel", "vae.unproj.bias", "vae.L0.block.conv2.bias", "vae.out.kernel"]
# a larger gradient is stored as every GRAD_STRIDE-th element of its flattened array (prime: the sample runs
# through every kernel tap and channel position)
SAMPLE_ABOVE = 1 << 16
GRAD_STRIDE = 17


def model_case(crop, out):
    shapes = R.param_shapes(crop=crop)
    p = R.init_params(shapes)
    x, y, eps, mask = R.synth_batch((1,) + crop)
    rr = ReferenceRunner(p, (1,) + crop + (2,))
    outs = rr.forward(x, eps=eps, training=True, dropout_mask=mask)
    loss = rr.loss(x, y, outs)
    macro, micro = rr.dice(y, outs[0])
    loss.backward()
    nv = rr.named_variables()
    d = {"y_pred": outs[0].detach().numpy().astype(np.float32),
         "y_vae": outs[1].detach().numpy().astype(np.float32),
         "z_mean": outs[2].detach().numpy(), "z_logvar": outs[3].detach().numpy(),
         "loss": np.float64(loss.item()), "macro": np.float64(macro.item()), "micro": np.float64(micro.item()),
         "grad_names": np.array(sorted(nv)),
         "grad_norms": np.array([float(nv[k].grad.norm()) for k in sorted(nv)])}
    for k in GRAD_KEYS:
        g = nv[k].grad.numpy().astype(np.float32)
        if g.size > SAMPLE_ABOVE:          # keeps the fixture file under 1 MB; its norm is in grad_norms
            d["grad_sample:" + k] = np.ascontiguousarray(g.reshape(-1)[::GRAD_STRIDE])
            d["grad_stride"] = np.int64(GRAD_STRIDE)
        else:
            d["grad:" + k] = g
    # inference call (VAE off) on the same weights
    yi = rr.forward(x, training=False, inference=True)[0]
    d["y_pred_inference"] = yi.detach().numpy().astype(np.float32)
    np.savez_compressed(out, **d)
    print(out, {k: getattr(v, "shape", None) for k, v in d.items() if not k.startswith("grad")})


def gn_cases(out):
    tf, _, _ = _import_reference()
    import importlib
    gn = importlib.import_module("layers.group_norm")
    rng = np.random.default_rng(11)
    d = {}
    for i, shp in enumerate([(1, 20, 6, 4, 16), (2, 5, 3, 3, 8), (1, 4, 4, 4, 32), (2, 2, 2, 2, 64)]):
        x = torch.from_numpy(rng.standard_normal(shp))
        layer = gn.GroupNormalization(groups=8, axis=-1)
        layer(x)
        with torch.no_grad():
            layer.gamma.copy_(torch.from_numpy(1 + 0.3 * rng.standard_normal(shp[-1])))
            layer.beta.copy_(torch.from_numpy(0.3 * rng.standard_normal(shp[-1])))
        y = layer(x)
        d[f"x{i}"], d[f"gamma{i}"], d[f"beta{i}"], d[f"y{i}"] = (x.numpy(), layer.gamma.detach().numpy(),
                                                                 layer.beta.detach().numpy(), y.detach().numpy())
    np.savez_compressed(out, **d)
    print(out)


if __name__ == "__main__":
    if not available():
        sys.exit(f"make_golden: no checkout of the original project at {REF} (install it at oracle/_ref/ or set "
                 "B3D_REFERENCE to its directory)")
    g = os.path.join(ROOT, "tests", "golden")
    os.makedirs(g, exist_ok=True)
    model_case((16, 16, 16), os.path.join(g, "model_16.npz"))
    gn_cases(os.path.join(g, "gn_cases.npz"))
