"""b3d — B200-native (sm_100a) hot path of the 3D U-Net + VAE brain-tumour segmenter of
vliu15/3d-brain-tumor-segmentation, behind the reference's own layer / model / loss API.

    from importlib import import_module
    b3d = import_module("3d-brain-tumor-segmentation_b200")
    model = b3d.Model()                     # same kwargs as the reference's model.Model
    y_pred, y_vae, z_mean, z_logvar = model(x, training=True, inference=False)

Importing this package loads csrc/libb3d.so (hand-written CUDA behind a C-ABI, include/b3d.h) and fails
loudly if it has not been built; nothing on the product path falls back to CPU or to library kernels.
"""
from . import _lib, ops  # noqa: F401  (loads the shared library)
from .layers import (GroupNormalization, ResnetBlock, ConvDownsample, MaxDownsample, ConvUpsample,  # noqa: F401
                     LinearUpsample, Encoder, Decoder, VariationalAutoencoder, get_downsampling, get_upsampling)
from .model import Model  # noqa: F401
from .util import DiceVAELoss, DiceCoefficient, ScheduledOptim  # noqa: F401
from . import train, infer, slab, data, metrics  # noqa: F401
from .data import parse_example, VolumeDataset  # noqa: F401
from .slab import (SlabContext, DistComm, PeerComm, ThreadComm, slab_bounds, sharded_inference,  # noqa: F401
                   GraphedInference)
from .infer import TestTimeAugmentor, pad_to_spatial_res  # noqa: F401
from .metrics import BRATS_REGIONS, predict_labels, segmentation_metrics  # noqa: F401
from .train import GradientTape, train_step, GraphedTrainStep, DataParallel, reduce_sum, TrainLog  # noqa: F401

__all__ = ["GroupNormalization", "ResnetBlock", "ConvDownsample", "MaxDownsample", "ConvUpsample",
           "LinearUpsample", "Encoder", "Decoder", "VariationalAutoencoder", "Model", "DiceVAELoss",
           "DiceCoefficient", "ScheduledOptim", "GradientTape", "train_step", "GraphedTrainStep"]
