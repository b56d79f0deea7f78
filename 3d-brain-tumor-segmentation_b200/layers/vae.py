"""VariationalAutoencoder — surface of /root/reference/layers/vae.py (:9-13 sample, :17-99 ctor,
:101-111 build, :114-143 call).  `eps` may be injected for deterministic parity runs; by default
it is drawn ~N(0,1) on every call, training or not, as the reference does (SURVEY F5)."""
import torch

from ..keras_compat import Layer, Conv3D, Dense, L2
from .. import ops
from .downsample import get_downsampling
from .upsample import get_upsampling
from .resnet import ResnetBlock


def sample(inputs, eps=None):
    """Samples from the Gaussian given by mean and log-variance (vae.py:9-13) from proj=[mean|logvar]."""
    proj = inputs
    if eps is None:
        eps = torch.randn((proj.shape[0], proj.shape[1] // 2), device=proj.device, dtype=torch.float32)
    return ops.vae_sample(proj, eps)


class VariationalAutoencoder(Layer):
    def __init__(self,
                 data_format='channels_last',
                 groups=8,
                 reduction=2,
                 l2_scale=1e-5,
                 downsampling='conv',
                 upsampling='conv',
                 base_filters=16,
                 depth=4,
                 out_ch=2):
        super().__init__()
        self.data_format = data_format
        self.l2_scale = l2_scale
        self.config = super().get_config()
        self.config.update({'groups': groups,
                            'reduction': reduction,
                            'downsampling': downsampling,
                            'upsampling': upsampling,
                            'base_filters': base_filters,
                            'depth': depth,
                            'out_ch': out_ch})
        Downsample = get_downsampling(downsampling)
        Upsample = get_upsampling(upsampling)

        # NB the reference passes kernel_regularizer= here, which ConvDownsample swallows (vae.py:53-57);
        # the conv still gets the default l2_scale=1e-5 regulariser.
        self.downsample = Downsample(filters=base_filters // 2, groups=groups, data_format=data_format,
                                     kernel_regularizer=L2(l2_scale))

        self.proj = Dense(units=base_filters * (2 ** (depth - 1)), kernel_regularizer=L2(l2_scale),
                          kernel_initializer='he_normal')
        self.latent_size = base_filters * (2 ** (depth - 2))

        self.upsample = Upsample(filters=base_filters * (2 ** (depth - 1)), groups=groups,
                                 data_format=data_format, l2_scale=l2_scale)

        self.levels = []
        for i in range(depth - 2, -1, -1):
            upsample = Upsample(filters=base_filters * (2 ** i), groups=groups, data_format=data_format,
                                l2_scale=l2_scale)
            conv = ResnetBlock(filters=base_filters * (2 ** i), groups=groups, reduction=reduction,
                               data_format=data_format, l2_scale=l2_scale)
            self.levels.append([upsample, conv])

        self.out = Conv3D(filters=out_ch, kernel_size=3, strides=1, padding='same', data_format=data_format,
                          kernel_regularizer=L2(l2_scale), kernel_initializer='he_normal')

    def build(self, input_shape, device):
        h, w, d = input_shape[1:-1]
        # vae.py:105-111 — the un-projection is sized from the first bottleneck shape seen
        self.unproj = Dense(units=h * w * d * 1 // 8, kernel_regularizer=L2(self.l2_scale),
                            kernel_initializer='he_normal', activation='relu')
        self._unflatten = (h // 2, w // 2, d // 2, 1)
        self.built = True

    def call(self, inputs, training=None, eps=None):
        inputs = self.downsample(inputs)
        inputs = inputs.reshape(inputs.shape[0], -1)            # Flatten (channels_last)
        inputs = self.proj(inputs)
        inputs, z_mean, z_logvar = sample(inputs, eps)
        inputs = self.unproj(inputs)
        inputs = inputs.reshape((inputs.shape[0],) + self._unflatten)
        inputs = self.upsample(inputs)
        for upsample, conv in self.levels:
            inputs = upsample(inputs, training=training)
            inputs = conv(inputs, training=training)
        inputs = self.out(inputs)
        return inputs, z_mean, z_logvar

    def get_config(self):
        self.config.update({'data_format': self.data_format,
                            'l2_scale': self.l2_scale})
        return self.config
