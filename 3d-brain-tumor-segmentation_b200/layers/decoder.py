"""Decoder — surface of /root/reference/layers/decoder.py (:9-63 ctor, :65-83 call)."""
from ..keras_compat import Layer, Conv3D, L2
from .. import ops
from .resnet import ResnetBlock
from .upsample import get_upsampling
from .encoder import _Concatenate


class Decoder(Layer):
    def __init__(self,
                 data_format='channels_last',
                 groups=8,
                 reduction=2,
                 l2_scale=1e-5,
                 upsampling='conv',
                 base_filters=16,
                 depth=4,
                 out_ch=3):
        super().__init__()
        self.config = super().get_config()
        self.data_format = data_format
        self.config.update({'data_format': data_format,
                            'groups': groups,
                            'reduction': reduction,
                            'l2_scale': l2_scale,
                            'upsampling': upsampling,
                            'base_filters': base_filters,
                            'depth': depth,
                            'out_ch': out_ch})
        Upsample = get_upsampling(upsampling)
        if Upsample is None:
            raise ValueError(f"unknown upsampling {upsampling!r}")

        self.levels = []
        for i in range(depth - 2, -1, -1):
            upsample = Upsample(filters=base_filters * (2 ** i), groups=groups, data_format=data_format,
                                l2_scale=l2_scale)
            res = _Concatenate(axis=-1)
            conv = ResnetBlock(filters=base_filters * (2 ** i), groups=groups, reduction=reduction,
                               data_format=data_format, l2_scale=l2_scale)
            self.levels.append([upsample, res, conv])

        # 1x1x1 conv to the class channels + sigmoid (glorot_normal, L2)
        self.out = Conv3D(filters=out_ch, kernel_size=1, strides=1, padding='same', activation='sigmoid',
                          data_format=data_format, kernel_regularizer=L2(l2_scale),
                          kernel_initializer='glorot_normal')

    def call(self, inputs, training=None):
        inputs, residuals = inputs
        for level, residual in zip(self.levels, residuals[::-1]):
            upsample, res, conv = level
            inputs = upsample(inputs, training=training)
            inputs = res([residual, inputs])           # order [encoder_residual, upsampled] (decoder.py:75)
            inputs = conv(inputs, training=training)
        return self.out(inputs)

    def get_config(self):
        return self.config
