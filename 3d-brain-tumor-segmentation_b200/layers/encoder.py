"""Encoder — surface of /root/reference/layers/encoder.py (:9-67 ctor, :69-101 call).

Per level i: (i+1) ResnetBlocks(F = base_filters * 2**i) with DenseNet-style concatenation
(`dense([inputs] + cache)` where `inputs is cache[-1]`, i.e. the last block output appears twice —
SURVEY F3, kept), concat of all block outputs (i > 0), ConvDownsample(F) except at the last level.
"""
from ..keras_compat import Layer
from .. import ops
from .resnet import ResnetBlock
from .downsample import get_downsampling


class _Concatenate(Layer):
    def __init__(self, axis=-1):
        super().__init__()
        self.axis = axis

    def call(self, xs, training=None):
        return ops.concat(list(xs))


class _Dropout(Layer):
    def __init__(self, rate):
        super().__init__()
        self.rate = rate
        self.seed = 0x5EED
        self._counter = None

    def call(self, x, training=None, mask=None):
        if not training:
            return x
        if mask is None and self._counter is None:
            import torch
            self._counter = torch.zeros(1, dtype=torch.int64, device=x.device)
        return ops.dropout(x, self.rate, True, mask, self.seed, self._counter)


class Encoder(Layer):
    def __init__(self,
                 data_format='channels_last',
                 groups=8,
                 reduction=2,
                 l2_scale=1e-5,
                 dropout=0.2,
                 downsampling='conv',
                 base_filters=16,
                 depth=4):
        super().__init__()
        self.config = super().get_config()
        self.data_format = data_format
        self.config.update({'data_format': data_format,
                            'groups': groups,
                            'reduction': reduction,
                            'l2_scale': l2_scale,
                            'downsampling': downsampling,
                            'base_filters': base_filters,
                            'depth': depth})
        Downsample = get_downsampling(downsampling)
        if Downsample is None:
            raise ValueError(f"unknown downsampling {downsampling!r}")

        self.dropout = _Dropout(rate=dropout)

        self.levels = []
        for i in range(depth):
            convs = []
            for j in range(i + 1):
                conv = ResnetBlock(filters=base_filters * (2 ** i), groups=groups, reduction=reduction,
                                   data_format=data_format, l2_scale=l2_scale)
                dense = _Concatenate(axis=-1) if j > 0 else None
                convs.append([conv, dense])
            concat = _Concatenate(axis=-1) if i > 0 else None
            downsample = Downsample(filters=base_filters * (2 ** i), groups=groups, data_format=data_format,
                                    l2_scale=l2_scale) if i < depth - 1 else None
            self.levels.append([convs, concat, downsample])

    def call(self, inputs, training=None, dropout_mask=None):
        inputs = self.dropout(inputs, training=training, mask=dropout_mask)
        residuals = []
        for i, level in enumerate(self.levels):
            convs, concat, downsample = level
            cache = []
            for conv, dense in convs:
                dup = 0
                if dense is not None:
                    if conv.built and self._can_dedup(cache):
                        # `inputs is cache[-1]`: [inputs] + cache lists it twice (encoder.py:85).  Feed [cache] only
                        # and let the block fold the duplicate's weight slice (exact; one K segment less)
                        inputs, dup = dense(cache), inputs.shape[-1]
                    else:
                        inputs = dense([inputs] + cache)
                inputs = conv(inputs, training=training, dup_first=dup) if dup else conv(inputs, training=training)
                cache.append(inputs)
            if concat is not None:
                inputs = concat(cache)
            residuals.append(inputs)
            if downsample is not None:
                inputs = downsample(inputs, training=training)
        return residuals

    @staticmethod
    def _can_dedup(cache):
        return (ops.FUSED["on"] and ops.twin_dtype(False) is not None
                and all(ops.sources(t) is not None for t in cache))

    def get_config(self):
        return self.config
