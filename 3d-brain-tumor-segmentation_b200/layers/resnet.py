"""ResnetBlock — same constructor / call surface as /root/reference/layers/resnet.py:8-113, :116-138.

    res  = ptwise(inputs);  res *= sigmoid(spatial(res)) + sigmoid(dense(relu(dense(GAP(res)))))
    x    = relu(GN(conv3(inputs)));  x = relu(GN(conv3(x)));  return res + x

B200 mapping: the pointwise conv emits the GAP sums from its epilogue, both 3x3x3 convs emit their GN
chunk statistics from theirs, and everything after the second conv (GN2 + ReLU + scSE scaling + add)
is ONE pass over HBM (csrc/block.cu).
"""
from ..keras_compat import Layer, Conv3D, Dense, L2
from .. import ops
from .group_norm import GroupNormalization


class _Activation(Layer):
    """tf.keras.layers.Activation('relu') placeholder: the ReLU is fused into the GN kernels."""

    def __init__(self, activation):
        super().__init__()
        self.activation = activation


class ResnetBlock(Layer):
    def __init__(self,
                 filters,
                 data_format='channels_last',
                 groups=8,
                 reduction=2,
                 l2_scale=1e-5):
        super().__init__()
        self.config = super().get_config()
        self.config.update({'filters': filters,
                            'data_format': data_format,
                            'reduction': reduction,
                            'l2_scale': l2_scale,
                            'groups': groups})
        self.filters, self.groups = filters, groups
        self.data_format = data_format
        # set by Decoder / VariationalAutoencoder on the block whose output feeds a narrow (2-3 channel) output conv: that
        # conv's weight gradient takes fp32 operands, so the output is kept in fp32 next to its 16-bit twin
        self.keep_f32_output = False
        self._fused_stats = data_format == 'channels_last'     # chunk statistics from the conv epilogue (F1 only)

        self.conv3d_ptwise = Conv3D(filters=filters, kernel_size=1, strides=1, padding='same',
                                    data_format=data_format, kernel_regularizer=L2(l2_scale),
                                    kernel_initializer='he_normal')
        if filters % reduction != 0:
            raise ValueError(
                'Reduction ratio, {}, must be a factor of number of channels, {}.'
                .format(reduction, filters))

        # channel squeeze-excitation (no biases); evaluated inside the fused epilogue
        self.dense_relu = Dense(units=filters // reduction, kernel_regularizer=L2(l2_scale),
                                kernel_initializer='he_normal', use_bias=False, activation='relu')
        self.dense_sigmoid = Dense(units=filters, kernel_regularizer=L2(l2_scale),
                                   kernel_initializer='he_normal', use_bias=False, activation=None)
        self.dense_sigmoid.activation = 'sigmoid'
        # spatial squeeze-excitation: Conv3D(1, k=1, no bias, sigmoid); evaluated inside the epilogue
        self.spatial = Conv3D(filters=1, kernel_size=1, strides=1, padding='same', data_format=data_format,
                              kernel_initializer='he_normal', kernel_regularizer=L2(l2_scale), use_bias=False,
                              activation='sigmoid')

        self.convs = []
        for gamma_init in ('ones', 'zeros'):
            self.convs.append([Conv3D(filters=filters, kernel_size=3, strides=1, padding='same',
                                      data_format=data_format, kernel_regularizer=L2(l2_scale),
                                      kernel_initializer='he_normal'),
                               GroupNormalization(groups=groups, axis=-1 if data_format == 'channels_last' else 1,
                                                  beta_initializer='zeros', gamma_initializer=gamma_init,
                                                  beta_regularizer=L2(l2_scale), gamma_regularizer=L2(l2_scale)),
                               _Activation('relu')])

    def build(self, input_shape, device):
        f = self.filters
        self.conv3d_ptwise.build(input_shape, device)
        self.dense_relu.build([input_shape[0], f], device)
        self.dense_sigmoid.build([input_shape[0], self.dense_relu.units], device)
        self.spatial.build(list(input_shape[:-1]) + [f], device)
        shp = list(input_shape)
        for conv, norm, _ in self.convs:
            conv.build(shp, device)
            shp = shp[:-1] + [f]
            norm.build(shp, device)
        self.built = True

    def call(self, inputs, training=None, dup_first=0):
        """dup_first = F > 0 (Encoder, inside a Model): the reference input is [a_last (F channels), a_0, .., a_last] and
        `inputs` holds only [a_0, .., a_last]; the two convs reading it use their kernels with the duplicate's weight
        slice folded into the last source's (SURVEY F3; exact)."""
        g = self.groups if self._fused_stats else 0
        box = {}                                          # the two data gradients w.r.t. `inputs` are summed in-kernel
        (conv1, norm1, _), (conv2, norm2, _) = self.convs
        kpt = ops.fold_dup(self.conv3d_ptwise.kernel, dup_first) if dup_first else None
        kc1 = ops.fold_dup(conv1.kernel, dup_first) if dup_first else None
        res, _, gap = self.conv3d_ptwise.call(inputs, want_gap=True, aux=True, share_x=True, grad_box=box, kernel=kpt)
        h1, st1, _ = conv1.call(inputs, gn_groups=g, aux=True, share_x=True, grad_box=box, kernel=kc1)
        a1 = norm1.call(h1, stats=st1, relu=True, operand_only=True)      # only conv2 reads it: 16-bit twin only
        h2, st2, _ = conv2.call(a1, gn_groups=g, aux=True)
        if st2 is None:                                   # chunk boundaries not voxel-aligned: unfused GN2
            a2 = norm2.call(h2, relu=True)
            return ops.block_epilogue(res, a2, None, None, None, self.spatial.kernel, gap,
                                      self.dense_relu.kernel, self.dense_sigmoid.kernel, self.groups, norm2.epsilon,
                                      keep_f32=self.keep_f32_output)
        return ops.block_epilogue(res, h2, st2, norm2.gamma, norm2.beta, self.spatial.kernel, gap,
                                  self.dense_relu.kernel, self.dense_sigmoid.kernel, self.groups, norm2.epsilon,
                                  keep_f32=self.keep_f32_output)

    def get_config(self):
        return self.config
