"""conv -> GroupNorm(1,C) [-> ReLU] units (drop-in for reference network/module/conv_gn_relu3.py:4-34): same constructors,
attribute names and state-dict keys; forward runs the C-ABI convolution + GroupNorm-apply kernels
(segmentation3d/_b200/blocks.py), and trains through blocks.run_module like every module here.  Built for the convolution shapes the library has kernels for: ksize 3 / stride 1 /
padding 1 (every use in the reference networks), ksize 2 / stride 2 / padding 0 (the second case of the reference's own
conv_gn_relu3_test.py) and ksize 1 / stride 1 / padding 0."""
import torch.nn as nn

from segmentation3d._b200 import blocks, lib
from segmentation3d.network._graph import Conv3dParams, GroupNormParams


_CONV_MODES = {(3, 1, 1): lib.CONV_K3, (2, 2, 0): lib.CONV_K2S2, (1, 1, 0): lib.CONV_K1}


def _conv_mode(ksize, stride, padding):
    if (ksize, stride, padding) not in _CONV_MODES:
        raise NotImplementedError('B200 build: ConvGnRelu3 has kernels for (ksize, stride, padding) in %s, got (%r, %r, %r)'
                                  % (sorted(_CONV_MODES), ksize, stride, padding))
    return _CONV_MODES[(ksize, stride, padding)]


class ConvGnRelu3(nn.Module):
    def __init__(self, in_channels, out_channels, ksize, stride, padding, do_act=True, bias=True):
        super(ConvGnRelu3, self).__init__()
        self._conv_mode = _conv_mode(ksize, stride, padding)
        self.conv = Conv3dParams(in_channels, out_channels, ksize)
        if not bias:
            self.conv.bias = None
        self.gn = GroupNormParams(out_channels)
        self.do_act = do_act
        if do_act:
            self.act = nn.ReLU(inplace=True)          # kept for the module tree; the ReLU runs inside the GroupNorm-apply kernel

    def _run(self, x_nd, dt, res=None, relu=None, tape=None):
        return blocks.conv_gn(x_nd, self.conv, self.gn, self._conv_mode, dt, self.do_act if relu is None else relu, res, tape=tape)

    def _forward(self, dt, tape, input):
        return blocks.to_ncdhw(self._run(blocks.to_ndhwc(input, dt, tape), dt, tape=tape), tape)

    def forward(self, input):
        blocks.check_input(input, self.conv.in_channels)
        return blocks.run_module(self, self._forward, input)


class BottConvGnRelu3(nn.Module):
    """bottleneck: C -> C/ratio -> C/ratio -> C, three k3 units."""

    def __init__(self, in_channels, out_channels, ksize, stride, padding, ratio, do_act=True, bias=True):
        super(BottConvGnRelu3, self).__init__()
        self.conv1 = ConvGnRelu3(in_channels, in_channels // ratio, ksize, stride, padding, do_act=True, bias=bias)
        self.conv2 = ConvGnRelu3(in_channels // ratio, in_channels // ratio, ksize, stride, padding, do_act=True, bias=bias)
        self.conv3 = ConvGnRelu3(in_channels // ratio, out_channels, ksize, stride, padding, do_act=do_act, bias=bias)

    def _run(self, x_nd, dt, res=None, relu=None, tape=None):
        y = self.conv2._run(self.conv1._run(x_nd, dt, tape=tape), dt, tape=tape)
        return self.conv3._run(y, dt, res, relu, tape=tape)

    def _forward(self, dt, tape, input):
        return blocks.to_ncdhw(self._run(blocks.to_ndhwc(input, dt, tape), dt, tape=tape), tape)

    def forward(self, input):
        blocks.check_input(input, self.conv1.conv.in_channels)
        return blocks.run_module(self, self._forward, input)
