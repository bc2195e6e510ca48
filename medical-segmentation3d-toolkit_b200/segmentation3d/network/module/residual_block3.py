"""Residual blocks (drop-in for reference network/module/residual_block3.py:5-46): relu(x + ops(x)) with `num_convs`
plain or bottleneck conv -> GroupNorm units; the residual add and the final ReLU run inside the last unit's GroupNorm-apply
kernel."""
import torch.nn as nn

from segmentation3d._b200 import blocks
from segmentation3d.network.module.conv_gn_relu3 import BottConvGnRelu3, ConvGnRelu3


class _ResidualBase(nn.Module):
    channels = 0

    def _run(self, x_nd, dt, tape=None):
        y = x_nd
        n = len(self.ops)
        for i, op in enumerate(self.ops):
            last = i == n - 1
            y = op._run(y, dt, res=x_nd if last else None, relu=True, tape=tape)     # last unit: relu(gn(conv) + x)
        return y

    def _forward(self, dt, tape, input):
        return blocks.to_ncdhw(self._run(blocks.to_ndhwc(input, dt, tape), dt, tape), tape)

    def forward(self, input):
        blocks.check_input(input, self.channels)
        return blocks.run_module(self, self._forward, input)


class ResidualBlock3(_ResidualBase):
    def __init__(self, channels, ksize, stride, padding, num_convs):
        super(ResidualBlock3, self).__init__()
        self.channels = channels
        layers = [ConvGnRelu3(channels, channels, ksize, stride, padding, do_act=(i != num_convs - 1)) for i in range(num_convs)]
        self.ops = nn.Sequential(*layers)
        self.act = nn.ReLU(inplace=True)


class BottResidualBlock3(_ResidualBase):
    def __init__(self, channels, ksize, stride, padding, ratio, num_convs):
        super(BottResidualBlock3, self).__init__()
        self.channels = channels
        layers = [BottConvGnRelu3(channels, channels, ksize, stride, padding, ratio, do_act=(i != num_convs - 1))
                  for i in range(num_convs)]
        self.ops = nn.Sequential(*layers)
        self.act = nn.ReLU(inplace=True)
