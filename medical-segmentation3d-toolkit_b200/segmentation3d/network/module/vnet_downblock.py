"""Down-sampling block (drop-in for reference network/module/vnet_downblock.py:5-22): conv k2 s2 C -> 2C, GroupNorm, ReLU,
then a (bottleneck) residual block."""
import torch.nn as nn

from segmentation3d._b200 import blocks, lib
from segmentation3d.network._graph import Conv3dParams, GroupNormParams
from segmentation3d.network.module.residual_block3 import BottResidualBlock3, ResidualBlock3


class DownBlock(nn.Module):
    def __init__(self, in_channels, num_convs, compression=False, ratio=4):
        super(DownBlock, self).__init__()
        out_channels = in_channels * 2
        self.down_conv = Conv3dParams(in_channels, out_channels, 2)
        self.down_gn = GroupNormParams(out_channels)
        self.down_act = nn.ReLU(inplace=True)
        if compression:
            self.rblock = BottResidualBlock3(out_channels, 3, 1, 1, ratio, num_convs)
        else:
            self.rblock = ResidualBlock3(out_channels, 3, 1, 1, num_convs)

    def _forward(self, dt, tape, input):
        out = blocks.conv_gn(blocks.to_ndhwc(input, dt, tape), self.down_conv, self.down_gn, lib.CONV_K2S2, dt, True, tape=tape)
        return blocks.to_ncdhw(self.rblock._run(out, dt, tape), tape)

    def forward(self, input):
        blocks.check_input(input, self.down_conv.in_channels)
        return blocks.run_module(self, self._forward, input)
