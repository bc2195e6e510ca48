"""Input block (drop-in for reference network/module/vnet_inblock.py:4-15): conv k3 p1 -> GroupNorm(1,C) -> ReLU."""
import torch.nn as nn

from segmentation3d._b200 import blocks, lib
from segmentation3d.network._graph import Conv3dParams, GroupNormParams


class InputBlock(nn.Module):
    def __init__(self, in_channels, out_channels):
        super(InputBlock, self).__init__()
        self.conv = Conv3dParams(in_channels, out_channels, 3)
        self.gn = GroupNormParams(out_channels)
        self.act = nn.ReLU(inplace=True)

    def _forward(self, dt, tape, input):
        x = blocks.to_ndhwc(input, dt, tape)
        return blocks.to_ncdhw(blocks.conv_gn(x, self.conv, self.gn, lib.CONV_K3, dt, True, tape=tape), tape)

    def forward(self, input):
        blocks.check_input(input, self.conv.in_channels)
        return blocks.run_module(self, self._forward, input)
