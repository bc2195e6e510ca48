"""Output block (drop-in for reference network/module/vnet_outblock.py:4-24): conv k3 -> GroupNorm -> ReLU -> conv k1 ->
GroupNorm -> channel softmax; returns fp32 probabilities [B, classes, D, H, W].  Trains with up to 16 classes (the
tail backward of the whole network); wider blocks run inference under torch.no_grad()."""
import torch.nn as nn

from segmentation3d._b200 import blocks
from segmentation3d.network._graph import Conv3dParams, GroupNormParams


class OutputBlock(nn.Module):
    def __init__(self, in_channels, out_channels):
        super(OutputBlock, self).__init__()
        self.conv1 = Conv3dParams(in_channels, out_channels, 3)
        self.gn1 = GroupNormParams(out_channels)
        self.act1 = nn.ReLU(inplace=True)
        self.conv2 = Conv3dParams(out_channels, out_channels, 1)
        self.gn2 = GroupNormParams(out_channels)
        self.softmax = nn.Softmax(dim=1)

    def _forward(self, dt, tape, input):
        return blocks.output_tail(blocks.to_ndhwc(input, dt, tape), self.conv1, self.gn1, self.conv2, self.gn2, dt, tape)

    def forward(self, input):
        blocks.check_input(input, self.conv1.in_channels)
        return blocks.run_module(self, self._forward, input)
