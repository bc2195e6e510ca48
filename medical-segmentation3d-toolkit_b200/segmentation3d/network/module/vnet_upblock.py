"""Up-sampling block (drop-in for reference network/module/vnet_upblock.py:6-23): transposed conv k2 s2 Cin -> Cout/2,
GroupNorm, ReLU, concat with the skip tensor (up-conv channels first), then a (bottleneck) residual block.  The concat is
formed in place: the GroupNorm-apply kernel writes the lower half of the buffer the skip tensor was copied into."""
import torch
import torch.nn as nn

from segmentation3d._b200 import blocks, lib
from segmentation3d.network._graph import ConvTranspose3dParams, GroupNormParams
from segmentation3d.network.module.residual_block3 import BottResidualBlock3, ResidualBlock3


class UpBlock(nn.Module):
    def __init__(self, in_channels, out_channels, num_convs, compression=False, ratio=4):
        super(UpBlock, self).__init__()
        self.up_conv = ConvTranspose3dParams(in_channels, out_channels // 2, 2)
        self.up_gn = GroupNormParams(out_channels // 2)
        self.up_act = nn.ReLU(inplace=True)
        if compression:
            self.rblock = BottResidualBlock3(out_channels, 3, 1, 1, ratio, num_convs)
        else:
            self.rblock = ResidualBlock3(out_channels, 3, 1, 1, num_convs)

    def _forward(self, dt, tape, input, skip):
        half = self.up_conv.out_channels
        x = blocks.to_ndhwc(input, dt, tape)
        raw, stats, conv = blocks.conv_raw(x, self.up_conv, lib.CONV_T2S2, dt)
        B, D, H, W, _ = raw.shape
        if tuple(skip.shape[2:]) != (D, H, W):
            raise ValueError('skip tensor must have the up-sampled spatial size %s, got %s' % ((D, H, W), tuple(skip.shape[2:])))
        cat = torch.empty((B, D, H, W, self.rblock.channels), dtype=raw.dtype, device=raw.device)
        cat[..., half:].copy_(skip.detach().permute(0, 2, 3, 4, 1))          # vnet_upblock.py:21: (up, skip) along channels
        blocks.gn_apply(raw, stats, self.up_gn, dt, True, out=cat, out_off=0)
        if tape is not None:        # the skip tensor's gradient is the upper channel window of the concat's gradient
            tape.input(1, blocks._View(cat, half, cat.shape[-1], cat.shape[-1] - half))
            tape.unit(x, self.up_conv, self.up_gn, lib.CONV_T2S2, conv, raw, stats, cat, 0, True, None)
        return blocks.to_ncdhw(self.rblock._run(cat, dt, tape), tape)

    def forward(self, input, skip):
        blocks.check_input(input, self.up_conv.in_channels)
        blocks.check_input(skip, self.rblock.channels - self.up_conv.out_channels)
        return blocks.run_module(self, self._forward, input, skip)
