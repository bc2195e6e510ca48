"""Parameter tree + forward of the V-shaped segmentation networks on the B200 kernels.

The reference builds VNet/VBNet from nn.Module blocks (network/module/*.py) whose forward runs
torch layers.  Here the module tree is only a PARAMETER CONTAINER with the reference's exact
attribute names (so `state_dict()` keys/shapes match SURVEY.md A.1, with or without the
DataParallel `module.` prefix) and the reference's construction-time random stream (so the same
seed gives bit-identical initial weights); `forward` hands the weights to the C-ABI kernel plan
(segmentation3d/_b200/plan.py).  No torch layer is ever executed and there is no CPU path.
"""
import math
import os

import torch
import torch.nn as nn

from segmentation3d._b200 import plan as _plan
from segmentation3d._b200.plan import NetPlan


class Conv3dParams(nn.Module):
    """weight/bias holder laid out like nn.Conv3d ([Cout,Cin,k,k,k]); class name contains
    'Conv3d' so the reference-style initialisers (module/weight_init.py) pick it up."""
    transposed = False

    def __init__(self, in_channels, out_channels, ksize):
        super().__init__()
        self.in_channels, self.out_channels, self.ksize = in_channels, out_channels, ksize
        shape = (in_channels, out_channels) if self.transposed else (out_channels, in_channels)
        self.weight = nn.Parameter(torch.empty(shape + (ksize,) * 3))
        self.bias = nn.Parameter(torch.empty(out_channels))
        # same draws as torch's _ConvNd.reset_parameters
        nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        fan_in, _ = nn.init._calculate_fan_in_and_fan_out(self.weight)
        if fan_in != 0:
            bound = 1 / math.sqrt(fan_in)
            nn.init.uniform_(self.bias, -bound, bound)

    def forward(self, *a, **k):
        raise RuntimeError('parameter holder: the network forward runs in libseg3d_b200.so')


class ConvTranspose3dParams(Conv3dParams):
    """holder laid out like nn.ConvTranspose3d ([Cin,Cout,k,k,k])."""
    transposed = True


class GroupNormParams(nn.Module):
    """gamma/beta holder of nn.GroupNorm(1, C) (eps 1e-5)."""

    def __init__(self, channels):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(channels))
        self.bias = nn.Parameter(torch.zeros(channels))

    def forward(self, *a, **k):
        raise RuntimeError('parameter holder: the network forward runs in libseg3d_b200.so')


class Block(nn.Module):
    """anonymous container node of the parameter tree"""

    def forward(self, *a, **k):
        raise RuntimeError('parameter holder: the network forward runs in libseg3d_b200.so')


def _residual_specs(prefix, ch, num_convs, bottleneck, ratio=4):
    out = []
    for i in range(num_convs):
        base = '%s.ops.%d' % (prefix, i)
        if bottleneck:
            mid = ch // ratio
            for j, (ci, co) in enumerate(((ch, mid), (mid, mid), (mid, ch)), 1):
                out += [('%s.conv%d.conv' % (base, j), 'conv', ci, co, 3), ('%s.conv%d.gn' % (base, j), 'gn', co)]
        else:
            out += [(base + '.conv', 'conv', ch, ch, 3), (base + '.gn', 'gn', ch)]
    return out


def network_specs(in_channels, out_channels, bottleneck_stages):
    """Ordered parameter spec of the V-shaped net (reference network/vnet.py:23-34, vbnet.py:24-35)."""
    s = [('in_block.conv', 'conv', in_channels, 16, 3), ('in_block.gn', 'gn', 16)]
    for cin, n in ((16, 1), (32, 2), (64, 3), (128, 3)):
        name = 'down_%d' % (2 * cin)
        s += [(name + '.down_conv', 'conv', cin, 2 * cin, 2), (name + '.down_gn', 'gn', 2 * cin)]
        s += _residual_specs(name + '.rblock', 2 * cin, n, name in bottleneck_stages)
    for cin, cout, n in ((256, 256, 3), (256, 128, 3), (128, 64, 2), (64, 32, 1)):
        name = 'up_%d' % cout
        s += [(name + '.up_conv', 'convT', cin, cout // 2, 2), (name + '.up_gn', 'gn', cout // 2)]
        s += _residual_specs(name + '.rblock', cout, n, name in bottleneck_stages)
    s += [('out_block.conv1', 'conv', 32, out_channels, 3), ('out_block.gn1', 'gn', out_channels),
          ('out_block.conv2', 'conv', out_channels, out_channels, 1), ('out_block.gn2', 'gn', out_channels)]
    return s


class VShapedNet(nn.Module):
    """Base of vnet.SegmentationNet / vbnet.SegmentationNet."""
    bottleneck_stages = ()
    arch = 'vnet'

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        for spec in network_specs(in_channels, out_channels, self.bottleneck_stages):
            path = spec[0].split('.')
            node = self
            for part in path[:-1]:
                if part not in node._modules:
                    node.add_module(part, Block())
                node = node._modules[part]
            if spec[1] == 'gn':
                leaf = GroupNormParams(spec[2])
            elif spec[1] == 'convT':
                leaf = ConvTranspose3dParams(spec[2], spec[3], spec[4])
            else:
                leaf = Conv3dParams(spec[2], spec[3], spec[4])
            node.add_module(path[-1], leaf)
        # execution mode: 'fp16' | 'bf16' (tensor cores, 2-byte storage) | 'fp32x' (tensor cores, split hi/lo operands:
        # strict parity) | 'fp32' (CUDA cores) | 'auto' (see resolve_mode).  SEG3D_MODE overrides the default.
        self.b200_mode = os.environ.get('SEG3D_MODE', 'auto')
        self._plans = {}            # resolved mode -> [NetPlan, weight key]
        self._weights_epoch = 0
        self._plan = None           # the plan of the most recent forward

    def max_stride(self):
        return 16

    def resolve_mode(self, train=False):
        """The mode a forward runs in.
        Inference, 'auto': binary nets run in fp16; nets with more than two classes run in 'fp32x' - measured on B200 and
        reproduced by oracle/reduced_precision.py, ANY half-precision operand rounding (weights alone, activations alone)
        flips enough near-tie voxels of a rare class of a random-init multi-class net to miss the per-class Dice >= 0.999 bar,
        and the default must meet the parity bars ('fp16' stays available explicitly).
        Training: the gradient buffers are stored in the mode's type and gradient magnitudes of ~1e-6 underflow fp16, so
        'auto', 'fp16' and the inference-only 'fp32x' train in bf16; 'bf16' and 'fp32' are taken as given."""
        mode = self.b200_mode
        if train:
            return mode if mode in ('bf16', 'fp32') else 'bf16'
        if mode == 'auto':
            return 'fp16' if self.out_channels <= 2 else 'fp32x'
        return mode

    def mark_weights_changed(self):
        """for code that writes the parameters behind torch's back (the C-ABI Adam kernel)"""
        self._weights_epoch += 1

    # -- kernel plan management -----------------------------------------------------------
    def _current_plan(self, train=False):
        params = list(self.parameters())
        dev = params[0].device
        _plan._require_cuda(dev, 'segmentation3d (B200 build) has no CPU path: move the network to a CUDA device')
        mode = self.resolve_mode(train)
        # weights changed <=> a parameter's version counter moved (torch in-place ops) or an optimiser that updates the
        # parameters through the C-ABI kernel (segmentation3d/_b200/optim.py) said so
        key = (str(dev), (self._weights_epoch,) + tuple(p._version for p in params), tuple(p.data_ptr() for p in params))
        entry = self._plans.get(mode)
        if entry is None or entry[1][0] != key[0] or entry[1][2] != key[2]:
            entry = self._plans[mode] = [NetPlan(self.state_dict(), mode=mode, device=dev, arch=self.arch), key]
            entry[0].bind_parameters(list(self.named_parameters()))
        elif entry[1] != key:
            entry[0].refresh(self.state_dict())            # same device and storage: re-pack the weights in place
            entry[1] = key
        self._plan = entry[0]
        return self._plan

    def forward(self, input):
        _plan._require_cuda(input.device, 'segmentation3d (B200 build) has no CPU path: pass a CUDA tensor')
        # differentiable when grad mode is on and the input or any parameter requires grad (the standalone modules' rule):
        # frozen parameters get no gradient and an input that requires grad gets one
        if torch.is_grad_enabled() and (input.requires_grad or any(p.requires_grad for p in self.parameters())):
            from segmentation3d._b200.autograd import train_forward
            return train_forward(self, input)
        with torch.no_grad():
            return self._current_plan().forward(input).clone()
