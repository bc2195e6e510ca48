"""Training cost of a network assembled from the standalone modules (network/module/*.py) against the whole-network plan,
and the achieved bandwidth of the modules' gradient layout boundary.

    python tools/bench_blocks_train.py [--batch 8] [--size 96] [--steps 5] [--warmup 2] [--out FILE]

Prints JSON lines (and writes them to --out): the card's name and power limit read in the same run; one bf16 training step
(train_step: forward, multi-class Dice loss, backward, FlatAdam) of VNet at batch x size^3 built from the blocks and as
`SegmentationNet`, in ms per step (CUDA events over --steps steps after --warmup); and seg3d_grad_to_ncdhw (two bf16
contributions of 32 channels, the skip half of a concat gradient) and seg3d_grad_from_ncdhw (32 channels) at the same
batch and size, in GB/s from the bytes each must move (computed from shapes) and as a share of the 7.7 TB/s HBM bound.
The working sets exceed the 126 MB L2."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'medical-segmentation3d-toolkit_b200'))
sys.path.insert(0, ROOT)

HBM_BPS = 7.7e12


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(',')]
    except Exception as e:      # noqa: BLE001 - reported, not hidden
        name, power, clk = torch.cuda.get_device_name(0), 'unknown (%s)' % e, 'unknown'
    return {'card': name, 'power_limit': power, 'max_sm_clock': clk}


class BlockVNet(nn.Module):
    """the reference's network/vnet.py written with the drop-in blocks"""

    def __init__(self, cin, cout):
        from segmentation3d.network.module.vnet_downblock import DownBlock
        from segmentation3d.network.module.vnet_inblock import InputBlock
        from segmentation3d.network.module.vnet_outblock import OutputBlock
        from segmentation3d.network.module.vnet_upblock import UpBlock
        super(BlockVNet, self).__init__()
        self.in_block = InputBlock(cin, 16)
        self.down_32 = DownBlock(16, 1)
        self.down_64 = DownBlock(32, 2)
        self.down_128 = DownBlock(64, 3)
        self.down_256 = DownBlock(128, 3)
        self.up_256 = UpBlock(256, 256, 3)
        self.up_128 = UpBlock(256, 128, 3)
        self.up_64 = UpBlock(128, 64, 2)
        self.up_32 = UpBlock(64, 32, 1)
        self.out_block = OutputBlock(32, cout)

    def forward(self, x):
        o16 = self.in_block(x)
        o32 = self.down_32(o16)
        o64 = self.down_64(o32)
        o128 = self.down_128(o64)
        o256 = self.down_256(o128)
        o = self.up_256(o256, o128)
        o = self.up_128(o, o64)
        o = self.up_64(o, o32)
        o = self.up_32(o, o16)
        return self.out_block(o)


def time_steps(net, crops, masks, steps, warmup):
    from segmentation3d.core.seg_train import make_optimizer, train_step
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    opt = make_optimizer(net, 1e-4)
    lf = MultiDiceLoss([0.5, 0.5], 2, True)
    for _ in range(warmup):
        train_step(net, opt, lf, crops, masks)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        loss = train_step(net, opt, lf, crops, masks)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps, float(loss.detach())


def time_kernel(fn, reps=20, warmup=3):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=8)
    ap.add_argument('--size', type=int, default=96)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    from segmentation3d._b200 import lib
    from segmentation3d.network import vnet
    lines = [card()]
    B, S = args.batch, args.size
    g = torch.Generator().manual_seed(0)
    crops = torch.randn((B, 1, S, S, S), generator=g).cuda()
    masks = (torch.rand((B, 1, S, S, S), generator=g) > 0.7).float().cuda()
    os.environ['SEG3D_MODE'] = 'bf16'
    for name, make in (('SegmentationNet', lambda: vnet.SegmentationNet(1, 2)), ('blocks', lambda: BlockVNet(1, 2))):
        torch.manual_seed(0)
        net = make().cuda()
        net.train()
        torch.cuda.reset_peak_memory_stats()
        ms, loss = time_steps(net, crops, masks, args.steps, args.warmup)
        lines.append({'what': 'bf16 train step, VNet %d x %d^3' % (B, S), 'net': name, 'ms_per_step': round(ms, 2),
                      'last_loss': round(loss, 5), 'peak_mem_gb': round(torch.cuda.max_memory_allocated() / 1e9, 2)})
        del net
        torch.cuda.empty_cache()
    lines.append({'what': 'block VNet step / SegmentationNet step', 'ratio': round(lines[2]['ms_per_step'] / lines[1]['ms_per_step'], 3)})

    nvox, C = S ** 3, 32
    dt = lib.BF16
    g64 = torch.randn((B, nvox, 64), device='cuda').to(torch.bfloat16)       # two concat-wide gradients, skip half = channels 32..63
    r64 = torch.randn((B, nvox, 64), device='cuda').to(torch.bfloat16)
    out = torch.empty((B, C, nvox), device='cuda')
    st = lib.stream_ptr()

    def to_ncdhw():
        lib.call('seg3d_grad_to_ncdhw', dt, 2, lib.ptr(g64), 64, 32, lib.ptr(r64), 64, 32, None, 0, 0, C, B, nvox, lib.ptr(out), st)

    def from_ncdhw():
        lib.call('seg3d_grad_from_ncdhw', dt, lib.ptr(out), C, B, nvox, lib.ptr(g64), C, 0, st)
    for name, fn, nbytes in (('seg3d_grad_to_ncdhw (2 x bf16 -> fp32, C=32)', to_ncdhw, B * nvox * C * (2 * 2 + 4)),
                             ('seg3d_grad_from_ncdhw (fp32 -> bf16, C=32)', from_ncdhw, B * nvox * C * (4 + 2))):
        ms = time_kernel(fn)
        lines.append({'what': name, 'shape': [B, C, S, S, S], 'ms': round(ms, 4), 'GB_per_s': round(nbytes / ms / 1e6, 1),
                      'share_of_hbm_bound': round(nbytes / HBM_BPS / (ms / 1e3), 3)})
    text = '\n'.join(json.dumps(x) for x in lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
