"""Training-step time of SegmentationNet (VNet, bf16) at 8 x 96^3 under the partial backward, alternating in one process:

  all           every parameter trainable, input without gradient (the benchmark's step)
  enc_frozen    in_block and down_* frozen
  out_only      only out_block trainable
  input_only    every parameter frozen, input gradient
  all_input     every parameter trainable, input gradient

A step is forward + Dice loss + backward + FlatAdam (when something is trainable), timed with CUDA events.  Also times
seg3d_conv3d_cin1_dgrad alone over many launches against its HBM bound (gy read at 16 bf16 channels + fp32 dx written,
36 B per voxel, at 7.7 TB/s).  Prints one JSON line per configuration and round.

    python tools/bench_partial_backward.py [--batch 8] [--size 96] [--steps 10] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'medical-segmentation3d-toolkit_b200'))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

HBM_BPS = 7.7e12


def card():
    try:
        return subprocess.check_output(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], text=True).strip()
    except Exception as e:          # the card name is part of every number printed
        return 'unknown (%s)' % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=8)
    ap.add_argument('--size', type=int, default=96)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--rounds', type=int, default=3)
    a = ap.parse_args()
    from oracle import init as oinit
    from segmentation3d._b200 import lib
    from segmentation3d.core.seg_train import make_optimizer
    from segmentation3d.loss.multi_dice_loss import MultiDiceLoss
    from segmentation3d.network import vnet
    assert torch.cuda.is_available(), 'needs a GPU'
    lib.load()
    print(json.dumps({'card': card()}))
    B, S = a.batch, a.size
    g = torch.Generator(device='cuda').manual_seed(0)
    crops = torch.randn((B, 1, S, S, S), generator=g, device='cuda')
    masks = (torch.rand((B, 1, S, S, S), generator=g, device='cuda') > 0.5).float()
    lf = MultiDiceLoss([1.0, 1.0], 2, False)
    sd = oinit.init_state_dict('vnet', 1, 2, 0)
    enc = ('in_block', 'down_')
    configs = {
        'all': (lambda n: True, False),
        'enc_frozen': (lambda n: not n.startswith(enc), False),
        'out_only': (lambda n: n.startswith('out_block'), False),
        'input_only': (lambda n: False, True),
        'all_input': (lambda n: True, True),
    }
    nets = {}
    for name, (trainable, _) in configs.items():
        net = vnet.SegmentationNet(1, 2)
        net.load_state_dict(sd)
        net.b200_mode = 'bf16'
        net = net.cuda().train()
        for n, p in net.named_parameters():
            p.requires_grad_(trainable(n))
        opt = make_optimizer(net, 1e-4) if any(p.requires_grad for p in net.parameters()) else None
        nets[name] = (net, opt)

    crops_g = crops.clone().requires_grad_(True)

    def step(name):
        net, opt = nets[name]
        x = crops_g if configs[name][1] else crops
        if opt is not None:
            opt.zero_grad()
        lf(net(x), masks).backward()
        if opt is not None:
            opt.step()
        crops_g.grad = None

    for name in configs:                   # warm-up: plans, backward state, optimiser adoption
        for _ in range(2):
            step(name)
    torch.cuda.synchronize()
    for r in range(a.rounds):
        for name in configs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                step(name)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.steps
            print(json.dumps({'round': r, 'config': name, 'batch': B, 'size': S, 'step_ms': round(ms, 3),
                              'patches_per_s': round(B * 1000.0 / ms, 1)}))
    # the input-gradient kernel alone
    gy = torch.randn((B, S, S, S, 16), generator=g, device='cuda').to(torch.bfloat16)
    w = torch.randn((27, 16), generator=g, device='cuda')
    dx = torch.empty((B, 1, S, S, S), device='cuda')
    for _ in range(5):
        lib.call('seg3d_conv3d_cin1_dgrad', lib.BF16, lib.ptr(gy), 16, lib.ptr(w), lib.ptr(dx), B, S, S, S, lib.stream_ptr())
    n = 50
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        lib.call('seg3d_conv3d_cin1_dgrad', lib.BF16, lib.ptr(gy), 16, lib.ptr(w), lib.ptr(dx), B, S, S, S, lib.stream_ptr())
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    nbytes = 36.0 * B * S ** 3
    bound_ms = nbytes / HBM_BPS * 1e3
    print(json.dumps({'kernel': 'seg3d_conv3d_cin1_dgrad', 'batch': B, 'size': S, 'ms': round(ms, 4), 'bytes': nbytes,
                      'hbm_bound_ms': round(bound_ms, 4), 'share_of_hbm_bound': round(bound_ms / ms, 3),
                      'note': 'working set %.0f MB, L2 126 MB: read from HBM' % (nbytes / 1e6)}))


if __name__ == '__main__':
    main()
